"""ORACLE (test infrastructure only) -- what the parity tests compare against, from the UNMODIFIED
reference (imported through oracle/ref_shims.py), so that those tests run without it:

  tests/golden/reference_parity.npz    arrays: the reference's limiter / spectrum helpers, stages.main and
                                       create_preview on the tests' seeded inputs
  tests/golden/reference_surface.json  the reference's Config attributes, log codes, checker warnings and
                                       checker errors

Each input below is the same seeded recipe its test builds; the SHA-256 of the input bytes is stored so a
test can tell "different input" from "different output".  Outputs a test compares bit for bit are
stored as the SHA-256 of their float64 bytes; outputs compared with a tolerance are stored whole, or, for
stages.main (three 4 MB arrays per case), as every EVERY-th frame plus 64 block sums of the output and
of its square, over which every frame counts.

    MATCHERING_REFERENCE_ROOT=<reference checkout> python oracle/make_golden_parity.py
"""
import hashlib
import json
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import port  # noqa: E402
from ref_shims import import_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
EVERY = 499
N_BLOCKS = 64

MAIN_CASES = [(44100, 6.0), (96000, 2.5)]                        # test_oracle_port.py::test_main_against_reference
PREVIEW_CASES = [(30000, False), (9000, True), (24000, False)]   # ::test_preview_pieces_against_reference
CONFIG_KW = dict(internal_sample_rate=48000, max_piece_size=7.5)  # test_cabi_and_surface.py


def digest(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def summarise(y: np.ndarray) -> dict:
    edges = np.linspace(0, y.shape[0], N_BLOCKS + 1).astype(np.int64)
    return dict(frames=y.shape[0], rows=y[::EVERY].astype(np.float64), block_edges=edges,
                block_sum=np.array([y[a:b].sum(axis=0) for a, b in zip(edges[:-1], edges[1:])]),
                block_sumsq=np.array([np.einsum("ij,ij->j", y[a:b], y[a:b]) for a, b in zip(edges[:-1], edges[1:])]))


def identities_inputs():
    rng = np.random.default_rng(5)
    g = np.abs(rng.standard_normal(5000)) * (rng.uniform(size=5000) > 0.7)
    pieces = rng.standard_normal((3, 20000))
    x = rng.standard_normal((1000, 2))
    return g, pieces, x


def main_inputs(sr, seconds):
    n = int(sr * seconds)
    return port.synth_target(n, 3).astype(np.float64), port.synth_reference(n - 777, 4).astype(np.float64)


def preview_inputs(n):
    target = 2.5 * port.synth_target(n, 41).astype(np.float64)
    result = port.synth_reference(n, 42).astype(np.float64) * (0.2 + np.abs(np.sin(np.linspace(0, 9, n))))[:, None]
    return target, result


def make_arrays(m) -> dict:
    from matchering import Config, Result, dsp, preview_creator, stages
    from matchering.limiter import hyrax
    from matchering.stage_helpers import match_frequencies as mf
    out = {}
    g, pieces, x = identities_inputs()
    out["identities_input_sha256"] = digest(np.concatenate([g, pieces.ravel(), x.ravel()]))
    sliding = getattr(hyrax, "__sliding_window_fast")
    for attack in (44, 45, 96):
        out[f"attack_max_{attack}_sha256"] = digest(sliding(g, attack, "attack"))
    for hold in (44, 45, 96, 3):
        out[f"hold_max_{hold}_sha256"] = digest(sliding(g, hold, "hold"))
    att, slided = getattr(hyrax, "__process_attack")(np.copy(g), Config())
    out["attack_envelope_sha256"], out["attack_gain"] = digest(slided), att
    out["average_fft"] = getattr(mf, "__average_fft")(pieces, 44100, 4096)
    mid, side = dsp.lr_to_ms(x)
    out["mid_sha256"], out["side_sha256"] = digest(mid), digest(side)

    for sr, seconds in MAIN_CASES:
        t, r = main_inputs(sr, seconds)
        key = f"main_{sr}"
        out[key + "_input_sha256"] = digest(np.concatenate([t.ravel(), r.ravel()]))
        cfg = Config(internal_sample_rate=sr, max_piece_size=1.0)
        for name, y in zip(("limited", "no_limiter", "normalized"), stages.main(t, r, cfg, True, True, True)):
            out.update({f"{key}_{name}_{k}": v for k, v in summarise(y).items()})

    saved = {}
    original_save = preview_creator.save
    preview_creator.save = lambda file, arr, sr, subtype, name: saved.__setitem__(name, arr.copy())
    try:
        for n, _ in PREVIEW_CASES:
            target, result = preview_inputs(n)
            key = f"preview_{n}"
            out[key + "_input_sha256"] = digest(np.concatenate([target.ravel(), result.ravel()]))
            cfg = Config(internal_sample_rate=2000, preview_size=6, preview_analysis_step=2)
            preview_creator.create_preview(target, result, cfg, Result("t.wav", "PCM_16"), Result("r.wav", "PCM_16"))
            for name in ("target", "result"):
                piece = saved[f"{name} preview"]
                out[f"{key}_{name}_shape"] = np.array(piece.shape)
                out[f"{key}_{name}_sha256"] = digest(piece)
    finally:
        preview_creator.save = original_save
    return out


def make_surface(m) -> dict:
    from matchering import Config
    from matchering.log.codes import Code as RefCode
    sys.modules.pop("test_checker_parity", None)
    import test_checker_parity  # its CASES: (label, array, expected) with arrays built from fixed seeds
    config = {k: (vars(v) if k == "limiter" else v) for k, v in vars(Config(**CONFIG_KW)).items()}
    warnings_seen = {}
    for label, array, _ in test_checker_parity.CASES:
        seen = []
        m.log(warning_handler=seen.append)
        try:
            m.checker.check(array.copy(), 44100, Config(), "target")
        finally:
            m.log()
        warnings_seen[label] = seen
    errors = {}
    for key, shape, kind in (("three_channels_22050", (3000, 3), "reference"), ("too_short_22050", (2000, 2), "target")):
        try:
            m.checker.check(np.zeros(shape), 22050, Config(), kind)
        except Exception as e:  # the reference's ModuleError
            errors[key] = {"type": type(e).__name__, "message": str(e)}
    return {"config_kwargs": CONFIG_KW, "config": config, "log_codes": {c.name: int(c) for c in RefCode},
            "checker_warnings": warnings_seen, "checker_errors": errors}


def main():
    warnings.simplefilter("ignore")
    m = import_reference()
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, "reference_parity.npz"), **make_arrays(m))
    with open(os.path.join(OUT, "reference_surface.json"), "w") as f:
        json.dump(make_surface(m), f, indent=1, sort_keys=True)
        f.write("\n")
    for name in ("reference_parity.npz", "reference_surface.json"):
        print(name, os.path.getsize(os.path.join(OUT, name)) // 1024, "KiB")


if __name__ == "__main__":
    main()
