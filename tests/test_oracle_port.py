"""oracle/port.py pinned against the golden vectors generated from the unmodified reference
(oracle/make_golden.py, oracle/make_golden_full.py, oracle/make_golden_parity.py)."""
import numpy as np
import pytest

import port
from make_golden_parity import EVERY, digest, identities_inputs, main_inputs, preview_inputs


def cfg_for(npz):
    return port.OracleConfig(max_piece_size=float(npz["max_piece_size_s"]))


def test_pipeline_small_matches_golden(golden):
    g = golden("pipeline_small.npz")
    cfg = cfg_for(g)
    tr = {}
    lim, plain, norm = port.main(g["target"].astype(np.float64), g["reference"].astype(np.float64), cfg,
                                 True, True, True, trace=tr)
    assert np.abs(lim - g["limited"]).max() < 1e-12
    assert np.abs(plain - g["no_limiter"]).max() < 1e-12
    assert np.abs(norm - g["normalized"]).max() < 2e-7  # stored as float32
    assert tr["target"]["divisions"] == int(g["target_divisions"]) and tr["target"]["piece"] == int(g["target_piece"])
    assert tr["reference"]["divisions"] == int(g["reference_divisions"])
    assert abs(tr["c0"] - float(g["rms_coefficient"])) < 1e-12
    assert abs(tr["final_coef"] - float(g["final_amplitude_coefficient"])) < 1e-15
    assert np.abs(tr["firs"]["mid"] - g["fir_mid"]).max() < 1e-13
    assert np.abs(tr["firs"]["side"] - g["fir_side"]).max() < 1e-13


def test_quiet_reference_matches_golden(golden):
    g = golden("pipeline_quiet_reference.npz")
    lim, plain, _ = port.main(g["target"].astype(np.float64), g["reference"].astype(np.float64), cfg_for(g),
                              True, True, False)
    assert np.abs(lim - g["limited"]).max() < 1e-12
    assert np.abs(plain - g["no_limiter"]).max() < 1e-12


def test_limiter_matches_golden(golden):
    g = golden("limiter.npz")
    x = g["x"].astype(np.float64)
    tr = {}
    assert np.abs(port.limit(x, port.OracleConfig(), trace=tr) - g["y_44100"]).max() < 1e-13
    assert np.abs(port.limit(x, port.OracleConfig(internal_sample_rate=96000)) - g["y_96000"]).max() < 1e-13
    assert np.abs(tr["a_env"] - g["envelope"]).max() < 1e-7
    assert np.abs(tr["g_att"] - g["gain_attack"]).max() < 1e-7
    assert np.abs(np.maximum(tr["hold_out"], tr["rel_out"]) - g["gain_release"]).max() < 1e-7
    assert abs(np.abs(g["y_44100"]).max() - port.OracleConfig().threshold) < 1e-9


def test_limiter_early_out_returns_input_object():
    x = 0.3 * port.synth_limiter_input(5000, 1).astype(np.float64)
    assert port.limit(x, port.OracleConfig()) is x


# ---- against the reference's outputs on the same seeded inputs (tests/golden/reference_parity.npz) ------
def test_identities_against_reference_helpers(golden):
    ref = golden("reference_parity.npz")
    g, pieces, x = identities_inputs()
    assert digest(np.concatenate([g, pieces.ravel(), x.ravel()])) == ref["identities_input_sha256"], "inputs differ from the golden's"
    for attack in (44, 45, 96):
        reach = (attack + 1 if not attack & 1 else attack) - 1
        assert digest(port.centred_max(g, reach)) == ref[f"attack_max_{attack}_sha256"]
    for hold in (44, 45, 96, 3):
        assert digest(port.trailing_max(g, hold)) == ref[f"hold_max_{hold}_sha256"]
    k = port.limiter_coefficients(port.OracleConfig())
    slided = port.centred_max(g, k["reach"])
    assert digest(slided) == ref["attack_envelope_sha256"]
    assert np.abs(port.one_pole_forward_backward(slided, k["c"]) - ref["attack_gain"]).max() < 1e-15
    flat = pieces.reshape(-1)
    got = port.average_spectrum(flat, 20000, np.ones(3, dtype=bool), 4096)
    assert np.abs(got - ref["average_fft"]).max() < 1e-15
    m2, s2 = port.mid_side(x)
    assert digest(m2) == ref["mid_sha256"] and digest(s2) == ref["side_sha256"]


def _compare_summary(y, ref, prefix, tol):
    """y against oracle/make_golden_parity.py's summary of the reference's output: the sampled rows at
    `tol`, and 64 block sums of y and of its square, in which every frame takes part."""
    assert y.shape[0] == int(ref[prefix + "frames"])
    assert np.abs(y[::EVERY] - ref[prefix + "rows"]).max() < tol
    edges = ref[prefix + "block_edges"]
    frames_per_block = np.diff(edges)[:, None]
    block_sum = np.array([y[a:b].sum(axis=0) for a, b in zip(edges[:-1], edges[1:])])
    block_sq = np.array([np.einsum("ij,ij->j", y[a:b], y[a:b]) for a, b in zip(edges[:-1], edges[1:])])
    # a per-sample error e moves a block's mean by at most e and its mean square by at most 2*peak*e
    peak = max(1.0, float(np.abs(y).max()))
    assert (np.abs(block_sum - ref[prefix + "block_sum"]) / frames_per_block).max() < tol
    assert (np.abs(block_sq - ref[prefix + "block_sumsq"]) / frames_per_block).max() < 2 * peak * tol


@pytest.mark.parametrize("sr,seconds", [(44100, 6.0), (96000, 2.5)])
def test_main_against_reference(golden, sr, seconds):
    ref = golden("reference_parity.npz")
    t, r = main_inputs(sr, seconds)
    key = f"main_{sr}_"
    assert digest(np.concatenate([t.ravel(), r.ravel()])) == ref[key + "input_sha256"], "inputs differ from the golden's"
    cfg = port.OracleConfig(internal_sample_rate=sr, max_piece_size=1.0)
    got = port.main(t, r, cfg, True, True, True)
    for name, y in zip(("limited", "no_limiter", "normalized"), got):
        _compare_summary(y, ref, key + name + "_", 1e-12)


@pytest.mark.parametrize("n,whole", [(30000, False), (9000, True), (12000 + 4000 * 3, False)])
def test_preview_pieces_against_reference(golden, n, whole):
    """oracle/port.py::preview_pieces against the pieces the unmodified create_preview passed to its two
    `save` calls, bit for bit."""
    ref = golden("reference_parity.npz")
    target, result = preview_inputs(n)
    key = f"preview_{n}_"
    assert digest(np.concatenate([target.ravel(), result.ravel()])) == ref[key + "input_sha256"], "inputs differ from the golden's"
    import matchering_b200 as mg
    cfg = mg.Config(internal_sample_rate=2000, preview_size=6, preview_analysis_step=2)
    index, t_piece, r_piece = port.preview_pieces(target, result, cfg)
    for name, piece in (("target", t_piece), ("result", r_piece)):
        assert piece.shape == tuple(ref[key + name + "_shape"]) and digest(piece) == ref[key + name + "_sha256"]
    assert (len(r_piece) == n) == whole
    if not whole:
        assert r_piece[0].tolist() == [0.0, 0.0] and r_piece[-1].tolist() == [0.0, 0.0]


def test_port_limiter_against_full_size_reference_golden(golden):
    """The first 40 s of BASELINE config 5's hour against the unmodified reference's decimated output
    (tests/golden/c5_limiter_hour.npz): the limiter is causal apart from its 88-sample look-ahead, so
    a prefix run equals the hour's prefix away from its own end."""
    g = golden("c5_limiter_hour.npz")
    n, every = int(g["frames"]), int(g["every"])
    m = 44100 * 40
    x = port.synth_limiter_input_prefix(n, m, int(g["seed"]))
    small = port.synth_limiter_input(5000, 3)
    assert np.array_equal(port.synth_limiter_input_prefix(5000, 1200, 3), small[:1200])
    y = port.limit(x.astype(np.float64), port.OracleConfig())
    keep = (m - 8192) // every
    assert np.abs(y[::every][:keep] - g["rows"][:keep]).max() < 1e-12
