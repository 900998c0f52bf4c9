"""Host-side checks that need no GPU: the C ABI library loads and exports every symbol the header
declares; the Python surface mirrors the reference's (Config/Result/log/process)."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "matchering_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mgb_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    from matchering_b200 import _native
    assert set(header_symbols()) == set(_native.PROTOTYPES)


def test_cuda_library_loads_and_exports_every_symbol():
    from matchering_b200 import _native, build
    path = build.build()  # no-op when up to date; nvcc cross-compiles without a GPU
    lib = C.CDLL(path)
    for name in header_symbols():
        assert hasattr(lib, name), name
    lib.mgb_version.restype = C.c_int
    assert lib.mgb_version() == 200
    assert C.sizeof(_native.HostBuffers) == 7 * 8
    # struct layouts the binding assumes (sizes of the C structs, computed from the header's fields)
    assert C.sizeof(_native.LimiterParams) == 8 + 6 * 4 + 8 + 4 * (_native.MGB_MAX_FILTER_ORDER + 1) * 8
    assert C.sizeof(_native.TrackLayout) == 4 * 8 + 4 * 4 + 8
    assert C.sizeof(_native.TrackState) == 6 * 8 + 16 * 8 + 2 * 8 + 4 + 4 * 4 + 3 * 4  # the last three: fir peaks + reserved


def test_emulator_library_exports_every_symbol():
    from emul_harness import emul_lib
    lib = emul_lib()
    for name in header_symbols():
        assert hasattr(lib, name), name


def test_argument_errors_are_reported_not_thrown():
    from emul_harness import EmulPlan, emul_lib
    import port
    from matchering_b200 import _native
    lib = emul_lib()
    ep = EmulPlan(port.OracleConfig(fft_size=1024))
    L = _native.TrackLayout()
    rc = lib.mgb_track_layout_init(C.byref(ep.struct), 500, 5000, C.byref(L))  # shorter than fft_size
    assert rc == _native.MGB_ERR_INVALID and b"longer than fft_size" in lib.mgb_last_error_string()
    with pytest.raises(ValueError):
        _native.check(lib, rc)
    assert lib.mgb_set_option(b"no_such_switch", 1) == _native.MGB_ERR_INVALID
    bad = _native.Plan()
    bad.fft_size = 256
    assert lib.mgb_track_layout_init(C.byref(bad), 10000, 10000, C.byref(L)) == _native.MGB_ERR_UNSUPPORTED


def test_config_matches_reference_defaults_and_asserts():
    import matchering_b200 as mg
    c = mg.Config()
    assert (c.internal_sample_rate, c.fft_size, c.rms_correction_steps, c.lin_log_oversampling) == (44100, 4096, 4, 4)
    assert c.max_piece_size == 15 * 44100 and c.threshold == (2 ** 15 - 61) / 2 ** 15 and c.min_value == 1e-6
    assert (c.lowess_frac, c.lowess_it, c.lowess_delta) == (0.0375, 0, 0.001)
    assert (c.limiter.attack, c.limiter.hold, c.limiter.release) == (1, 1, 3000)
    assert c.preview_size == 30 * 44100 and c.limiter is mg.Config().limiter  # shared default, like the reference
    for bad in (dict(threshold=1.5), dict(fft_size=1000), dict(min_value=0.5), dict(max_piece_size=0.01),
                dict(internal_sample_rate=44100.0), dict(rms_correction_steps=-1), dict(allow_equality=1)):
        with pytest.raises(AssertionError):
            mg.Config(**bad)
    with pytest.raises(AssertionError):
        mg.LimiterConfig(hold_filter_order=0)


def reference_surface():
    """The reference's Config attributes and log codes (tests/golden/reference_surface.json, written by
    oracle/make_golden_parity.py from the unmodified reference)."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_surface.json")) as f:
        return json.load(f)


def test_config_attribute_parity_with_reference():
    import matchering_b200 as mg
    ref = reference_surface()
    assert ref["config_kwargs"] == dict(internal_sample_rate=48000, max_piece_size=7.5)
    ours = mg.Config(internal_sample_rate=48000, max_piece_size=7.5)
    for name, value in ref["config"].items():
        if name == "limiter":
            assert vars(ours.limiter) == value
        else:
            assert getattr(ours, name) == value, name


def test_results_and_log_surface():
    import matchering_b200 as mg
    from matchering_b200.log import Code, ModuleError, info, warning
    r = mg.Result("out.wav", "PCM_24", use_limiter=False, normalize=False)
    assert (r.file, r.subtype, r.use_limiter, r.normalize) == ("out.wav", "PCM_24", False, False)
    assert mg.pcm16("a.wav").subtype == "PCM_16" and mg.pcm24("a.wav").subtype == "PCM_24"
    with pytest.raises(TypeError):
        mg.Result("out.xyz", "PCM_16")
    with pytest.raises(TypeError):
        mg.Result("out.wav", "VORBIS")
    seen = []
    mg.log(seen.append, show_codes=True)
    try:
        info(Code.INFO_MATCHING_LEVELS)
        warning(Code.WARNING_TARGET_IS_CLIPPING)
    finally:
        mg.log()
    assert seen[0] == "2004: Matching levels" and seen[1].startswith("3001: Audio clipping")
    assert int(Code.ERROR_VALIDATION) == 4202 and str(ModuleError(Code.ERROR_VALIDATION)).startswith("4202: Validation failed")


def test_log_codes_match_reference():
    from matchering_b200.log import Code
    assert {c.name: int(c) for c in Code} == reference_surface()["log_codes"]


def test_wav_roundtrip_and_checker(tmp_path):
    import matchering_b200 as mg
    from matchering_b200 import wavio
    from matchering_b200.log import ModuleError
    rng = np.random.default_rng(0)
    x = np.clip(0.5 * rng.standard_normal((5000, 2)), -1, 1)
    for subtype, tol in (("PCM_16", 1.6 / 32768), ("PCM_24", 1.6 / 8388608), ("PCM_32", 1e-9), ("FLOAT", 1e-7), ("DOUBLE", 0)):  # write scales by 2^(b-1)-1, read by 2^-(b-1), as libsndfile does
        path = str(tmp_path / f"x_{subtype}.wav")
        wavio.write(path, x, 44100, subtype)
        y, sr = mg.load(path, "target", str(tmp_path))
        assert sr == 44100 and y.shape == x.shape and np.abs(y - x).max() <= tol
    mono, sr = mg.check(x[:, :1].copy(), 44100, mg.Config(), "reference")
    assert mono.shape == (5000, 2) and sr == 44100
    with pytest.raises(ModuleError):
        mg.check(x[:100], 44100, mg.Config(), "target")  # shorter than fft_size
    import torch
    if torch.cuda.is_available():
        resampled, sr = mg.check(x, 22050, mg.Config(), "target")
        assert sr == 44100 and resampled.shape == (10000, 2)
    else:  # resampling is a device kernel (csrc/resample.cu): no CPU fallback
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            mg.check(x, 22050, mg.Config(), "target")


def test_process_without_results_or_gpu(tmp_path):
    import matchering_b200 as mg
    with pytest.raises(RuntimeError):
        mg.process("t.wav", "r.wav", [])
    import torch
    if not torch.cuda.is_available():
        from matchering_b200 import stages
        x = np.zeros((10000, 2))
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            stages.main(x, x, mg.Config())
