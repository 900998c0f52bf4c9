"""matchering_b200.checker against the UNMODIFIED reference's checker (matchering/checker.py:75-137):
the clipping / limiter warning rule, the order of the checks and the rate-scaled minimum length.
What the reference's checker reported on these cases is stored in tests/golden/reference_surface.json
(oracle/make_golden_parity.py)."""
import json
import os

import numpy as np
import pytest

import matchering_b200 as mg
from matchering_b200 import checker
from matchering_b200.log import Code, ModuleError

CLIP, LIM = int(Code.WARNING_TARGET_IS_CLIPPING), int(Code.WARNING_TARGET_LIMITER_IS_APPLIED)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_surface.json")


@pytest.fixture(scope="module")
def reference_checker():
    with open(GOLDEN) as f:
        surface = json.load(f)
    return surface["checker_warnings"], surface["checker_errors"]


def _noise(n=6000, seed=0, scale=0.5):
    return np.random.default_rng(seed).uniform(-scale, scale, (n, 2))


def _with_peaks(peak, count, n=6000, seed=0):
    x = _noise(n, seed)
    idx = np.random.default_rng(seed + 1).choice(n, count, replace=False)
    x[idx, 0] = peak * np.where(np.arange(count) % 2 == 0, 1.0, -1.0)
    return x


# (label, array, expected warning codes in order) -- verified against the reference below
CASES = [
    ("24-bit +FS x 20 -> clipping", _with_peaks(8388607 / 8388608, 20), [CLIP]),
    ("24-bit +FS x 8 (at the threshold, not above)", _with_peaks(8388607 / 8388608, 8), []),
    ("float 1.5 x 200 -> limiter (not close to 1.0)", _with_peaks(1.5, 200), [LIM]),
    ("float 1.5 x 20 -> nothing", _with_peaks(1.5, 20), []),
    ("0.9 x 9 -> limiter? no: 9 <= 128", _with_peaks(0.9, 9), []),
    ("0.9 x 129 -> limiter", _with_peaks(0.9, 129), [LIM]),
    ("0.9 x 128 -> nothing", _with_peaks(0.9, 128), []),
    ("1.0 x 129 -> clipping wins", _with_peaks(1.0, 129), [CLIP]),
    ("1.000001 x 9 -> clipping (isclose)", _with_peaks(1.000001, 9), [CLIP]),
]


@pytest.mark.parametrize("label,array,expected", CASES, ids=[c[0] for c in CASES])
def test_peak_warning_rule(label, array, expected):
    peak, hits = checker._count_max_peaks(array)
    code = checker.peak_warning(peak, hits, mg.Config())
    assert ([int(code)] if code is not None else []) == expected


@pytest.mark.parametrize("label,array,expected", CASES, ids=[c[0] for c in CASES])
def test_peak_warning_rule_matches_live_reference(reference_checker, label, array, expected):
    seen = reference_checker[0][label]  # the reference's warnings on this array
    from matchering_b200.log.explanations import explain
    assert seen == [explain(Code(c), False) for c in expected]
    ours = []
    mg.log(warning_handler=ours.append)
    try:
        out, sr = checker.check(array.copy(), 44100, mg.Config(), "target")
    finally:
        mg.log()
    assert ours == seen and sr == 44100 and np.array_equal(out, array)


def test_check_order_and_scaled_minimum_length(reference_checker):
    """Length is judged at the SOURCE rate against fft_size * rate // internal_rate, before channels
    and before resampling (matchering/checker.py:95-110)."""
    ref_errors = reference_checker[1]  # what the reference's checker raised on the same two arrays
    cfg_ours = mg.Config()
    # 3000 frames at 22050 Hz: >= 4096 * 22050 // 44100 = 2048 -> accepted by the length check, and the
    # 3-channel error comes before any resampling
    x3 = np.zeros((3000, 3))
    with pytest.raises(ModuleError) as e:
        checker.check(x3, 22050, cfg_ours, "reference")
    for err in (ref_errors["three_channels_22050"], {"type": type(e.value).__name__, "message": str(e.value)}):
        assert err["type"] == "ModuleError"
        assert err["message"].startswith(f"{int(Code.ERROR_REFERENCE_NUM_OF_CHANNELS_IS_EXCEEDED)}:")
    # 2000 frames at 22050 Hz: below the scaled minimum
    x2 = np.zeros((2000, 2))
    with pytest.raises(ModuleError) as e:
        checker.check(x2, 22050, cfg_ours, "target")
    for err in (ref_errors["too_short_22050"], {"type": type(e.value).__name__, "message": str(e.value)}):
        assert err["type"] == "ModuleError"
        assert err["message"].startswith(f"{int(Code.ERROR_TARGET_LENGTH_IS_TOO_SMALL)}:")
    # too long is judged at the source rate as well
    class Fake:  # only .shape is looked at before the error
        shape = (cfg_ours.max_length * 22050 + 1, 2)
    with pytest.raises(ModuleError) as e:
        checker.check(Fake(), 22050, cfg_ours, "target")
    assert e.value.code == Code.ERROR_TARGET_LENGTH_IS_EXCEEDED
