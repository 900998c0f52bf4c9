"""ORACLE (test infrastructure only) -- import the UNMODIFIED reference here.

`import matchering` from /root/reference fails in this image because three
third-party packages are absent: soundfile (``matchering/results.py:22``),
resampy (``matchering/checker.py:22``) and statsmodels (``matchering/dsp.py:22``).
This module injects stand-ins into ``sys.modules`` BEFORE the import so that the
reference's own ``stages.main`` / ``limiter.limit`` / helpers run unmodified:

* soundfile, resampy: file I/O and resampling only, off the hot path.
* statsmodels.api.nonparametric.lowess -> oracle/lowess.py (the one piece of
  hot-path arithmetic that is a restatement; see that file's header).

Needs a checkout of the reference (MATCHERING_REFERENCE_ROOT).  Used by the
oracle/make_golden*.py scripts, which store what the tests compare against
under tests/golden/.
"""
import os
import sys
import types
import warnings

REFERENCE_ROOT = os.environ.get("MATCHERING_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "matchering"))


def import_reference():
    """Return the reference package (module object named ``matchering``)."""
    if "matchering" in sys.modules and getattr(sys.modules["matchering"], "__mgb_shimmed__", False):
        return sys.modules["matchering"]
    if not reference_available():
        raise ImportError(f"reference tree not found at {REFERENCE_ROOT}")
    here = os.path.dirname(os.path.abspath(__file__))
    if here not in sys.path:
        sys.path.insert(0, here)
    import lowess as _lowess  # oracle/lowess.py
    import numpy as np

    if "soundfile" not in sys.modules:
        sf = types.ModuleType("soundfile")
        sf.check_format = lambda fmt, subtype=None, endian=None: True

        def _no_io(*a, **k):
            raise RuntimeError("soundfile shim: no file I/O in the oracle")

        sf.read = _no_io
        sf.write = _no_io
        sys.modules["soundfile"] = sf
    if "resampy" not in sys.modules:
        rs = types.ModuleType("resampy")

        def _no_rs(*a, **k):
            raise RuntimeError("resampy shim: no resampling in the oracle")

        rs.resample = _no_rs
        sys.modules["resampy"] = rs
    if "statsmodels.api" not in sys.modules:
        sm_pkg = types.ModuleType("statsmodels")
        sm_api = types.ModuleType("statsmodels.api")
        nonparam = types.SimpleNamespace()

        def _lowess_shim(endog, exog, frac=2.0 / 3.0, it=3, delta=0.0, **kw):
            fitted = _lowess.lowess(endog, exog, frac, it, delta)
            return np.column_stack([np.asarray(exog, dtype=float), fitted])

        nonparam.lowess = _lowess_shim
        sm_api.nonparametric = nonparam
        sm_pkg.api = sm_api
        sys.modules["statsmodels"] = sm_pkg
        sys.modules["statsmodels.api"] = sm_api
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import matchering  # noqa: the reference itself
    matchering.__mgb_shimmed__ = True
    return matchering
