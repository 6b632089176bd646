"""The rule that sends a row to the log-space step (csrc/em_kernels.cuh: row_needs_logspace,
flag when !(t >= 2^-960)), rehearsed in numpy fp64 on window_cases: the pass arithmetic of
window_cases.model_pass, a flagged iteration redone by the long-double log-space formula, against
tile_cases.ld_iterate.  Every iteration the rule leaves in linear space must agree with the
reference within the tolerance of the GPU tests; the old rule (t == 0) leaves rows in linear
space whose coefficient w / t overflows, and the proportions become NaN.  No GPU needed."""
import numpy as np
import pytest

from tile_cases import ld_iterate
from window_cases import (LEVELS, LN_THETA, MODES, SCALES, THETA, model_iterate, rule_new,
                          rule_old, window_case)

LN_TOL = 1e-12       # test_tile_kernels_gpu.LN_TOL
K = 3

_TRAJ = {}


def _case(layout, mode, level):
    key = (layout, mode, level)
    if key not in _TRAJ:
        mat, w, lnp, _ = window_case(layout, mode, level)
        _TRAJ[key] = (mat, w, lnp, ld_iterate(mat, w, lnp, K))
    return _TRAJ[key]


def _ld_step(mat, w):
    return lambda lnp: ld_iterate(mat, w, lnp, 1)[1]


def _ln_err(got, want):
    """Largest relative log error on finite entries; inf when the -inf patterns differ or an
    entry the reference keeps finite is not."""
    want = np.asarray(want, dtype=np.longdouble)
    if not np.array_equal(np.isneginf(got), np.isneginf(want)):
        return np.inf
    fin = np.isfinite(want)
    if not np.isfinite(got[fin]).all():
        return np.inf
    return float((np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))).max())


def test_theta_constants():
    assert THETA == np.ldexp(1.0, -960) and np.log(THETA) == pytest.approx(LN_THETA, abs=1e-12)
    # the coefficient bound: w * 2^960 summed over a total weight below 2^63 stays finite
    assert np.isfinite(np.ldexp(1.0, 63) / THETA)
    # subnormal terms (at most 2^-1075 each) move t by less than an ulp, up to 2^62 columns
    assert np.ldexp(1.0, 62 - 1075) / THETA < np.finfo(np.float64).eps


@pytest.mark.parametrize("layout", ["rows", "narrow"])
@pytest.mark.parametrize("mode", MODES)
def test_new_rule_matches_long_double(layout, mode):
    """Flagged at every level below theta, not above it; every case, at every weight scale,
    follows the long-double trajectory for K iterations, and every iteration left in linear
    space is within the GPU tolerance."""
    for level in LEVELS:
        mat, w, lnp, traj = _case(layout, mode, level)
        for scale in SCALES:
            ws = w * scale
            got, flags = model_iterate(mat, ws, lnp, K, rule_new, _ld_step(mat, ws))
            assert flags[0] == (level < LN_THETA), (level, scale, flags)
            for k in range(1, K + 1):
                err = _ln_err(got[k], traj[k])
                assert err <= LN_TOL, (level, scale, k, flags, err)


@pytest.mark.parametrize("mode", MODES)
def test_old_rule_leaves_nan_in_the_window(mode):
    """With t == 0 as the test, every level from e^-740 to e^-705 goes through linear space and
    gives NaN proportions at every weight scale, and e^-700 does at scales 1e3 and 1e6 (normal t,
    coefficient overflow).  The new rule flags every case that gives NaN."""
    for level in LEVELS:
        mat, w, lnp, traj = _case("rows", mode, level)
        for scale in SCALES:
            ws = w * scale
            got_old, flags_old = model_iterate(mat, ws, lnp, 1, rule_old, _ld_step(mat, ws))
            nan_old = not flags_old[0] and np.isnan(got_old[1]).any()
            must = (-740.0 <= level <= -705.0) or (level == -700.0 and scale >= 1e3)
            if must:
                assert nan_old, (level, scale, flags_old)
            if nan_old:
                _, flags_new = model_iterate(mat, ws, lnp, 1, rule_new, _ld_step(mat, ws))
                assert flags_new[0], (level, scale)
        if level == -760.0:      # exactly 0: both rules flag it
            assert model_iterate(mat, w, lnp, 1, rule_old, _ld_step(mat, w))[1][0]
