"""Host rules of the log-likelihood and the contributor likelihood-ratio test
(mixemt_b200.likelihood), no GPU: the boundary p-value against scipy's chi-square tail halved,
the starts of the constrained refits, the statistic of an LRTResult, every argument error of
log_likelihood and contributor_lrt (raised before the device is touched), and rows mode
rejected."""
import io
import math

import numpy as np
import pytest
from scipy.stats import chi2

from mixemt_b200 import likelihood
from conftest import make_args


@pytest.mark.parametrize("d", [1e-12, 1e-3, 0.5, 1.0, 2.705543, 3.841459, 10.0, 50.0, 300.0])
def test_pvalue_is_half_the_chi2_tail(d):
    want = chi2.sf(d, 1) / 2
    assert abs(likelihood.boundary_pvalue(d) - want) <= 1e-12 * want


def test_pvalue_at_zero_and_infinity():
    """D = 0 carries the point mass of the mixture: p = 1; D = inf: p = 0 (scipy's tail too)."""
    assert likelihood.boundary_pvalue(0.0) == 1.0
    assert likelihood.boundary_pvalue(math.inf) == 0.0 == chi2.sf(math.inf, 1) / 2


def test_null_start_drops_the_column_and_renormalises():
    p = np.array([0.5, 0.2, 0.0, 0.3, 1e-300])
    for c in (0, 1, 3, 4):
        s = likelihood.null_start(p, c)
        assert s[c] == -np.inf and s[2] == -np.inf
        rest = [j for j in range(5) if j not in (c, 2)]
        assert abs(np.exp(s[rest]).sum() - 1.0) < 1e-15
        q = p[rest] / p[rest].sum()
        assert np.allclose(np.exp(s[rest]), q, rtol=1e-13, atol=0)


def test_statistic_and_report():
    ll = np.array([-100.0, -100.0, -103.0, -np.inf, -99.0])
    lnp = np.log(np.tile([0.5, 0.25, 0.125, 0.125], (5, 1)))
    res = likelihood.LRTResult([0, 1, 2, 3], ll, lnp, np.arange(5), np.ones(5), 2)
    assert res.loglik_full == -100.0
    assert np.array_equal(res.statistic, [0.0, 6.0, np.inf, 0.0])   # a better null clips to 0
    assert res.pvalue[0] == 1.0 and res.pvalue[2] == 0.0 and res.pvalue[3] == 1.0
    assert abs(res.pvalue[1] - chi2.sf(6.0, 1) / 2) < 1e-15
    assert res.lnprops_full.shape == (4,) and res.lnprops_null.shape == (4, 4)
    out = io.StringIO()
    res.report(["A", "B", "C", "D"], out)
    lines = out.getvalue().splitlines()
    assert len(lines) == 4 and lines[1].startswith("B\t0.250000\tD=6\t")


MAT = np.log(np.array([[0.5, 0.3, 0.2], [0.1, 0.6, 0.3], [0.2, 0.2, 0.6], [0.3, 0.3, 0.4]]))
W = np.array([1.0, 2.0, 0.5, 3.0])


@pytest.mark.parametrize("mat,weights,props", [
    (MAT, W, [0.5, 0.5]),                       # wrong length
    (MAT, W, [[0.2, 0.3, 0.5], [0.5, 0.5]]),    # ragged
    (MAT, W, np.ones((2, 2, 3))),               # 3-d
    (MAT, W, np.ones((0, 3))),                  # no vector
    (MAT, W, [0.2, np.nan, 0.5]),
    (MAT, W, [0.2, -0.1, 0.5]),
    (MAT, W, [0.2, np.inf, 0.5]),
    (MAT, W, [[0.2, 0.3, 0.5], [0.0, 0.0, 0.0]]),
    (MAT, [1.0, 2.0, np.nan, 1.0], [0.2, 0.3, 0.5]),
    (MAT, [1.0, 2.0, np.inf, 1.0], [0.2, 0.3, 0.5]),
    (MAT, [1.0, -2.0, 1.0, 1.0], [0.2, 0.3, 0.5]),
    (MAT, [1.0, 2.0, 1.0], [0.2, 0.3, 0.5]),
    (MAT[0], W, [0.2, 0.3, 0.5]),               # 1-d matrix
])
def test_log_likelihood_errors(mat, weights, props):
    with pytest.raises(ValueError):
        likelihood.log_likelihood(mat, np.asarray(weights, dtype=np.float64), props)


P = np.array([0.5, 0.3, 0.2])


@pytest.mark.parametrize("weights,props,columns", [
    (W, P, []),
    (W, P, [0, 0]),
    (W, P, [3]),
    (W, P, [-1]),
    (W, P, [1.0]),
    (W, [0.5, 0.5, 0.0], [2]),                  # nothing to test
    (W, [0.0, 1.0, 0.0], [1]),                  # no mass without it
    (W, [0.5, np.nan, 0.2], [0]),
    (W, [0.0, 0.0, 0.0], [0]),
    (W, [0.5, 0.5], [0]),
    (W, [0.5, -0.2, 0.7], [0]),
    ([1.0, 2.0, np.nan, 1.0], P, [0]),
    ([1.0, -1.0, 1.0, 1.0], P, [0]),
    ([1.0, 1.0, 1.0], P, [0]),
])
def test_contributor_lrt_errors(weights, props, columns):
    with pytest.raises(ValueError):
        likelihood.contributor_lrt(MAT, np.asarray(weights, dtype=np.float64), make_args(),
                                   np.asarray(props, dtype=np.float64), columns)


def test_rows_mode_is_rejected():
    with pytest.raises(ValueError):
        likelihood.contributor_lrt(MAT, W, make_args(b200_shard="rows"), P, [0])


def test_non_integer_weights_are_accepted_by_the_checks():
    """The bootstrap's integer rule does not apply: fractional weights pass validation."""
    w = likelihood._weights([0.5, 1.25, 0.0, 3.0], 4)
    assert w.dtype == np.float64 and w[1] == 1.25
