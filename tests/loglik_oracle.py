"""Long-double restatement of the log-likelihood (csrc/loglik.cu, mixemt_b200.likelihood) and
of the contributor likelihood-ratio test for the tests: the refits are oracle_np.run_em
restarts, the log-likelihoods tile_cases._ld_lse in long double, the p-value scipy's chi-square
tail halved."""
import numpy as np
from scipy.stats import chi2

from oracle import oracle_np
from tile_cases import _ld_lse


def ld_row_loglik(mat, lnp):
    """l_i = logsumexp_j(M_ij + ln pi_j) per row in long double (-inf without a finite term)."""
    z = np.asarray(lnp, dtype=np.longdouble) + np.asarray(mat, dtype=np.longdouble)
    return _ld_lse(z, 1)


def ld_loglik(mat, w, lnp):
    """(sum_i w_i l_i over the rows of nonzero weight, sum_i w_i |l_i| over its finite terms):
    the value and the scale of its tolerance."""
    li = ld_row_loglik(mat, lnp)
    wl = np.asarray(w, dtype=np.longdouble)
    terms = wl[wl != 0] * li[wl != 0]
    return terms.sum(), np.abs(terms[np.isfinite(terms)]).sum()


def starts(props, columns):
    """The unconstrained start and one start per column with that column at 0, in log space."""
    p = np.asarray(props, dtype=np.float64)
    out = []
    for c in [None] + list(columns):
        q = p.copy()
        if c is not None:
            q[c] = 0.0
        with np.errstate(divide="ignore"):
            out.append(np.log(q) - np.log(q.sum()))
    return np.array(out)


def lrt(mat, w, props, columns, max_iter, tol):
    """The whole test: {loglik (1 + K), statistic (K), pvalue (K), props (1 + K, H),
    iterations (1 + K), scale}."""
    lls, scales, fits, iters = [], [], [], []
    for s in starts(props, columns):
        o_props, _, it = oracle_np.run_em(mat, w, s.reshape(1, -1), max_iter, tol)
        with np.errstate(divide="ignore"):
            ll, scale = ld_loglik(mat, w, np.log(o_props))
        lls.append(ll)
        scales.append(scale)
        fits.append(o_props)
        iters.append(it[0])
    lls = np.array(lls)
    d = np.where(lls[1:] == -np.inf, np.inf, np.maximum(0, 2 * (lls[0] - lls[1:])))
    p = np.array([1.0 if x == 0 else chi2.sf(float(x), 1) / 2 for x in d])
    return dict(loglik=lls, statistic=d, pvalue=p, props=np.array(fits),
                iterations=np.array(iters), scale=max(scales))
