"""Log-likelihood of a fit, and a likelihood-ratio test of whether each contributor is present.

The mixture log-likelihood of proportions ``pi`` is

    l(pi) = sum_i w_i logsumexp_j(M_ij + ln pi_j)

(csrc/loglik.cu: up to 16 vectors per read of the matrix).  The reference reports none; with it
two fits can be compared, e.g. restarts that ended in different optima.

``contributor_lrt`` tests each column ``c`` in turn: it refits from the fit with ``pi_c`` held at
0 (EM's multiplicative M-step keeps a zero proportion at exactly zero) and compares the
maximised log-likelihood with the unconstrained one, ``D = 2 (l_full - l_null)``.  The
proportion lies on the boundary of its range under the null, so ``D`` follows the chi-bar-square
mixture ``0.5 chi2_0 + 0.5 chi2_1`` (Self and Liang 1987): ``p = 0.5 erfc(sqrt(D / 2))`` for
``D > 0`` and 1 for ``D = 0``.  The unconstrained fit and the K constrained ones are refitted
side by side on class tiles (csrc/em.cu: mxb_em_refit), from the same starting point and with
the same stopping rule.
"""
import ctypes
import math
import sys

import numpy

from . import _lib, sharding
from ._lib import lib, check, ptr
from .bootstrap import _deal_tasks, start_from_props
from .consumers import _collective, _shard_mark
from .runtime import OnDevice, get_context, matrix_shape


def _weights(weights, n_rows):
    w = _lib.as_f64(numpy.asarray(weights).reshape(-1))
    if w.shape[0] != n_rows:
        raise ValueError("weights has %d entries for %d rows" % (w.shape[0], n_rows))
    if not numpy.isfinite(w).all() or (w < 0).any():
        raise ValueError("weights must be finite and non-negative")
    return w


def _lnprops(props, n_cols):
    """``(K x H log-proportions normalised per vector, whether props was one vector)``."""
    p = numpy.asarray(props, dtype=numpy.float64)
    single = p.ndim == 1
    if single:
        p = p.reshape(1, -1)
    if p.ndim != 2 or p.shape[0] < 1 or p.shape[1] != n_cols:
        raise ValueError("props must have shape (%d,) or (K, %d), not %s"
                         % (n_cols, n_cols, numpy.shape(props)))
    if numpy.isnan(p).any():
        raise ValueError("props holds NaN")
    if not numpy.isfinite(p).all() or (p < 0).any():
        raise ValueError("props must be finite and non-negative")
    sums = p.sum(axis=1)
    if not (sums > 0).all():
        raise ValueError("every proportion vector must have a positive sum")
    with numpy.errstate(divide="ignore"):
        return numpy.ascontiguousarray(numpy.log(p) - numpy.log(sums)[:, None]), single


def _loglik(dev, w, lnp):
    """``mxb_matrix_loglik`` of the K x H log-proportions ``lnp`` over ``dev``'s rows."""
    lnp = numpy.ascontiguousarray(lnp, dtype=numpy.float64)
    out = numpy.zeros(lnp.shape[0])
    check(lib.mxb_matrix_loglik(dev.ctx.handle, dev.handle, ptr(w), ptr(lnp), lnp.shape[0],
                                ptr(out)))
    return out


def log_likelihood(read_hap_mat, weights, props, sharded=False):
    """``sum_i weights[i] * logsumexp_j(read_hap_mat[i, j] + log(props[j]))`` for linear-scale
    ``props``, each vector normalised to sum 1 first (``run_em`` returns a geometric mean that
    does not).  ``props`` of shape (H,) gives a float, (K, H) an ndarray of K values.  Weights
    need not be integers; a row of weight 0 adds exactly 0.  ``read_hap_mat`` is a host ndarray,
    a resident ndarray or a ``DeviceMatrix``.  On a row shard (``sharded=True``, or a
    ``DeviceMatrix`` with ``row_shard``) each rank passes its rows and weights, and every rank
    returns the total of the whole matrix."""
    n, h = matrix_shape(read_hap_mat)
    lnp, single = _lnprops(props, h)
    mark, ctx = _shard_mark(read_hap_mat, sharded)
    if mark is None:
        w = _weights(weights, n)
        with OnDevice(read_hap_mat) as dev:
            out = _loglik(dev, w, lnp)
    else:
        out, err = numpy.zeros(lnp.shape[0]), None
        try:
            w = _weights(weights, n)
            with OnDevice(read_hap_mat, ctx) as dev:
                out = _loglik(dev, w, lnp)
        except Exception as exc:      # local failure: reported through the sum
            err = exc
        out = _collective(err, lambda ok: sharding.sum_ranks(out, ctx.allreduce_host, ok))
    return float(out[0]) if single else out


def boundary_pvalue(statistic):
    """P(D >= statistic) under ``0.5 chi2_0 + 0.5 chi2_1``: ``0.5 erfc(sqrt(D / 2))`` for
    D > 0 (half the chi-square(1) tail), 1 for D = 0."""
    d = float(statistic)
    return 0.5 * math.erfc(math.sqrt(d / 2.0)) if d > 0 else 1.0


def null_start(props, column):
    """The start of the refit without ``column``: ``props`` with that column set to 0,
    renormalised over the others, in log space (-inf for a zero)."""
    q = numpy.array(props, dtype=numpy.float64).reshape(-1)
    q[column] = 0.0
    with numpy.errstate(divide="ignore"):
        return numpy.log(q) - numpy.log(q.sum())


def _columns(columns, props):
    arr = numpy.asarray(columns).reshape(-1)
    if arr.size and arr.dtype.kind not in "iu":
        raise ValueError("columns must be integer column indexes")
    cols = [int(c) for c in arr]
    h = len(props)
    if not cols:
        raise ValueError("no columns to test")
    if len(set(cols)) != len(cols):
        raise ValueError("columns holds duplicates")
    for c in cols:
        if not 0 <= c < h:
            raise ValueError("column %d out of range (%d haplogroups)" % (c, h))
        if props[c] == 0:
            raise ValueError("the proportion of column %d is 0: nothing to test" % c)
        if not numpy.delete(props, c).sum() > 0:
            raise ValueError("column %d holds all the mass: no fit without it" % c)
    return cols


class LRTResult:
    """``columns`` the tested columns; ``loglik_full`` the log-likelihood of the unconstrained
    refit and ``loglik_null`` (K,) of each refit without its column; ``statistic`` (K,)
    ``D = max(0, 2 (loglik_full - loglik_null))`` (+inf when the null fit cannot explain the
    reads); ``pvalue`` (K,) the boundary p-value (:func:`boundary_pvalue`); ``lnprops_full``
    (H,) and ``lnprops_null`` (K, H) the refits' log-proportions; ``iterations`` and
    ``converged`` of all 1 + K refits, the unconstrained one first; ``slots`` the refits
    iterated per launch."""

    def __init__(self, columns, loglik, lnprops, iterations, converged, slots):
        self.columns = list(columns)
        self.loglik_full = float(loglik[0])
        self.loglik_null = numpy.asarray(loglik[1:], dtype=numpy.float64)
        with numpy.errstate(invalid="ignore"):
            d = numpy.maximum(0.0, 2.0 * (self.loglik_full - self.loglik_null))
        self.statistic = numpy.where(self.loglik_null == -numpy.inf, numpy.inf, d)
        self.pvalue = numpy.array([boundary_pvalue(x) for x in self.statistic])
        self.lnprops_full = lnprops[0]
        self.lnprops_null = lnprops[1:]
        self.iterations = iterations
        self.converged = converged
        self.slots = slots

    def report(self, haplogroups, out=None):
        """One line per tested column on ``out`` (default ``sys.stdout``): haplogroup, its
        proportion in the unconstrained refit, D and p."""
        out = sys.stdout if out is None else out
        for k, c in enumerate(self.columns):
            out.write("%s\t%.6f\tD=%.6g\tp=%.3g\n" % (haplogroups[c],
                                                     math.exp(self.lnprops_full[c]),
                                                     self.statistic[k], self.pvalue[k]))


def _refit(dev, w, starts, max_iter, tol):
    k, h = starts.shape
    lnp = numpy.zeros((max(1, k), h))
    iters = numpy.zeros(max(1, k), dtype=numpy.int64)
    conv = numpy.zeros(max(1, k), dtype=numpy.int32)
    slots = ctypes.c_int32(1)
    if k > 0:
        check(lib.mxb_em_refit(dev.ctx.handle, dev.handle, ptr(w), ptr(starts), k, int(max_iter),
                               float(tol), ptr(lnp), ptr(iters), ptr(conv), ctypes.byref(slots)))
    return lnp[:k], iters[:k], conv[:k], slots.value


def contributor_lrt(read_hap_mat, weights, args, props, columns, tolerance=None):
    """Likelihood-ratio test of each column in ``columns`` of the fit ``props`` (what
    ``run_em`` returned for ``read_hap_mat`` and ``weights``).  The unconstrained fit and one
    fit per column with that column's proportion held at 0 are refitted from ``props``
    normalised (the column dropped and the rest renormalised), each as one ``run_em`` restart
    with ``args.max_iter`` and ``tolerance`` (default ``args.tolerance``), so that both sides
    stop by the same rule; their log-likelihoods give the statistics.  ``read_hap_mat`` is a
    host ndarray, a resident ndarray or a ``DeviceMatrix``.  With ``args.b200_shard ==
    "restarts"`` the refits are dealt to the ranks in contiguous blocks and every rank returns
    the same result.

    Returns an :class:`LRTResult`."""
    shard = getattr(args, "b200_shard", None)
    if shard == "rows":
        raise ValueError("a row-sharded likelihood-ratio test is not supported; use "
                         "b200_shard='restarts'")
    n, h = matrix_shape(read_hap_mat)
    w = _weights(weights, n)
    p = numpy.asarray(props, dtype=numpy.float64).reshape(-1)
    if (p < 0).any() or numpy.isinf(p).any():
        raise ValueError("props must be finite and non-negative")
    full = start_from_props(p, h)
    cols = _columns(columns, p)
    starts = numpy.ascontiguousarray(numpy.vstack([full] + [null_start(p, c) for c in cols]))
    tol = args.tolerance if tolerance is None else tolerance
    n_fits = len(starts)

    ctx = get_context()
    with OnDevice(read_hap_mat, ctx) as dev:
        lnp, iters, conv, slots = _deal_tasks(
            ctx, shard, n_fits, lambda k0, k: _refit(dev, w, starts[k0:k0 + k], args.max_iter, tol))
        loglik = _loglik(dev, w, lnp)
    if getattr(args, "verbose", False):
        sys.stderr.write("LRT: %d columns, %d refits per launch, iterations mean %.1f, %d of %d "
                         "converged\n" % (len(cols), slots, iters.mean(), int(conv.sum()),
                                          n_fits))
    return LRTResult(cols, loglik, lnp, iters, conv, slots)
