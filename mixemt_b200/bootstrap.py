"""Nonparametric bootstrap confidence intervals for the mixture proportions.

The reference gives one proportion per haplogroup and no uncertainty.  A bootstrap
replicate resamples the fragments with replacement (``W = sum(weights)`` draws over
the signature rows), refits from the fit being bootstrapped, and the spread of the
replicates' proportions gives percentile intervals.  The draw is counter-based
(Philox4x32-10, csrc/bootstrap.cu), so replicate ``b`` depends only on the matrix,
the weights, the start, the seed, ``b``, ``max_iter`` and ``tolerance``.  The refits
run on the GPU, several replicates per launch over class tiles (csrc/em.cu:
run_bootstrap).
"""
import ctypes
import sys

import numpy

from . import _lib, sharding
from ._lib import lib, check, ptr
from .runtime import DeviceMatrix, get_context, lookup_resident


class BootstrapResult:
    """``props`` (n_boot, H): each replicate's proportions (linear scale, as ``run_em``
    returns them); ``lnprops`` the same in log space; ``iterations`` and ``converged``
    per replicate; ``seed`` the seed of the draws; ``slots`` the replicates iterated per
    launch."""

    def __init__(self, lnprops, iterations, converged, seed, slots):
        self.lnprops = lnprops
        self.props = numpy.exp(lnprops)
        self.iterations = iterations
        self.converged = converged
        self.seed = seed
        self.slots = slots

    def interval(self, level=0.95):
        """Percentile interval ``(lo, hi)`` per haplogroup over the replicates."""
        if not 0.0 < level < 1.0:
            raise ValueError("level must lie in (0, 1)")
        tail = 100.0 * (1.0 - level) / 2.0
        lo, hi = numpy.percentile(self.props, [tail, 100.0 - tail], axis=0)
        return lo, hi


def _validate(weights, props, n_rows, n_cols, n_boot):
    w = _lib.as_f64(numpy.asarray(weights).reshape(-1))
    if w.shape[0] != n_rows:
        raise ValueError("weights has %d entries for %d rows" % (w.shape[0], n_rows))
    if not numpy.isfinite(w).all() or (w < 0).any() or (numpy.floor(w) != w).any():
        raise ValueError("bootstrap weights must be finite, non-negative integers")
    total = w.sum()
    if not 1 <= total < 2.0 ** 32:
        raise ValueError("bootstrap weights must sum to at least 1 and less than 2^32")
    p = numpy.asarray(props, dtype=numpy.float64).reshape(-1)
    if p.shape[0] != n_cols:
        raise ValueError("props has %d entries for %d haplogroups" % (p.shape[0], n_cols))
    if numpy.isnan(p).any():
        raise ValueError("props holds NaN")
    if not p.sum() > 0:
        raise ValueError("props must have a positive sum")
    if int(n_boot) < 1:
        raise ValueError("n_boot must be at least 1")
    with numpy.errstate(divide="ignore"):
        start = numpy.log(p) - numpy.log(p.sum())
    return w, numpy.ascontiguousarray(start)


def _run(dev, w, start, boot0, n_boot, seed, args):
    h = dev.shape[1]
    lnp = numpy.zeros((max(1, n_boot), h))
    iters = numpy.zeros(max(1, n_boot), dtype=numpy.int64)
    conv = numpy.zeros(max(1, n_boot), dtype=numpy.int32)
    slots = ctypes.c_int32(1)
    if n_boot > 0:
        check(lib.mxb_em_bootstrap(dev.ctx.handle, dev.handle, ptr(w), ptr(start), int(boot0),
                                   int(n_boot), int(seed), int(args.max_iter),
                                   float(args.tolerance), ptr(lnp), ptr(iters), ptr(conv),
                                   ctypes.byref(slots)))
    return lnp[:n_boot], iters[:n_boot], conv[:n_boot], slots.value


def bootstrap_props(read_hap_mat, weights, args, props, n_boot=100, seed=None):
    """Bootstrap the fit ``props`` (what ``run_em`` returned for ``read_hap_mat`` and
    ``weights``): ``n_boot`` replicates, each one ``run_em`` restart (``args.max_iter``,
    ``args.tolerance``) on resampled fragment counts, started from ``props``
    normalised; zero proportions stay zero.  ``read_hap_mat`` is a host ndarray, a
    resident ndarray or a ``DeviceMatrix``, as ``run_em`` takes it.  ``seed=None``
    draws one from the global ``numpy.random`` stream.  With ``args.b200_shard ==
    "restarts"`` the replicates are dealt to the ranks in contiguous blocks.

    Returns a :class:`BootstrapResult`."""
    shard = getattr(args, "b200_shard", None)
    if shard == "rows":
        raise ValueError("a row-sharded bootstrap is not supported; use b200_shard='restarts'")
    dev = None
    if isinstance(read_hap_mat, DeviceMatrix):
        dev = read_hap_mat
        n, h = dev.shape
    else:
        if isinstance(read_hap_mat, numpy.ndarray):
            dev = lookup_resident(read_hap_mat)
        mat = read_hap_mat if dev is not None else _lib.as_f64(read_hap_mat)
        if mat.ndim != 2:
            raise ValueError("read_hap_mat must be 2-dimensional")
        n, h = mat.shape
    n_boot = int(n_boot)
    w, start = _validate(weights, props, n, h, n_boot)
    if seed is not None and not 0 <= int(seed) < 2 ** 64:
        raise ValueError("seed must lie in [0, 2^64)")

    ctx = get_context()
    fan_out = False
    if shard == "restarts":
        ctx.init_comm_from_torch()
        fan_out = ctx.world > 1
    if seed is None:
        draw = lambda: numpy.array([numpy.random.randint(0, 2 ** 53, dtype=numpy.int64)])
        if fan_out:
            seed = int(sharding.share_from_rank0(draw, (1,), ctx.rank, ctx.allreduce_host)[0])
        else:
            seed = int(draw()[0])
    seed = int(seed)
    owned = dev is None
    if owned:
        dev = DeviceMatrix.from_host(ctx, mat)
    try:
        if fan_out:
            mine = sharding.restart_shard(n_boot, ctx.rank, ctx.world)
            boot0 = mine[0] if mine else 0
            lnp, iters, conv, slots = _run(dev, w, start, boot0, len(mine), seed, args)
            lnp, iters, conv = sharding.merge_bootstrap(lnp, iters, conv, boot0, n_boot,
                                                        ctx.allreduce_host)
        else:
            lnp, iters, conv, slots = _run(dev, w, start, 0, n_boot, seed, args)
    finally:
        if owned:
            dev.free()
    if getattr(args, "verbose", False):
        sys.stderr.write("Bootstrap: %d replicates (seed %d), %d per launch, iterations mean "
                         "%.1f, %d converged\n" % (n_boot, seed, slots, iters.mean(),
                                                   int(conv.sum())))
    return BootstrapResult(lnp, iters, conv, seed, slots)


def boot_counts(weights, seed, boot0=0, n_boot=1):
    """The resampled fragment counts of replicates ``boot0 .. boot0 + n_boot - 1``:
    ``(n_boot, N)`` uint32, drawn on the GPU (``mxb_boot_counts``)."""
    w = _lib.as_f64(numpy.asarray(weights).reshape(-1))
    out = numpy.zeros((int(n_boot), w.shape[0]), dtype=numpy.uint32)
    check(lib.mxb_boot_counts(get_context().handle, ptr(w), w.shape[0], int(seed), int(boot0),
                              int(n_boot), ptr(out)))
    return out
