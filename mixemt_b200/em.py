"""B200 drop-in for ``mixemt.em`` (reference mixemt/em.py:23-165).

Same function names, arguments, return values and stderr messages as the
reference; the iteration loop runs on the GPU (csrc/em.cu) behind the C-ABI.
Random initialisation stays on the host and consumes the legacy global
``numpy.random`` stream exactly like the reference does (one Dirichlet draw of
length H per restart, em.py:36; SURVEY.md F6).
"""
import ctypes
import sys

import numpy

from . import _lib
from ._lib import lib, check, ptr
from . import sharding
from .runtime import (DeviceMatrix, RowShard, get_context, lookup_resident, remember_resident,
                      resident_mode)


def init_props(nhaps, alpha=1.0):
    """Random start: Dirichlet(alpha, ..., alpha), or uniform for alpha=inf
    (reference em.py:23-36)."""
    if alpha == float("inf"):
        return numpy.full(nhaps, 1.0 / nhaps)
    return numpy.random.dirichlet(numpy.full(nhaps, alpha).tolist())


def converged(prop, last_prop, tolerance=0.0001):
    """``sum |exp(prop) - exp(last_prop)| < tolerance`` on log-proportions
    (reference em.py:39-54).  The GPU loop applies the same test on device."""
    return numpy.abs(numpy.exp(prop) - numpy.exp(last_prop)).sum() < tolerance


def em_step(read_hap_mat, weights, ln_props, read_mix_mat):
    """One EM iteration (reference em.py:57-91).

    ``read_mix_mat`` is overwritten in place with the log responsibilities
    ``(M + ln_props) - logsumexp_rows(...)`` and returned together with the new
    log-proportions."""
    ctx = get_context()
    mat = _lib.as_f64(read_hap_mat)
    n, h = mat.shape
    wts = _lib.as_f64(numpy.asarray(weights).reshape(-1))
    props = _lib.as_f64(ln_props)
    direct = (isinstance(read_mix_mat, numpy.ndarray) and read_mix_mat.dtype == numpy.float64
              and read_mix_mat.flags["C_CONTIGUOUS"] and read_mix_mat.shape == (n, h)
              and read_mix_mat.flags.writeable)
    out = read_mix_mat if direct else numpy.empty((n, h))
    new_props = numpy.empty(h)
    check(lib.mxb_em_step(ctx.handle, ptr(mat), ptr(wts), ptr(props), n, h, ptr(out),
                          ptr(new_props)))
    if not direct:
        read_mix_mat[...] = out
    return read_mix_mat, new_props


def _draw_inits(n_multi, nhaps, alpha):
    inits = numpy.empty((n_multi, nhaps))
    for i in range(n_multi):
        inits[i] = numpy.log(init_props(nhaps, alpha=alpha))
    return inits


def _report(verbose, first_run, iters, conv):
    """The reference's progress lines (em.py:119-135), emitted after the fact."""
    if not verbose:
        return
    for k in range(len(iters)):
        sys.stderr.write("Starting EM run %d...\n" % (first_run + k + 1))
        sys.stderr.write('.' * int(iters[k] // 10))
        if conv[k]:
            sys.stderr.write("\nConverged! (%d)\n" % iters[k])


def run_em_device(dev_mat, weights, args, keep_device=False, want_host=True, inits=None):
    """``run_em`` on a matrix that already lives in HBM (``DeviceMatrix``).

    Returns ``(props, read_mix, info, read_mix_dev)``: ``read_mix`` is the host
    ndarray (``want_host``) or ``None``; ``read_mix_dev`` the HBM-resident
    ``DeviceMatrix`` (``keep_device``) or ``None``."""
    ctx = dev_mat.ctx
    n, h = dev_mat.shape
    n_multi = int(args.n_multi)
    if n_multi < 1:
        raise TypeError("run_em needs n_multi >= 1")
    wts = _lib.as_f64(numpy.asarray(weights).reshape(-1))
    if wts.shape[0] != n:
        raise ValueError("weights has %d entries for %d rows" % (wts.shape[0], n))
    shard = getattr(args, "b200_shard", None)
    verbose = getattr(args, "verbose", False)
    flags = 0
    mine = list(range(n_multi))
    if shard == "rows":
        ctx.init_comm_from_torch()
        flags |= _lib.MXB_EM_SHARDED
    elif shard == "restarts":
        ctx.init_comm_from_torch()
        if ctx.world > 1:
            flags |= _lib.MXB_EM_RAW
            mine = sharding.restart_shard(n_multi, ctx.rank, ctx.world)
    if inits is None:
        if shard in ("rows", "restarts") and ctx.world > 1:
            # every rank must start every restart from the same proportions (the fused tail
            # takes one convergence decision for all ranks): rank 0 draws from its global
            # numpy.random stream, as the reference would, and the draws are shared
            inits = sharding.share_from_rank0(
                lambda: _draw_inits(n_multi, h, args.init_alpha), (n_multi, h), ctx.rank,
                ctx.allreduce_host)
        else:
            inits = _draw_inits(n_multi, h, args.init_alpha)
    inits = _lib.as_f64(inits)

    props = numpy.zeros(h)
    iters = numpy.zeros(max(1, len(mine)), dtype=numpy.int64)
    conv = numpy.zeros(max(1, len(mine)), dtype=numpy.int32)
    read_mix = _lib.result_empty((n, h)) if (want_host and not (flags & _lib.MXB_EM_RAW)) else None
    mix_handle = ctypes.c_void_p()
    need_dev = keep_device or bool(flags & _lib.MXB_EM_RAW)
    if mine:
        my_inits = numpy.ascontiguousarray(inits[mine])
        check(lib.mxb_run_em_dev(ctx.handle, dev_mat.handle, ptr(wts), ptr(my_inits), len(mine),
                                 int(args.max_iter), float(args.tolerance), flags, ptr(props),
                                 ptr(read_mix), ctypes.byref(mix_handle) if need_dev else None,
                                 ptr(iters), ptr(conv)))
        _report(verbose, 0, iters[:len(mine)], conv[:len(mine)])
    mix_dev = DeviceMatrix(ctx, mix_handle) if (need_dev and mix_handle.value) else None
    if mix_dev is not None and shard == "rows" and ctx.world > 1:
        # the kept read matrix holds this rank's rows: the consumers work on it as a shard
        mix_dev.row_shard = dev_mat.row_shard or RowShard()

    if flags & _lib.MXB_EM_RAW:
        # restart fan-out: combine the per-rank partial results (em.py:145-163)
        if mix_dev is None:
            # no restart landed on this rank: neutral element of logaddexp
            mix_dev = DeviceMatrix.from_host(ctx, numpy.full((n, h), -numpy.inf))
        props = sharding.combine_restart_props(props, n_multi, ctx.allreduce_host)
        mix_dev.fold_ranks(numpy.log(n_multi) if n_multi > 1 else 0.0)
        if want_host:
            read_mix = mix_dev.to_host()
    info = {"iterations": iters[:len(mine)].tolist(), "converged": conv[:len(mine)].tolist(),
            "restarts": mine}
    if not keep_device and mix_dev is not None:
        mix_dev.free()
        mix_dev = None
    return props, read_mix, info, mix_dev


def run_em(read_hap_mat, weights, args):
    """
    Runs the EM algorithm on the read x haplogroup log-likelihood matrix
    (reference em.py:94-165): ``args.n_multi`` restarts from Dirichlet draws,
    each iterated until ``sum |d props| < args.tolerance`` or ``args.max_iter``.

    Returns ``(res_props, res_read_mix)``: the proportions on the linear scale
    (geometric mean over restarts, not renormalised -- em.py:155-163) and the
    N x H log responsibilities at the *previous* proportions of the final
    iteration, averaged over restarts in linear space (em.py:156, :161).
    Inputs are not modified.
    """
    ctx = get_context()
    dev = None
    owned = False
    if isinstance(read_hap_mat, DeviceMatrix):
        dev = read_hap_mat
    elif isinstance(read_hap_mat, numpy.ndarray):
        dev = lookup_resident(read_hap_mat)
    if dev is None:
        mat = _lib.as_f64(read_hap_mat)
        if mat.ndim != 2:
            raise ValueError("read_hap_mat must be 2-dimensional")
        dev = DeviceMatrix.from_host(ctx, mat)
        owned = True
    keep = resident_mode(args)
    try:
        props, read_mix, _, mix_dev = run_em_device(dev, weights, args, keep_device=keep)
    finally:
        if owned:
            dev.free()
    if keep and mix_dev is not None and read_mix is not None:
        # opt-in residency: the consumers in mixemt_b200.consumers find the HBM copy of
        # the result through the (read-only) host array, see runtime.remember_resident
        read_mix.flags.writeable = False
        remember_resident(read_mix, mix_dev)
    return props, read_mix
