"""Device-side forms of the functions that consume ``run_em``'s results
(SURVEY.md 8f, rows N2-N4).  Same names, arguments and return values as the
reference functions they mirror; the N x H matrices are read where they live,
in HBM, so only O(N) or O(H) numbers cross PCIe:

    reduce_em_matrix          mixemt/preprocess.py:230-251
    find_contribs_from_reads  mixemt/assemble.py:102-124 (_find_contribs_from_reads)
    read_votes                mixemt/stats.py:34-46      (the argmax in report_read_votes)
    assign_read_indexes       mixemt/assemble.py:267-334
    save_npy / load_npy       bin/mixemt:214-245, :168-211 (the .npy halves of -s / -l)

Every matrix argument may be a ``DeviceMatrix``, an ndarray that
``build_em_matrix`` / ``run_em`` handed out in resident mode (its HBM copy is
reused), or any other ndarray (uploaded first: there is no host code path).

Rows mode (``args.b200_shard = "rows"`` with more than one rank): a matrix whose
``DeviceMatrix.row_shard`` is set, or any matrix passed with ``sharded=True``, is
this rank's slice of the rows.  Every rank then calls the same consumer;
contributor lists, kept columns, row indexes and .npy files are those of the whole
matrix (collectives: O(H) host all-reduces through ``Context.allreduce_host``).
An error on one rank is raised on every rank before anyone waits in a later
collective (``sharding.RankFailed`` on the ranks that did not fail).
"""
import collections
import ctypes

import numpy

from . import sharding
from ._lib import lib, check, ptr
from .runtime import (DeviceMatrix, OnDevice, RowShard, get_context, lookup_resident,
                      remember_resident, resident_mode)


def _shard_mark(mat, sharded):
    """``(mark, ctx)``: the ``RowShard`` of a consumer's matrix argument (a resident
    ndarray has it on its HBM copy; ``sharded=True`` makes a new one), ``None`` for a
    whole matrix or in a world of one rank."""
    dev = mat if isinstance(mat, DeviceMatrix) else \
        (lookup_resident(mat) if isinstance(mat, numpy.ndarray) else None)
    if dev is None and not sharded:
        return None, None
    ctx = dev.ctx if dev is not None else get_context()
    mark = dev.row_shard if dev is not None else None
    if mark is None and sharded:
        mark = RowShard()
    return (mark if ctx.world > 1 else None), ctx


def _collective(err, call):
    """``call(ok)`` for a collective that carries this rank's ok flag (``err is None``);
    a rank that failed raises its own ``err``, the others ``sharding.RankFailed``."""
    try:
        return call(err is None)
    except sharding.RankFailed:
        if err is not None:
            raise err
        raise


def _offsets(mark, n_local, ctx, err=None):
    """``(lo, n_total)`` of a marked shard; the first call computes them (a collective
    that carries ``err``), later ones read the mark."""
    if mark.lo is None:
        mark.lo, mark.n_total = _collective(err, lambda ok: sharding.shard_offsets(
            n_local, ctx.rank, ctx.world, ctx.allreduce_host, ok))
    return mark.lo, mark.n_total


def gather_columns(dev_mat, indexes):
    """``dev_mat[:, indexes]`` as a new ``DeviceMatrix`` (a row shard stays one)."""
    cols = numpy.ascontiguousarray(indexes, dtype=numpy.int64)
    handle = ctypes.c_void_p()
    check(lib.mxb_matrix_gather_cols(dev_mat.ctx.handle, dev_mat.handle, ptr(cols), len(cols),
                                     ctypes.byref(handle)))
    out = DeviceMatrix(dev_mat.ctx, handle)
    out.row_shard = dev_mat.row_shard
    return out


def reduce_em_matrix(em_mat, haplogroups, contrib_props, sharded=False):
    """
    Keeps only the columns of the haplogroups listed in ``contrib_props``
    (reference preprocess.py:230-251).  Returns ``(matrix, new_haps)``: a
    ``DeviceMatrix`` when ``em_mat`` is one, otherwise a host ndarray whose HBM
    copy stays registered so that the refinement ``run_em`` (bin/mixemt:318)
    starts without a host->device copy.

    On a row shard every rank must keep the same columns, or the refinement
    ``run_em`` would enter its per-iteration collectives with a different H on each
    rank: when the ranks disagree, every rank raises ``ValueError``.
    """
    haps_to_keep = {con[1] for con in contrib_props}
    indexes = [i for i in range(len(haplogroups)) if haplogroups[i] in haps_to_keep]
    new_haps = [haplogroups[i] for i in indexes]
    was_resident = isinstance(em_mat, numpy.ndarray) and lookup_resident(em_mat) is not None
    mark, ctx = _shard_mark(em_mat, sharded)
    if mark is None:
        with OnDevice(em_mat) as dev:
            small = gather_columns(dev, indexes)
    else:
        small, err = None, None
        try:
            with OnDevice(em_mat, ctx) as dev:
                small = gather_columns(dev, indexes)
            small.row_shard = mark
        except Exception as exc:      # local failure: reported through the agreement
            err = exc
        if not _collective(err, lambda ok: sharding.agree(indexes, ctx.allreduce_host, ok)):
            small.free()
            raise ValueError("reduce_em_matrix: the ranks keep different columns (%d here); "
                             "every rank must pass the same contributors" % len(indexes))
    if isinstance(em_mat, DeviceMatrix):
        return small, new_haps
    host = small.to_host()
    if was_resident or resident_mode():
        # opt-in residency only: the HBM copy stays registered behind a read-only array
        host.flags.writeable = False
        remember_resident(host, small)
    else:
        small.free()    # the reference hands back a fresh writable array (preprocess.py:251)
    return host, new_haps


def vote_count(read_hap_mat, wts):
    """``(votes[H], argmax[N])``: weighted votes per haplogroup column from the
    row maxima (first maximum, like ``numpy.argmax(read_hap_mat, 1)``)."""
    with OnDevice(read_hap_mat) as dev:
        n, h = dev.shape
        weights = _weights_for(wts, n)
        votes = numpy.zeros(h, dtype=numpy.int64)
        best = numpy.empty(n, dtype=numpy.int64)
        check(lib.mxb_matrix_vote_count(dev.ctx.handle, dev.handle, ptr(weights), ptr(votes),
                                        ptr(best)))
    return votes, best


def _weights_for(wts, n):
    weights = numpy.ascontiguousarray(numpy.asarray(wts).reshape(-1), dtype=numpy.int64)
    if weights.shape[0] != n:
        raise ValueError("wts has %d entries for %d rows" % (weights.shape[0], n))
    return weights


def vote_first(read_hap_mat, wts, row0=0):
    """``(votes[H], first[H])``: the votes of :func:`vote_count` and, per column, the
    smallest ``row0 + r`` whose first row maximum it is (-1: none).  Only these 2H
    numbers come back from the device."""
    with OnDevice(read_hap_mat) as dev:
        n, h = dev.shape
        weights = _weights_for(wts, n)
        votes = numpy.zeros(h, dtype=numpy.int64)
        first = numpy.empty(h, dtype=numpy.int64)
        check(lib.mxb_matrix_vote_first(dev.ctx.handle, dev.handle, ptr(weights), int(row0),
                                        ptr(votes), ptr(first)))
    return votes, first


def find_contribs_from_reads(read_hap_mat, wts, args, sharded=False):
    """
    Column indexes of the haplogroups whose reads (rows voting for them with
    their multiplicity) reach ``args.min_reads`` -- reference
    assemble.py:102-124, in the reference's order (first appearance among the
    row maxima).  On a row shard (``wts`` = this rank's weights) every rank
    returns the list of the whole matrix.
    """
    mark, ctx = _shard_mark(read_hap_mat, sharded)
    if mark is None:
        votes, first = vote_first(read_hap_mat, wts)
        return sharding.contrib_order(votes, first, args.min_reads)
    n, h = read_hap_mat.shape
    err = None
    try:
        _weights_for(wts, n)
    except ValueError as exc:
        err = exc
    lo, _ = _offsets(mark, n, ctx, err)
    votes, first = numpy.zeros(h, dtype=numpy.int64), numpy.full(h, -1, dtype=numpy.int64)
    if err is None:
        try:
            votes, first = vote_first(read_hap_mat, wts, lo)
        except Exception as exc:
            err = exc
    votes, first = _collective(err, lambda ok: sharding.merge_votes(votes, first,
                                                                    ctx.allreduce_host, ok))
    return sharding.contrib_order(votes, first, args.min_reads)


def read_votes(read_hap_mat):
    """``numpy.argmax(read_hap_mat, 1)`` of stats.report_read_votes (stats.py:39)."""
    with OnDevice(read_hap_mat) as dev:
        return dev.argmax_rows()


def assign_rows(read_hap_mat, props, con_indexes, min_fold):
    """int32 per row: position in ``con_indexes`` of the contributor the row is
    assigned to, or -1 (unassigned)."""
    cols = numpy.ascontiguousarray(con_indexes, dtype=numpy.int64)
    log_props = numpy.log(numpy.asarray(props, dtype=numpy.float64))   # assemble.py:300
    con_ln = numpy.ascontiguousarray(log_props[cols])
    with OnDevice(read_hap_mat) as dev:
        out = numpy.empty(dev.shape[0], dtype=numpy.int32)
        check(lib.mxb_assign_reads(dev.ctx.handle, dev.handle, ptr(cols), ptr(con_ln), len(cols),
                                   float(numpy.log(min_fold)), ptr(out)))
    return out


def assign_read_indexes(contribs, em_results, haps, reads, min_fold, sharded=False):
    """
    Maps contributor names to the set of row indexes assigned to them, plus
    ``'unassigned'`` (reference assemble.py:267-334): a row goes to the
    contributor with the highest ``read_mix - log(props)`` if it leads the next
    contributor by at least ``log(min_fold)``.  On a row shard ``reads`` are this
    rank's rows and the sets hold global row indexes ``lo + i``.
    """
    props, read_hap_mat = em_results
    mark, ctx = _shard_mark(read_hap_mat, sharded)
    assigned, err = None, None
    try:
        if len(contribs) > 1:
            cols = [haps.index(group) for _, group, _ in contribs]
            assigned = assign_rows(read_hap_mat, props, cols, min_fold)[:len(reads)]
    except Exception as exc:
        if mark is None:
            raise
        err = exc
    lo = 0
    if mark is not None:
        lo, _ = _offsets(mark, read_hap_mat.shape[0], ctx, err)
        if err is not None:
            raise err
    contrib_reads = collections.defaultdict(set)
    if assigned is not None:
        for k, (name, _, _) in enumerate(contribs):
            rows = numpy.nonzero(assigned == k)[0]
            if len(rows):
                contrib_reads[name].update((rows + lo).tolist())
        rows = numpy.nonzero(assigned < 0)[0]
        if len(rows):
            contrib_reads['unassigned'].update((rows + lo).tolist())
    else:
        contrib_reads[contribs[0][0]].update(range(lo, lo + len(reads)))
    return contrib_reads


# ---- .npy streaming (N4) -------------------------------------------------------
_CHUNK_BYTES = 256 << 20


def _write_rows(dev, handle):
    """``dev``'s rows, downloaded in chunks of ``_CHUNK_BYTES``, at ``handle``'s position."""
    n, h = dev.shape
    rows_per = max(1, _CHUNK_BYTES // max(8 * h, 1))
    buf = numpy.empty((min(rows_per, max(n, 1)), h), dtype=numpy.float64)
    for r0 in range(0, n, rows_per):
        k = min(rows_per, n - r0)
        check(lib.mxb_matrix_download_rows(dev.ctx.handle, dev.handle, r0, k, ptr(buf)))
        buf[:k].tofile(handle)


def save_npy(mat, path, sharded=False):
    """``numpy.save(path, mat)`` for a matrix that lives in HBM: the file is
    written in row chunks, so no N x H host copy is needed (bin/mixemt:240-242
    saves the EM input and result matrices this way).

    On a row shard every rank passes the same path on one node's filesystem and
    the file holds the whole matrix: rank 0 writes the header and sizes the file,
    then each rank writes its rows at their offset (two barriers)."""
    with OnDevice(mat) as dev:
        n, h = dev.shape
        if not str(path).endswith(".npy"):
            path = str(path) + ".npy"          # numpy.save appends the suffix
        mark, ctx = _shard_mark(dev, sharded)
        if mark is None:
            header, _ = sharding.npy_layout(n, h)
            with open(path, "wb") as handle:
                handle.write(header)
                _write_rows(dev, handle)
            return path
        lo, n_total = _offsets(mark, n, ctx)
        header, offset = sharding.npy_layout(n_total, h, lo)
        err = None
        if ctx.rank == 0:
            try:
                with open(path, "wb") as handle:
                    handle.write(header)
                    handle.truncate(len(header) + n_total * h * 8)
            except Exception as exc:
                err = exc
        _collective(err, lambda ok: sharding.barrier(ctx.allreduce_host, ok))
        try:
            with open(path, "r+b") as handle:
                handle.seek(offset)
                _write_rows(dev, handle)
        except Exception as exc:
            err = exc
        _collective(err, lambda ok: sharding.barrier(ctx.allreduce_host, ok))
    return path


def load_npy(path, ctx=None, sharded=False):
    """``numpy.load(path)`` straight into HBM (bin/mixemt:199-203): returns a
    ``DeviceMatrix``; the file is read in row chunks.  With ``sharded=True`` and
    more than one rank, each rank loads its rows ``sharding.row_shard(n, rank,
    world)`` and the result is marked as a row shard."""
    from numpy.lib import format as npy_format
    ctx = ctx or get_context()
    with open(path, "rb") as handle:
        version = npy_format.read_magic(handle)
        if version == (1, 0):
            shape, fortran, dtype = npy_format.read_array_header_1_0(handle)
        else:
            shape, fortran, dtype = npy_format.read_array_header_2_0(handle)
        if len(shape) != 2 or fortran or dtype != numpy.dtype("<f8"):
            raise ValueError("%s: expected a C-ordered 2-d float64 array, found %s %s%s"
                             % (path, shape, dtype, " (Fortran order)" if fortran else ""))
        n_total, h = shape
        lo, hi = 0, n_total
        shard = sharded and ctx.world > 1
        if shard:
            lo, hi = sharding.row_shard(n_total, ctx.rank, ctx.world)
            handle.seek(lo * h * 8, 1)
        n = hi - lo
        dev = DeviceMatrix.empty(ctx, n, h)
        rows_per = max(1, _CHUNK_BYTES // max(8 * h, 1))
        for r0 in range(0, n, rows_per):
            k = min(rows_per, n - r0)
            buf = numpy.fromfile(handle, dtype=numpy.float64, count=k * h)
            if buf.size != k * h:
                dev.free()
                raise ValueError("%s: truncated file" % path)
            check(lib.mxb_matrix_upload_rows(ctx.handle, dev.handle, r0, k, ptr(buf)))
    if shard:
        dev.row_shard = RowShard(lo, n_total)
    return dev
