"""Host-side rules of the multi-GPU modes (SURVEY.md 8e).  Pure numpy; the
collectives are passed in as callables so that the same code runs over NCCL
(``Context.allreduce_host`` / device kernels) and, in the CPU tests, over a
world_size-2 gloo group.

* rows mode:     signature rows are split into contiguous balanced shards; each
                 EM iteration all-reduces the H partial column sums T_j.
* restarts mode: the matrix is replicated, the restarts are dealt in contiguous
                 blocks, and the per-rank results are combined as the reference
                 combines restarts (em.py:145-163): log-proportions are summed
                 and divided by n_multi, read matrices are folded with
                 logaddexp and shifted by -log(n_multi).
* rows-mode consumers: each rank knows only its shard of the read matrix, so the
                 votes of find_contribs_from_reads, the kept columns of
                 reduce_em_matrix, global row indexes and .npy files are formed from
                 O(H) all-reduces and the shards' offsets.

The fp64 all-reduces carry integers exactly while they stay below 2**53.  A
collective that may be the first one of a call carries an ``ok`` flag as an extra
element: when any rank passes ``ok=False`` every rank raises ``RankFailed``, so no
rank is left waiting in a later collective.
"""
import io

import numpy as np
from numpy.lib import format as npy_format

_EXACT = 2.0 ** 53


class RankFailed(ValueError):
    """A rank could not take part in a row-sharded call (raised on every rank)."""


def _fail_flag(ok):
    return 0.0 if ok else 1.0


def _raise_if_failed(flag):
    if flag:
        raise RankFailed("a rank failed in a row-sharded call; see that rank's error")


def row_shard(n_rows, rank, world):
    """Contiguous balanced row range [lo, hi) of ``rank``."""
    return (n_rows * rank) // world, (n_rows * (rank + 1)) // world


def restart_shard(n_multi, rank, world):
    """Indices of the restarts ``rank`` runs: contiguous balanced blocks, so that folding the
    ranks' partial results in rank order adds the restarts in restart order (em.py:155-156)."""
    return list(range((n_multi * rank) // world, (n_multi * (rank + 1)) // world))


def combine_restart_props(local_sum_lnprops, n_multi, allreduce):
    """em.py:155 + :158-163 across ranks: ``allreduce(arr, "sum")`` in place."""
    total = allreduce(np.ascontiguousarray(local_sum_lnprops, dtype=np.float64), "sum")
    if n_multi > 1:
        total = total / n_multi
    return np.exp(total)


def fold_read_mix(local_mix, n_multi, allreduce):
    """log(sum over ranks of exp(local_mix)) - log(n_multi), computed as
    max-shift + sum so that it needs only max/sum all-reduces; ``local_mix`` is
    this rank's logaddexp fold of its restarts (all -inf when it ran none).  A
    collective-only statement of what ``mxb_matrix_fold_ranks`` computes on the
    GPUs (there: all-to-all of row shards + logaddexp in rank order), used by
    the gloo tests."""
    mx = allreduce(np.array(local_mix, dtype=np.float64, copy=True), "max")
    with np.errstate(invalid="ignore"):
        lin = np.where(np.isinf(mx), np.where(mx < 0, 0.0, 1.0), np.exp(local_mix - mx))
    lin = allreduce(np.ascontiguousarray(lin), "sum")
    with np.errstate(divide="ignore"):
        out = np.where(np.isinf(mx), mx, mx + np.log(lin))
    return out - (np.log(n_multi) if n_multi > 1 else 0.0)


def share_from_rank0(make, shape, rank, allreduce):
    """Rank 0 evaluates ``make()`` (e.g. the Dirichlet draws of em.py:36 from its global
    numpy.random stream); every rank returns that array.  Shared as a sum all-reduce of
    zeros on the other ranks -- ``-inf`` entries (a zero proportion) survive a sum, a NaN
    would not and is rejected."""
    if rank == 0:
        arr = np.ascontiguousarray(make(), dtype=np.float64).reshape(shape)
        if np.isnan(arr).any():
            raise ValueError("initial log-proportions hold NaN")
    else:
        arr = np.zeros(shape, dtype=np.float64)
    return allreduce(arr, "sum")


def shard_offsets(n_local, rank, world, allreduce, ok=True):
    """``(lo, n_total)`` of this rank's ``n_local`` rows, the shards laid end to end in
    rank order: one sum all-reduce of the ``world`` shard sizes (arbitrary or empty
    boundaries work) plus the ok flag."""
    vec = np.zeros(world + 1)
    vec[rank] = n_local
    vec[world] = _fail_flag(ok)
    vec = allreduce(vec, "sum")
    _raise_if_failed(vec[world])
    n_total = vec[:world].sum()
    assert n_total < _EXACT, "row count not exact in fp64"
    return int(vec[:rank].sum()), int(n_total)


def merge_votes(votes, first, allreduce, ok=True):
    """The ranks' ``(votes[H], first[H])`` of ``mxb_matrix_vote_first`` merged into
    those of the whole matrix: votes summed, first rows (-1 = absent) reduced to
    their minimum as the maximum of their negations."""
    h = len(votes)
    vec = np.empty(h + 1)
    vec[:h] = votes
    vec[h] = _fail_flag(ok)
    vec = allreduce(vec, "sum")
    _raise_if_failed(vec[h])
    assert vec[:h].sum() < _EXACT, "total weight not exact in fp64"
    first = np.asarray(first)
    neg = np.ascontiguousarray(np.where(first >= 0, -first.astype(np.float64), -np.inf))
    neg = allreduce(neg, "max")
    with np.errstate(invalid="ignore"):
        merged = np.where(np.isfinite(neg), -neg, -1.0)
    return vec[:h].astype(np.int64), merged.astype(np.int64)


def contrib_order(votes, first, min_reads):
    """Column indexes of ``_find_contribs_from_reads`` (assemble.py:102-124): every column
    that some row votes for (also with 0 votes, from rows of weight 0), ordered by its
    first row like the reference's dict, then those with ``votes >= min_reads``."""
    first = np.asarray(first)
    seen = np.nonzero(first >= 0)[0]
    order = seen[np.argsort(first[seen], kind="stable")]
    return [int(j) for j in order if votes[j] >= min_reads]


def agree(vector, allreduce, ok=True):
    """True on every rank when all ranks hold the same integer vector: the lengths, then
    the elements, compared as max == min (max all-reduces of ``v`` and ``-v``)."""
    vec = np.asarray(vector, dtype=np.float64).reshape(-1)
    assert vec.size == 0 or np.abs(vec).max() < _EXACT, "values not exact in fp64"
    n = float(vec.size)
    head = allreduce(np.array([_fail_flag(ok), n, -n]), "max")
    _raise_if_failed(head[0])
    if head[1] != -head[2]:
        return False
    both = allreduce(np.concatenate([vec, -vec]), "max")
    return bool(np.array_equal(both[:vec.size], -both[vec.size:]))


def barrier(allreduce, ok=True):
    """All-reduce of one flag: returns once every rank got here, raises ``RankFailed``
    on every rank when one of them passes ``ok=False``."""
    _raise_if_failed(allreduce(np.array([_fail_flag(ok)]), "sum")[0])


def npy_layout(n_total, h, lo=0):
    """``(header, offset)``: the bytes ``numpy.save`` writes before the data of a C-ordered
    float64 ``(n_total, h)`` array, and the file offset of row ``lo``."""
    buf = io.BytesIO()
    npy_format.write_array_header_1_0(buf, {"descr": "<f8", "fortran_order": False,
                                            "shape": (int(n_total), int(h))})
    header = buf.getvalue()
    return header, len(header) + int(lo) * int(h) * 8


def merge_bootstrap(lnprops, iters, conv, boot0, n_boot, allreduce):
    """Bootstrap fan-out: this rank's replicates ``boot0 .. boot0 + len(lnprops) - 1`` (its
    ``restart_shard`` block) placed into zero rows of the ``(n_boot, H)`` log-proportions and
    the iteration counts and converged flags behind them, then one sum all-reduce.  Adding
    zeros is exact (``-inf`` survives), so every rank gets what one rank running all
    replicates computes."""
    lnprops = np.asarray(lnprops, dtype=np.float64)   # (replicates of this rank, H)
    h = lnprops.shape[1]
    buf = np.zeros((n_boot, h + 2))
    k = len(iters)
    buf[boot0:boot0 + k, :h] = lnprops
    buf[boot0:boot0 + k, h] = iters
    buf[boot0:boot0 + k, h + 1] = conv
    assert np.abs(buf[:, h]).max(initial=0) < _EXACT, "iteration counts not exact in fp64"
    buf = allreduce(np.ascontiguousarray(buf), "sum")
    return buf[:, :h], buf[:, h].astype(np.int64), buf[:, h + 1].astype(np.int32)
