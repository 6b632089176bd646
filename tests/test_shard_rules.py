"""Host rules of the rows-mode consumers (mixemt_b200.sharding) over world-size-2 and -3
gloo groups on the CPU: each rank's votes and first rows are computed in numpy, as
mxb_matrix_vote_first computes them on its GPU, and merged with the sharding rules; the
merged contributor lists must equal the reference's on the whole matrix."""
import io
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mixemt_b200 import sharding
from oracle import oracle_np
from conftest import load_golden


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gloo_allreduce(arr, op):
    t = torch.from_numpy(arr)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return arr


def local_votes(shard, wts, lo):
    """What mxb_matrix_vote_first returns for a shard starting at global row lo."""
    h = shard.shape[1]
    votes = np.zeros(h, dtype=np.int64)
    first = np.full(h, -1, dtype=np.int64)
    if len(shard):
        best = np.argmax(shard, 1)
        np.add.at(votes, best, np.asarray(wts, dtype=np.int64))
        seen, idx = np.unique(best, return_index=True)
        first[seen] = idx + lo
    return votes, first


def voting(cols, h, wts):
    """A matrix whose row r has its first maximum in column cols[r]."""
    mat = np.full((len(cols), h), -1.0)
    mat[np.arange(len(cols)), cols] = 0.0
    return mat, np.asarray(wts, dtype=np.int64)


def cases():
    """(name, matrix, weights, {world: shard bounds}, min_reads values)."""
    out = []
    for seed in (71, 72):
        _, mix, wts = oracle_np.synthetic_em_result(seed)
        n = len(mix)
        out.append(("s%d" % seed, mix, wts,
                    {2: [sharding.row_shard(n, r, 2) for r in range(2)],
                     3: [(0, 17), (17, 17), (17, n)]}, (1, 60, 400)))
    # column 3 first appears on rank 1, whose local order (3, 5, 2, 1) is not the global one
    mat, w = voting([5, 2, 3, 5, 2, 1], 7, [1, 1, 1, 1, 1, 1])
    out.append(("order", mat, w, {2: [(0, 2), (2, 6)], 3: [(0, 1), (1, 3), (3, 6)]}, (0, 1, 2)))
    # column 4 reaches 50 only in the sum over the ranks
    mat, w = voting([4, 0, 4, 1], 6, [30, 60, 30, 70])
    out.append(("sum", mat, w, {2: [(0, 2), (2, 4)], 3: [(0, 1), (1, 2), (2, 4)]}, (50, 61)))
    # rows of weight 0: their columns appear with 0 votes and count at min_reads = 0
    mat, w = voting([2, 0, 3, 2, 1], 5, [0, 4, 0, 3, 0])
    out.append(("zero", mat, w, {2: [(0, 3), (3, 5)], 3: [(0, 1), (1, 1), (1, 5)]}, (0, 1, 4)))
    # empty shards and uneven hand-made boundaries
    rs = np.random.RandomState(3)
    mat = -rs.gamma(2.0, 3.0, size=(10, 9))
    mat[rs.rand(10, 9) < 0.3] = 0.0
    w = rs.randint(0, 20, size=10)
    out.append(("uneven", mat, w, {2: [(0, 0), (0, 10)], 3: [(0, 1), (1, 9), (9, 10)]},
                (0, 5, 20)))
    return out


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = {}
        for name, mat, wts, bounds, min_reads in cases():
            lo, hi = bounds[world][rank]
            got_lo, n_total = sharding.shard_offsets(hi - lo, rank, world, gloo_allreduce)
            votes, first = local_votes(mat[lo:hi], wts[lo:hi], got_lo)
            votes, first = sharding.merge_votes(votes, first, gloo_allreduce)
            res[name] = (got_lo, n_total, [sharding.contrib_order(votes, first, m)
                                           for m in min_reads])
        res["agree_same"] = sharding.agree([4, 9, 2], gloo_allreduce)
        res["agree_value"] = sharding.agree([4, 9, 2 + (rank == world - 1)], gloo_allreduce)
        res["agree_length"] = sharding.agree(list(range(3 + (rank == 1))), gloo_allreduce)
        res["agree_empty"] = sharding.agree([], gloo_allreduce)
        try:      # one rank's failure reaches every rank through the ok flag
            sharding.shard_offsets(5, rank, world, gloo_allreduce, ok=rank != 1)
            res["flag"] = "no error"
        except sharding.RankFailed:
            res["flag"] = "raised"
        try:
            sharding.agree([1], gloo_allreduce, ok=rank != world - 1)
            res["flag_agree"] = "no error"
        except sharding.RankFailed:
            res["flag_agree"] = "raised"
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module", params=[2, 3])
def world_results(request):
    world = request.param
    mgr = mp.get_context("spawn").Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, free_port(), out), nprocs=world, join=True)
    res = dict(out)
    mgr.shutdown()
    return world, res


def test_merged_votes_give_the_reference_contributors(world_results):
    world, res = world_results
    g = load_golden("golden_consumers.npz")
    for name, mat, wts, bounds, min_reads in cases():
        want = [oracle_np.find_contribs_from_reads(mat, wts, m) for m in min_reads]
        if name in ("s71", "s72"):
            assert want == [g["%s_contribs_r%d" % (name, m)].tolist() for m in min_reads]
        for rank in range(world):
            lo, n_total, got = res[rank][name]
            assert (lo, n_total) == (bounds[world][rank][0], len(mat))
            assert got == want, (name, rank)


def test_handmade_cases_cover_their_edges():
    by_name = {c[0]: c for c in cases()}
    _, mat, w, _, _ = by_name["order"]
    assert oracle_np.find_contribs_from_reads(mat, w, 0) == [5, 2, 3, 1]
    _, mat, w, _, _ = by_name["sum"]
    assert oracle_np.find_contribs_from_reads(mat, w, 50) == [4, 0, 1]
    _, mat, w, _, _ = by_name["zero"]
    assert oracle_np.find_contribs_from_reads(mat, w, 0) == [2, 0, 3, 1]


def test_agree_and_failure_flags_reach_every_rank(world_results):
    world, res = world_results
    for rank in range(world):
        r = res[rank]
        assert r["agree_same"] is True and r["agree_empty"] is True
        assert r["agree_value"] is False and r["agree_length"] is False
        assert r["flag"] == "raised" and r["flag_agree"] == "raised"


def test_single_rank_order_matches_reference():
    _, mix, wts = oracle_np.synthetic_em_result(71)
    votes, first = local_votes(mix, wts, 0)
    for m in (0, 1, 60, 400):
        assert sharding.contrib_order(votes, first, m) == \
            oracle_np.find_contribs_from_reads(mix, wts, m)


@pytest.mark.parametrize("bounds", [[(0, 1237)], [(0, 600), (600, 1237)],
                                    [(0, 0), (0, 411), (411, 411), (411, 1237)]])
def test_npy_layout_shards_give_numpy_save_bytes(tmp_path, bounds):
    rs = np.random.RandomState(4)
    mat = rs.randn(1237, 61)
    mat[3, 5] = -np.inf
    ref = io.BytesIO()
    np.save(ref, mat)
    n, h = mat.shape
    path = str(tmp_path / "shards.npy")
    header, _ = sharding.npy_layout(n, h)
    with open(path, "wb") as f:          # rank 0
        f.write(header)
        f.truncate(len(header) + n * h * 8)
    for lo, hi in reversed(bounds):      # the ranks, in any order
        head, offset = sharding.npy_layout(n, h, lo)
        assert head == header and offset == len(header) + lo * h * 8
        with open(path, "r+b") as f:
            f.seek(offset)
            mat[lo:hi].tofile(f)
    assert open(path, "rb").read() == ref.getvalue()
