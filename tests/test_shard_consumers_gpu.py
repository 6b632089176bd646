"""Rows-mode consumers on one B200: 2 and 3 processes share device 0, each holding a
row shard, and talk through a gloo group that replaces their context's
``allreduce_host`` (the consumers' collectives are host-side only; NCCL cannot put two
ranks on one GPU).  The results must be those of the whole matrix: the reference's
outputs in tests/golden/golden_consumers.npz, the CPU oracle, the one-process run."""
import hashlib
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mixemt_b200 import consumers, sharding
from oracle import oracle_np
from conftest import load_golden, make_args
from shard_pipeline_check import build17_fragments

pytestmark = pytest.mark.gpu

SEEDS = (71, 72)
MIN_READS = (1, 60, 400)


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gloo_allreduce(arr, op="sum"):
    t = torch.from_numpy(arr)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return arr


def digest(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


def decode_assign(res, n):
    out = np.full(n, -2, dtype=np.int32)
    for name, rows in res.items():
        out[sorted(rows)] = -1 if name == 'unassigned' else int(name[3:]) - 1
    return out


def _synthetic(rank, world, ctx, tmp):
    from mixemt_b200.runtime import DeviceMatrix, RowShard
    g = load_golden("golden_consumers.npz")
    res = {}
    for seed in SEEDS:
        props, mix, wts = oracle_np.synthetic_em_result(seed)
        haps = ["hg%d" % j for j in range(mix.shape[1])]
        lo, hi = sharding.row_shard(len(mix), rank, world)
        dev = DeviceMatrix.from_host(ctx, mix[lo:hi])
        dev.row_shard = RowShard()
        r = {"lo": lo, "hi": hi}
        r["contribs"] = [consumers.find_contribs_from_reads(dev, wts[lo:hi],
                                                            make_args(min_reads=m))
                         for m in MIN_READS]
        r["offsets"] = (dev.row_shard.lo, dev.row_shard.n_total)
        r["contribs_host"] = consumers.find_contribs_from_reads(
            mix[lo:hi], wts[lo:hi], make_args(min_reads=60), sharded=True)
        top = g["s%d_top" % seed].tolist()
        contribs = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(top)]
        r["assign"] = {}
        for tag, fold, cons in (("f2", 2.0, contribs), ("f1p2", 1.2, contribs[:2]),
                                ("single", 2.0, contribs[:1])):
            got = consumers.assign_read_indexes(cons, (props, dev), haps,
                                                list(range(hi - lo)), fold)
            r["assign"][tag] = {k: sorted(v) for k, v in got.items()}
        red, new_haps = consumers.reduce_em_matrix(dev, haps, contribs)
        r["reduced"] = red.to_host()
        r["reduced_marked"] = red.row_shard is dev.row_shard
        r["new_haps"] = new_haps
        red_host, _ = consumers.reduce_em_matrix(mix[lo:hi], haps, contribs, sharded=True)
        r["reduced_host"] = red_host
        consumers._CHUNK_BYTES = 8 * mix.shape[1] * 7      # 7-row chunks: ragged writes
        path = consumers.save_npy(dev, os.path.join(tmp, "s%d" % seed))
        back = consumers.load_npy(path, sharded=True)
        r["loaded"] = back.to_host()
        r["loaded_offsets"] = (back.row_shard.lo, back.row_shard.n_total)
        r["path"] = path
        res[seed] = r
    return res


def _errors(rank, world, ctx, tmp):
    from mixemt_b200.runtime import DeviceMatrix, RowShard
    _, mix, wts = oracle_np.synthetic_em_result(71)
    haps = ["hg%d" % j for j in range(mix.shape[1])]
    lo, hi = sharding.row_shard(len(mix), rank, world)
    dev = DeviceMatrix.from_host(ctx, mix[lo:hi])
    dev.row_shard = RowShard()
    out = {}
    # contributor lists that differ between the ranks
    mine = [["hap1", haps[3], 0.5], ["hap2", haps[10 + rank], 0.5]]
    try:
        consumers.reduce_em_matrix(dev, haps, mine)
        out["reduce"] = "returned"
    except ValueError as exc:
        out["reduce"] = type(exc).__name__
    # a weights vector of the wrong length on the last rank only, before and after the
    # offsets are known (the ok flag rides on shard_offsets, then on the vote merge)
    for when in ("offsets", "merge"):
        if when == "merge":
            consumers.find_contribs_from_reads(dev, wts[lo:hi], make_args(min_reads=1))
        w = wts[lo:hi] if rank != world - 1 else wts[lo:hi - 1]
        fresh = DeviceMatrix.from_host(ctx, mix[lo:hi]) if when == "offsets" else dev
        if when == "offsets":
            fresh.row_shard = RowShard()
        try:
            consumers.find_contribs_from_reads(fresh, w, make_args(min_reads=1))
            out[when] = "returned"
        except sharding.RankFailed:
            out[when] = "RankFailed"
        except ValueError:
            out[when] = "ValueError"
    # the ranks are still in step afterwards
    out["after"] = consumers.find_contribs_from_reads(dev, wts[lo:hi], make_args(min_reads=60))
    return out


def _build17(rank, world, ctx, tmp):
    from mixemt_b200.preprocess import build_em_input_arrays
    phylo, frag_ptr, pos, base = build17_fragments()
    args = make_args(b200_shard="rows")
    dmat, w, haps, red = build_em_input_arrays(frag_ptr, pos, base, phylo.refseq, phylo, args,
                                               keep_device=True)
    host, w_host, _, _ = build_em_input_arrays(frag_ptr, pos, base, phylo.refseq, phylo, args)
    r = {"offsets": (dmat.row_shard.lo, dmat.row_shard.n_total), "n_rows": red.n_rows,
         "shape": dmat.shape, "digest": digest(dmat.to_host()), "digest_host": digest(host),
         "weights": np.asarray(w), "weights_host": np.asarray(w_host)}
    r["contribs"] = consumers.find_contribs_from_reads(dmat, w, make_args(min_reads=10))
    props = np.full(len(haps), 1.0 / len(haps))
    cons = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(r["contribs"][:3])]
    got = consumers.assign_read_indexes(cons, (props, dmat), haps, list(range(dmat.shape[0])),
                                        1.5)
    r["assign"] = {k: sorted(v) for k, v in got.items()}
    return r


JOBS = {"synthetic": _synthetic, "errors": _errors, "build17": _build17}


def _worker(rank, world, port, job, tmp, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), MIXEMT_B200_DEVICE="0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from mixemt_b200.runtime import get_context
        ctx = get_context()
        ctx.rank, ctx.world = rank, world
        ctx.allreduce_host = gloo_allreduce
        out[rank] = JOBS[job](rank, world, ctx, tmp)
    finally:
        dist.destroy_process_group()


def run_ranks(job, world, tmp, timeout=300):
    """Runs ``job`` on ``world`` processes; every process must exit, with status 0, in time."""
    spawn = mp.get_context("spawn")
    mgr = spawn.Manager()
    out = mgr.dict()
    port = free_port()
    procs = [spawn.Process(target=_worker, args=(r, world, port, job, str(tmp), out))
             for r in range(world)]
    for p in procs:
        p.start()
    deadline = time.time() + timeout
    for p in procs:
        p.join(max(1.0, deadline - time.time()))
    late = [p for p in procs if p.is_alive()]
    for p in late:
        p.kill()
        p.join()
    assert not late, "%d rank(s) still running after %d s" % (len(late), timeout)
    assert [p.exitcode for p in procs] == [0] * world
    res = dict(out)
    mgr.shutdown()
    return res


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_consumers_match_reference(world, tmp_path):
    res = run_ranks("synthetic", world, tmp_path)
    g = load_golden("golden_consumers.npz")
    for seed in SEEDS:
        props, mix, wts = oracle_np.synthetic_em_result(seed)
        haps = ["hg%d" % j for j in range(mix.shape[1])]
        want = [g["s%d_contribs_r%d" % (seed, m)].tolist() for m in MIN_READS]
        assert want == [oracle_np.find_contribs_from_reads(mix, wts, m) for m in MIN_READS]
        ref = tmp_path / "ref.npy"
        np.save(str(ref), mix)
        cols = g["s%d_reduced_cols" % seed].tolist()
        for rank in range(world):
            r = res[rank][seed]
            lo, hi = r["lo"], r["hi"]
            assert r["contribs"] == want, (seed, rank)
            assert r["contribs_host"] == want[1]
            assert r["offsets"] == (lo, len(mix)) == r["loaded_offsets"]
            assert [haps.index(x) for x in r["new_haps"]] == cols
            assert r["reduced_marked"]
            assert np.array_equal(r["reduced"], g["s%d_reduced" % seed][lo:hi])
            assert np.array_equal(r["reduced_host"], g["s%d_reduced" % seed][lo:hi])
            assert np.array_equal(r["loaded"], mix[lo:hi])
        for tag in ("f2", "f1p2", "single"):
            union = {}
            for rank in range(world):
                for name, rows in res[rank][seed]["assign"][tag].items():
                    assert not set(rows) & set(union.get(name, ()))
                    union.setdefault(name, []).extend(rows)
            assert np.array_equal(decode_assign(union, len(mix)), g["s%d_assign_%s" % (seed, tag)])
        path = res[0][seed]["path"]
        assert open(path, "rb").read() == open(str(ref), "rb").read()   # byte-identical


def test_failures_reach_every_rank(tmp_path):
    world = 3
    res = run_ranks("errors", world, tmp_path, timeout=240)
    _, mix, wts = oracle_np.synthetic_em_result(71)
    for rank in range(world):
        r = res[rank]
        assert r["reduce"] == "ValueError"
        want = "ValueError" if rank == world - 1 else "RankFailed"
        assert r["offsets"] == want and r["merge"] == want, (rank, r)
        assert r["after"] == oracle_np.find_contribs_from_reads(mix, wts, 60)


def test_sharded_build_matches_one_process_build(tmp_path):
    from mixemt_b200.preprocess import build_em_input_arrays
    world = 2
    res = run_ranks("build17", world, tmp_path)
    phylo, frag_ptr, pos, base = build17_fragments()
    full, w, haps, red = build_em_input_arrays(frag_ptr, pos, base, phylo.refseq, phylo)
    n = red.n_rows
    want = oracle_np.find_contribs_from_reads(full, w, 10)
    assert len(want) >= 2
    props = np.full(len(haps), 1.0 / len(haps))
    cons = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(want[:3])]
    assign = consumers.assign_read_indexes(cons, (props, full), haps, list(range(n)), 1.5)
    union = {}
    for rank in range(world):
        r = res[rank]
        lo, hi = sharding.row_shard(n, rank, world)
        assert r["offsets"] == (lo, n) and r["n_rows"] == n and r["shape"] == (hi - lo, len(haps))
        assert r["digest"] == digest(full[lo:hi]) == r["digest_host"]     # bit for bit
        assert np.array_equal(r["weights"], w[lo:hi]) and np.array_equal(r["weights_host"], w[lo:hi])
        assert r["contribs"] == want
        for name, rows in r["assign"].items():
            union.setdefault(name, set()).update(rows)
    assert union == {k: set(v) for k, v in assign.items()}


def test_vote_first_at_build17_width():
    rs = np.random.RandomState(6)
    n, h = 4099, 5408
    mix = -rs.gamma(2.0, 5.0, size=(n, h))
    mix[rs.rand(n, h) < 0.2] = 0.0
    mix[0] = -np.inf                      # all -inf: argmax 0
    mix[1] = 0.0                          # all equal: argmax 0
    mix[2, -1] = 1.0                      # maximum in the last column
    mix[3, 100] = mix[3, 200] = np.nan    # NaN wins, the first one
    mix[4000:, 17] = 5.0                  # a column first reached late
    wts = rs.randint(0, 1000, size=n).astype(np.int64)
    best = np.argmax(mix, 1)
    assert best[0] == 0 and best[1] == 0 and best[2] == h - 1 and best[3] == 100
    seen, idx = np.unique(best, return_index=True)
    for row0 in (0, 1, 10_000_019):
        votes, first = consumers.vote_first(mix, wts, row0)
        want_first = np.full(h, -1, dtype=np.int64)
        want_first[seen] = idx + row0
        assert np.array_equal(first, want_first)
        assert np.array_equal(votes, np.bincount(best, weights=wts, minlength=h).astype(np.int64))
    votes, first = consumers.vote_first(mix[:0], wts[:0], 5)
    assert not votes.any() and (first == -1).all()
