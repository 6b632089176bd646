"""Row- and restart-sharded EM at any world size up to 8, against long double; launched by
torchrun (see test_multirank_gpu.py):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W \\
        --master-addr 127.0.0.1 --master-port P tests/multirank_check.py REFS.npz

REFS.npz is written once, before the launch, by write_references(W, path): the matrices, the
starts and the long-double references (tile_cases.ld_iterate / ld_read_mix) of every case, so
that the ranks do no reference work of their own.  The exchange is the one the context picks:
peer stores inside the EM tail, or NCCL under MXB_NO_P2P=1.

Row cases: every rank runs a sharded session on its row_shard, k = 1 and 3 iterations (and 6
with a dying column) without a convergence test; the proportions must match the reference in
log space (rank_cases.assert_ln_close, 1e-12), the rank's rows of the read matrix within
1e-11, and every rank must hold the same bits.  The layout flags of mxb_em_pass_bytes (0: class
tiles, -1: fp64 rows or the general path) are gathered and must be the ones the case intends.
The widths put the session on the general path with the split tail (H = 3, 130, 1000 and 9000,
which is wider than the fused tail), and on fp64 rows at NC = 1, 2, 3, 5, 7 and 8 column chunks
and on class tiles (H = 1024, 1040, 2049, 4097, 6145, 8192), with the peer tail or the split
tail.  No world size of 2, 4 or 8 divides the 301 rows.  Further cases: fewer rows than ranks,
a rank whose weights are all 0, tiles on the first half of the ranks and fp64 rows on the rest,
and rows that underflow in linear space on the last rank only, then on a middle rank only
(logspace_shards_check.underflowing_case), followed by run_em from that start and from one
that never underflows, with the C oracle's iteration counts.

Restart cases: run_em_device(b200_shard="restarts") with n_multi = 1, W - 1, W and W + 3 on a
narrow and a wide matrix, and on one with fewer rows than ranks (empty fold ranges): the
proportions are exp(mean_i traj_i[k]), the read matrix logaddexp_i(ld_read_mix(traj_i[k-1]))
- log(n_multi).
"""
import functools
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from logspace_shards_check import underflowing_case  # noqa: E402
from rank_cases import start_lnprops  # noqa: E402
from tile_cases import class_matrix, ld_iterate, ld_read_mix  # noqa: E402
from test_tile_plan import ROWS  # noqa: E402

N_ROWS = 301
GENERAL_WIDTHS = (3, 130, 1000, 9000)
STREAM_WIDTHS = (1024, 1040, 2049, 4097, 6145, 8192)   # NC = 1, 2 (ragged), 3, 5, 7, 8
RESTART_K = 3


def row_shard(n, rank, world):
    return (n * rank) // world, (n * (rank + 1)) // world


def width_matrix(h, n, seed):
    """n x h with 2 .. 40 column classes per batch of 128 rows (so that every shard compresses
    to class tiles); from H = 64 on, a dead column and a dying one."""
    rs = np.random.RandomState(seed)
    big = h >= 64
    ncls = rs.randint(3 if big else 2, min(h, 40) + 1, size=-(-n // ROWS))
    return class_matrix(ncls, h, n, "random", seed, dead=big, dying=big)


def random_matrix(h, n, seed):
    """n x h of distinct values: no class tiles."""
    rs = np.random.RandomState(seed)
    return -rs.gamma(2.0, 3.0, size=(n, h)), rs.randint(1, 50, size=n).astype(np.float64)


@functools.lru_cache(maxsize=None)
def _width_ref(h):
    mat, w, _, j_dying = width_matrix(h, N_ROWS, h)
    lnp = start_lnprops(h, h + 1, j_dying)
    return _row_ref(mat, w, lnp, (1, 3, 6) if j_dying is not None else (1, 3))


def _row_ref(mat, w, lnp, ks):
    traj = ld_iterate(mat, w, lnp, max(ks))
    arrays = {"mat": mat, "w": w, "lnp": lnp, "traj": traj.astype(np.float64)}
    for k in ks:
        arrays["mix%d" % k] = ld_read_mix(mat, traj[k - 1]).astype(np.float64)
    return arrays, list(ks)


@functools.lru_cache(maxsize=None)
def _under_ref(layout, lo, hi, max_iter=60, tol=1e-6):
    from oracle import oracle_c
    mat, w, bad, good = underflowing_case(
        layout, bad_rows=lambda n: slice(lo, min(hi, lo + n // 4)))
    arrays, ks = _row_ref(mat, w, bad[0], (1, 3))
    arrays["good"] = good[0]
    for tag, start in (("bad", bad), ("good", good)):
        o_p, _, o_it = oracle_c.run_em(mat, w, start, max_iter, tol)
        arrays["o_p_" + tag], arrays["o_it_" + tag] = o_p, np.asarray(o_it)
    return arrays, ks, max_iter, tol


@functools.lru_cache(maxsize=None)
def _restart_mat(name, h, n):
    if name == "tiny":
        mat, w = random_matrix(h, n, 17)
        return mat, w, None
    mat, w, _, j_dying = width_matrix(h, n, h + 2)
    return mat, w, j_dying


@functools.lru_cache(maxsize=None)
def _restart_traj(name, h, n, i):
    mat, w, j_dying = _restart_mat(name, h, n)
    lnp = start_lnprops(h, 100 + i, j_dying)
    return lnp, ld_iterate(mat, w, lnp, RESTART_K)


def _restart_ref(name, h, n, n_multis):
    mat, w, _ = _restart_mat(name, h, n)
    k = RESTART_K
    runs = [_restart_traj(name, h, n, i) for i in range(max(n_multis))]
    arrays = {"mat": mat, "w": w, "inits": np.stack([lnp for lnp, _ in runs])}
    for nm in n_multis:
        trajs = [t for _, t in runs[:nm]]
        arrays["props%d" % nm] = (sum(t[k] for t in trajs) / nm).astype(np.float64)
        with np.errstate(divide="ignore"):
            mix = ld_read_mix(mat, trajs[0][k - 1])
            for t in trajs[1:]:
                mix = np.logaddexp(mix, ld_read_mix(mat, t[k - 1]))
            arrays["mix%d" % nm] = (mix - np.log(np.longdouble(nm))).astype(np.float64)
    return arrays


def cases(world):
    """(specs, arrays): the case list for `world` ranks and the arrays behind it, keyed
    "<case index>_<name>"."""
    specs, arrays = [], {}

    def add(spec, arr):
        spec["key"] = "%d_" % len(specs)
        specs.append(spec)
        arrays.update({spec["key"] + k: v for k, v in arr.items()})

    every = lambda flag: [flag] * world   # noqa: E731
    for h in GENERAL_WIDTHS + STREAM_WIDTHS:
        arr, ks = _width_ref(h)
        runs = [{"no_pack": True, "want": every(-1)}]     # fp64 rows, or the general path
        if h in STREAM_WIDTHS:
            runs.insert(0, {"no_pack": False, "want": every(0)})
        add({"kind": "rows", "name": "H%d" % h, "ks": ks, "runs": runs}, arr)

    # fewer rows than ranks: the ranks without rows still take part in every exchange
    n = max(1, world - 3)
    mat, w = random_matrix(1040, n, 11)
    arr, ks = _row_ref(mat, w, start_lnprops(1040, 12), (1, 3))
    add({"kind": "rows", "name": "rows%d" % n, "ks": ks,
         "runs": [{"no_pack": True, "want": every(-1)}]}, arr)

    if world > 1:   # one rank without weight
        mat, w, _, j_dying = width_matrix(2049, N_ROWS, 13)
        lo, hi = row_shard(N_ROWS, world // 2, world)
        w = w.copy()
        w[lo:hi] = 0.0
        arr, ks = _row_ref(mat, w, start_lnprops(2049, 14, j_dying), (1, 3, 6))
        add({"kind": "rows", "name": "zero_weight_rank%d" % (world // 2), "ks": ks,
             "runs": [{"no_pack": False, "want": every(0)}]}, arr)

    # class tiles on the first world // 2 ranks, fp64 rows on the others, under one tail
    split = row_shard(N_ROWS, world // 2, world)[0]
    mat, w = random_matrix(2049, N_ROWS, 15)
    if split:
        mat[:split], w[:split], _, _ = width_matrix(2049, split, 16)
    arr, ks = _row_ref(mat, w, start_lnprops(2049, 17), (1, 3))
    add({"kind": "rows", "name": "mixed", "ks": ks,
         "runs": [{"no_pack": False, "want": [0] * (world // 2) + [-1] * (world - world // 2)}]},
        arr)

    # underflow in linear space on one rank only, the last and then a middle one
    for layout, flag in (("fp64", -1), ("tiles", 0)):
        n = 300 if layout == "fp64" else 1280
        for r in sorted({world - 1, world // 2}, reverse=True):
            lo, hi = row_shard(n, r, world)
            arr, ks, max_iter, tol = _under_ref(layout, lo, hi)
            add({"kind": "rows", "name": "underflow_%s_rank%d" % (layout, r), "ks": ks,
                 "runs": [{"no_pack": False, "want": every(flag)}],
                 "run_em": {"max_iter": max_iter, "tol": tol}}, arr)

    n_multis = sorted({1, max(1, world - 1), world, world + 3})
    for name, h, n, nms in (("narrow", 130, N_ROWS, n_multis), ("wide", 4097, N_ROWS, n_multis),
                            ("tiny", 1040, max(1, world - 1), [1, world + 3])):
        add({"kind": "restarts", "name": "restarts_%s%dx%d" % (name, n, h), "k": RESTART_K,
             "n_multi": nms}, _restart_ref(name, h, n, tuple(nms)))
    return specs, arrays


def write_references(world, path):
    specs, arrays = cases(world)
    np.savez(path, meta=json.dumps({"world": world, "cases": specs}), **arrays)
    return len(specs)


def main():
    import torch
    import torch.distributed as dist
    from conftest import make_args
    from mixemt_b200 import em, sharding
    from mixemt_b200._lib import lib
    from mixemt_b200.runtime import DeviceMatrix, get_context
    from rank_cases import Session, assert_ln_close, assert_mix_close

    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = get_context()
    ctx.init_comm_from_torch()
    refs = np.load(sys.argv[1])
    meta = json.loads(str(refs["meta"]))
    assert meta["world"] == world, (meta["world"], world)

    def gather(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    def same_on_every_rank(arr):
        got = gather(np.asarray(arr).tobytes())
        assert all(g == got[0] for g in got), "ranks disagree"

    lines = []
    for case in meta["cases"]:
        key = case["key"]
        get = lambda name: refs[key + name]   # noqa: E731
        mat, w = get("mat"), get("w")
        n, h = mat.shape
        err_ln = err_mix = 0.0
        if case["kind"] == "rows":
            lo, hi = sharding.row_shard(n, rank, world)
            dev = DeviceMatrix.from_host(ctx, mat[lo:hi])
            w_mine = np.ascontiguousarray(w[lo:hi])
            traj, lnp = get("traj"), get("lnp")
            flags = []
            for run in case["runs"]:
                if run["no_pack"]:
                    os.environ["MXB_EM_NO_PACK"] = "1"
                else:
                    os.environ.pop("MXB_EM_NO_PACK", None)
                s = Session(dev, w_mine, sharded=True)
                try:
                    got = gather(s.pass_bytes()[0])
                    assert got == run["want"], (case["name"], got, run["want"])
                    flags.append(got)
                    for k in case["ks"]:
                        latest, prev, mix = s.iterate(lnp, k)
                        err_ln = max(err_ln, assert_ln_close(latest, traj[k]),
                                     assert_ln_close(prev, traj[k - 1]))
                        err_mix = max(err_mix, assert_mix_close(mix, get("mix%d" % k)[lo:hi]))
                        same_on_every_rank(latest)
                finally:
                    s.close()
            os.environ.pop("MXB_EM_NO_PACK", None)
            if case["name"] == "mixed" and world > 1:
                assert {0, -1} <= set(flags[0]), flags
            what = "flags=%s" % ",".join("".join("T" if f == 0 else "r" for f in fl) for fl in flags)
            if "run_em" in case:
                # run_em from the start that underflows, then from one that never does: the
                # ranks redo the iteration together and their mailboxes stay in step
                a = make_args(max_iter=case["run_em"]["max_iter"], tolerance=case["run_em"]["tol"],
                              n_multi=1, b200_shard="rows")
                for tag, start in (("bad", lnp), ("good", get("good"))):
                    p, _, info, _ = em.run_em_device(dev, w_mine, a, inits=start.reshape(1, h),
                                                     want_host=False)
                    assert info["iterations"] == get("o_it_" + tag).tolist(), \
                        (case["name"], tag, info, get("o_it_" + tag))
                    assert np.abs(p - get("o_p_" + tag)).max() < 1e-9, (case["name"], tag)
                    same_on_every_rank(p)
                    what += " run_em:%s=%s" % (tag, info["iterations"])
            dev.free()
        else:
            k = case["k"]
            dev = DeviceMatrix.from_host(ctx, mat)
            inits = get("inits")
            for nm in case["n_multi"]:
                a = make_args(max_iter=k, tolerance=0.0, n_multi=nm, b200_shard="restarts")
                props, mix, info, _ = em.run_em_device(dev, w, a, inits=inits[:nm])
                mine = sharding.restart_shard(nm, rank, world)
                assert info["restarts"] == mine and info["iterations"] == [k] * len(mine), info
                want = get("props%d" % nm)
                live = want > -700.0
                with np.errstate(divide="ignore"):
                    err_ln = max(err_ln, assert_ln_close(np.log(props[live]), want[live]))
                assert (props[~live] < 1e-300).all(), case["name"]
                err_mix = max(err_mix, assert_mix_close(mix, get("mix%d" % nm)))
                same_on_every_rank(props)
                same_on_every_rank(mix)
            dev.free()
            what = "n_multi=%s" % case["n_multi"]
        worst = gather((err_ln, err_mix))
        lines.append("%-26s %5d x %-5d %s ln_err=%.1e mix_err=%.1e"
                     % (case["name"], n, h, what, max(e[0] for e in worst),
                        max(e[1] for e in worst)))

    dist.barrier()
    if rank == 0:
        how = "p2p" if lib.mxb_comm_p2p_enabled(ctx.handle) else "nccl"
        print("\n".join(lines))
        print("MULTIRANK_OK world=%d exchange=%s cases=%d device=%s"
              % (world, how, len(lines), torch.cuda.get_device_name(local)))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
