"""Row-sharded log-space rescue on 2 GPUs, launched by torchrun (see
test_logspace_rescue_gpu.py):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 \
        --master-addr 127.0.0.1 --master-port 29519 tests/logspace_shards_check.py [level]

For fp64 rows and for class tiles, every rank runs run_em on its row shard of a matrix whose
rows underflow in linear space at the first iteration; all ranks redo that iteration in log
space together.  Proportions and iteration counts must equal the CPU oracle on the whole
matrix, and all ranks must hand back the same bits.  A following run that never underflows
must succeed too (the peer mailboxes are still in step).  Rank 0 reports the time of one
rescued iteration next to one plain iteration of the same session.  The optional argument is
ln pi_0 of the underflowing start (default -760, exactly 0 in fp64; -730 makes t subnormal).
"""
import ctypes
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def underflowing_case(layout, level=-760.0, bad_rows=None):
    """Rows whose mass sits ~800 log units below their best haplotype, which starts with a
    proportion of e^level (e^-760 is 0 in fp64): s_i = sum_j L_ij pi_j is about e^level.
    bad_rows(n) gives those rows (default the first quarter)."""
    rs = np.random.RandomState(5)
    if layout == "fp64":
        n, h = 300, 1100
        mat = -rs.gamma(2.0, 3.0, size=(n, h))
    else:   # blocks of 64 identical columns: the shards run over class tiles
        n, h = 1280, 5408
        mat = np.repeat(-rs.gamma(2.0, 3.0, size=(n, h // 64 + 1)), 64, axis=1)[:, :h].copy()
    mat[:, 0] = 0.0
    mat[slice(0, n // 4) if bad_rows is None else bad_rows(n), 1:] -= 800.0
    wts = rs.randint(1, 5, size=n).astype(np.float64)
    bad = np.full(h, -np.log(h - 1.0))
    bad[0] = level
    good = np.full(h, -np.log(float(h)))
    return mat, wts, bad.reshape(1, h), good.reshape(1, h)


def main():
    import torch
    import torch.distributed as dist
    from conftest import make_args
    from mixemt_b200 import em, sharding
    from mixemt_b200._lib import lib, check, ptr
    from mixemt_b200.runtime import DeviceMatrix, get_context
    from oracle import oracle_c

    level = float(sys.argv[1]) if len(sys.argv) > 1 else -760.0
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = get_context()
    ctx.init_comm_from_torch()

    report = []
    for layout in ("fp64", "tiles"):
        mat, wts, bad, good = underflowing_case(layout, level)
        n, h = mat.shape
        lo, hi = sharding.row_shard(n, rank, world)
        shard = DeviceMatrix.from_host(ctx, mat[lo:hi])
        w_mine = wts[lo:hi].copy()

        sess = ctypes.c_void_p()
        check(lib.mxb_em_create(ctx.handle, shard.handle, ptr(w_mine), 1, ctypes.byref(sess)))
        nb, flag = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nb), ctypes.byref(flag)))
        assert flag.value == (0 if layout == "tiles" else -1), (layout, flag.value)
        # one iteration from each start, same session: plain, then rescued in log space
        ms = {}
        for name, init in (("plain", good), ("rescue", bad)):
            it, conv = ctypes.c_int64(), ctypes.c_int32()
            best = None
            for _ in range(3):
                check(lib.mxb_em_set_lnprops(sess, ptr(init[0].copy())))
                dist.barrier()
                t0 = time.perf_counter()
                check(lib.mxb_em_iterate(sess, 1, -1.0, ctypes.byref(it), ctypes.byref(conv)))
                dt = (time.perf_counter() - t0) * 1e3
                best = dt if best is None else min(best, dt)
            assert it.value == 1, (name, it.value)
            ms[name] = best
        lib.mxb_em_destroy(sess)

        a = make_args(max_iter=60, tolerance=1e-6, n_multi=1, b200_shard="rows")
        p, m, info, _ = em.run_em_device(shard, w_mine, a, inits=bad)
        o_p, o_m, o_it = oracle_c.run_em(mat, wts, bad, a.max_iter, a.tolerance)
        assert info["iterations"] == list(o_it), (layout, info, o_it)
        err_p = np.abs(p - o_p).max()
        assert err_p < 1e-9, (layout, err_p)
        fin = np.isfinite(o_m[lo:hi])
        err_m = np.abs(m[fin] - o_m[lo:hi][fin]).max()
        assert err_m < 1e-8, (layout, err_m)
        gathered = [None] * world
        dist.all_gather_object(gathered, p.tobytes())
        assert all(g == gathered[0] for g in gathered), "ranks disagree on the proportions"

        # a run that never underflows, in the same process: the mailboxes are still in step
        p2, _, info2, _ = em.run_em_device(shard, w_mine, a, inits=good)
        o_p2, _, o_it2 = oracle_c.run_em(mat, wts, good, a.max_iter, a.tolerance)
        assert info2["iterations"] == list(o_it2), (layout, info2, o_it2)
        assert np.abs(p2 - o_p2).max() < 1e-9, (layout, np.abs(p2 - o_p2).max())
        report.append("%s: %dx%d iters=%s dprops=%.1e plain_iter_ms=%.3f rescue_iter_ms=%.3f"
                      % (layout, n, h, info["iterations"], err_p, ms["plain"], ms["rescue"]))
        shard.free()

    dist.barrier()
    if rank == 0:
        how = "p2p" if lib.mxb_comm_p2p_enabled(ctx.handle) else "nccl"
        name = torch.cuda.get_device_name(local)
        print("LOGSPACE_SHARDS_OK world=%d exchange=%s level=%g device=%s | %s"
              % (world, how, level, name, " | ".join(report)))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
