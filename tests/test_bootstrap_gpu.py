"""The bootstrap on the GPU (csrc/bootstrap.cu, csrc/em.cu: run_bootstrap): the draws equal the
numpy restatement bit for bit, every replicate is the run_em restart on its counts from the
bootstrapped fit (class tiles: within 1e-13 of run_em_device, fp64 rows: bit-identical), a
replicate does not depend on how many are asked for or on the slot it ran in, uneven runs
refill their slots, an underflowing replicate is redone in log space on its own slot, and the
restart fan-out over 2 and 3 processes equals one process."""
import ctypes
import os
import socket
import time

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from mixemt_b200 import bootstrap, em, synth
from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
from mixemt_b200.runtime import DeviceMatrix, get_context
from oracle import oracle_np
from bootstrap_oracle import boot_counts
from conftest import make_args

pytestmark = pytest.mark.gpu

SEED = 77


@pytest.fixture
def no_pack():
    old = os.environ.get("MXB_EM_NO_PACK")
    os.environ["MXB_EM_NO_PACK"] = "1"
    yield
    if old is None:
        os.environ.pop("MXB_EM_NO_PACK")
    else:
        os.environ["MXB_EM_NO_PACK"] = old


@pytest.fixture(scope="module")
def build17(phylo17):
    """Build-17 mixture in the reference's row order (class tiles) and its fit."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 3000, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    wts = mix.weights.astype(np.float64)
    dev = DeviceMatrix.from_host(get_context(), mat)
    np.random.seed(3)
    props, _ = em.run_em(dev, wts, make_args(max_iter=400, tolerance=1e-5))
    yield mat, wts, props, dev
    dev.free()


def _start(props):
    with np.errstate(divide="ignore"):
        return np.log(props) - np.log(props.sum())


def _single(dev, counts, start, max_iter, tol):
    """One run_em restart on the counts from start (mxb_run_em_dev with MXB_EM_RAW): its final
    log-proportions, iterations and converged flag."""
    from mixemt_b200 import _lib
    from mixemt_b200._lib import lib, check, ptr
    lnp = np.zeros(dev.shape[1])
    it, cv = np.zeros(1, dtype=np.int64), np.zeros(1, dtype=np.int32)
    wts, init = _lib.as_f64(counts), np.ascontiguousarray(start)   # alive during the call
    check(lib.mxb_run_em_dev(dev.ctx.handle, dev.handle, ptr(wts),
                             ptr(init), 1, max_iter, tol, _lib.MXB_EM_RAW,
                             ptr(lnp), None, None, ptr(it), ptr(cv)))
    return lnp, int(it[0]), int(cv[0])


def test_counts_equal_numpy_draw():
    w = np.random.RandomState(2).randint(0, 6, size=257).astype(np.float64)
    w[[0, 5, 256]] = 0
    for seed in (0, 1, 2 ** 53 - 1):
        for boot0 in (0, 1000):
            for n_boot in (1, 37):
                got = bootstrap.boot_counts(w, seed, boot0, n_boot)
                want = np.array([boot_counts(w, seed, boot0 + k) for k in range(n_boot)])
                assert np.array_equal(got, want), (seed, boot0, n_boot)


def _check_replicates(build17, res, n_check, tol, exact, max_iter=400, t=1e-5):
    mat, wts, props, dev = build17
    start = _start(props)
    for b in range(n_check):
        c = bootstrap.boot_counts(wts, res.seed, b)[0]
        lnp, it, cv = _single(dev, c, start, max_iter, t)
        assert (res.iterations[b], res.converged[b]) == (it, cv), b
        assert np.array_equal(np.isfinite(lnp), np.isfinite(res.lnprops[b]))
        if exact:
            assert np.array_equal(res.lnprops[b], lnp), b
        else:
            assert np.abs(res.props[b] - np.exp(lnp)).max() < tol, b


def test_replicates_equal_run_em_on_their_counts(build17):
    mat, wts, props, dev = build17
    res = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=400, tolerance=1e-5), props,
                                    n_boot=6, seed=SEED)
    assert res.slots >= 1 and res.props.shape == (6, mat.shape[1])
    _check_replicates(build17, res, 6, 1e-13, exact=False)
    # against the oracle (two replicates, 40 iterations: the numpy restatement is slow)
    start = _start(props)
    short = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=40, tolerance=1e-5), props,
                                      n_boot=2, seed=SEED)
    for b in range(2):
        c = bootstrap.boot_counts(wts, SEED, b)[0].astype(np.float64)
        o_props, _, o_it = oracle_np.run_em(mat, c, start.reshape(1, -1), 40, 1e-5)
        assert o_it == [short.iterations[b]]
        assert np.abs(short.props[b] - o_props).max() < 1e-10
    lo, hi = res.interval(0.9)
    assert (lo <= hi).all()


def test_fp64_rows_are_bit_identical(build17, no_pack):
    mat, wts, props, dev = build17
    res = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=400, tolerance=1e-5), props,
                                    n_boot=3, seed=SEED)
    assert res.slots == 1
    _check_replicates(build17, res, 3, 0.0, exact=True)


def test_replicates_do_not_depend_on_n_boot(build17):
    mat, wts, props, dev = build17
    a = make_args(max_iter=60, tolerance=1e-6)
    ref = bootstrap.bootstrap_props(dev, wts, a, props, n_boot=40, seed=SEED)
    r = ref.slots
    again = bootstrap.bootstrap_props(dev, wts, a, props, n_boot=40, seed=SEED)
    assert np.array_equal(again.lnprops, ref.lnprops)
    for n in sorted({1, max(1, r - 1), r + 3}):
        res = bootstrap.bootstrap_props(dev, wts, a, props, n_boot=n, seed=SEED)
        assert np.array_equal(res.lnprops, ref.lnprops[:n]), n
        assert np.array_equal(res.iterations, ref.iterations[:n])


@pytest.mark.parametrize("max_iter", [0, 1, 7])
def test_uneven_runs_and_short_max_iter(build17, max_iter):
    """A tiny tolerance: every replicate stops at max_iter, except ones that converge; slots
    are refilled as they finish."""
    mat, wts, props, dev = build17
    res = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=max_iter, tolerance=1e-300),
                                    props, n_boot=5, seed=SEED + 1)
    if max_iter == 0:
        assert (res.iterations == 0).all() and (res.converged == 0).all()
        assert np.array_equal(res.lnprops, np.tile(_start(props), (5, 1)))
    else:
        assert (res.iterations == max_iter).all()
    _check_replicates(build17, res, 5, 1e-13, exact=False, max_iter=max_iter, t=1e-300)


def test_zero_props_stay_zero(build17):
    mat, wts, props, dev = build17
    p = props.copy()
    p[np.argsort(p)[:100]] = 0.0
    res = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=50, tolerance=1e-6), p,
                                    n_boot=5, seed=SEED)
    assert (res.props[:, p == 0] == 0).all()
    assert np.isneginf(res.lnprops[:, p == 0]).all()


def _abi_bootstrap(dev, wts, start, n_boot, seed, max_iter, tol, boot0=0):
    """mxb_em_bootstrap from log-proportions (a start that no proportion vector represents)."""
    from mixemt_b200._lib import lib, check, ptr
    h = dev.shape[1]
    lnp = np.zeros((n_boot, h))
    it, cv = np.zeros(n_boot, dtype=np.int64), np.zeros(n_boot, dtype=np.int32)
    slots = ctypes.c_int32()
    check(lib.mxb_em_bootstrap(dev.ctx.handle, dev.handle, ptr(wts), ptr(start), boot0, n_boot,
                               seed, max_iter, tol, ptr(lnp), ptr(it), ptr(cv),
                               ctypes.byref(slots)))
    return lnp, it, cv, slots.value


def test_underflowing_replicate_is_redone_in_log_space():
    """Column 0 starts at e^-760 (0 in fp64): the linear-space pass underflows at the first
    iteration (checked first), every replicate goes through the log-space step on its own slot
    and matches its run_em restart and the oracle."""
    from test_logspace_rescue_gpu import _underflowing_matrix, _layout_and_underflow, _init
    mat, wts = _underflowing_matrix("tiles")
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    try:
        start = _init(mat.shape[1], True)
        _, under = _layout_and_underflow(ctx, dev, wts, start)
        assert under
        lnp, it, cv, _ = _abi_bootstrap(dev, wts, start, 3, SEED, 30, 1e-8)
        for b in range(3):
            c = bootstrap.boot_counts(wts, SEED, b)[0].astype(np.float64)
            want, w_it, w_cv = _single(dev, c, start, 30, 1e-8)
            assert (it[b], cv[b]) == (w_it, w_cv)
            assert np.abs(np.exp(lnp[b]) - np.exp(want)).max() < 1e-13
            o_props, _, o_it = oracle_np.run_em(mat, c, start.reshape(1, -1), 30, 1e-8)
            assert o_it == [it[b]]
            assert np.abs(np.exp(lnp[b]) - o_props).max() < 1e-10
    finally:
        dev.free()


def test_refilled_slots_equal_independent_runs(build17):
    """n_boot = 2 R + 3 with a tolerance the replicates reach after different numbers of
    iterations: slots are refilled at different times, and every replicate, also those that ran
    in a refilled slot, equals the run_em restart on its own counts."""
    mat, wts, props, dev = build17
    r = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=1, tolerance=1e-5), props,
                                  n_boot=1, seed=SEED).slots
    n_boot = 2 * r + 3
    res = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=1000, tolerance=1e-3), props,
                                    n_boot=n_boot, seed=SEED + 2)
    assert len(set(res.iterations.tolist())) > 1, res.iterations
    _check_replicates(build17, res, n_boot, 1e-13, exact=False, max_iter=1000, t=1e-3)


def test_one_underflowing_slot_leaves_the_others_untouched():
    """Only some replicates draw the one row of weight 1 whose likelihood underflows from an
    e^-760 start: those are redone in log space on their slots and match their run_em restarts
    and the oracle; the others of the same passes are bit-identical to runs of their own."""
    from test_logspace_rescue_gpu import _underflowing_matrix, _layout_and_underflow, _init
    mat, wts = _underflowing_matrix("tiles")
    n = mat.shape[0]
    wts[:n // 4] = 0.0
    wts[0] = 1.0
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    try:
        start = _init(mat.shape[1], True)
        _, under = _layout_and_underflow(ctx, dev, wts, start)
        assert under
        n_boot = 19
        lnp, it, cv, r = _abi_bootstrap(dev, wts, start, n_boot, SEED, 30, 1e-8)
        counts = bootstrap.boot_counts(wts, SEED, 0, n_boot).astype(np.float64)
        flagged = counts[:, :n // 4].sum(1) > 0
        assert flagged.any() and not flagged.all()
        for b in range(n_boot):
            want, w_it, w_cv = _single(dev, counts[b], start, 30, 1e-8)
            assert (it[b], cv[b]) == (w_it, w_cv), b
            assert np.abs(np.exp(lnp[b]) - np.exp(want)).max() < 1e-13, b
            if not flagged[b]:
                alone, a_it, _, _ = _abi_bootstrap(dev, wts, start, 1, SEED, 30, 1e-8, boot0=b)
                assert np.array_equal(lnp[b], alone[0]) and a_it[0] == it[b], b
        for b in (int(np.argmax(flagged)), int(np.argmin(flagged))):
            o_props, _, o_it = oracle_np.run_em(mat, counts[b], start.reshape(1, -1), 30, 1e-8)
            assert o_it == [it[b]]
            assert np.abs(np.exp(lnp[b]) - o_props).max() < 1e-10
    finally:
        dev.free()


def test_launch_economy(build17):
    """n_boot = R replicates with a fixed number of iterations launch the kernels of one
    replicate's iterations: the launches beyond one replicate are resampling launches only."""
    mat, wts, props, dev = build17
    ctx = dev.ctx
    a = make_args(max_iter=5, tolerance=-1.0)
    one = bootstrap.bootstrap_props(dev, wts, a, props, n_boot=1, seed=SEED)
    r = one.slots
    l0 = ctx.launch_count
    bootstrap.bootstrap_props(dev, wts, a, props, n_boot=1, seed=SEED)
    l1 = ctx.launch_count - l0
    l0 = ctx.launch_count
    bootstrap.bootstrap_props(dev, wts, a, props, n_boot=r, seed=SEED)
    lr = ctx.launch_count - l0
    per_replicate = 4          # draw, counts -> weights, set proportions, reset control block
    assert lr - l1 == (r - 1) * per_replicate
    # and one replicate's iterations cost what one run_em restart's do (4 per tiled iteration)
    l0 = ctx.launch_count
    em.run_em_device(dev, wts, a, want_host=False, inits=_start(props).reshape(1, -1))
    run = ctx.launch_count - l0
    assert l1 - per_replicate == run - 2         # run_em: set proportions + reset


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gloo_allreduce(arr, op):
    import torch
    t = torch.from_numpy(arr)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return arr


def _worker(rank, world, port, mat, wts, props, n_boot, mode, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), MIXEMT_B200_DEVICE="0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ctx = get_context()
        ctx.rank, ctx.world = rank, world
        ctx.allreduce_host = gloo_allreduce
        a = make_args(max_iter=60, tolerance=1e-6, b200_shard=mode)
        try:
            np.random.seed(5)
            res = bootstrap.bootstrap_props(mat, wts, a, props, n_boot=n_boot)
            out[rank] = (res.lnprops, res.iterations, res.converged, res.seed)
        except ValueError:
            out[rank] = "ValueError"
    finally:
        dist.destroy_process_group()


def _run_ranks(world, args):
    spawn = mp.get_context("spawn")
    mgr = spawn.Manager()
    out = mgr.dict()
    port = free_port()
    procs = [spawn.Process(target=_worker, args=(r, world, port) + args + (out,))
             for r in range(world)]
    for p in procs:
        p.start()
    deadline = time.time() + 300
    for p in procs:
        p.join(max(1.0, deadline - time.time()))
    late = [p for p in procs if p.is_alive()]
    for p in late:
        p.kill()
        p.join()
    assert not late and [p.exitcode for p in procs] == [0] * world
    res = dict(out)
    mgr.shutdown()
    return res


@pytest.mark.parametrize("world", [2, 3])
def test_restart_fan_out_equals_one_process(build17, world):
    mat, wts, props, dev = build17
    np.random.seed(5)
    one = bootstrap.bootstrap_props(dev, wts, make_args(max_iter=60, tolerance=1e-6), props,
                                    n_boot=7)
    res = _run_ranks(world, (mat, wts, props, 7, "restarts"))
    for rank in range(world):
        lnp, it, cv, seed = res[rank]
        assert seed == one.seed
        assert np.array_equal(lnp, one.lnprops) and np.array_equal(it, one.iterations)
        assert np.array_equal(cv, one.converged)
    rows = _run_ranks(world, (mat, wts, props, 7, "rows"))
    assert all(rows[r] == "ValueError" for r in range(world))
