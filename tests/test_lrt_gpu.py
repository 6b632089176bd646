"""The contributor likelihood-ratio test on the GPU (csrc/em.cu: mxb_em_refit through run_tasks,
mixemt_b200.likelihood.contributor_lrt): every refit equals a one-restart run_em from its start
(class tiles: within 1e-13, fp64 rows: bit-identical), the dropped column stays exactly 0, a
refit does not depend on which other columns are tested, uneven refits refill their slots and a
short max_iter hands back the starts, the statistic is the log-likelihood difference, the whole
result matches the long-double oracle on the reference's toy mixture and on a reduced
contributor matrix, and the restart fan-out over 2 and 3 processes equals one process."""
import io
import os
import socket
import time

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from mixemt_b200 import consumers, em, likelihood, synth
from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
from mixemt_b200.runtime import DeviceMatrix, get_context
from conftest import make_args
import loglik_oracle

pytestmark = pytest.mark.gpu


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
    """Build-17 mixture in the reference's row order (class tiles), its fit and the columns of
    its six largest proportions."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 3000, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    wts = mix.weights.astype(np.float64)
    dev = DeviceMatrix.from_host(get_context(), mat)
    np.random.seed(3)
    props, _ = em.run_em(dev, wts, make_args(max_iter=400, tolerance=1e-5))
    top = [int(c) for c in np.argsort(props)[::-1][:6]]
    yield mat, wts, props, dev, top, haps
    dev.free()


def _single(dev, w, start, max_iter, tol):
    """One run_em restart from start (mxb_run_em_dev with MXB_EM_RAW)."""
    from mixemt_b200 import _lib
    from mixemt_b200._lib import lib, check, ptr
    lnp = np.zeros(dev.shape[1])
    it, cv = np.zeros(1, dtype=np.int64), np.zeros(1, dtype=np.int32)
    init = np.ascontiguousarray(start)
    check(lib.mxb_run_em_dev(dev.ctx.handle, dev.handle, ptr(_lib.as_f64(w)), ptr(init), 1,
                             max_iter, tol, _lib.MXB_EM_RAW, ptr(lnp), None, None, ptr(it),
                             ptr(cv)))
    return lnp, int(it[0]), int(cv[0])


def _check_refits(dev, w, props, res, max_iter, tol, exact):
    starts = loglik_oracle.starts(props, res.columns)
    fits = np.vstack([res.lnprops_full, res.lnprops_null])
    for k, s in enumerate(starts):
        lnp, it, cv = _single(dev, w, s, max_iter, tol)
        assert (res.iterations[k], res.converged[k]) == (it, cv), k
        assert np.array_equal(np.isfinite(lnp), np.isfinite(fits[k])), k
        if exact:
            assert np.array_equal(fits[k], lnp), k
        else:
            assert np.abs(np.exp(fits[k]) - np.exp(lnp)).max() < 1e-13, k


def test_refits_equal_one_restart_runs(build17):
    mat, wts, props, dev, top, _ = build17
    a = make_args(max_iter=400, tolerance=1e-5)
    res = likelihood.contributor_lrt(dev, wts, a, props, top)
    assert res.slots >= 1 and res.lnprops_null.shape == (6, mat.shape[1])
    _check_refits(dev, wts, props, res, 400, 1e-5, exact=False)
    for k, c in enumerate(top):     # zeros stay zero
        assert res.lnprops_null[k, c] == -np.inf
    assert np.isneginf(res.lnprops_null[:, props == 0]).all()
    # the statistic is the difference of log_likelihood at the refits
    full = likelihood.log_likelihood(dev, wts, np.exp(res.lnprops_full))
    null = likelihood.log_likelihood(dev, wts, np.exp(res.lnprops_null))
    scale = float(loglik_oracle.ld_loglik(mat, wts, res.lnprops_full)[1])
    assert abs(res.loglik_full - full) <= 1e-12 * scale
    want = np.maximum(0.0, 2 * (full - null))
    assert np.abs(res.statistic - want).max() <= 4e-12 * scale


def test_fp64_rows_are_bit_identical(build17, no_pack):
    mat, wts, props, dev, top, _ = build17
    res = likelihood.contributor_lrt(dev, wts, make_args(max_iter=400, tolerance=1e-5), props,
                                     top[:3])
    assert res.slots == 1
    _check_refits(dev, wts, props, res, 400, 1e-5, exact=True)


def test_refits_do_not_depend_on_the_batch(build17):
    mat, wts, props, dev, top, _ = build17
    a = make_args(max_iter=60, tolerance=1e-6)
    ref = likelihood.contributor_lrt(dev, wts, a, props, top)
    again = likelihood.contributor_lrt(dev, wts, a, props, top)
    assert np.array_equal(again.lnprops_null, ref.lnprops_null)
    assert np.array_equal(again.statistic, ref.statistic)
    for sub in ([top[2]], top[3:0:-1], [top[5], top[0]]):
        res = likelihood.contributor_lrt(dev, wts, a, props, sub)
        assert np.array_equal(res.lnprops_full, ref.lnprops_full)
        assert res.loglik_full == ref.loglik_full
        for k, c in enumerate(sub):
            i = top.index(c)
            assert np.array_equal(res.lnprops_null[k], ref.lnprops_null[i]), c
            assert res.loglik_null[k] == ref.loglik_null[i] and res.statistic[k] == ref.statistic[i]
            assert res.iterations[1 + k] == ref.iterations[1 + i]


@pytest.mark.parametrize("max_iter", [0, 1, 7])
def test_short_max_iter(build17, max_iter):
    mat, wts, props, dev, top, _ = build17
    res = likelihood.contributor_lrt(dev, wts, make_args(max_iter=max_iter, tolerance=1e-300),
                                     props, top[:4])
    if max_iter == 0:
        assert (res.iterations == 0).all() and (res.converged == 0).all()
        starts = loglik_oracle.starts(props, top[:4])
        assert np.array_equal(np.vstack([res.lnprops_full, res.lnprops_null]), starts)
    else:
        assert (res.iterations == max_iter).all()
    _check_refits(dev, wts, props, res, max_iter, 1e-300, exact=False)


def test_refilled_slots_equal_independent_runs(build17):
    """More refits than slots, stopping after different numbers of iterations: slots are
    refilled at different times, and every refit equals its one-restart run."""
    mat, wts, props, dev, top, _ = build17
    r = likelihood.contributor_lrt(dev, wts, make_args(max_iter=1), props, top[:1]).slots
    cols = [int(c) for c in np.argsort(props)[::-1][:min(2 * r + 3, 40)]]
    res = likelihood.contributor_lrt(dev, wts, make_args(max_iter=1000, tolerance=1e-3), props,
                                     cols)
    assert len(set(res.iterations.tolist())) > 1, res.iterations
    _check_refits(dev, wts, props, res, 1000, 1e-3, exact=False)


def _against_oracle(mat, w, props, cols, max_iter, tol):
    res = likelihood.contributor_lrt(mat, w, make_args(max_iter=max_iter, tolerance=tol), props,
                                     cols)
    o = loglik_oracle.lrt(mat, w, props, cols, max_iter, tol)
    assert res.iterations.tolist() == o["iterations"].tolist()
    fits = np.exp(np.vstack([res.lnprops_full, res.lnprops_null]))
    assert np.abs(fits - o["props"]).max() < 1e-10
    lls = np.concatenate([[res.loglik_full], res.loglik_null])
    assert np.abs(lls - o["loglik"].astype(np.float64)).max() <= 1e-10 * o["scale"]
    for k in range(len(cols)):
        d, od = res.statistic[k], float(o["statistic"][k])
        if np.isinf(od):
            assert d == od
        else:
            assert abs(d - od) <= 1e-9 * max(od, 1.0), (k, d, od)
            assert abs(res.pvalue[k] - o["pvalue"][k]) <= 1e-9 * max(o["pvalue"][k], 1e-300) \
                + 1e-12
    return res, o


def test_toy_mixture_against_the_oracle(golden_toy):
    """The reference's 10 x 9 toy (em_test.py:104-116: B 0.8, E 0.2): its fit, then B, E and
    the next largest column."""
    mat = golden_toy["em_mat"]
    w = np.ones(10)
    np.random.seed(1)
    props, _ = em.run_em(mat, w, make_args())
    other = [int(c) for c in np.argsort(props)[::-1] if c not in (1, 4) and props[c] > 0][0]
    _against_oracle(mat, w, props, [1, 4, other], 1000, 1e-4)


def test_reduced_contributor_matrix_against_the_oracle(build17):
    """The refinement matrix of bin/mixemt:311-320: the contributor columns of the fit
    (reduce_em_matrix), refitted, then each contributor tested (fp64 rows, H = 4)."""
    mat, wts, props, dev, top, haps = build17
    contribs = [("hap%d" % (i + 1), haps[c], props[c]) for i, c in enumerate(top[:4])]
    small, new_haps = consumers.reduce_em_matrix(mat, haps, contribs)
    np.random.seed(2)
    sprops, _ = em.run_em(small, wts, make_args(max_iter=500, tolerance=1e-6))
    cols = [new_haps.index(h) for _, h, _ in contribs]
    res, _ = _against_oracle(small, wts, sprops, cols, 500, 1e-6)
    out = io.StringIO()
    res.report(new_haps, out)
    assert len(out.getvalue().splitlines()) == 4


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gloo_allreduce(arr, op):
    import torch
    t = torch.from_numpy(arr)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return arr


def _worker(rank, world, port, mat, wts, props, cols, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), MIXEMT_B200_DEVICE="0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ctx = get_context()
        ctx.rank, ctx.world = rank, world
        ctx.allreduce_host = gloo_allreduce
        a = make_args(max_iter=60, tolerance=1e-6, b200_shard="restarts")
        res = likelihood.contributor_lrt(mat, wts, a, props, cols)
        out[rank] = (res.lnprops_full, res.lnprops_null, res.iterations, res.converged,
                     res.loglik_full, res.loglik_null, res.statistic)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_restart_fan_out_equals_one_process(build17, world):
    mat, wts, props, dev, top, _ = build17
    cols = top[:4]
    one = likelihood.contributor_lrt(dev, wts, make_args(max_iter=60, tolerance=1e-6), props,
                                     cols)
    spawn = mp.get_context("spawn")
    mgr = spawn.Manager()
    out = mgr.dict()
    port = free_port()
    procs = [spawn.Process(target=_worker, args=(r, world, port, mat, wts, props, cols, out))
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
    want = (one.lnprops_full, one.lnprops_null, one.iterations, one.converged, one.loglik_full,
            one.loglik_null, one.statistic)
    for rank in range(world):
        for got, w in zip(res[rank], want):
            assert np.array_equal(got, w), rank
