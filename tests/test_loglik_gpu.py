"""The log-likelihood kernel (csrc/loglik.cu, mixemt_b200.likelihood.log_likelihood) on the GPU:
within 1e-12 of long double (relative to sum_i w_i |l_i|) on -inf matrices, random widths,
zero weights on impossible rows, zero proportions, rows whose likelihood is tiny but not zero
(log-space redo) and the Build-17 mixture; every vector bit-identical to its value computed
alone and across calls whatever K; and a row-sharded call over 2 and 3 processes on one GPU
equal to the whole matrix and identical on every rank."""
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mixemt_b200 import em, likelihood, synth
from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
from mixemt_b200.runtime import DeviceMatrix, get_context
from conftest import make_args
from loglik_oracle import ld_loglik
from window_cases import MODES, window_case

pytestmark = pytest.mark.gpu

INF = np.inf


def _norm_ln(props):
    p = np.atleast_2d(np.asarray(props, dtype=np.float64))
    with np.errstate(divide="ignore"):
        return np.log(p) - np.log(p.sum(1, keepdims=True))


def check_ld(mat, w, props, tol=1e-12):
    """log_likelihood of the (K, H) props against long double."""
    got = likelihood.log_likelihood(mat, w, np.atleast_2d(props))
    for k, lnp in enumerate(_norm_ln(props)):
        want, scale = ld_loglik(mat, w, lnp)
        if want == -INF:
            assert got[k] == -INF, k
        else:
            assert np.isfinite(got[k]), k
            assert abs(got[k] - float(want)) <= tol * max(float(scale), 1e-300), \
                (k, got[k], float(want), float(scale))
    return got


@pytest.mark.parametrize("wts", [[1, 1, 1], [2, 1, 1], [0.5, 0, 3]])
def test_em_test_inf_matrix(wts):
    """em_test.py:35-65's 3 x 3 matrix of 0 / -inf, with a single vector and with several."""
    mat = np.array([[0.0, -INF, -INF], [-INF, 0.0, -INF], [-INF, -INF, 0.0]])
    w = np.array(wts, dtype=np.float64)
    props = np.array([[0.6, 0.2, 0.2], [0.5, 0.5, 0.0], [1.0, 0.0, 0.0]])
    got = check_ld(mat, w, props)
    assert got[2] == (-INF if (w[1:] > 0).any() else 0.0)
    one = likelihood.log_likelihood(mat, w, props[0])
    assert isinstance(one, float) and one == got[0]


def _random(n, h, seed):
    rs = np.random.RandomState(seed)
    mat = -rs.gamma(2.0, 3.0, size=(n, h))
    mat[rs.rand(n, h) < 0.1] = -INF
    w = rs.randint(0, 6, size=n).astype(np.float64) * rs.choice([1.0, 0.25], size=n)
    props = rs.dirichlet(np.ones(h), size=3)
    return mat, w, props


@pytest.mark.parametrize("h", [1, 31, 32, 33, 5408])
def test_random_widths(h):
    n = 300 if h < 5408 else 64
    mat, w, props = _random(n, h, h)
    if h > 1:
        props[1, : h // 2] = 0.0          # zero proportions
    check_ld(mat, w, props)


def test_zero_weight_rows_without_a_finite_term():
    mat, w, props = _random(200, 40, 7)
    mat[[3, 50, 199]] = -INF
    w[[3, 50, 199]] = 0.0
    got = check_ld(mat, w, props)
    assert np.isfinite(got).all()
    w[50] = 1.0
    assert (likelihood.log_likelihood(mat, w, props) == -INF).all()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("level", [-760.0, -740.0, -708.4, -700.0, -665.0, -600.0])
def test_tiny_row_likelihoods_take_the_log_space_redo(mode, level):
    """window_cases: a quarter of the rows have sum_j L_ij pi_j about e^level, some below the
    2^-960 rule (redone in log space), some above it; both match long double."""
    mat, w, lnp, _ = window_case("rows", mode, level)
    check_ld(mat, w, np.exp(lnp))


def test_log_space_redo_keeps_proportions_exp_would_lose():
    """ln pi_0 = -760: pi_0 is 0 in fp64, so only the redo from the log-proportions gives the
    window rows a finite value (the Python front normalises linear proportions, so this is the
    C-ABI)."""
    from mixemt_b200._lib import lib, check, ptr
    mat, w, lnp, q = window_case("rows", "pi", -760.0)
    lnp = np.ascontiguousarray(lnp.reshape(1, -1))
    dev = DeviceMatrix.from_host(get_context(), mat)
    try:
        out = np.zeros(1)
        check(lib.mxb_matrix_loglik(dev.ctx.handle, dev.handle, ptr(w), ptr(lnp), 1, ptr(out)))
    finally:
        dev.free()
    want, scale = ld_loglik(mat, w, lnp[0])
    assert np.isfinite(out[0]) and abs(out[0] - float(want)) <= 1e-12 * float(scale)


@pytest.fixture(scope="module")
def build17(phylo17):
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 3000, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    wts = mix.weights.astype(np.float64)
    np.random.seed(3)
    props, _ = em.run_em(mat, wts, make_args(max_iter=400, tolerance=1e-5))
    return mat, wts, props


def _vectors(props, k, seed=1):
    rs = np.random.RandomState(seed)
    out = np.tile(props, (k, 1)) * rs.uniform(0.5, 1.5, size=(k, len(props)))
    out[1::3, np.argsort(props)[-1]] = 0.0
    return out


def test_build17_mixture(build17):
    mat, wts, props = build17
    check_ld(mat, wts, np.vstack([props, _vectors(props, 3)]))


@pytest.mark.parametrize("k", [1, 16, 17, 40])
def test_vectors_do_not_depend_on_the_batch(build17, k):
    mat, wts, props = build17
    dev = DeviceMatrix.from_host(get_context(), mat)
    try:
        vecs = _vectors(props, k)
        got = likelihood.log_likelihood(dev, wts, vecs)
        again = likelihood.log_likelihood(dev, wts, vecs)
        assert np.array_equal(got, again)
        for i in sorted({0, k // 2, k - 1}):
            assert likelihood.log_likelihood(dev, wts, vecs[i]) == got[i], i
        if k > 1:
            assert np.array_equal(likelihood.log_likelihood(dev, wts, vecs[::-1]), got[::-1])
    finally:
        dev.free()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gloo_allreduce(arr, op="sum"):
    t = torch.from_numpy(arr)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return arr


def _worker(rank, world, port, mat, wts, props, out):
    from mixemt_b200 import sharding
    from mixemt_b200.runtime import RowShard
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), MIXEMT_B200_DEVICE="0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ctx = get_context()
        ctx.rank, ctx.world = rank, world
        ctx.allreduce_host = gloo_allreduce
        lo, hi = sharding.row_shard(len(mat), rank, world)
        host = likelihood.log_likelihood(mat[lo:hi], wts[lo:hi], props, sharded=True)
        dev = DeviceMatrix.from_host(ctx, mat[lo:hi])
        dev.row_shard = RowShard()
        marked = likelihood.log_likelihood(dev, wts[lo:hi], props)
        dev.free()
        try:    # a rank with bad weights: every rank raises
            likelihood.log_likelihood(mat[lo:hi], wts[lo:hi][:-1] if rank == 1 else wts[lo:hi],
                                      props, sharded=True)
            failed = None
        except ValueError as exc:
            failed = type(exc).__name__
        out[rank] = (host, marked, failed)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_row_shards_equal_the_whole_matrix(build17, world):
    mat, wts, props = build17
    vecs = np.vstack([props, _vectors(props, 4)])
    whole = likelihood.log_likelihood(mat, wts, vecs)
    spawn = mp.get_context("spawn")
    mgr = spawn.Manager()
    out = mgr.dict()
    port = free_port()
    procs = [spawn.Process(target=_worker, args=(r, world, port, mat, wts, vecs, out))
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
    scale = max(float(ld_loglik(mat, wts, lnp)[1]) for lnp in _norm_ln(vecs))
    for rank in range(world):
        host, marked, failed = res[rank]
        assert np.array_equal(host, res[0][0]) and np.array_equal(marked, host)
        assert np.abs(host - whole).max() <= 1e-12 * scale
        assert failed is not None
