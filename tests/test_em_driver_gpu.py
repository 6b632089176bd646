"""The EM driver (csrc/em.cu: em_poll_loop and run_tasks) takes the same decisions for one
restart slot and for two: restarts combined on the device equal independent runs combined in
restart order, max_iter 0 and 1 give the reference's results, a session iterated with
mxb_em_iterate hands back what run_em computes, and em_step launches no more kernels than one
iteration of run_em."""
import ctypes
import math
import os

import numpy as np
import pytest

from mixemt_b200 import _lib, em, synth
from mixemt_b200._lib import check, lib, ptr
from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
from mixemt_b200.runtime import DeviceMatrix, get_context
from oracle import oracle_np
from conftest import make_args

pytestmark = pytest.mark.gpu


def _close_mix(a, b, tol):
    fin = np.isfinite(b)
    return np.array_equal(a[~fin], b[~fin]) and np.abs(a[fin] - b[fin]).max() < tol


def _combine(props, mixes):
    """em.py:145-163 in numpy: sums and logaddexp folds in restart order, then averaged."""
    k = len(props)
    acc, mix = props[0].copy(), mixes[0].copy()
    for i in range(1, k):
        acc += props[i]
        mix = np.logaddexp(mix, mixes[i])
    if k > 1:
        acc /= k
        mix = mix - np.log(k)
    return np.array([math.exp(v) for v in acc]), mix


@pytest.fixture(scope="module")
def build17(phylo17):
    """Build-17 mixture in the reference's row order: compresses into class tiles."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)],
                             4000, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    inits = np.log(np.random.RandomState(1).dirichlet([1.0] * mat.shape[1], size=3))
    dev = DeviceMatrix.from_host(get_context(), mat)
    yield mat, mix.weights.astype(np.float64), inits, dev
    dev.free()


@pytest.fixture(scope="module")
def steps17(build17):
    """oracle_np.em_step at each init: (read matrix, new log-proportions) per restart."""
    mat, wts, inits, _ = build17
    return [oracle_np.em_step(mat, wts, init) for init in inits]


@pytest.fixture
def layout_env(request):
    old = {v: os.environ.pop(v, None) for v in ("MXB_EM_NO_PACK", "MXB_EM_NO_BATCH",
                                                "MXB_EM_SPLIT_TAIL", "MXB_EM_FORCE_GENERAL")}
    os.environ.update(request.param)
    yield request.param
    for v, val in old.items():
        os.environ.pop(v, None)
        if val is not None:
            os.environ[v] = val


LAYOUTS = [{}, {"MXB_EM_NO_PACK": "1"}, {"MXB_EM_NO_PACK": "1", "MXB_EM_NO_BATCH": "1"},
           {"MXB_EM_NO_PACK": "1", "MXB_EM_SPLIT_TAIL": "1"}, {"MXB_EM_FORCE_GENERAL": "1"}]


def _raw_run(dev, wts, init, max_iter, tol):
    """One restart through mxb_run_em_dev with MXB_EM_RAW: its final log-proportions and its
    read matrix, neither averaged."""
    ctx = dev.ctx
    h = dev.shape[1]
    props = np.zeros(h)
    iters, conv = np.zeros(1, dtype=np.int64), np.zeros(1, dtype=np.int32)
    handle = ctypes.c_void_p()
    check(lib.mxb_run_em_dev(ctx.handle, dev.handle, ptr(wts), ptr(np.ascontiguousarray(init)),
                             1, max_iter, tol, _lib.MXB_EM_RAW, ptr(props), None,
                             ctypes.byref(handle), ptr(iters), ptr(conv)))
    m = DeviceMatrix(ctx, handle)
    mix = m.to_host()
    m.free()
    return props, mix, int(iters[0]), int(conv[0])


@pytest.mark.parametrize("layout_env", LAYOUTS, indirect=True,
                         ids=["tiles", "rows", "rows1", "rows_split", "general"])
def test_restarts_equal_independent_runs(build17, layout_env):
    """Three restarts in one call (one slot over class tiles, two slots over fp64 rows, one slot
    with MXB_EM_NO_BATCH=1, one slot over fp64 rows with the split tail, the general path)
    against three single-restart calls combined in numpy."""
    mat, wts, inits, dev = build17
    a = make_args(n_multi=3, max_iter=400, tolerance=1e-5)
    props, mix, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    runs = [_raw_run(dev, wts, init, a.max_iter, a.tolerance) for init in inits]
    assert info["iterations"] == [r[2] for r in runs] and min(info["iterations"]) > 20
    assert info["converged"] == [r[3] for r in runs]
    want_props, want_mix = _combine([r[0] for r in runs], [r[1] for r in runs])
    assert np.array_equal(props, want_props)
    assert _close_mix(mix, want_mix, 1e-13)


@pytest.mark.parametrize("max_iter", [0, 1])
@pytest.mark.parametrize("n_multi", [1, 3])
@pytest.mark.parametrize("layout_env", LAYOUTS[:2], indirect=True, ids=["tiles", "rows"])
def test_zero_and_one_iteration(build17, steps17, layout_env, n_multi, max_iter):
    """max_iter 0: every restart hands back its init (em.py:126 never iterates) and the read
    matrix of the inits; max_iter 1: one em_step per restart, as oracle_np.run_em."""
    mat, wts, inits, dev = build17
    inits = inits[:n_multi]
    a = make_args(n_multi=n_multi, max_iter=max_iter, tolerance=1e-4)
    props, mix, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    steps = steps17[:n_multi]
    if max_iter == 0:
        assert info["iterations"] == [0] * n_multi and info["converged"] == [0] * n_multi
        want_props, want_mix = _combine(list(inits), [s[0] for s in steps])
        assert np.array_equal(props, want_props)
        assert _close_mix(mix, want_mix, 1e-9)
    else:
        o_props, o_mix, o_iters = oracle_np.run_em(mat, wts, inits, 1, a.tolerance)
        assert info["iterations"] == o_iters == [1] * n_multi
        assert info["converged"] == [0] * n_multi
        assert np.abs(props - o_props).max() < 1e-11
        assert _close_mix(mix, o_mix, 1e-9)


def test_em_step_launches_one_iteration(golden_toy):
    """em_step is run_em with one restart and max_iter 1: it enqueues one iteration's kernels,
    not a chunk of them."""
    mat = golden_toy["em_mat"]
    wts = np.arange(1, mat.shape[0] + 1, dtype=np.float64)
    ctx = get_context()
    init = np.log(np.full(mat.shape[1], 1.0 / mat.shape[1]))
    l0 = ctx.launch_count
    em.em_step(mat, wts, init, np.empty_like(mat))
    step = ctx.launch_count - l0
    dev = DeviceMatrix.from_host(ctx, mat)
    l0 = ctx.launch_count
    em.run_em_device(dev, wts, make_args(max_iter=1), inits=init.reshape(1, -1))
    one = ctx.launch_count - l0
    dev.free()
    assert 0 < step <= one


@pytest.mark.parametrize("max_iter", [0, 1, 400])
def test_session_iterate_equals_run_em(build17, max_iter):
    """mxb_em_set_lnprops + mxb_em_iterate continue from the set proportions with the same
    driver as run_em: the latest log-proportions (mxb_em_get_lnprops 0) equal run_em's with
    MXB_EM_RAW, the read matrix (mxb_em_read_mix) is formed from the ones before them, which
    mxb_em_get_lnprops 1 returns (the init when no iteration ran)."""
    mat, wts, inits, dev = build17
    ctx = dev.ctx
    n, h = mat.shape
    want_props, want_mix, want_it, want_conv = _raw_run(dev, wts, inits[0], max_iter, 1e-5)
    sess, mix_h = ctypes.c_void_p(), ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
    try:
        check(lib.mxb_em_set_lnprops(sess, ptr(np.ascontiguousarray(inits[0]))))
        it, cv = ctypes.c_int64(), ctypes.c_int32()
        check(lib.mxb_em_iterate(sess, max_iter, 1e-5, ctypes.byref(it), ctypes.byref(cv)))
        latest, prev = np.empty(h), np.empty(h)
        check(lib.mxb_em_get_lnprops(sess, 0, ptr(latest)))
        check(lib.mxb_em_get_lnprops(sess, 1, ptr(prev)))
        check(lib.mxb_matrix_alloc(ctx.handle, n, h, ctypes.byref(mix_h)))
        mix_dev = DeviceMatrix(ctx, mix_h)
        check(lib.mxb_em_read_mix(sess, mix_dev.handle, 0, 0.0))
        mix = mix_dev.to_host()
        mix_dev.free()
    finally:
        lib.mxb_em_destroy(sess)
    assert (it.value, cv.value) == (want_it, want_conv)
    assert np.array_equal(latest, want_props)
    assert np.array_equal(mix, want_mix)
    if max_iter <= 1:   # no iteration, or one from the init: the previous proportions are the init
        assert np.array_equal(prev, inits[0])
    if max_iter == 0:
        assert np.array_equal(latest, inits[0])
    else:
        assert want_it == max_iter or want_conv == 1
