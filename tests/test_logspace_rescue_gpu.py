"""Rows whose mixture likelihood underflows in linear space, in the sessions that iterate two
restarts per pass and in row-sharded sessions: the flagged iteration is redone in log space
(em.py:80-89, max-shifted logsumexp) and the run goes on, where it used to end with
NumericRangeError."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import make_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _close_mix(a, b, tol):
    fin = np.isfinite(b)
    return np.array_equal(fin, np.isfinite(a)) and np.abs(a[fin] - b[fin]).max() < tol


def _underflowing_matrix(layout="fp64"):
    """test_underflowing_rows_are_redone_in_log_space's matrices: a quarter of the rows sit
    ~800 log units below their best haplotype (column 0) everywhere else."""
    rs = np.random.RandomState(5)
    if layout == "fp64":
        n, h = 300, 1100
        mat = -rs.gamma(2.0, 3.0, size=(n, h))
    else:   # blocks of 64 identical columns: class tiles
        n, h = 1280, 5408
        mat = np.repeat(-rs.gamma(2.0, 3.0, size=(n, h // 64 + 1)), 64, axis=1)[:, :h].copy()
    mat[:, 0] = 0.0
    mat[: n // 4, 1:] -= 800.0
    wts = rs.randint(1, 5, size=n).astype(np.float64)
    return mat, wts


def _init(h, underflows):
    """A start with proportion e^-760 (0 in fp64) on column 0 makes those rows' likelihood
    underflow at the first iteration; a uniform start does not."""
    if underflows:
        lnp = np.full(h, -np.log(h - 1.0))
        lnp[0] = -760.0
        return lnp
    return np.full(h, -np.log(float(h)))


def _layout_and_underflow(ctx, dev, wts, lnp):
    """(layout flag of mxb_em_pass_bytes, whether the linear-space pass flags an underflow at
    the first iteration from lnp: mxb_em_iterate_fixed stops with MXB_ERR_RANGE then)."""
    from mixemt_b200 import _lib
    from mixemt_b200._lib import lib, check, ptr
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
    try:
        nb, flag = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nb), ctypes.byref(flag)))
        check(lib.mxb_em_set_lnprops(sess, ptr(np.ascontiguousarray(lnp))))
        rc = lib.mxb_em_iterate_fixed(sess, 1, None, None)
        assert rc in (_lib.MXB_OK, _lib.MXB_ERR_RANGE), rc
    finally:
        lib.mxb_em_destroy(sess)
    return flag.value, rc == _lib.MXB_ERR_RANGE


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["fp64", "tiles"])
def test_single_restart_redoes_underflowing_iteration(layout):
    """One restart on one GPU, from a start that does underflow at the first iteration (the
    precondition is checked: the linear-space pass alone stops there)."""
    from mixemt_b200 import em
    from mixemt_b200.runtime import DeviceMatrix, get_context
    from oracle import oracle_c
    mat, wts = _underflowing_matrix(layout)
    inits = _init(mat.shape[1], True).reshape(1, -1)
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    flag, underflows = _layout_and_underflow(ctx, dev, wts, inits[0])
    assert flag == (0 if layout == "tiles" else -1) and underflows
    a = make_args(max_iter=60, tolerance=1e-6)
    p, m, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    o_p, o_m, o_it = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert info["iterations"] == list(o_it)
    assert np.abs(p - o_p).max() < 1e-9
    assert _close_mix(m, o_m, 1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["UF", "FU", "UU", "UFU"])
def test_restart_pairs_redo_underflowing_iterations(pattern):
    """n_multi = len(pattern) restarts, two per pass (em_pass_pair_kernel); 'U' starts
    underflow, 'F' starts do not, so a pair may hold one of each.  Iteration counts equal the
    oracle's, results are within 1e-9 (props) and 1e-8 (read matrix) of the oracle and
    bit-identical to the restarts run one at a time (MXB_EM_NO_BATCH=1)."""
    from mixemt_b200 import em
    from mixemt_b200.runtime import DeviceMatrix, get_context
    from oracle import oracle_c
    mat, wts = _underflowing_matrix()
    h = mat.shape[1]
    inits = np.array([_init(h, c == "U") for c in pattern])
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    # fp64 rows (the noise does not compress into class tiles): the pair path applies; the
    # 'U' start underflows, the 'F' start does not
    assert _layout_and_underflow(ctx, dev, wts, _init(h, True)) == (-1, True)
    assert _layout_and_underflow(ctx, dev, wts, _init(h, False)) == (-1, False)

    a = make_args(n_multi=len(pattern), max_iter=60, tolerance=1e-6)
    p_b, m_b, info_b, _ = em.run_em_device(dev, wts, a, inits=inits)
    os.environ["MXB_EM_NO_BATCH"] = "1"
    try:
        p_s, m_s, info_s, _ = em.run_em_device(dev, wts, a, inits=inits)
    finally:
        del os.environ["MXB_EM_NO_BATCH"]
    o_p, o_m, o_it = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert info_b["iterations"] == list(o_it) == info_s["iterations"]
    assert info_b["converged"] == info_s["converged"]
    assert np.abs(p_b - o_p).max() < 1e-9
    assert _close_mix(m_b, o_m, 1e-8)
    assert np.array_equal(p_b, p_s)
    assert np.array_equal(m_b, m_s)


@pytest.mark.gpu
@pytest.mark.parametrize("exchange", ["p2p", "nccl"])
def test_row_shards_redo_underflowing_iterations(exchange):
    """World size 2, row-sharded, fp64 rows and class tiles, column sums exchanged by peer
    stores in the tail kernel or by ncclAllReduce (MXB_NO_P2P=1): see logspace_shards_check.py."""
    from mixemt_b200 import _lib
    if _lib.lib.mxb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ)
    env["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 2) // 2))
    if exchange == "nccl":
        env["MXB_NO_P2P"] = "1"
    else:
        env.pop("MXB_NO_P2P", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29519" if exchange == "p2p" else "29520",
           os.path.join(ROOT, "tests", "logspace_shards_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert res.returncode == 0 and "LOGSPACE_SHARDS_OK" in res.stdout, \
        res.stdout[-2000:] + res.stderr[-4000:]
    assert ("exchange=%s" % exchange) in res.stdout, res.stdout[-2000:]
    print(res.stdout.strip().splitlines()[-1])
