"""Rows whose mixture likelihood t = sum_j L_ij pi_j is tiny but not zero (window_cases: e^-760
to e^-600, entered through pi, through L or through a product of two normal factors, weights
scaled by 1, 1e3 and 1e6) in every EM pass, against the long-double reference
(tile_cases.ld_iterate / ld_read_mix) with the tolerances of rank_cases.py.  A row
with t < 2^-960 (csrc/em_kernels.cuh: row_needs_logspace) is redone in log space; above it the
linear-space pass must stay finite and accurate.  The flag probe pins the boundary from both
sides."""
import os
import subprocess
import sys

import numpy as np
import pytest

from mixemt_b200 import _lib, bootstrap, em
from mixemt_b200.runtime import DeviceMatrix, get_context
from oracle import oracle_c
from bootstrap_oracle import boot_counts
from conftest import make_args
from test_logspace_rescue_gpu import _layout_and_underflow
from rank_cases import Session, assert_ln_close, assert_mix_close
from tile_cases import ld_iterate, ld_read_mix
from window_cases import LN_THETA, MODES, SCALES, levels_of, plain_start, window_case

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 3
SEED = 17

# path -> (window_cases layout, environment, layout flag of mxb_em_pass_bytes)
PATHS = {
    "rows_nc2": ("rows", {"MXB_EM_NO_PACK": "1"}, -1),           # em_pass_fast_kernel<2>
    "rows_nc8": ("rows8", {"MXB_EM_NO_PACK": "1"}, -1),          # em_pass_fast_kernel<8>
    "general_h3": ("narrow", {}, -1),                            # em_rowdot_kernel
    "general_h9000": ("wide", {"MXB_EM_NO_PACK": "1"}, -1),
    "general_forced": ("rows", {"MXB_EM_FORCE_GENERAL": "1"}, -1),
    "tiles": ("tiles", {}, 0),                                   # tile_pass_kernel
}

_CASES = {}
_DEV = {}


def case(layout, mode, level):
    """Matrix, weights (scale 1), window start and its long-double trajectory (K iterations)."""
    key = (layout, mode, level)
    if key not in _CASES:
        mat, w, lnp, _ = window_case(layout, mode, level)
        _CASES[key] = (mat, w, lnp, ld_iterate(mat, w, lnp, K))
    return _CASES[key]


def plain(layout, mode, level):
    """The trajectory of a uniform start on the same matrix."""
    key = (layout, mode, level, "plain")
    if key not in _CASES:
        mat, w, _, _ = case(layout, mode, level)
        lnp = plain_start(mat.shape[1])
        _CASES[key] = (mat, w, lnp, ld_iterate(mat, w, lnp, K))
    return _CASES[key]


def device(layout, mode, level):
    # the "pi" matrices do not depend on the level
    key = (layout, mode, None if mode == "pi" else level)
    if key not in _DEV:
        _DEV[key] = DeviceMatrix.from_host(get_context(), case(layout, mode, level)[0])
    return _DEV[key]


@pytest.fixture(scope="module", autouse=True)
def _free_cache():
    yield
    for d in _DEV.values():
        d.free()
    _DEV.clear()
    _CASES.clear()


@pytest.fixture
def env():
    saved = {}

    def set_(**kw):
        for k, v in kw.items():
            saved.setdefault(k, os.environ.get(k))
            os.environ[k] = v
    yield set_
    for k, v in saved.items():
        os.environ.pop(k, None)
        if v is not None:
            os.environ[k] = v


def _params(paths):
    return [pytest.param(p, m, lv, id="%s-%s-%.2f" % (p, m, lv))
            for p in paths for m in MODES for lv in levels_of(PATHS[p][0])]


@pytest.mark.parametrize("path,mode,level", _params(PATHS))
def test_window_sessions(path, mode, level, env):
    """k = 1 and 3 iterations through mxb_em_iterate at every weight scale: ln pi within 1e-12
    of the reference with its -inf pattern, the read matrix within 1e-11, nothing NaN.  The
    first pass flags a row (mxb_em_iterate_fixed(1) stops with MXB_ERR_RANGE) exactly when the
    level is below ln 2^-960."""
    layout, variables, want_layout = PATHS[path]
    env(**variables)
    mat, w, lnp, traj = case(layout, mode, level)
    dev = device(layout, mode, level)
    for scale in SCALES:
        ws = w * scale
        flag, flagged = _layout_and_underflow(dev.ctx, dev, ws, lnp)
        assert flag == want_layout
        assert flagged == (level < LN_THETA), (scale, flagged)
        s = Session(dev, ws)
        try:
            for k in (1, K):
                latest, prev, mix = s.iterate(lnp, k)
                assert not np.isnan(latest).any() and not np.isnan(mix).any(), (scale, k)
                assert_ln_close(latest, traj[k])
                assert_ln_close(prev, traj[k - 1])
                assert_mix_close(mix, ld_read_mix(mat, traj[k - 1]))
        finally:
            s.close()


@pytest.mark.parametrize("mode,level",
                         [pytest.param(m, lv, id="%s-%.2f" % (m, lv))
                          for m in MODES for lv in levels_of("rows")])
def test_window_restart_pairs(mode, level, env):
    """Two restarts per pass (em_pass_pair_kernel), one window start and one uniform start, in
    both orders: equal to the reference and bit-identical to one restart at a time."""
    env(MXB_EM_NO_PACK="1")
    mat, w, lnp, traj = case("rows", mode, level)
    _, _, lnp_u, traj_u = plain("rows", mode, level)
    dev = device("rows", mode, level)
    a = make_args(n_multi=2, max_iter=K, tolerance=0.0)
    for scale in (1.0, 1e6):
        ws = w * scale
        for inits, trajs in (((lnp, lnp_u), (traj, traj_u)), ((lnp_u, lnp), (traj_u, traj))):
            inits = np.stack(inits)
            os.environ.pop("MXB_EM_NO_BATCH", None)
            p_b, m_b, info_b, _ = em.run_em_device(dev, ws, a, inits=inits)
            env(MXB_EM_NO_BATCH="1")
            p_s, m_s, info_s, _ = em.run_em_device(dev, ws, a, inits=inits)
            os.environ.pop("MXB_EM_NO_BATCH")
            assert info_b["iterations"] == info_s["iterations"] == [K, K]
            want = (trajs[0][K] + trajs[1][K]) / 2      # run_em averages ln pi (em.py:155-160)
            live = want > -700.0
            assert_ln_close(np.log(p_b[live]), want[live])
            assert (p_b[~live] < 1e-300).all()
            with np.errstate(divide="ignore"):
                want_mix = np.logaddexp(ld_read_mix(mat, trajs[0][K - 1]),
                                        ld_read_mix(mat, trajs[1][K - 1]))
                want_mix -= np.log(np.longdouble(2))
            assert not np.isnan(m_b).any()
            assert_mix_close(m_b, want_mix)
            assert np.array_equal(p_b, p_s) and np.array_equal(m_b, m_s)


@pytest.mark.parametrize("mode,level",
                         [pytest.param(m, lv, id="%s-%.2f" % (m, lv))
                          for m in MODES for lv in levels_of("rows")])
def test_window_em_step(mode, level):
    """The drop-in em.em_step (one iteration of one restart, fp64 rows and H = 3)."""
    for layout in ("rows", "narrow"):
        mat, w, lnp, traj = case(layout, mode, level)
        for scale in SCALES:
            mix = np.empty_like(mat)
            mix, new = em.em_step(mat, w * scale, lnp, mix)
            assert not np.isnan(new).any() and not np.isnan(mix).any()
            assert_ln_close(new, traj[1])
            assert_mix_close(mix, ld_read_mix(mat, traj[0]))


BOOT_LEVELS = (-740.0, -700.0, LN_THETA - 0.5, LN_THETA + 0.5)


def _boot(mode, level, scale, k):
    """2R replicates of k iterations, R the session's slots: (matrix, weights, start, ln pi, R)."""
    mat, w, lnp, _ = case("tiles", mode, level)
    dev = device("tiles", mode, level)
    a = make_args(max_iter=k, tolerance=0.0)
    wb = _lib.as_f64(w * scale)
    _, _, _, slots = bootstrap._run(dev, wb, np.ascontiguousarray(lnp), 0, 1, SEED, a)
    assert slots > 1
    got, iters, conv, _ = bootstrap._run(dev, wb, np.ascontiguousarray(lnp), 0, 2 * slots, SEED,
                                         a)
    assert (iters == k).all() and not np.isnan(got).any()
    return mat, w * scale, lnp, got, slots


@pytest.mark.parametrize("mode,level",
                         [pytest.param(m, lv, id="%s-%.2f" % (m, lv))
                          for m in MODES for lv in BOOT_LEVELS])
def test_window_bootstrap_on_tiles(mode, level):
    """Bootstrap replicates side by side on slotted class tiles (tile_pass_kernel<..., true>),
    2R replicates so that the slots are refilled: the first replicate of the first round and
    the last of the second match K iterations of the reference on their fragment counts."""
    mat, wb, lnp, got, slots = _boot(mode, level, 1.0, K)
    for b in (0, 2 * slots - 1):
        counts = boot_counts(wb, SEED, b).astype(np.float64)
        assert_ln_close(got[b], ld_iterate(mat, counts, lnp, K)[K])


def test_window_bootstrap_every_replicate():
    """Every one of 2R replicates from a start at e^-700 with weights 1e3..4e3 (normal t whose
    coefficients overflow), one iteration each."""
    mat, wb, lnp, got, slots = _boot("product", -700.0, 1e3, 1)
    for b in range(2 * slots):
        counts = boot_counts(wb, SEED, b).astype(np.float64)
        assert_ln_close(got[b], ld_iterate(mat, counts, lnp, 1)[1])


@pytest.mark.parametrize("layout,starts", [
    ("rows", (("pi", -720.0, 1.0), ("product", -700.0, 1e3))),
    ("tiles", (("L", -730.0, 1.0), ("pi", -705.0, 1e6))),
])
def test_window_runs_converge_like_the_oracle(layout, starts, env):
    """Two window starts per layout run to convergence: the iteration counts of the oracle and
    proportions within 1e-9, read matrix within 1e-8."""
    if layout == "rows":
        env(MXB_EM_NO_PACK="1")
    for mode, level, scale in starts:
        mat, w, lnp, _ = case(layout, mode, level)
        ws = w * scale
        dev = device(layout, mode, level)
        a = make_args(max_iter=60, tolerance=1e-6)
        p, m, info, _ = em.run_em_device(dev, ws, a, inits=lnp.reshape(1, -1))
        o_p, o_m, o_it = oracle_c.run_em(mat, ws, lnp.reshape(1, -1), a.max_iter, a.tolerance)
        assert info["iterations"] == list(o_it), (mode, level, info["iterations"], o_it)
        assert np.abs(p - o_p).max() < 1e-9
        fin = np.isfinite(o_m)
        assert np.array_equal(fin, np.isfinite(m)) and np.abs(m[fin] - o_m[fin]).max() < 1e-8


@pytest.mark.parametrize("exchange", ["p2p", "nccl"])
def test_window_row_shards(exchange):
    """World size 2, row-sharded, from a start at e^-730 (subnormal t): see
    logspace_shards_check.py."""
    if _lib.lib.mxb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ)
    env["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 2) // 2))
    if exchange == "nccl":
        env["MXB_NO_P2P"] = "1"
    else:
        env.pop("MXB_NO_P2P", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29523" if exchange == "p2p" else "29524",
           os.path.join(ROOT, "tests", "logspace_shards_check.py"), "-730"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert res.returncode == 0 and "LOGSPACE_SHARDS_OK" in res.stdout, \
        res.stdout[-2000:] + res.stderr[-4000:]
    assert ("exchange=%s" % exchange) in res.stdout and "level=-730" in res.stdout, \
        res.stdout[-2000:]
