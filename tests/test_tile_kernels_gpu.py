"""The class-tile kernels (tile_pi_kernel, tile_pass_kernel, tile_gather_kernel, em_finish_kernel
and their slotted variants) at every row width and class layout of tile_cases.CASES, against
k iterations of the reference in long double (tile_cases.ld_iterate), column by column in log
space: |ln pi_dev - ln pi_ref| <= 1e-12 max(1, |ln pi_ref|) on finite entries and the same -inf
pattern.  The starts put columns at 1e-200, 1e-295 and exactly 0, so both branches of the
finish run; a dying column (200 log units below every row's best) crosses the window in which
pi * T underflows while pi does not.  The same matrices run over fp64 rows, two restarts per
pass, and as bootstrap replicates; tiny and ragged row counts; and a matrix with a constructed
hash collision falls back to fp64 rows."""
import ctypes
import os

import numpy as np
import pytest

from mixemt_b200 import _lib, bootstrap, em
from mixemt_b200._lib import check, lib, ptr
from mixemt_b200.runtime import DeviceMatrix, get_context
from oracle import oracle_c
from bootstrap_oracle import boot_counts
from conftest import make_args
from test_tile_plan import ROWS
from tile_cases import (CASES, case_matrix, class_matrix, colliding_column, ld_iterate,
                        ld_read_mix, predicted_pass_bytes)

pytestmark = pytest.mark.gpu

LN_TOL = 1e-12
MIX_TOL = 1e-11
SEED = 91


def assert_ln_close(got, want, tol=LN_TOL):
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.longdouble)
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), \
        np.flatnonzero(np.isneginf(got) != np.isneginf(want))[:10]
    fin = np.isfinite(want)
    assert np.isfinite(got[fin]).all()
    if fin.any():
        err = np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))
        assert float(err.max()) <= tol, (float(err.max()), np.flatnonzero(fin)[np.argmax(err)])


def assert_mix_close(got, want, tol=MIX_TOL):
    want = np.asarray(want, dtype=np.longdouble)
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    assert float(np.abs(got[fin] - want[fin]).max()) <= tol


def start_lnprops(h, seed, dying=None):
    """A Dirichlet draw with columns at 1e-200, 1e-295 and 0 (the dying column at 1e-3)."""
    rs = np.random.RandomState(seed)
    p = rs.dirichlet([1.0] * h)
    cols = rs.permutation(h)
    q = max(1, h // 16)
    p[cols[:q]] = 1e-200
    p[cols[q:2 * q]] = 1e-295
    p[cols[2 * q:3 * q]] = 0.0
    if dying is not None:
        p[dying] = 1e-3
    with np.errstate(divide="ignore"):
        return np.log(p)


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


class Session:
    def __init__(self, dev, w):
        self.dev, self.w = dev, np.ascontiguousarray(w, dtype=np.float64)
        self.h = ctypes.c_void_p()
        check(lib.mxb_em_create(dev.ctx.handle, dev.handle, ptr(self.w), 0, ctypes.byref(self.h)))

    def pass_bytes(self):
        nbytes, layout = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_em_pass_bytes(self.h, ctypes.byref(nbytes), ctypes.byref(layout)))
        return layout.value, nbytes.value

    def iterate(self, lnp, k):
        """k iterations from lnp without a convergence test: (latest, previous, read matrix)."""
        n, h = self.dev.shape
        start = np.ascontiguousarray(lnp, dtype=np.float64)
        check(lib.mxb_em_set_lnprops(self.h, ptr(start)))
        it, cv = ctypes.c_int64(), ctypes.c_int32()
        check(lib.mxb_em_iterate(self.h, k, -1.0, ctypes.byref(it), ctypes.byref(cv)))
        assert (it.value, cv.value) == (k, 0)
        latest, prev = np.empty(h), np.empty(h)
        check(lib.mxb_em_get_lnprops(self.h, 0, ptr(latest)))
        check(lib.mxb_em_get_lnprops(self.h, 1, ptr(prev)))
        mh = ctypes.c_void_p()
        check(lib.mxb_matrix_alloc(self.dev.ctx.handle, n, h, ctypes.byref(mh)))
        mix_dev = DeviceMatrix(self.dev.ctx, mh)
        try:
            check(lib.mxb_em_read_mix(self.h, mix_dev.handle, 0, 0.0))
            mix = mix_dev.to_host()
        finally:
            mix_dev.free()
        return latest, prev, mix

    def close(self):
        lib.mxb_em_destroy(self.h)


def check_session(dev, mat, w, lnp, traj, ks, want_layout, want_bytes=None):
    s = Session(dev, w)
    try:
        layout, nbytes = s.pass_bytes()
        assert layout == want_layout
        if want_bytes is not None:
            assert nbytes == want_bytes
        for k in ks:
            latest, prev, mix = s.iterate(lnp, k)
            assert_ln_close(latest, traj[k])
            assert_ln_close(prev, traj[k - 1])
            assert_mix_close(mix, ld_read_mix(mat, traj[k - 1]))
    finally:
        s.close()


_CACHE = {}


def case_data(case):
    """Matrix, weights, start, long-double trajectory (6 iterations) and device copy."""
    name = case[0]
    if name not in _CACHE:
        mat, w, j_dead, j_dying = case_matrix(case)
        lnp = start_lnprops(mat.shape[1], len(name), j_dying)
        traj = ld_iterate(mat, w, lnp, 6 if j_dying is not None else 3)
        _CACHE[name] = (mat, w, lnp, traj, j_dying, DeviceMatrix.from_host(get_context(), mat))
    return _CACHE[name]


@pytest.fixture(scope="module", autouse=True)
def _free_cache():
    yield
    for v in _CACHE.values():
        v[-1].free()
    _CACHE.clear()


def _ks(j_dying):
    return (1, 3, 6) if j_dying is not None else (1, 3)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_widths_sweep_on_tiles(case):
    """Layout 0 and exactly the pass bytes of the intended classes: the device found them."""
    name, h, n, ncls, *_ = case
    mat, w, lnp, traj, j_dying, dev = case_data(case)
    if h < 1024:      # below the fast path's 1024 columns: the general path (em_update_kernel)
        check_session(dev, mat, w, lnp, traj, _ks(j_dying), -1)
        return
    check_session(dev, mat, w, lnp, traj, _ks(j_dying), 0, predicted_pass_bytes(ncls, n, h))
    if j_dying is not None:
        assert np.isfinite(traj[6][j_dying]) and traj[6][j_dying] < -800.0


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_widths_sweep_on_fp64_rows(case, env):
    """The same matrices over fp64 rows (em_pass_fast_kernel), and two restarts per pass
    (em_pass_pair_kernel) through run_em_device."""
    mat, w, lnp, traj, j_dying, dev = case_data(case)
    env(MXB_EM_NO_PACK="1")
    ks = _ks(j_dying)
    check_session(dev, mat, w, lnp, traj, ks, -1)
    k = ks[-1]
    lnp2 = start_lnprops(mat.shape[1], 7, j_dying)
    traj2 = ld_iterate(mat, w, lnp2, k)
    props, mix, info, _ = em.run_em_device(dev, w, make_args(n_multi=2, max_iter=k, tolerance=0.0),
                                           inits=np.stack([lnp, lnp2]))
    assert info["iterations"] == [k, k]
    want = (traj[k] + traj2[k]) / 2
    live = want > -700.0
    assert_ln_close(np.log(props[live]), want[live])
    assert (props[~live] < 1e-300).all()
    with np.errstate(divide="ignore"):
        want_mix = np.logaddexp(ld_read_mix(mat, traj[k - 1]), ld_read_mix(mat, traj2[k - 1])) \
            - np.log(np.longdouble(2))
    assert_mix_close(mix, want_mix)


@pytest.mark.parametrize("name", ["lg3_to_6", "lg8_to_9", "narrow_wide_narrow"])
def test_slotted_kernels_bootstrap(name):
    """Bootstrap replicates iterate side by side (tile_*_kernel<..., true>); 2R replicates, so
    slots are refilled; each is k iterations of the reference on its counts."""
    case = next(c for c in CASES if c[0] == name)
    mat, w, lnp, _, j_dying, dev = case_data(case)
    wb = np.where(w > 100, 1000.0, w)               # integer weights with a modest total
    k = 3
    a = make_args(max_iter=k, tolerance=0.0)
    _, _, _, slots = bootstrap._run(dev, _lib.as_f64(wb), np.ascontiguousarray(lnp), 0, 1, SEED, a)
    assert slots > 1
    n_boot = 2 * slots
    got, iters, conv, _ = bootstrap._run(dev, _lib.as_f64(wb), np.ascontiguousarray(lnp), 0,
                                         n_boot, SEED, a)
    assert (iters == k).all() and (conv == 0).all()
    for b in (0, slots - 1, slots, n_boot - 1):
        counts = boot_counts(wb, SEED, b).astype(np.float64)
        assert_ln_close(got[b], ld_iterate(mat, counts, lnp, k)[k])


@pytest.mark.parametrize("n", [3, 31, 33, 127, 128, 129, 257])
def test_tiny_and_ragged_rows_on_tiles(n):
    nb = -(-n // ROWS)
    ncls = [4, 6, 5][:nb]
    mat, w, _, j_dying = class_matrix(ncls, 1024, n, "random", n, dead=True, dying=True)
    lnp = start_lnprops(1024, n, j_dying)
    traj = ld_iterate(mat, w, lnp, 6)
    dev = DeviceMatrix.from_host(get_context(), mat)
    try:
        check_session(dev, mat, w, lnp, traj, (1, 6), 0, predicted_pass_bytes(ncls, n, 1024))
    finally:
        dev.free()


@pytest.fixture(scope="module")
def collision():
    """A compressible matrix in which column jb of batch 1 hashes like column ja but differs
    from it in two cells."""
    mat, w, _, _ = class_matrix([5, 7, 6, 4], 1024, 4 * ROWS - 3, "random", 5)
    r0, ja = ROWS, 10
    block = mat[r0:r0 + ROWS]
    jb = next(j for j in range(mat.shape[1]) if not np.array_equal(block[:, j], block[:, ja]))
    mat[r0:r0 + ROWS, jb] = colliding_column(block[:, ja], 1)
    return mat, w, jb


def _layout(dev, w, capfd):
    """Layout of a new session and what its creation printed."""
    capfd.readouterr()
    s = Session(dev, w)
    layout = s.pass_bytes()[0]
    s.close()
    return layout, capfd.readouterr().err


def test_hash_collision_falls_back(collision, env, capfd):
    mat, w, jb = collision
    k = 3
    lnp = start_lnprops(mat.shape[1], 2)
    traj = ld_iterate(mat, w, lnp, k)
    dev = DeviceMatrix.from_host(get_context(), mat)
    try:
        env(MXB_TIMING="1")
        layout, err = _layout(dev, w, capfd)
        assert layout == -1
        assert "[mxb tiles] not used: hash collision" in err
        check_session(dev, mat, w, lnp, traj, (1, k), -1)
        props, mix, info, _ = em.run_em_device(dev, w, make_args(max_iter=k, tolerance=0.0),
                                               inits=lnp.reshape(1, -1))
        o_props, o_mix, o_it = oracle_c.run_em(mat, w, lnp.reshape(1, -1), k, 0.0)
        assert info["iterations"] == list(o_it) == [k]
        assert np.abs(props - o_props).max() < 1e-12
        assert_mix_close(mix, o_mix, 1e-9)
    finally:
        dev.free()
    # one ulp further: no collision, tiles, the same results
    moved = mat.copy()
    moved[ROWS + 1, jb] = np.nextafter(mat[ROWS + 1, jb], 0.0)
    traj_m = ld_iterate(moved, w, lnp, k)
    dev = DeviceMatrix.from_host(get_context(), moved)
    try:
        layout, err = _layout(dev, w, capfd)
        assert layout == 0 and "not used" not in err
        check_session(dev, moved, w, lnp, traj_m, (1, k), 0)
    finally:
        dev.free()


def test_hash_collision_bootstrap_falls_back(collision):
    """A bootstrap session on the colliding matrix keeps fp64 rows (one slot); its replicates
    equal run_em restarts on their counts bit for bit."""
    mat, w, _ = collision
    k = 3
    lnp = start_lnprops(mat.shape[1], 3)
    dev = DeviceMatrix.from_host(get_context(), mat)
    try:
        a = make_args(max_iter=k, tolerance=0.0)
        got, iters, conv, slots = bootstrap._run(dev, _lib.as_f64(w), np.ascontiguousarray(lnp),
                                                 0, 3, SEED, a)
        assert slots == 1 and (iters == k).all()
        counts = bootstrap.boot_counts(w, SEED, 0, 3)
        for b in range(3):
            c = _lib.as_f64(counts[b])
            out = np.zeros(mat.shape[1])
            it, cv = np.zeros(1, dtype=np.int64), np.zeros(1, dtype=np.int32)
            check(lib.mxb_run_em_dev(dev.ctx.handle, dev.handle, ptr(c), ptr(lnp), 1, k, 0.0,
                                     _lib.MXB_EM_RAW, ptr(out), None, None, ptr(it), ptr(cv)))
            assert np.array_equal(got[b], out), b
    finally:
        dev.free()
