"""What the EM session tests share: the starts with columns at 1e-200, 1e-295 and 0, a thin
wrapper over one mxb_em session (one process, or one rank's row shard of a sharded run), and
the comparisons with the long-double references of tile_cases (ld_iterate, ld_read_mix).
Used by test_tile_kernels_gpu.py, test_row_likelihood_window_gpu.py and multirank_check.py."""
import ctypes

import numpy as np

from mixemt_b200._lib import check, lib, ptr
from mixemt_b200.runtime import DeviceMatrix

LN_TOL = 1e-12
MIX_TOL = 1e-11


def assert_ln_close(got, want, tol=LN_TOL):
    """|ln pi_dev - ln pi_ref| <= tol max(1, |ln pi_ref|) on finite entries and the same -inf
    pattern; returns the worst relative error."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.longdouble)
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), \
        np.flatnonzero(np.isneginf(got) != np.isneginf(want))[:10]
    fin = np.isfinite(want)
    assert np.isfinite(got[fin]).all()
    if not fin.any():
        return 0.0
    err = np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))
    assert float(err.max()) <= tol, (float(err.max()), np.flatnonzero(fin)[np.argmax(err)])
    return float(err.max())


def assert_mix_close(got, want, tol=MIX_TOL):
    """Read matrices: the same -inf pattern, finite cells within tol; returns the worst error."""
    want = np.asarray(want, dtype=np.longdouble)
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    err = float(np.abs(got[fin] - want[fin]).max()) if fin.any() else 0.0
    assert err <= tol, err
    return err


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


class Session:
    """One mxb_em session on `dev` (sharded: this rank's rows of a row-sharded run; every rank
    creates and iterates its session in the same order)."""

    def __init__(self, dev, w, sharded=False):
        self.dev, self.w = dev, np.ascontiguousarray(w, dtype=np.float64)
        self.h = ctypes.c_void_p()
        check(lib.mxb_em_create(dev.ctx.handle, dev.handle, ptr(self.w), int(sharded),
                                ctypes.byref(self.h)))

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
        if n == 0:      # a rank of a row-sharded run without rows
            return latest, prev, np.empty((0, h))
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
