"""Device memory of every allocating entry point is given back, and every allocation failure
is a clean MemoryError.

Leak check: on a fresh context each entry point leaves no live device bytes once the test has
freed what it was handed, and mxb_ctx_trim leaves no cached bytes.  Failure sweep: with
MXB_DEBUG_FAIL_ALLOC=k the k-th device allocation of a fresh context fails; the call either
raises MemoryError or returns exactly what a clean run returns (a session whose class tiles
could not be set up equals a clean MXB_EM_NO_PACK=1 run), leaves no live bytes, and a second
call on the same context equals the clean run bit for bit."""
import ctypes
import os

import numpy as np
import pytest

from mixemt_b200 import _lib, synth
from mixemt_b200._lib import lib, check, ptr
from mixemt_b200.preprocess import HapVarBaseMatrix

c_i64, c_i32, c_f32 = ctypes.c_int64, ctypes.c_int32, ctypes.c_float


def _mem(ctx):
    live, cached = c_i64(), c_i64()
    check(lib.mxb_ctx_mem_stats(ctx.handle, ctypes.byref(live), ctypes.byref(cached)))
    return live.value, cached.value


class _Handles(object):
    """Device handles a case creates, destroyed however the case ends."""

    def __init__(self):
        self.items = []

    def add(self, destroy, handle):
        self.items.append((destroy, handle))
        return handle

    def close(self):
        for destroy, h in reversed(self.items):
            if h.value:
                destroy(h)
        self.items = []


def _upload(ctx, hs, a):
    m = hs.add(lib.mxb_matrix_destroy, ctypes.c_void_p())
    check(lib.mxb_matrix_upload(ctx.handle, ptr(np.ascontiguousarray(a)), a.shape[0], a.shape[1],
                                ctypes.byref(m)))
    return m


def _download(ctx, m, shape):
    out = np.empty(shape)
    check(lib.mxb_matrix_download(ctx.handle, m, ptr(out)))
    return out


# ---- inputs ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def inputs(phylo17):
    rs = np.random.RandomState(11)
    toy = np.log(rs.dirichlet(np.ones(24), size=96))                     # general path
    noise = -rs.gamma(2.0, 3.0, size=(2000, 1100))                       # fp64 rows
    uf = -rs.gamma(2.0, 3.0, size=(300, 1100))                           # underflowing rows
    uf[:, 0] = 0.0
    uf[:75, 1:] -= 800.0
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq,
                             [("H1", 0.4), ("L3e", 0.3), ("U5a1", 0.2), ("M7", 0.1)], 2000,
                             err=0.01, seed=21)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    csr = mix.csr(tables)
    return dict(toy=toy, noise=noise, uf=uf, tables=tables, csr=csr,
                w_toy=rs.randint(1, 4, size=96).astype(np.float64),
                w_noise=rs.randint(1, 5, size=2000).astype(np.float64),
                w_uf=rs.randint(1, 5, size=300).astype(np.float64),
                w_mix=mix.weights.astype(np.float64))


@pytest.fixture(scope="module")
def build17(inputs):
    """The Build-17 mixture's matrix (class tiles)."""
    from mixemt_b200.runtime import Context
    ctx = Context()
    try:
        return _build(ctx, inputs, counts=False)[0]
    finally:
        ctx.close()


def _inits(h, k, seed=3):
    rs = np.random.RandomState(seed)
    return np.ascontiguousarray(np.log(rs.dirichlet(np.ones(h), size=k)))


# ---- cases: fn(ctx, inputs) -> tuple of result arrays; everything created is freed -----------

def _phylo(ctx, hs, t):
    ph = hs.add(lib.mxb_phylo_destroy, ctypes.c_void_p())
    check(lib.mxb_phylo_pack(ctx.handle, t.n_pos, t.n_hap, t.n_sym, ptr(t.hit), ptr(t.miss),
                             ptr(t.ref_code), ptr(t.marker_ptr), ptr(t.marker_pos_idx),
                             ptr(t.marker_code), ctypes.byref(ph)))
    return ph


def _build(ctx, inp, counts=True):
    t, csr = inp["tables"], inp["csr"]
    n = csr.n_rows
    hs = _Handles()
    try:
        ph = _phylo(ctx, hs, t)
        out = np.empty((n, t.n_hap))
        cnt = np.empty((n, t.n_hap), np.int32) if counts else None
        routes = np.empty(n, np.int32)
        dev = hs.add(lib.mxb_matrix_destroy, ctypes.c_void_p())
        ms = c_f32()
        check(lib.mxb_build_matrix(ctx.handle, ph, n, ptr(csr.row_ptr), ptr(csr.pos_idx),
                                   ptr(csr.base_code), ptr(out), ptr(cnt), ptr(routes),
                                   ctypes.byref(dev), ctypes.byref(ms)))
        again = _download(ctx, dev, out.shape)
        assert again.tobytes() == out.tobytes()
        return (out, routes) + ((cnt,) if counts else ())
    finally:
        hs.close()


def case_matrix(ctx, inp):
    hs = _Handles()
    try:
        a = inp["noise"]
        m = _upload(ctx, hs, a)
        b = np.empty((100, a.shape[1]))
        check(lib.mxb_matrix_download_rows(ctx.handle, m, 50, 100, ptr(b)))
        check(lib.mxb_matrix_upload_rows(ctx.handle, m, 0, 100, ptr(b)))
        empty = hs.add(lib.mxb_matrix_destroy, ctypes.c_void_p())
        check(lib.mxb_matrix_alloc(ctx.handle, 0, 7, ctypes.byref(empty)))
        return (_download(ctx, m, a.shape),)
    finally:
        hs.close()


def case_build(ctx, inp):
    return _build(ctx, inp)


def case_build_dense(ctx, inp):
    os.environ["MXB_BUILD_DENSE"] = "1"
    try:
        return _build(ctx, inp)
    finally:
        del os.environ["MXB_BUILD_DENSE"]


def _run_em(ctx, a, w, n_multi, keep=False, inits=None, max_iter=40):
    hs = _Handles()
    try:
        m = _upload(ctx, hs, a)
        n, h = a.shape
        inits = _inits(h, n_multi) if inits is None else inits
        props = np.empty(h)
        mix = None if keep else np.empty((n, h))
        mix_dev = hs.add(lib.mxb_matrix_destroy, ctypes.c_void_p())
        iters = np.empty(n_multi, np.int64)
        conv = np.empty(n_multi, np.int32)
        check(lib.mxb_run_em_dev(ctx.handle, m, ptr(w), ptr(inits), n_multi, max_iter, 1e-6, 0,
                                 ptr(props), ptr(mix), ctypes.byref(mix_dev) if keep else None,
                                 ptr(iters), ptr(conv)))
        if keep:
            mix = _download(ctx, mix_dev, (n, h))
        return props, mix, iters, conv
    finally:
        hs.close()


def case_em_tiles(ctx, inp):
    return _run_em(ctx, inp["build17"], inp["w_mix"], 1)


def case_em_rows(ctx, inp):
    return _run_em(ctx, inp["noise"], inp["w_noise"], 1)


def case_em_row_pairs(ctx, inp):
    return _run_em(ctx, inp["noise"], inp["w_noise"], 2)


def case_em_general(ctx, inp):
    return _run_em(ctx, inp["toy"], inp["w_toy"], 2)


def case_em_keep_device(ctx, inp):
    return _run_em(ctx, inp["noise"], inp["w_noise"], 1, keep=True)


def case_logspace_rescue(ctx, inp):
    h = inp["uf"].shape[1]
    lnp = np.full((1, h), -np.log(h - 1.0))
    lnp[0, 0] = -760.0
    return _run_em(ctx, inp["uf"], inp["w_uf"], 1, inits=lnp)


def case_em_step(ctx, inp):
    a = inp["noise"]
    mix, props = np.empty(a.shape), np.empty(a.shape[1])
    check(lib.mxb_em_step(ctx.handle, ptr(a), ptr(inp["w_noise"]), ptr(_inits(a.shape[1], 1)[0]),
                          a.shape[0], a.shape[1], ptr(mix), ptr(props)))
    return mix, props


def _session(ctx, a, w, range_stop):
    n, h = a.shape
    hs = _Handles()
    try:
        m = _upload(ctx, hs, a)
        em = hs.add(lib.mxb_em_destroy, ctypes.c_void_p())
        check(lib.mxb_em_create(ctx.handle, m, ptr(w), 0, ctypes.byref(em)))
        out = []
        if range_stop:   # a start whose rows underflow: the fixed run stops after its first pass
            lnp = np.full(h, -np.log(h - 1.0))
            lnp[0] = -760.0
            check(lib.mxb_em_set_lnprops(em, ptr(lnp)))
            rc = lib.mxb_em_iterate_fixed(em, 3, None, None)
            if rc != _lib.MXB_ERR_RANGE:
                check(rc)
                raise AssertionError("iterate_fixed did not stop")
        uniform = np.full(h, -np.log(float(h)))
        check(lib.mxb_em_set_lnprops(em, ptr(uniform)))
        check(lib.mxb_em_iterate_fixed(em, 3, None, None))
        got = np.empty(h)
        check(lib.mxb_em_get_lnprops(em, 0, ptr(got)))
        out.append(got)
        ms = (c_f32 * 4)()
        check(lib.mxb_em_set_lnprops(em, ptr(uniform)))
        check(lib.mxb_em_profile(em, 2, ms))
        check(lib.mxb_em_set_lnprops(em, ptr(uniform)))
        iters, conv = c_i64(), c_i32()
        check(lib.mxb_em_iterate(em, 40, 1e-6, ctypes.byref(iters), ctypes.byref(conv)))
        for which in (0, 1):
            got = np.empty(h)
            check(lib.mxb_em_get_lnprops(em, which, ptr(got)))
            out.append(got)
        dst = hs.add(lib.mxb_matrix_destroy, ctypes.c_void_p())
        check(lib.mxb_matrix_alloc(ctx.handle, n, h, ctypes.byref(dst)))
        check(lib.mxb_em_read_mix(em, dst, 0, 0.0))
        out.append(_download(ctx, dst, (n, h)))
        out.append(np.array([iters.value, conv.value]))
        return tuple(out)
    finally:
        hs.close()


def case_session_rows(ctx, inp):
    return _session(ctx, inp["uf"], inp["w_uf"], True)


def case_session_tiles(ctx, inp):
    return _session(ctx, inp["build17"], inp["w_mix"], False)


def _bootstrap(ctx, a, w):
    hs = _Handles()
    try:
        m = _upload(ctx, hs, a)
        h, nb = a.shape[1], 5
        start = np.full(h, -np.log(float(h)))
        lnp = np.empty((nb, h))
        iters, conv = np.empty(nb, np.int64), np.empty(nb, np.int32)
        slots = c_i32()
        check(lib.mxb_em_bootstrap(ctx.handle, m, ptr(w), ptr(start), 0, nb, 7, 30, 1e-6,
                                   ptr(lnp), ptr(iters), ptr(conv), ctypes.byref(slots)))
        return lnp, iters, conv
    finally:
        hs.close()


def case_bootstrap_tiles(ctx, inp):
    return _bootstrap(ctx, inp["build17"], inp["w_mix"])


def case_bootstrap_rows(ctx, inp):
    return _bootstrap(ctx, inp["noise"], inp["w_noise"])


def case_boot_counts(ctx, inp):
    w = inp["w_noise"]
    out = np.empty((3, w.shape[0]), np.uint32)
    check(lib.mxb_boot_counts(ctx.handle, ptr(w), w.shape[0], 5, 2, 3, ptr(out)))
    return (out,)


def case_consumers(ctx, inp):
    a = inp["build17"]
    n, h = a.shape
    hs = _Handles()
    try:
        m = _upload(ctx, hs, a)
        w = np.ascontiguousarray(inp["w_mix"].astype(np.int64))
        cols = np.array([5, 0, h - 1, 17], np.int64)
        g = hs.add(lib.mxb_matrix_destroy, ctypes.c_void_p())
        check(lib.mxb_matrix_gather_cols(ctx.handle, m, ptr(cols), len(cols), ctypes.byref(g)))
        gathered = _download(ctx, g, (n, len(cols)))
        votes, am = np.empty(h, np.int64), np.empty(n, np.int64)
        check(lib.mxb_matrix_vote_count(ctx.handle, m, ptr(w), ptr(votes), ptr(am)))
        votes2, first = np.empty(h, np.int64), np.empty(h, np.int64)
        check(lib.mxb_matrix_vote_first(ctx.handle, m, ptr(w), 10, ptr(votes2), ptr(first)))
        assign = np.empty(n, np.int32)
        ln = np.log(np.array([0.4, 0.3, 0.2, 0.1]))
        check(lib.mxb_assign_reads(ctx.handle, m, ptr(cols), ptr(ln), len(cols), np.log(2.0),
                                   ptr(assign)))
        am2 = np.empty(n, np.int64)
        check(lib.mxb_matrix_argmax_rows(ctx.handle, m, ptr(am2)))
        return gathered, votes, am, votes2, first, assign, am2
    finally:
        hs.close()


def case_fold_ranks(ctx, inp):
    hs = _Handles()
    try:
        a = inp["toy"]
        m = _upload(ctx, hs, a)
        check(lib.mxb_matrix_fold_ranks(ctx.handle, m, np.log(3.0)))
        return (_download(ctx, m, a.shape),)
    finally:
        hs.close()


def case_phylo(ctx, inp):
    hs = _Handles()
    try:
        _phylo(ctx, hs, inp["tables"])
        return ()
    finally:
        hs.close()


CASES = {k[5:]: v for k, v in sorted(globals().items()) if k.startswith("case_")}
COPIES = {"matrix"}            # pure copies: leak check only


def _same(a, b):
    return len(a) == len(b) and all(
        x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()
        for x, y in zip(a, b))


def _fresh(fail_at=None):
    from mixemt_b200.runtime import Context
    if fail_at is not None:
        os.environ["MXB_DEBUG_FAIL_ALLOC"] = str(fail_at)
    try:
        return Context()
    finally:
        os.environ.pop("MXB_DEBUG_FAIL_ALLOC", None)


@pytest.fixture
def inp(inputs, build17):
    return dict(inputs, build17=build17)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_no_device_memory_left_behind(name, inp):
    ctx = _fresh()
    try:
        assert _mem(ctx) == (0, 0)
        CASES[name](ctx, inp)
        live, _ = _mem(ctx)
        assert live == 0, "%s left %d live device bytes" % (name, live)
        check(lib.mxb_ctx_trim(ctx.handle))
        assert _mem(ctx) == (0, 0)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(set(CASES) - COPIES))
def test_every_allocation_failure_is_clean(name, inp):
    fn = CASES[name]
    ctx = _fresh()
    try:
        clean = fn(ctx, inp)
        os.environ["MXB_EM_NO_PACK"] = "1"
        try:
            fp64_rows = fn(ctx, inp)
        finally:
            del os.environ["MXB_EM_NO_PACK"]
    finally:
        ctx.close()
    for k in range(1, 200):
        ctx = _fresh(fail_at=k)
        try:
            try:
                got = fn(ctx, inp)
            except MemoryError:
                got = None
            assert got is None or _same(got, clean) or _same(got, fp64_rows), \
                "%s: allocation %d failed and the result changed" % (name, k)
            assert _mem(ctx)[0] == 0, "%s: allocation %d failed and left live bytes" % (name, k)
            # the call made k - 1 allocations when the next one is number k
            probe = ctypes.c_void_p()
            rc = lib.mxb_matrix_alloc(ctx.handle, 1, 1, ctypes.byref(probe))
            lib.mxb_matrix_destroy(probe)
            if rc == _lib.MXB_ERR_NOMEM:
                assert got is not None and _same(got, clean)
                return
            check(rc)
            assert _same(fn(ctx, inp), clean), "%s: second call after failure %d" % (name, k)
            assert _mem(ctx)[0] == 0
        finally:
            ctx.close()
    raise AssertionError("%s: more than 200 allocations" % name)
