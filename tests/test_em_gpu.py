"""Kernel 2 parity: CUDA em_step / run_em (through the C-ABI) against the
reference's own unit tests, its golden outputs and the CPU oracle.

Tolerances (north star): proportions within 1e-6 absolute (asserted much
tighter where the reference result is well conditioned), identical
read-to-haplotype argmax assignments, log responsibilities within 1e-9
absolute wherever they are finite."""
import math

import numpy as np
import pytest

import mixemt_b200
from mixemt_b200 import em, synth
from mixemt_b200.preprocess import HapVarBaseMatrix, build_em_matrix, build_matrix_from_csr
from mixemt_b200.runtime import DeviceMatrix, get_context
from oracle import oracle_c, oracle_np
from conftest import make_args, load_golden

pytestmark = pytest.mark.gpu

PROP_TOL = 1e-6


def close_mix(a, b, tol=1e-9):
    fin = np.isfinite(a) & np.isfinite(b)
    same_inf = np.array_equal(np.isfinite(a), np.isfinite(b)) and \
        np.array_equal(a[~fin], b[~fin])
    return same_inf and (np.abs(a[fin] - b[fin]).max() if fin.any() else 0.0) < tol


# ---- the reference's own tests (mixemt/test/em_test.py) ------------------------
def test_init_props():
    props = em.init_props(10)
    assert len(props) == 10 and abs(props.sum() - 1.0) < 1e-9
    assert np.array_equal(em.init_props(4, float("inf")), np.array([0.25] * 4))


def test_converged():
    prev = np.array([math.log(1.0)] * 10)
    cur = np.array([math.log(2.0)] * 10)
    assert em.converged(cur, cur) and em.converged(prev, prev)
    assert not em.converged(prev, cur) and not em.converged(cur, prev)
    close = np.array(cur)
    close[3] = math.log(2.0001)
    assert em.converged(cur, prev, 20.0)
    assert not em.converged(cur, close)
    assert em.converged(cur, close, 0.001)


@pytest.mark.parametrize("wts,key", [([1, 1, 1], "step_w111"), ([2, 1, 1], "step_w211")])
def test_em_step_simple(wts, key, golden_toy):
    """em_test.py:35-65: identity-like 3 x 3 matrix of 0 / -inf."""
    inf = float("inf")
    in_mat = np.array([[0.0, -inf, -inf], [-inf, 0.0, -inf], [-inf, -inf, 0.0]])
    props = np.log(np.array([0.6, 0.2, 0.2]))
    mix_mat = np.empty_like(in_mat)
    res_mat, res_props = em.em_step(in_mat, np.array(wts), props, mix_mat)
    assert res_mat is mix_mat
    assert np.all(in_mat == mix_mat)
    want = np.log(np.array(wts, dtype=float) / sum(wts))
    # the reference asserts exact equality; device log() is within 1 ulp of libm
    assert np.abs(res_props - want).max() <= 2.3e-16
    assert np.abs(res_props - golden_toy[key + "_props"]).max() <= 2.3e-16
    assert np.array_equal(res_mat, golden_toy[key + "_mix"])


def test_em_step_toy_golden(golden_toy):
    mat = golden_toy["em_mat"]
    mix = np.empty_like(mat)
    res_mat, res_props = em.em_step(mat, np.arange(1, 11), golden_toy["step_toy_start"], mix)
    assert np.abs(res_props - golden_toy["step_toy_props"]).max() < 1e-13
    assert np.abs(res_mat - golden_toy["step_toy_mix"]).max() < 1e-13
    # non-contiguous / wrong-dtype destination is still written in place
    dest = np.zeros((10, 18))[:, ::2]
    out, _ = em.em_step(mat, np.arange(1, 11), golden_toy["step_toy_start"], dest)
    assert out is dest and np.array_equal(dest, res_mat)


@pytest.mark.parametrize("n_multi", [1, 10])
def test_em_runs_recover_truth(n_multi, golden_toy):
    """em_test.py:104-116."""
    mat = golden_toy["em_mat"]
    true_props = np.array([0.0, 0.8, 0.0, 0.0, 0.2, 0.0, 0.0, 0.0, 0.0])
    true_haps = np.full_like(mat, -np.inf)
    true_haps[0:8, 1] = 0.0
    true_haps[8:10, 4] = 0.0
    props, read_mix = em.run_em(mat, np.ones(10), make_args(n_multi=n_multi))
    assert np.allclose(props, true_props, atol=0.02)
    assert np.allclose(np.exp(read_mix), np.exp(true_haps), atol=0.05)


# ---- golden outputs of the reference -----------------------------------------------
@pytest.mark.parametrize("n_multi", [1, 4, 10])
def test_run_em_toy_golden(n_multi, golden_toy):
    mat = golden_toy["em_mat"].copy()
    before = mat.copy()
    np.random.seed(int(golden_toy["run_%d_seed" % n_multi]))
    props, read_mix = em.run_em(mat, np.ones(10), make_args(n_multi=n_multi))
    assert np.array_equal(mat, before)                      # inputs untouched
    assert props.shape == (9,) and read_mix.shape == (10, 9)
    assert np.abs(props - golden_toy["run_%d_props" % n_multi]).max() < 1e-10
    assert close_mix(read_mix, golden_toy["run_%d_mix" % n_multi])
    if n_multi > 1:   # geometric mean of restarts is not renormalised (SURVEY F4)
        assert abs(props.sum() - golden_toy["run_%d_props" % n_multi].sum()) < 1e-12


def test_run_em_iteration_counts(golden_toy, capsys):
    """'Converged! (n)' lines carry the reference's iteration counts."""
    import re
    np.random.seed(int(golden_toy["run_10_seed"]))
    em.run_em(golden_toy["em_mat"], np.ones(10), make_args(n_multi=10, verbose=True))
    err = capsys.readouterr().err
    its = [int(x) for x in re.findall(r"Converged! \((\d+)\)", err)]
    assert its == golden_toy["run_10_iters"].tolist()
    assert err.count("Starting EM run") == 10


def test_run_em_exhausts_max_iter(golden_toy):
    """for/else branch em.py:141-143 + uniform start (alpha = inf)."""
    props, read_mix = em.run_em(golden_toy["em_mat"], np.arange(1, 11),
                                make_args(init_alpha=float("inf"), max_iter=7))
    assert np.abs(props - golden_toy["run_exhaust_props"]).max() < 1e-13
    assert close_mix(read_mix, golden_toy["run_exhaust_mix"], 1e-12)


def _em17_inputs(phylo17, gold, tag):
    haps = sorted(phylo17.hap_var)
    reads = str(gold[tag + "_reads"]).split("\n")
    if tag == "b":
        haps = [haps[j] for j in gold["b_cols"].tolist()]
    mat = build_em_matrix(phylo17.refseq, phylo17, reads, haps, make_args())
    return mat, gold[tag + "_weights"]


def test_run_em_build17_full_width_trajectory(phylo17):
    """192 signatures x 5408 haplotypes, 150 iterations from a seeded Dirichlet
    start, never converging: the whole trajectory must track the reference
    (fast TMA-ring kernel path, H >= 1024)."""
    gold = load_golden("golden_em17.npz")
    mat, wts = _em17_inputs(phylo17, gold, "a")
    assert abs(mat.sum() - gold["a_mat_checksum"][0]) == 0.0
    np.random.seed(int(gold["a_seed"]))
    props, read_mix = em.run_em(mat, wts, make_args(max_iter=int(gold["a_max_iter"]),
                                                    tolerance=float(gold["a_tol"])))
    assert np.abs(props - gold["a_props"]).max() < 1e-12
    assert close_mix(read_mix[:6], gold["a_mix_rows"])
    assert np.array_equal(np.argmax(read_mix, 1), gold["a_argmax"])


@pytest.mark.parametrize("tag,n_multi", [("b1", 1), ("b3", 3)])
def test_run_em_build17_converged(phylo17, tag, n_multi, capsys):
    """600 signatures x 512 haplotypes to convergence (general kernel path):
    same iteration counts, proportions and assignments as the reference."""
    import re
    gold = load_golden("golden_em17.npz")
    mat, wts = _em17_inputs(phylo17, gold, "b")
    np.random.seed(int(gold[tag + "_seed"]))
    props, read_mix = em.run_em(mat, wts, make_args(n_multi=n_multi, max_iter=5000, verbose=True))
    its = [int(x) for x in re.findall(r"Converged! \((\d+)\)", capsys.readouterr().err)]
    assert its == gold[tag + "_iters"].tolist()
    assert np.abs(props - gold[tag + "_props"]).max() < 1e-9 < PROP_TOL
    assert close_mix(read_mix[:6], gold[tag + "_mix_rows"])
    assert np.array_equal(np.argmax(read_mix, 1), gold[tag + "_argmax"])


# ---- against the oracle on seeded inputs ------------------------------------------
def _random_problem(n, h, seed, spread=30.0):
    rs = np.random.RandomState(seed)
    mat = -rs.gamma(2.0, spread / 2.0, size=(n, h))
    mat[rs.rand(n, h) < 0.3] = mat.max()             # ties at the row maximum
    wts = rs.randint(1, 50, size=n)
    inits = np.log(rs.dirichlet([1.0] * h, size=3))
    return mat, wts, inits


@pytest.mark.parametrize("n,h", [(1, 1), (7, 1), (5, 2), (64, 3), (300, 33), (257, 1023),
                                 (100, 1024), (149, 1040), (500, 2049), (311, 5408),
                                 (40, 8192), (33, 9000)])
def test_run_em_vs_oracle_shapes(n, h):
    """Every kernel path (general, TMA ring with NC = 1..8, wider than the ring)
    and ragged shapes: H = 1, H not a multiple of the vector width, N smaller
    than the grid."""
    mat, wts, inits = _random_problem(n, h, seed=n * 7 + h)
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    a = make_args(n_multi=3, max_iter=60, tolerance=1e-7)
    props, read_mix, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    dev.free()
    o_props, o_mix, o_iters = oracle_c.run_em(mat, wts, inits, 60, 1e-7)
    assert info["iterations"] == o_iters
    assert np.abs(props - o_props).max() < 1e-11
    assert close_mix(read_mix, o_mix)


def test_em_step_vs_numpy_oracle():
    mat, wts, inits = _random_problem(50, 1500, seed=1)
    mix = np.empty_like(mat)
    _, new = em.em_step(mat, wts, inits[0], mix)
    o_mix, o_new = oracle_np.em_step(mat, wts, inits[0])
    assert np.abs(new - o_new).max() < 1e-12 and np.abs(mix - o_mix).max() < 1e-11


def test_zero_weights_and_dead_columns():
    """scipy drops zero-weight rows (_logsumexp.py:205-206); an all -inf column
    gets proportion 0 and -inf log responsibilities."""
    mat, wts, inits = _random_problem(40, 1200, seed=5)
    wts = wts.astype(float)
    wts[::3] = 0.0
    mat[:, 7] = -np.inf
    mat[3, :100] = -np.inf
    o_props, o_mix, o_iters = oracle_c.run_em(mat, wts, inits[:1], 40, 1e-9)
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    props, read_mix, info, _ = em.run_em_device(dev, wts, make_args(max_iter=40, tolerance=1e-9),
                                                inits=inits[:1])
    assert props[7] == 0.0 and np.all(np.isneginf(read_mix[:, 7]))
    assert np.abs(props - o_props).max() < 1e-12 and close_mix(read_mix, o_mix)


def test_dying_components_stay_in_log_space():
    """A column that is never the best explanation decays geometrically; after
    thousands of iterations its proportion underflows fp64 but its
    log-proportion must keep tracking the reference (SURVEY section 7)."""
    rs = np.random.RandomState(3)
    n, h = 64, 1100
    mat = np.full((n, h), -40.0)
    mat[np.arange(n), rs.randint(0, 4, size=n)] = 0.0   # four live columns
    mat[:, 10] = -3.0                                    # plausible but dominated
    inits = np.log(np.full((1, h), 1.0 / h))
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    a = make_args(max_iter=4000, tolerance=0.0)
    props, read_mix, info, _ = em.run_em_device(dev, np.ones(n), a, inits=inits)
    o_props, o_mix, _ = oracle_c.run_em(mat, np.ones(n), inits, 4000, 0.0)
    assert np.abs(props - o_props).max() < 1e-12
    fin = np.isfinite(o_mix)
    assert o_mix[fin].min() < -800.0                     # far below exp() underflow
    assert np.allclose(read_mix[fin], o_mix[fin], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("h,layout,gaps", [
    (1100, "rows", (50.0, 200.0, 400.0)),
    (5408, "tiles", (50.0, 200.0, 400.0)),
    (3, "general", (50.0, 200.0)),
    (9000, "general", (50.0, 200.0, 400.0)),
])
def test_fast_dying_components_stay_in_log_space(h, layout, gaps):
    """Columns 50 to 400 log units below every row's best decay so fast that
    pi * T underflows while pi is still above 1e-290: their log-proportions
    must stay finite and track the reference as in
    test_dying_components_stay_in_log_space (em_finish_kernel, em_update_kernel),
    on class tiles, fp64 rows and the general path."""
    import ctypes
    import os
    from mixemt_b200._lib import lib, check, ptr
    rs = np.random.RandomState(3)
    n = 64
    if layout == "tiles":   # blocks of 64 identical columns: class tiles
        mat = np.repeat(np.full((n, h // 64 + 1), -40.0), 64, axis=1)[:, :h].copy()
    else:
        mat = np.full((n, h), -40.0)
    mat[np.arange(n), rs.randint(0, min(4, h), size=n)] = 0.0   # up to four live columns
    dying = np.arange(h - len(gaps), h)
    for j, g in zip(dying, gaps):
        mat[:, j] = -g - rs.uniform(0.0, 5.0, size=n)
    init = np.full(h, 1.0 / h)
    init[dying] = 1e-3
    inits = np.log(init).reshape(1, h)
    max_iter = 40
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    wts = np.ones(n)
    if layout == "rows":     # the matrix compresses: keep fp64 rows on purpose
        os.environ["MXB_EM_NO_PACK"] = "1"
    try:
        sess = ctypes.c_void_p()
        check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
        nbytes, flag = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nbytes), ctypes.byref(flag)))
        lib.mxb_em_destroy(sess)
        assert flag.value == (0 if layout == "tiles" else -1)
        a = make_args(max_iter=max_iter, tolerance=0.0)
        props, read_mix, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    finally:
        os.environ.pop("MXB_EM_NO_PACK", None)
        dev.free()
    o_props, o_mix, _ = oracle_c.run_em(mat, wts, inits, max_iter, 0.0)
    assert np.abs(props - o_props).max() < 1e-12
    fin = np.isfinite(o_mix)
    assert o_mix[fin].min() < -800.0                     # far below exp() underflow
    assert np.allclose(read_mix[fin], o_mix[fin], rtol=1e-9, atol=1e-9)
    assert close_mix(read_mix, o_mix)


# ---- size-independent properties at scale ------------------------------------------
def test_properties_config1_shape(phylo17):
    """Config-1 shape (10k fragments x 5408): proportions sum to 1, the true
    contributors dominate, duplicating rows == doubling weights, and a row
    permutation leaves the proportions unchanged."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 10000, seed=1)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    _, _, dmat, _ = build_matrix_from_csr(tables, mix.csr(tables), want_host=False,
                                          keep_device=True)
    inits = np.log(np.random.RandomState(0).dirichlet([1.0] * len(haps), size=1))
    a = make_args(max_iter=300, tolerance=1e-4)
    props, _, info, mix_dev = em.run_em_device(dmat, mix.weights, a, inits=inits,
                                               keep_device=True, want_host=False)
    assert abs(props.sum() - 1.0) < 1e-9
    votes = np.bincount(mix_dev.argmax_rows(), weights=mix.weights, minlength=len(haps))
    assert {haps[i].split('/')[0][:2] for i in np.argsort(votes)[::-1][:2]} <= {"H1", "L3", "H", "L"}
    host = dmat.to_host()
    perm = np.random.RandomState(1).permutation(host.shape[0])
    d2 = DeviceMatrix.from_host(dmat.ctx, host[perm])
    p2, _, _, _ = em.run_em_device(d2, mix.weights[perm], a, inits=inits, want_host=False)
    assert np.abs(props - p2).max() < 1e-9
    d3 = DeviceMatrix.from_host(dmat.ctx, np.concatenate([host, host[:1000]]))
    w3 = np.concatenate([mix.weights, mix.weights[:1000]])
    w4 = mix.weights.copy()
    w4[:1000] *= 2
    p3, _, _, _ = em.run_em_device(d3, w3, a, inits=inits, want_host=False)
    p4, _, _, _ = em.run_em_device(dmat, w4, a, inits=inits, want_host=False)
    assert np.abs(p3 - p4).max() < 1e-9
    for d in (dmat, d2, d3, mix_dev):
        d.free()


def test_resident_matrix_reuse(phylo17):
    """build_em_matrix(args.b200_resident) hands out a read-only array whose HBM
    copy run_em reuses; results equal the plain host path."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 500, seed=4)
    a = make_args(max_iter=30, tolerance=1e-9, b200_resident=True)
    mat = build_em_matrix(phylo17.refseq, phylo17, mix.signatures, haps, a)
    assert not mat.flags.writeable
    from mixemt_b200.runtime import lookup_resident
    assert lookup_resident(mat) is not None
    np.random.seed(3)
    p1, m1 = em.run_em(mat, mix.weights, a)
    np.random.seed(3)
    p2, m2 = em.run_em(mat.copy(), mix.weights, a)
    assert np.array_equal(p1, p2) and np.array_equal(m1, m2)


def test_install_patches_reference_entry_points():
    import types
    fake = types.SimpleNamespace(preprocess=types.SimpleNamespace(build_em_matrix=None),
                                 em=types.SimpleNamespace(run_em=None, em_step=None))
    mixemt_b200.install(fake)
    assert fake.preprocess.build_em_matrix is mixemt_b200.preprocess.build_em_matrix
    assert fake.em.run_em is mixemt_b200.em.run_em and fake.em.em_step is mixemt_b200.em.em_step


@pytest.mark.parametrize("n_multi", [2, 5])
def test_batched_restarts_equal_sequential(n_multi):
    """run_em with n_multi > 1 iterates two restarts per read of the matrix
    (em_pass_pair_kernel); the results must equal the one-at-a-time path
    (MXB_EM_NO_BATCH=1) and the oracle, restart by restart."""
    import os
    from mixemt_b200.runtime import DeviceMatrix, get_context
    rs = np.random.RandomState(11)
    n, h = 2500, 5408
    mat = -rs.gamma(2.0, 8.0, size=(n, h))
    mat[rs.rand(n, h) < 0.4] = 0.0
    mat[:, :40] += 3.0                                  # a few strong components
    wts = rs.randint(1, 50, size=n)
    inits = np.log(rs.dirichlet([1.0] * h, size=n_multi))
    a = make_args(n_multi=n_multi, max_iter=90, tolerance=3e-3)
    dev = DeviceMatrix.from_host(get_context(), mat)
    p_b, m_b, info_b, _ = em.run_em_device(dev, wts, a, inits=inits)
    os.environ["MXB_EM_NO_BATCH"] = "1"
    try:
        p_s, m_s, info_s, _ = em.run_em_device(dev, wts, a, inits=inits)
    finally:
        del os.environ["MXB_EM_NO_BATCH"]
    assert info_b["iterations"] == info_s["iterations"]
    assert info_b["converged"] == info_s["converged"]
    assert len(set(info_b["iterations"])) > 1 or n_multi == 2   # slots are refilled mid-run
    assert np.abs(p_b - p_s).max() < 1e-13
    assert close_mix(m_b, m_s, 1e-10)
    o_p, o_m, o_it = oracle_c.run_em(mat, wts.astype(np.float64), inits, a.max_iter, a.tolerance)
    assert list(o_it) == info_b["iterations"]
    assert np.abs(p_b - o_p).max() < 1e-10
    assert close_mix(m_b, o_m)


@pytest.mark.parametrize("n_extra,n_multi", [(0, 1), (37, 1), (150, 3)])
def test_class_tiles_equal_fp64_rows(phylo17, n_extra, n_multi):
    """A matrix built from string-sorted signatures runs over class tiles (em_tiles.cuh: per
    128-row batch the bit-identical columns collapse into classes; tile_pi / tile_pass /
    tile_gather kernels).  The same non-negative terms enter every sum, regrouped; results must
    equal the fp64-row pass (MXB_EM_NO_PACK=1) to rounding with identical iteration counts,
    and the oracle.  Noise rows in the middle make batches whose columns are all distinct
    (16 warps per row).  With a few thousand rows over the whole genome nearly every batch is
    wide and the pass's CTAs hold two segments of different widths whose row counts are not
    multiples of the rows handled at a time: the case in which the warps of a wide row must
    agree anew on the buffer of their partial dot products at every batch."""
    import ctypes
    import os
    from mixemt_b200._lib import lib, check, ptr
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)],
                             4000, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    wts = mix.weights.astype(np.float64)
    if n_extra:
        rs = np.random.RandomState(3)
        noise = mat[:n_extra] - rs.gamma(2.0, 1.0, size=(n_extra, mat.shape[1]))
        mat = np.ascontiguousarray(np.vstack([mat[:1500], noise, mat[1500:]]))
        wts = np.concatenate([wts[:1500], rs.randint(1, 9, size=n_extra).astype(np.float64),
                              wts[1500:]])
    n, h = mat.shape
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    # the session reports what its pass reads: tiles, far fewer bytes than the fp64 rows
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
    nbytes, flag = ctypes.c_int64(), ctypes.c_int64()
    check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nbytes), ctypes.byref(flag)))
    lib.mxb_em_destroy(sess)
    assert flag.value == 0 and nbytes.value < 0.5 * n * h * 8

    inits = np.log(np.random.RandomState(1).dirichlet([1.0] * h, size=n_multi))
    a = make_args(max_iter=400, tolerance=1e-5, n_multi=n_multi)
    p_c, m_c, info_c, _ = em.run_em_device(dev, wts, a, inits=inits)
    os.environ["MXB_EM_NO_PACK"] = "1"
    try:
        sess = ctypes.c_void_p()
        check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
        check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nbytes), ctypes.byref(flag)))
        lib.mxb_em_destroy(sess)
        assert flag.value == -1 and nbytes.value == n * ((h + 15) // 16 * 16) * 8
        p_f, m_f, info_f, _ = em.run_em_device(dev, wts, a, inits=inits)
    finally:
        del os.environ["MXB_EM_NO_PACK"]
    assert info_c["iterations"] == info_f["iterations"] and min(info_c["iterations"]) > 20
    assert np.abs(p_c - p_f).max() < 1e-13
    assert close_mix(m_c, m_f, 1e-10)
    o_p, o_m, o_it = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert list(o_it) == info_c["iterations"]
    assert np.abs(p_c - o_p).max() < 1e-10
    assert close_mix(m_c, o_m)


def test_class_tiles_fall_back_on_unsorted_rows(phylo17):
    """Rows in random order share no column classes within a batch: the session keeps the
    fp64 rows (and still equals the oracle)."""
    import ctypes
    from mixemt_b200._lib import lib, check, ptr
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.6), ("L3e", 0.4)], 3000, seed=6)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    perm = np.random.RandomState(2).permutation(mat.shape[0])
    mat, wts = np.ascontiguousarray(mat[perm]), mix.weights[perm].astype(np.float64)
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
    nbytes, flag = ctypes.c_int64(), ctypes.c_int64()
    check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nbytes), ctypes.byref(flag)))
    lib.mxb_em_destroy(sess)
    assert flag.value == -1
    inits = np.log(np.random.RandomState(1).dirichlet([1.0] * mat.shape[1], size=1))
    a = make_args(max_iter=60, tolerance=1e-9)
    p, m, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    o_p, o_m, o_it = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert np.abs(p - o_p).max() < 1e-10 and close_mix(m, o_m)


def test_config1_to_convergence_against_oracle(phylo17):
    """BASELINE.json config 1 (H1 70 % + L3e 30 %, 10 000 fragments x 5408 Build-17
    haplogroups) from a Dirichlet(1) start to convergence at the reference's default
    tolerance: same iteration count as the CPU oracle, proportions within 1e-6 (north star),
    identical argmax votes and identical read-to-contributor assignments
    (assemble.py:267-334 restated in oracle_np)."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 10000, seed=1)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _, dmat, _ = build_matrix_from_csr(tables, mix.csr(tables), keep_device=True)
    wts = mix.weights.astype(np.float64)
    inits = np.log(np.random.RandomState(5).dirichlet([1.0] * len(haps), size=1))
    a = make_args(max_iter=10000, tolerance=1e-4)
    props, read_mix, info, _ = em.run_em_device(dmat, wts, a, inits=inits)
    o_props, o_mix, o_iters = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert info["converged"] == [1] and info["iterations"] == list(o_iters)
    assert info["iterations"][0] > 300
    assert np.abs(props - o_props).max() < PROP_TOL
    assert np.array_equal(np.argmax(read_mix, 1), np.argmax(o_mix, 1))
    top = np.argsort(props)[::-1][:2]
    assert [haps[i] for i in top] == ["H1", "L3e"]
    contribs = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(top.tolist())]
    got = oracle_np.assign_read_indexes(contribs, (props, read_mix), haps, len(wts), 2.0)
    want = oracle_np.assign_read_indexes(contribs, (o_props, o_mix), haps, len(wts), 2.0)
    assert got == want
    from mixemt_b200 import consumers
    dev_assign = consumers.assign_read_indexes(contribs, (props, read_mix), haps,
                                               [[i] for i in range(len(wts))], 2.0)
    assert {k: set(v) for k, v in dev_assign.items()} == want
    dmat.free()


@pytest.mark.parametrize("h,layout", [(1100, "fp64"), (5408, "tiles")])
def test_underflowing_rows_are_redone_in_log_space(h, layout):
    """Rows whose mixture likelihood underflows in linear space (all the remaining mass sits
    on haplotypes ~800 log units worse than the row's best one) used to abort the run with a
    NumericRangeError; the reference's log-space arithmetic (em.py:80-89) stays finite.  The
    flagged iteration is redone in log space on the device and the run continues; results
    equal the oracle."""
    rs = np.random.RandomState(5)
    n = 300 if layout == "fp64" else 1280
    if layout == "fp64":
        mat = -rs.gamma(2.0, 3.0, size=(n, h))
    else:   # column classes: blocks of 64 identical columns -> runs over class tiles
        mat = np.repeat(-rs.gamma(2.0, 3.0, size=(n, h // 64 + 1)), 64, axis=1)[:, :h].copy()
    mat[:, 0] = 0.0
    mat[: n // 4, 1:] -= 800.0          # these rows only make sense under column 0 ...
    init = np.full(h, 1.0)
    init[0] = 1e-300                     # ... which starts with (almost) no mass
    inits = np.log(init / init.sum()).reshape(1, h)
    wts = rs.randint(1, 5, size=n).astype(np.float64)
    a = make_args(max_iter=60, tolerance=1e-6)
    dev = DeviceMatrix.from_host(get_context(), mat)
    props, read_mix, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    o_props, o_mix, o_iters = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert info["iterations"] == list(o_iters)
    assert np.abs(props - o_props).max() < 1e-9
    assert close_mix(read_mix, o_mix, 1e-8)


def test_pinned_result_pool_and_stage_times():
    """Results of the drop-in calls can live in pooled pinned host memory (mxb_host_alloc):
    same values as with pageable results, ordinary writable arrays, blocks reused after the
    arrays die; the stage timer reports where a call spent its time (bench e2e.breakdown_ms)."""
    import ctypes
    import gc
    import os
    from mixemt_b200 import _lib
    from mixemt_b200._lib import lib, check
    rs = np.random.RandomState(2)
    n, h = 4000, 1200
    mat = -rs.gamma(2.0, 5.0, size=(n, h))
    wts = rs.randint(1, 9, size=n)
    a = make_args(max_iter=15, tolerance=1e-9)
    np.random.seed(5)
    p0, m0 = em.run_em(mat, wts, a)
    assert _lib.pinned_mode() == "auto"
    _lib.reserve_pinned(m0.nbytes, 1)
    check(lib.mxb_stage_timing(1))
    np.random.seed(5)
    p1, m1 = em.run_em(mat, wts, a)
    stage = (ctypes.c_double * 6)()
    check(lib.mxb_stage_times(stage, 6))
    check(lib.mxb_stage_timing(0))
    assert np.array_equal(p0, p1) and np.array_equal(m0, m1)
    assert m1.flags.writeable and m1.flags.c_contiguous
    # the pooled block is handed out again once the array is gone
    addr = m1.ctypes.data
    del m1
    gc.collect()
    np.random.seed(5)
    _, m2 = em.run_em(mat, wts, a)
    assert m2.ctypes.data == addr and np.array_equal(m0, m2)
    assert stage[0] > 0 and stage[2] > 0 and stage[4] > 0      # h2d, iterations, d2h
    os.environ["MIXEMT_B200_PINNED"] = "0"
    try:
        np.random.seed(5)
        _, m3 = em.run_em(mat, wts, a)
    finally:
        del os.environ["MIXEMT_B200_PINNED"]
    assert m3.ctypes.data != addr and np.array_equal(m0, m3)
    del m2
    gc.collect()
    _lib.trim_pinned()


@pytest.mark.parametrize("h", [1040, 1500, 3000, 4961, 8000, 8192])
def test_class_tiles_other_widths(h):
    """Class tiles at widths other than Build 17's 5408: the class-sum kernel reads its chunks
    as 4, 8, 12 or 16 entries per thread depending on H, the sort uses as many items; -U gives
    H = 4961.  Columns come in blocks of equal columns of varying width (1..200), rows 300-330
    are noise (every column its own class)."""
    import ctypes
    from mixemt_b200._lib import lib, check, ptr
    rs = np.random.RandomState(h)
    n = 700
    widths = []
    while sum(widths) < h:
        widths.append(int(rs.randint(1, 200)))
    base = -rs.gamma(2.0, 3.0, size=(n, len(widths)))
    mat = np.repeat(base, widths, axis=1)[:, :h].copy()
    mat = mat[:, rs.permutation(h)]                      # classes are not contiguous columns
    mat[300:330] -= rs.gamma(2.0, 1.0, size=(30, h))
    wts = rs.randint(0, 6, size=n).astype(np.float64)   # some zero weights
    ctx = get_context()
    dev = DeviceMatrix.from_host(ctx, mat)
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(wts), 0, ctypes.byref(sess)))
    nbytes, flag = ctypes.c_int64(), ctypes.c_int64()
    check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nbytes), ctypes.byref(flag)))
    lib.mxb_em_destroy(sess)
    assert flag.value == 0, "expected class tiles"
    inits = np.log(rs.dirichlet([1.0] * h, size=1))
    a = make_args(max_iter=80, tolerance=1e-7)
    props, read_mix, info, _ = em.run_em_device(dev, wts, a, inits=inits)
    o_props, o_mix, o_iters = oracle_c.run_em(mat, wts, inits, a.max_iter, a.tolerance)
    assert info["iterations"] == list(o_iters)
    assert np.abs(props - o_props).max() < 1e-10
    assert close_mix(read_mix, o_mix)
