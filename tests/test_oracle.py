"""Pins the CPU oracle (oracle/oracle_np.py, oracle/oracle.c) to the
reference: against the golden vectors the unmodified reference produced
(oracle/make_golden.py, oracle/live_cases.py), and against the live reference
where it is installed."""
import numpy as np
import pytest

from mixemt_b200.preprocess import HapVarBaseMatrix, parse_signatures
from oracle import live_cases, oracle_c, oracle_np, refload
from conftest import load_golden, make_args


def seeded_inits(seed, n_multi, h):
    np.random.seed(seed)
    return np.array([np.log(np.random.dirichlet([1.0] * h)) for _ in range(n_multi)])


def test_build_toy_golden(toy_phylo, golden_toy):
    haps = list("ABCDEFGHI")
    for key, mat_key in (("build_reads", "build_mat"), ("em_reads", "em_mat")):
        reads = str(golden_toy[key]).split("\n")
        for fn in (oracle_np.build_matrix_loops, oracle_np.build_matrix_fast):
            mat, _ = fn("AAAAAAAAA", toy_phylo, reads, haps)
            assert np.array_equal(mat, golden_toy[mat_key])
        t = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, haps).pack()
        csr, _ = parse_signatures(reads, t)
        mat, cnt = oracle_c.build_matrix(t, csr)
        assert np.array_equal(mat, golden_toy[mat_key])
        assert np.array_equal(cnt, oracle_np.build_matrix_loops("AAAAAAAAA", toy_phylo, reads, haps)[1])


@pytest.mark.parametrize("fixture,gold", [("phylo17", "golden_build17.npz"),
                                          ("phylo17_cfg5", "golden_build17_cfg5.npz")])
def test_build17_golden(fixture, gold, request):
    phylo = request.getfixturevalue(fixture)
    g = load_golden(gold)
    reads = str(g["reads"]).split("\n")
    haps = sorted(phylo.hap_var)
    t = HapVarBaseMatrix(phylo.refseq, phylo, haps).pack()
    csr, err = parse_signatures(reads, t)
    assert err is None
    mat, cnt = oracle_c.build_matrix(t, csr)
    assert np.array_equal(mat, g["mat"])                        # bit-exact
    rows = [0, len(reads) - 2, len(reads) - 1]                  # incl. the odd-base rows
    py, py_cnt = oracle_np.build_matrix_fast(phylo.refseq, phylo, [reads[i] for i in rows], haps)
    assert np.array_equal(py, g["mat"][rows]) and np.array_equal(py_cnt, cnt[rows])


def test_em_step_golden(golden_toy):
    inf = float("inf")
    in_mat = np.array([[0.0, -inf, -inf], [-inf, 0.0, -inf], [-inf, -inf, 0.0]])
    start = np.log(np.array([0.6, 0.2, 0.2]))
    for key, wts in (("step_w111", [1, 1, 1]), ("step_w211", [2, 1, 1])):
        mix, new = oracle_np.em_step(in_mat, np.array(wts), start)
        assert np.array_equal(mix, golden_toy[key + "_mix"])
        assert np.array_equal(new, golden_toy[key + "_props"])   # exact, like em_test.py:48
        mix, new = oracle_c.em_step(in_mat, np.array(wts, dtype=float), start)
        assert np.array_equal(mix, golden_toy[key + "_mix"])
        assert np.abs(new - golden_toy[key + "_props"]).max() < 3e-16
    mat = golden_toy["em_mat"]
    for impl, tol in ((oracle_np, 0.0), (oracle_c, 1e-13)):
        mix, new = impl.em_step(mat, np.arange(1, 11).astype(float), golden_toy["step_toy_start"])
        assert np.abs(new - golden_toy["step_toy_props"]).max() <= tol
        assert np.abs(mix - golden_toy["step_toy_mix"]).max() <= tol
    mix2, new2 = oracle_np.em_step_scipy(mat, np.arange(1, 11), golden_toy["step_toy_start"],
                                         np.empty_like(mat))
    assert np.array_equal(new2, golden_toy["step_toy_props"])


@pytest.mark.parametrize("n_multi", [1, 4, 10])
def test_run_em_toy_golden(n_multi, golden_toy):
    mat = golden_toy["em_mat"]
    inits = seeded_inits(int(golden_toy["run_%d_seed" % n_multi]), n_multi, 9)
    for impl, tol in ((oracle_np, 1e-15), (oracle_c, 1e-12)):
        props, mix, iters = impl.run_em(mat, np.ones(10), inits, 1000, 1e-4)
        assert list(iters) == golden_toy["run_%d_iters" % n_multi].tolist()
        assert np.abs(props - golden_toy["run_%d_props" % n_multi]).max() <= tol
        assert np.abs(mix - golden_toy["run_%d_mix" % n_multi]).max() <= max(tol, 1e-15) * 1e3


def test_run_em_exhaust_golden(golden_toy):
    inits = np.log(np.full((1, 9), 1.0 / 9))
    for impl in (oracle_np, oracle_c):
        props, mix, iters = impl.run_em(golden_toy["em_mat"], np.arange(1, 11).astype(float),
                                        inits, 7, 1e-4)
        assert list(iters) == [7]
        assert np.abs(props - golden_toy["run_exhaust_props"]).max() < 1e-14
        assert np.abs(mix - golden_toy["run_exhaust_mix"]).max() < 1e-12


def test_run_em_build17_golden(phylo17):
    """Build-17 sub-problem (600 x 512) to convergence: the C oracle reproduces
    the reference's iteration counts, proportions and assignments."""
    g = load_golden("golden_em17.npz")
    haps = sorted(phylo17.hap_var)
    haps_b = [haps[j] for j in g["b_cols"].tolist()]
    reads = str(g["b_reads"]).split("\n")
    t = HapVarBaseMatrix(phylo17.refseq, phylo17, haps_b).pack()
    csr, _ = parse_signatures(reads, t)
    mat, _ = oracle_c.build_matrix(t, csr, want_counts=False)
    for tag, n_multi in (("b1", 1), ("b3", 3)):
        inits = seeded_inits(int(g[tag + "_seed"]), n_multi, len(haps_b))
        props, mix, iters = oracle_c.run_em(mat, g["b_weights"], inits, 5000, 1e-4)
        assert list(iters) == g[tag + "_iters"].tolist()
        assert np.abs(props - g[tag + "_props"]).max() < 1e-10
        assert np.abs(mix[:6] - g[tag + "_mix_rows"]).max() < 1e-9
        assert np.array_equal(np.argmax(mix, 1), g[tag + "_argmax"])


def test_against_live_reference(phylo17):
    """The oracles against the reference's build_em_matrix and run_em on 12 Build-17 reads
    (tests/golden/golden_live.npz, oracle/live_cases.py); where the reference is installed,
    the stored outputs against the reference itself."""
    g = live_cases.load_golden()
    haps = sorted(phylo17.hap_var)
    reads, wts = str(g["b17_reads"]).split("\n"), g["b17_weights"]
    want = g["b17_mat"]
    if refload.available():
        _, ref_pre, ref_em = refload.load()
        assert (reads, wts.tolist()) == tuple(map(list, live_cases.build17_reads(phylo17)))
        assert np.array_equal(ref_pre.build_em_matrix(phylo17.refseq, phylo17, reads, haps,
                                                      make_args()), want)
    t = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    csr, _ = parse_signatures(reads, t)
    assert np.array_equal(oracle_c.build_matrix(t, csr)[0], want)
    sub = live_cases.build17_sub(want)
    seed, n_multi, max_iter = (live_cases.RUN_EM_SEED, live_cases.RUN_EM_MULTI,
                               live_cases.RUN_EM_MAX_ITER)
    p_ref, m_ref = g["b17_props"], g["b17_mix"]
    if refload.available():
        np.random.seed(seed)
        p_live, m_live = ref_em.run_em(sub, wts, make_args(n_multi=n_multi, max_iter=max_iter))
        assert np.array_equal(p_live, p_ref) and np.array_equal(m_live, m_ref)
    inits = seeded_inits(seed, n_multi, sub.shape[1])
    p_np, m_np, _ = oracle_np.run_em(sub, wts, inits, max_iter, 1e-4)
    p_c, m_c, _ = oracle_c.run_em(sub, wts, inits, max_iter, 1e-4)
    assert np.array_equal(p_np, p_ref) and np.array_equal(m_np, m_ref)
    assert np.abs(p_c - p_ref).max() < 1e-13 and np.abs(m_c - m_ref).max() < 1e-10


# ---- consumers of the EM result (SURVEY.md 8f N2/N3) ---------------------------
@pytest.mark.parametrize("seed", [71, 72])
def test_consumers_golden(seed):
    g = load_golden("golden_consumers.npz")
    props, mix, wts = oracle_np.synthetic_em_result(seed)
    haps = ["hg%d" % j for j in range(mix.shape[1])]
    for min_reads in (1, 60, 400):
        got = oracle_np.find_contribs_from_reads(mix, wts, min_reads)
        assert got == g["s%d_contribs_r%d" % (seed, min_reads)].tolist()
    top = g["s%d_top" % seed].tolist()
    contribs = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(top)]
    for tag, fold, cons in (("f2", 2.0, contribs), ("f1p2", 1.2, contribs[:2]),
                            ("single", 2.0, contribs[:1])):
        res = oracle_np.assign_read_indexes(cons, (props, mix), haps, len(mix), fold)
        assert np.array_equal(live_cases.decode_assign(res, len(mix)), g["s%d_assign_%s" % (seed, tag)])
    red, new_haps = oracle_np.reduce_em_matrix(mix, haps, contribs)
    assert np.array_equal(red, g["s%d_reduced" % seed])
    assert [haps.index(x) for x in new_haps] == g["s%d_reduced_cols" % seed].tolist()


def test_consumers_live_reference():
    """The consumers' restatements against the reference's assemble / reduce_em_matrix on a
    150 x 40 stand-in (tests/golden/golden_live.npz); where the reference is installed, the
    stored outputs against the reference itself."""
    g = live_cases.load_golden()
    props, mix, wts, haps, contribs = live_cases.consumers_case()
    n, min_reads, fold = len(mix), live_cases.CONSUMERS_MIN_READS, live_cases.CONSUMERS_FOLD
    want_red, want_cols = g["c_reduced"], [haps[j] for j in g["c_reduced_cols"].tolist()]
    if refload.available():
        refload.load()
        from mixemt import assemble, preprocess as ref_pre
        assert assemble._find_contribs_from_reads(mix, wts, make_args(min_reads=min_reads)) == \
            g["c_contribs"].tolist()
        ref = assemble.assign_read_indexes(contribs, (props, mix), haps, list(range(n)), fold)
        assert np.array_equal(live_cases.decode_assign(ref, n), g["c_assign"])
        a = ref_pre.reduce_em_matrix(mix, haps, contribs)
        assert np.array_equal(a[0], want_red) and a[1] == want_cols
    assert oracle_np.find_contribs_from_reads(mix, wts, min_reads) == g["c_contribs"].tolist()
    got = oracle_np.assign_read_indexes(contribs, (props, mix), haps, n, fold)
    assert np.array_equal(live_cases.decode_assign(got, n), g["c_assign"])
    b = oracle_np.reduce_em_matrix(mix, haps, contribs)
    assert np.array_equal(b[0], want_red) and b[1] == want_cols


def test_em_step_fuzz_against_live_reference():
    """The oracles' em_step against the reference's own (em.py:57-91, scipy logsumexp) on small
    random inputs with the edge values the domain has: -inf cells, ties among the row and
    column maxima, a row that fits no haplotype (NaN, like the reference), zero weights,
    components with zero proportion.  numpy restatement: bit-identical, NaN for NaN; C port:
    the same non-finite pattern and within 1e-12.  The reference's outputs are stored in
    tests/golden/golden_live.npz; where the reference is installed, they are checked against
    it too."""
    import warnings
    g = live_cases.load_golden()
    ref_em = refload.load()[2] if refload.available() else None
    zo = po = 0
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        for it, (mat, wts, lp) in enumerate(live_cases.em_step_cases()):
            n, h = mat.shape
            z_ref = g["step_z"][zo:zo + n * h].reshape(n, h)
            p_ref = g["step_p"][po:po + h]
            zo, po = zo + n * h, po + h
            if ref_em is not None:
                z_live, p_live = ref_em.em_step(mat, wts, lp, np.empty_like(mat))
                assert np.array_equal(z_live, z_ref, equal_nan=True), it
                assert np.array_equal(p_live, p_ref, equal_nan=True), it
            z_np, p_np = oracle_np.em_step(mat, wts, lp)
            assert np.array_equal(z_np, z_ref, equal_nan=True), it
            assert np.array_equal(p_np, p_ref, equal_nan=True), it
            z_c, p_c = oracle_c.em_step(mat, wts.astype(np.float64), lp)
            for got, want in ((z_c, z_ref), (p_c, p_ref)):
                fin = np.isfinite(want)
                assert np.array_equal(got[~fin], want[~fin], equal_nan=True), it
                assert not fin.any() or np.abs(got[fin] - want[fin]).max() < 1e-12, it
    assert (zo, po) == (g["step_z"].size, g["step_p"].size)
