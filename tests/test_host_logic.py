"""Host-side logic that needs no GPU: signature parsing (C), table packing,
the synthetic generator, and the Build-17 fixture."""
import collections

import numpy as np
import pytest

from mixemt_b200 import synth
from mixemt_b200.preprocess import (HapVarBaseMatrix, parse_signatures, pos_from_var, der_allele)
from oracle import oracle_np


def py_pos_obs(sig):
    """What preprocess.pos_obs_from_sig (reference :151-160) returns."""
    out = []
    for var in sig.split(','):
        pos, obs = var.split(':')
        out.append((int(pos), obs))
    return out


def test_variant_string_helpers():
    for var, pos, der in [("A73G", 72, "G"), ("(C16519T)", 16518, "T"), ("T152C!", 151, "C"),
                          ("(T195C!)", 194, "C"), ("G1438a", 1437, "A"), ("C150T!!", 149, "T")]:
        assert pos_from_var(var) == pos and der_allele(var) == der
        assert oracle_np.variant_pos(var) == pos and oracle_np.variant_der(var) == der


def test_markers_match_reference_unit_test(toy_phylo):
    """reference preprocess_test.py:34-53."""
    hvb = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, mut_wt=0.02, mut_max=0.6)
    markers = {'A': {1: 'T', 3: 'T', 0: 'G'},
               'B': {0: 'G', 2: 'T', 4: 'T', 5: 'T', 7: 'T'},
               'C': {0: 'G', 2: 'T', 5: 'T'},
               'D': {0: 'G', 2: 'T', 4: 'T', 6: 'T', 8: 'T'},
               'E': {0: 'G', 2: 'T', 3: 'T', 4: 'T', 6: 'T'},
               'F': {0: 'G', 2: 'T', 4: 'T', 5: 'T'},
               'G': {0: 'G', 2: 'T', 4: 'T', 6: 'T'},
               'H': {0: 'G', 2: 'T', 4: 'T'},
               'I': {0: 'G'}}
    assert hvb.markers == markers
    assert hvb.markers == oracle_np.marker_table(toy_phylo, "AAAAAAAAA")


def test_probs_match_reference_unit_tests(toy_phylo):
    """reference preprocess_test.py:55-79."""
    hvb = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, mut_wt=0.10, mut_max=0.50)
    assert hvb._prob(hvb.markers['I'], 0, 'G') == 1.0 - 0.1
    assert hvb._prob(hvb.markers['I'], 4, 'A') == 1.0 - 0.2
    assert hvb._prob(hvb.markers['I'], 0, 'A') == 0.1 / 3.0
    assert hvb._prob(hvb.markers['I'], 4, 'T') == 0.2 / 3.0


def test_pack_tables(toy_phylo):
    t = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, list("ABCDEFGHI")).pack()
    assert t.positions.tolist() == list(range(9)) and t.n_hap == 9 and t.n_pos == 9
    assert t.symbols == ['A', 'G', 'T']
    assert t.sym2code[ord('A')] == 0 and t.sym2code[ord('T')] == 2 and t.sym2code[ord('C')] == 255
    assert np.array_equal(t.hit[:2], np.log([0.99, 0.99]))      # one mutation each
    assert t.miss[3] == np.log(0.02 / 3.0)                      # A4T occurs twice
    assert int(t.marker_ptr[-1]) == sum(len(m) for m in t.markers.values())


def test_pack_keeps_phylo_counts_as_is(toy_phylo):
    """SURVEY F3: ignore_sites doubles the counts; the tables must follow
    phylo.variants, never recount from the tree."""
    doubled = type(toy_phylo)({p: collections.Counter({b: 2 * c for b, c in cnt.items()})
                               for p, cnt in toy_phylo.variants.items()},
                              toy_phylo.hap_var, toy_phylo.refseq)
    a = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, list("ABC")).pack()
    b = HapVarBaseMatrix("AAAAAAAAA", doubled, list("ABC")).pack()
    assert np.allclose(np.exp(b.miss) * 3, 2 * np.exp(a.miss) * 3)


def test_unknown_haplogroup_is_a_keyerror(toy_phylo):
    with pytest.raises(KeyError):
        HapVarBaseMatrix("AAAAAAAAA", toy_phylo, ["A", "nope"]).pack()


@pytest.mark.parametrize("sig", ["1:A,2:T,3:A", "9:G", " 4 :T,5:AC,6:", "+7:a,1_0:T"])
def test_parse_matches_python(toy_phylo, sig):
    variants = dict(toy_phylo.variants)
    variants[9] = collections.Counter("A")
    variants[10] = collections.Counter("C")
    phylo = type(toy_phylo)(variants, toy_phylo.hap_var, "AAAAAAAAAAAA")
    t = HapVarBaseMatrix("AAAAAAAAAAAA", phylo, list("ABCDEFGHI")).pack()
    csr, err = parse_signatures([sig], t)
    assert err is None
    want = py_pos_obs(sig)
    assert csr.row_ptr.tolist() == [0, len(want)]
    assert [int(t.positions[i]) for i in csr.pos_idx] == [p for p, _ in want]
    for code, (_, obs) in zip(csr.base_code.tolist(), want):
        assert (t.symbols[code] if code != 255 else None) == (obs if obs in t.symbols else None)


@pytest.mark.parametrize("sig", ["", "1A", "1:A:C", "1:A,,2:T", "x:A", "1 2:A", "1:A,", "1__0:A",
                                 "_1:A", "1_:A"])
def test_parse_malformed_is_valueerror_like_python(toy_phylo, sig):
    t = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, list("ABC")).pack()
    with pytest.raises(ValueError):
        py_pos_obs(sig)
    _, err = parse_signatures(["1:A", sig, "77:A"], t)
    assert err == (1, "value", None)


def test_parse_error_order(toy_phylo):
    t = HapVarBaseMatrix("AAAAAAAAA", toy_phylo, list("ABC")).pack()
    assert parse_signatures(["1:A", "77:A", "bad"], t)[1] == (1, "key", 77)
    assert parse_signatures(["1:A", "2:T,-3:A"], t)[1] == (1, "key", -3)
    assert parse_signatures(["1:A", "99999999999:T"], t)[1][:2] == (1, "key")
    # a malformed field later in the same row still wins (whole row is parsed first)
    assert parse_signatures(["77:A,oops"], t)[1] == (0, "value", None)
    many = ["1:A"] * 5000 + ["5:T,66:A"] + ["1:A"] * 5000 + ["zzz"]
    assert parse_signatures(many, t)[1] == (5000, "key", 66)


def test_fixture_has_build17_shape(phylo17, phylo17_cfg5):
    assert len(phylo17.hap_var) == 5408 and len(phylo17.variants) == 4070
    assert len(phylo17.refseq) == 16569
    for hap in ("H1", "L3e", "U5a1", "M7", "D4a"):
        assert hap in phylo17.hap_var
    t = HapVarBaseMatrix(phylo17.refseq, phylo17, sorted(phylo17.hap_var)).pack()
    assert t.symbols == ['A', 'C', 'G', 'T'] and int(t.marker_ptr[-1]) == 263826
    assert len(set(np.round(np.exp(t.miss) * 3, 12))) == 44        # 44 distinct mut_prob
    assert len(phylo17_cfg5.variants) < 4070 and "custom_hap1" in phylo17_cfg5.hap_var


def test_synth_is_deterministic_and_well_formed(phylo17):
    a = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 3000, seed=1)
    b = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.7), ("L3e", 0.3)], 3000, seed=1)
    assert a.signatures == b.signatures and np.array_equal(a.weights, b.weights)
    assert a.signatures == sorted(a.signatures) and len(set(a.signatures)) == a.n_rows
    assert a.weights.sum() <= 3000 and a.weights.min() >= 1
    t = HapVarBaseMatrix(phylo17.refseq, phylo17, ["H1", "L3e"]).pack()
    csr, err = parse_signatures(a.signatures, t)
    direct = a.csr(t)
    assert err is None and np.array_equal(csr.row_ptr, direct.row_ptr)
    assert np.array_equal(csr.pos_idx, direct.pos_idx)
    assert np.array_equal(csr.base_code, direct.base_code)
    k = np.diff(csr.row_ptr)
    assert 10 <= k.min() and k.max() <= 200 and 60 < k.mean() < 100


def test_parse_fuzz_against_python():
    """Random short strings over the characters that matter to ``int()`` and to the two
    splits: the C parser accepts, rejects (ValueError) and reports unknown positions (KeyError)
    exactly where ``pos_obs_from_sig`` + the table lookup would (preprocess.py:151-160, :79-84)."""
    import random
    from mixemt_b200.phylo_tables import PhyloTables
    variants = {p: collections.Counter("A") for p in range(40)}
    phylo = PhyloTables(variants, {"X": ["A1G"]}, "A" * 64)
    t = HapVarBaseMatrix("A" * 64, phylo, ["X"]).pack()
    rnd = random.Random(7)
    alphabet = "0123456789:,_+- \tACGTx\n"
    for _ in range(20000):
        sig = "".join(rnd.choice(alphabet) for _ in range(rnd.randint(0, 12)))
        try:
            want = py_pos_obs(sig)
        except ValueError:
            want = None
        csr, err = parse_signatures([sig], t)
        if want is None:
            assert err is not None and err[1] == "value", sig
            continue
        outside = [p for p, _ in want if not 0 <= p < 40]
        if outside:
            assert err == (0, "key", outside[0]), sig
        else:
            assert err is None, sig
            assert [int(t.positions[i]) for i in csr.pos_idx] == [p for p, _ in want], sig


def test_table_packing_fuzz_against_live_reference():
    """Random small trees with the variant spellings Phylotree has -- '(A73G)', 'T152C!',
    'C150T!!', lower-case derived bases, back mutations onto the reference base, several
    variants of one haplogroup at one position, markers at positions that are not variant
    sites (SURVEY F8), mutation counts past the 0.5 cap -- and signatures with repeated and
    unsorted positions and 'N' observations: the product's host tables (HapVarBaseMatrix.pack,
    parse_signatures) evaluated by the CPU oracle give the reference's build_em_matrix
    (preprocess.py:177-198) bit for bit.  The reference's matrices are stored in
    tests/golden/golden_live.npz (oracle/live_cases.py); where the reference is installed,
    they are checked against it too."""
    import argparse
    from oracle import live_cases, oracle_c, refload
    g = live_cases.load_golden()
    ref_pre = refload.load()[1] if refload.available() else None
    off = 0
    for it, (refseq, phylo, haps, reads) in enumerate(live_cases.packing_cases()):
        want = g["pack_mats"][off:off + len(reads) * len(haps)].reshape(len(reads), len(haps))
        off += want.size
        if ref_pre is not None:
            live = ref_pre.build_em_matrix(refseq, phylo, reads, haps, argparse.Namespace(verbose=False))
            assert np.array_equal(live, want), it
        tables = HapVarBaseMatrix(refseq, phylo, haps).pack()
        csr, err = parse_signatures(reads, tables)
        assert err is None
        got, counts = oracle_c.build_matrix(tables, csr)
        assert np.array_equal(got, want), it
        assert (counts >= 0).all() and (counts <= np.diff(csr.row_ptr)[:, None]).all()
    assert off == g["pack_mats"].size


@pytest.mark.parametrize("exotic", [None, "A0G", "A3é"])
def test_marker_csr_both_packing_paths(toy_phylo, exotic):
    """pack() flattens the marker tables with numpy; a table with a negative position ('A0G')
    or a non-ASCII derived base takes the per-entry loop.  Both must give the CSR a plain
    Python walk over ``markers`` gives."""
    import types
    hap_var = {h: list(v) for h, v in toy_phylo.hap_var.items()}
    if exotic:
        hap_var[sorted(hap_var)[1]].append(exotic)
    phylo = types.SimpleNamespace(variants=toy_phylo.variants, hap_var=hap_var,
                                  refseq=toy_phylo.refseq)
    haps = sorted(hap_var)
    t = HapVarBaseMatrix(toy_phylo.refseq, phylo, haps).pack()
    pos_index = {int(p): i for i, p in enumerate(t.positions)}
    ptr, pos, code = [0], [], []
    for hap in haps:
        for p, der in t.markers[hap].items():
            if p in pos_index:
                pos.append(pos_index[p])
                code.append(t.symbols.index(der))
        ptr.append(len(pos))
    assert t.marker_ptr.tolist() == ptr and t.marker_ptr.dtype == np.int64
    assert t.marker_pos_idx.tolist() == pos and t.marker_pos_idx.dtype == np.int32
    assert t.marker_code.tolist() == code and t.marker_code.dtype == np.uint8
