"""The build-kernel cases of build_cases.py land on the limits they are named after, the restated
routing agrees with a plain per-cell walk, and every case can tell a reordered sum from the
reference's (no GPU needed)."""
import numpy as np
import pytest

import build_cases as bc
from oracle import oracle_c


@pytest.mark.parametrize("name", bc.CASE_NAMES)
def test_case_lands_on_its_boundary(name):
    c = bc.case(name)
    lists = bc.DeviationLists(c.tables)
    routes = bc.predict_routes(c.tables, c.csr)
    for i, want in enumerate(c.want):
        st = bc.row_stats(lists, c.csr, i)
        got = dict(K=st["K"], carry=st["carry"], n_dense=st["n_dense"], route=int(routes[i]))
        for key in ("K", "carry", "n_dense", "route"):
            if key in want:
                assert got[key] == want[key], (i, key, got)
        if "items" in want:
            tier_name, w, n = want["items"]
            items = bc.warp_items(st, bc.TIER1 if tier_name == "t1" else bc.TIER2)
            assert items[w] == n, (i, items)
        if "a_of" in want:
            assert list(st["a"][:len(want["a_of"])]) == want["a_of"], (i, st["a"])
        if "first_dev" in want:
            on_warp0 = st["glist"][::bc.TIER1.warps]
            assert st["first"][on_warp0].min() == want["first_dev"], i


def test_cases_cover_every_limit():
    ks, carries, a_vals, items, paths, widths, k_mod8 = set(), set(), set(), set(), set(), set(), set()
    pool_hits = set()
    for c in bc.cases():
        widths.add(c.tables.n_hap)
        routes = bc.predict_routes(c.tables, c.csr)
        paths.update((routes % 4).tolist())
        lists = bc.DeviationLists(c.tables)
        for i, want in enumerate(c.want):
            st = bc.row_stats(lists, c.csr, i)
            ks.add(st["K"])
            carries.add(st["carry"])
            a_vals.update(st["a"].tolist())
            items.update(st["items"].tolist())
            if "items" in want:
                pool_hits.add(want["items"])
            if "first_dev" in want:
                k_mod8.add((want["first_dev"] == st["K"] - 1, st["K"] % 8))
    assert {0, 1, 7, 8, 9, 31, 32, 33, 255, 256, 257, 511, 512, 513, 1024, 1025} <= ks
    assert {1536, 1537, 8064, 8065} <= carries
    assert {1, 2, 5, 6, 31, 32, 33} <= a_vals and 32 in items
    assert {("t1", 0, 146), ("t1", 0, 147), ("t1", 6, 146), ("t1", 6, 147),
            ("t2", 0, 273), ("t2", 0, 274), ("t2", 14, 273), ("t2", 14, 274)} <= pool_hits
    assert {("t1", 0, n) for n in (1, 31, 32, 33, 63, 64, 65, 97)} <= pool_hits
    assert {(True, r) for r in range(1, 8)} <= k_mod8
    assert paths == {0, 1, 2, 3}
    assert {1, 4, 31, 32, 33, 5404, 5406, 5632, 5633, 8191, 8192, 8193, 10241} <= widths


def _per_cell_walk(tables, csr, row, base_ref):
    """Deviating observations per 32-column group, from the expected-symbol table cell by cell:
    a cell deviates when its outcome differs from the outcome most of its plane's cells have."""
    exp = oracle_c.expected_table(tables)
    k0, k1 = int(csr.row_ptr[row]), int(csr.row_ptr[row + 1])
    n_groups = -(-max(tables.n_hap, 1) // 32)
    a = np.zeros(n_groups, dtype=np.int64)
    for k in range(k0, k1):
        p, c = int(csr.pos_idx[k]), int(csr.base_code[k])
        match = (exp[:, p] == c) if c != 255 else np.zeros(tables.n_hap, dtype=bool)
        base = (c == tables.ref_code[p]) if base_ref else 2 * int(match.sum()) > tables.n_hap
        dev = np.zeros(n_groups * 32, dtype=bool)
        dev[:tables.n_hap] = match != base
        a += dev.reshape(n_groups, 32).any(1)
    return a


@pytest.mark.parametrize("base_ref", [False, True])
def test_deviation_counts_equal_a_per_cell_walk(base_ref):
    for c in bc.cases():
        lists = bc.DeviationLists(c.tables, base_ref)
        rows = range(c.csr.n_rows) if c.csr.n_rows <= 8 else range(0, c.csr.n_rows, 7)
        for i in rows:
            st = bc.row_stats(lists, c.csr, i)
            assert np.array_equal(st["a"], _per_cell_walk(c.tables, c.csr, i, base_ref)), (c, i)


def _columns(entries):
    g, d = entries
    bits = np.unpackbits(d.astype("<u4").view(np.uint8).reshape(-1, 4), axis=1, bitorder="little")
    return np.nonzero(bits)[1] + 32 * np.repeat(g, bits.sum(1).astype(np.int64))


def test_majority_baseline_ties_count_as_no_match():
    """'planes': a symbol carried by exactly half of the 64 haplotypes has the baseline "no
    match", so its deviations are its 32 carriers; a derived allele on 40 of them has the
    baseline "match", so its deviations are the 24 others; the "other" plane has none."""
    c = bc.case("planes")
    lists = bc.DeviationLists(c.tables)
    exp = bc.expected(c.tables)
    by_count = {int((exp[:, p] != 0).sum()): p for p in range(c.tables.n_pos)}
    p_half, p_major = by_count[32], by_count[45]
    assert np.array_equal(_columns(lists.entries(lists.plane(p_half, 1))),
                          np.nonzero(exp[:, p_half] == 1)[0])
    assert np.array_equal(_columns(lists.entries(lists.plane(p_half, 0))),
                          np.nonzero(exp[:, p_half] == 0)[0])
    assert np.array_equal(_columns(lists.entries(lists.plane(p_major, 2))),
                          np.nonzero(exp[:, p_major] != 2)[0])
    for code in (4, 255):
        assert lists.entries(lists.plane(p_major, code))[0].size == 0
    ref_lists = bc.DeviationLists(c.tables, base_ref=True)    # marker-free baseline
    assert np.array_equal(_columns(ref_lists.entries(ref_lists.plane(p_major, 2))),
                          np.nonzero(exp[:, p_major] == 2)[0])


def _sorted_order_sums(tables, csr):
    exp = oracle_c.expected_table(tables)
    out = np.zeros((csr.n_rows, tables.n_hap))
    for i in range(csr.n_rows):
        k0, k1 = int(csr.row_ptr[i]), int(csr.row_ptr[i + 1])
        if k1 == k0:
            continue
        p, c = csr.pos_idx[k0:k1], csr.base_code[k0:k1]
        match = (exp[:, p].T == c[:, None]) & (c[:, None] != 255)
        terms = np.where(match, tables.hit[p][:, None], tables.miss[p][:, None])
        out[i] = np.cumsum(np.sort(terms, axis=0), axis=0)[-1]   # sequential, sorted order
    return out


@pytest.mark.parametrize("name", bc.CASE_NAMES)
def test_case_is_order_sensitive(name):
    """Summing each cell's terms in sorted order instead of signature order changes some cells
    of every case, so a kernel that reorders additions cannot pass the bit-exact comparison."""
    c = bc.case(name)
    ref, _ = oracle_c.build_matrix(c.tables, c.csr)
    alt = _sorted_order_sums(c.tables, c.csr)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(alt), fin)
    assert (alt[fin] != ref[fin]).any()
    assert np.abs(alt[fin] - ref[fin]).max() <= 1e-9 * np.abs(ref[fin]).max()
