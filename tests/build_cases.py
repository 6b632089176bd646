"""Packed tables and signature rows that sit on the routing limits of the matrix-build kernel
(csrc/build.cu), and a restatement of that routing, for tests/test_build_cases.py (CPU) and
tests/test_build_kernels_gpu.py.

The class kernel finishes a row in tier 1 when it has at most 256 observations, at most 1536
deviation entries and at most 146 chain items on every work warp; tier 2 takes what is left up to
512 observations, 8064 entries and 273 items per warp, and build_dense_row the rest.  A 32-column
group with more than 32 deviating observations is walked by the per-group dense loop; up to five
take the straight-line pattern code, one takes no cross-lane work at all.  Tables wider than 8192
columns go to build_matrix_dense_kernel.  predict_routes restates all of this from the packed
tables (the majority-baseline deviation lists of mxb_phylo_pack) and gives the code that
mxb_build_matrix reports per row: path + 4 * dense groups.

The tables are built from an expected-symbol matrix exp[H, P] (haplotype j expects symbol
exp[j, p] at position p) and the rows directly as a CSR, so K and every observation are exact.
hit / miss are drawn log-uniformly over twelve orders of magnitude (a few are -inf), so any change
in the order of a cell's additions changes its last bits."""
import copy

import numpy as np

from mixemt_b200.preprocess import HapVarBaseMatrix, SignatureCSR

N_SYM = 4                      # symbol codes 0..3; codes >= N_SYM (4, 255) use the all-zero plane


class Tier(object):
    """Pool sizes of one launch of build_matrix_kernel (build.cu: Tier1, Tier2)."""

    def __init__(self, path, threads, entries, items, obs_words):
        self.path = path
        self.obs = obs_words * 32
        self.entries = entries
        self.warps = threads // 32 - 1            # the last warp runs the prefix chain
        self.pool = (items - 1) // self.warps     # item 0 is the baseline class


TIER1 = Tier(0, 256, 1536, 1024, 8)
TIER2 = Tier(1, 512, 8064, 4096, 16)
assert (TIER1.pool, TIER1.warps, TIER2.pool, TIER2.warps) == (146, 7, 273, 15)
MAX_CLASS_HAP = 256 * 32       # kGroupsLarge: wider tables take build_matrix_dense_kernel
DENSE_ROW, DENSE_KERNEL = 2, 3
MAX_CLASS_A = 32               # a group with more deviating observations is walked densely


# ---- tables ------------------------------------------------------------------------------------
def make_tables(exp, ref_code, hit, miss, n_sym=N_SYM):
    """A HapVarBaseMatrix holding just the fields that to_device (mxb_phylo_pack) and
    oracle_c.build_matrix read: markers are the cells of exp that differ from ref_code."""
    exp = np.ascontiguousarray(exp, dtype=np.uint8)
    n_hap, n_pos = exp.shape
    t = HapVarBaseMatrix.__new__(HapVarBaseMatrix)
    t._device = None
    t.n_hap, t.n_pos, t.n_sym = n_hap, n_pos, n_sym
    t.hit = np.ascontiguousarray(hit, dtype=np.float64)
    t.miss = np.ascontiguousarray(miss, dtype=np.float64)
    t.ref_code = np.ascontiguousarray(ref_code, dtype=np.uint8)
    hap, pos = np.nonzero(exp != t.ref_code[None, :])
    t.marker_ptr = np.zeros(n_hap + 1, dtype=np.int64)
    np.cumsum(np.bincount(hap, minlength=n_hap), out=t.marker_ptr[1:])
    t.marker_pos_idx = pos.astype(np.int32)
    t.marker_code = np.ascontiguousarray(exp[hap, pos])
    return t


def repacked(tables):
    """The same tables, packed again by the next to_device (which reads MXB_BUILD_BASE_REF)."""
    t = copy.copy(tables)
    t._device = None
    return t


def expected(tables):
    """exp[H, P] from the marker CSR (what oracle_c.expected_table gives)."""
    exp = np.tile(tables.ref_code, (tables.n_hap, 1))
    hap = np.repeat(np.arange(tables.n_hap), np.diff(tables.marker_ptr))
    exp[hap, tables.marker_pos_idx] = tables.marker_code
    return exp


# ---- the routing, restated -------------------------------------------------------------------
class DeviationLists(object):
    """Sparse deviation lists of mxb_phylo_pack, one plane at a time: the plane's bitset is the
    reference plane with every marker moved to its own symbol's plane; the baseline outcome is
    "match" when more than half of the haplotypes match (a tie is "no match"), or, with base_ref
    (MXB_BUILD_BASE_REF), when the symbol is the reference's; the entries are the non-zero words
    of bits XOR baseline, past-the-end columns masked off."""

    def __init__(self, tables, base_ref=False):
        self.t = tables
        self.base_ref = base_ref
        self.n_planes = tables.n_sym + 1
        self.n_groups = -(-max(tables.n_hap, 1) // 32)
        hap = np.repeat(np.arange(tables.n_hap), np.diff(tables.marker_ptr))
        order = np.argsort(tables.marker_pos_idx, kind="stable")
        self._m_hap = hap[order]
        self._m_code = tables.marker_code[order]
        self._m_ptr = np.searchsorted(tables.marker_pos_idx[order], np.arange(tables.n_pos + 1))
        self._cache = {}

    def plane(self, p, c):
        return p * self.n_planes + min(int(c), self.n_planes - 1)

    def entries(self, plane):
        """(group indexes ascending, D words) of one plane."""
        hit = self._cache.get(plane)
        if hit is not None:
            return hit
        t = self.t
        p, a = divmod(plane, self.n_planes)
        match = np.zeros(self.n_groups * 32, dtype=bool)
        if a < t.n_sym:
            if a == t.ref_code[p]:
                match[:t.n_hap] = True
            lo, hi = self._m_ptr[p], self._m_ptr[p + 1]
            match[self._m_hap[lo:hi]] = self._m_code[lo:hi] == a
        base = (a == t.ref_code[p]) if self.base_ref else 2 * int(match.sum()) > t.n_hap
        dev = match.copy()
        if base:
            dev[:t.n_hap] = ~dev[:t.n_hap]
        words = np.packbits(dev.reshape(-1, 32), axis=1, bitorder="little").view("<u4")[:, 0]
        g = np.nonzero(words)[0]
        self._cache[plane] = hit = (g, words[g].astype(np.uint32))
        return hit


def row_stats(lists, csr, row):
    """What the class kernel works out for one row (phases 1 and 2 of build_matrix_kernel):
    K, a[g] (deviating observations per group), carry (their sum = the entry count), the
    non-empty groups in ascending order (dense ones keep their list slot), items[g] (distinct
    non-zero lane patterns of a group with a <= 32, 0 for a dense group), first[g] (the group's
    first deviating observation, -1 if none) and the number of dense groups."""
    k0, k1 = int(csr.row_ptr[row]), int(csr.row_ptr[row + 1])
    n_groups = lists.n_groups
    ent_k, ent_g, ent_d = [], [], []
    for k in range(k1 - k0):
        g, d = lists.entries(lists.plane(int(csr.pos_idx[k0 + k]), csr.base_code[k0 + k]))
        ent_k.append(np.full(len(g), k))
        ent_g.append(g)
        ent_d.append(d)
    cat = (lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt))
    ent_k, ent_g, ent_d = cat(ent_k, np.int64), cat(ent_g, np.int64), cat(ent_d, np.uint64)
    a = np.bincount(ent_g, minlength=n_groups)
    order = np.lexsort((ent_k, ent_g))          # by group, then by observation
    ent_k, ent_g, ent_d = ent_k[order], ent_g[order], ent_d[order]
    start = np.concatenate(([0], np.cumsum(a)))
    e = np.arange(len(ent_g)) - start[ent_g]    # rank of k among the group's deviating k
    first = np.full(n_groups, -1)
    first[ent_g[e == 0]] = ent_k[e == 0]
    cls = a[ent_g] <= MAX_CLASS_A
    lanes = np.arange(32, dtype=np.uint64)
    bits = ((ent_d[cls, None] >> lanes) & np.uint64(1)) << e[cls, None].astype(np.uint64)
    pat = np.zeros((n_groups, 32), dtype=np.uint64)
    np.add.at(pat, ent_g[cls], bits)
    s = np.sort(pat, axis=1)
    items = (s[:, 1:] != s[:, :-1]).sum(1) + 1 - (s[:, 0] == 0)
    items[a > MAX_CLASS_A] = 0
    glist = np.nonzero(a)[0]
    return dict(K=k1 - k0, a=a, carry=int(a.sum()), glist=glist, items=items, first=first,
                n_dense=int((a > MAX_CLASS_A).sum()))


def warp_items(st, tier):
    """Chain items per work warp: list slot gi goes to warp gi mod tier.warps."""
    slot = np.arange(len(st["glist"])) % tier.warps
    return np.bincount(slot, weights=st["items"][st["glist"]], minlength=tier.warps).astype(int)


def tier_route(st, tier):
    """Route code when the tier finishes the row, None when it passes the row on."""
    if st["K"] > tier.obs or st["carry"] > tier.entries or warp_items(st, tier).max() > tier.pool:
        return None
    return tier.path + 4 * st["n_dense"]


def predict_routes(tables, csr, two_tiers=True, base_ref=False):
    """The route code mxb_build_matrix reports for every row (two_tiers=False: MXB_BUILD_TIERS=2;
    base_ref: tables packed with MXB_BUILD_BASE_REF)."""
    n = csr.n_rows
    if tables.n_hap > MAX_CLASS_HAP:
        return np.full(n, DENSE_KERNEL, dtype=np.int32)
    lists = DeviationLists(tables, base_ref)
    out = np.empty(n, dtype=np.int32)
    for row in range(n):
        st = row_stats(lists, csr, row)
        r = tier_route(st, TIER1) if two_tiers else None
        if r is None:
            r = tier_route(st, TIER2)
        out[row] = DENSE_ROW if r is None else r
    return out


# ---- case builder ------------------------------------------------------------------------------
class Case(object):
    def __init__(self, name, tables, csr, want):
        self.name, self.tables, self.csr, self.want = name, tables, csr, want

    def __repr__(self):
        return "Case(%s: H=%d, %d rows)" % (self.name, self.tables.n_hap, self.csr.n_rows)


def group_entries(ks, n_items, rs, lanes=32):
    """Entries (k, lane mask) of one group whose deviating observations are ks (ascending) and
    whose lanes show exactly n_items distinct non-zero patterns: lanes picked at random get the
    patterns 1..n_items, the others keep the baseline, and the lane of the largest pattern also
    deviates at every observation past its bits, so that every observation has a deviating lane."""
    a = len(ks)
    bl = n_items.bit_length()
    assert list(ks) == sorted(set(ks)) and 1 <= n_items <= lanes and bl <= a, (ks, n_items)
    chosen = rs.permutation(lanes)[:n_items]
    pats = {int(lane): i + 1 for i, lane in enumerate(chosen)}
    pats[int(chosen[-1])] |= ((1 << a) - 1) & ~((1 << bl) - 1)
    masks = [sum(1 << lane for lane, pt in pats.items() if pt >> e & 1) for e in range(a)]
    assert all(masks)
    return list(zip(ks, masks))


def dense_entries(ks, rs, lanes=32):
    """Entries of a group walked densely (more than 32 deviating observations), random lanes."""
    return [(k, int(rs.randint(1, 1 << lanes))) for k in ks]


class Builder(object):
    """Collects positions (columns of exp, reference code 0) and rows, then packs a Case.  Every
    position gets its own hit / miss; positions are renumbered at random at the end, so the
    order of a row is not the order of the table."""

    def __init__(self, name, n_hap, seed):
        self.name, self.n_hap = name, n_hap
        self.rs = np.random.RandomState(seed)
        self.cols = []
        self.rows = []
        self.want = []

    def position(self, col=None):
        self.cols.append(np.zeros(self.n_hap, np.uint8) if col is None else
                         np.asarray(col, dtype=np.uint8))
        return len(self.cols) - 1

    def row(self, pos, codes, **want):
        self.rows.append((list(pos), list(codes)))
        self.want.append(want)

    def dev_row(self, dev, **want):
        """A row with one new position per observation k where the columns dev[k] (fewer than
        half of all) carry symbol 1; the row observes the reference base or symbol 1 at random, so
        that in both cases observation k deviates from its plane's baseline exactly at dev[k]."""
        pos, codes = [], []
        for cols in dev:
            col = np.zeros(self.n_hap, np.uint8)
            col[np.asarray(cols, dtype=np.int64)] = 1
            assert 2 * int(col.sum()) < self.n_hap or not col.any()
            pos.append(self.position(col))
            codes.append(int(self.rs.randint(2)))
        self.row(pos, codes, **want)

    def group_row(self, n_obs, groups, **want):
        """groups: {g: [(k, lane mask), ...]}; observation k deviates at 32 g + the mask's lanes."""
        dev = [[] for _ in range(n_obs)]
        for g, ents in groups.items():
            for k, mask in ents:
                dev[k].extend(32 * g + lane for lane in range(32) if mask >> lane & 1)
        self.dev_row(dev, **want)

    def random_row(self, n_obs, p_dev=0.3, max_cols=4):
        """Observation k deviates with probability p_dev, at 1..max_cols random columns."""
        dev = []
        for _ in range(n_obs):
            if self.rs.rand() < p_dev:
                dev.append(self.rs.choice(self.n_hap, self.rs.randint(1, max_cols + 1)))
            else:
                dev.append([])
        return dev

    def warp_row(self, n_obs, tier, loads, first=None, **want):
        """A row whose work warps carry the chain items of loads {warp: items} and every other
        warp one item per group.  Each loaded warp gets ceil(items / 32) groups (32 items each,
        the rest in its last one), and all groups 0 .. n-1 are non-empty, so group g takes list
        slot g and work warp g mod tier.warps.  With `first`, every group deviates first at that
        observation or later, and the first group of the lowest loaded warp exactly there."""
        rs = self.rs
        m = max(-(-n // 32) for n in loads.values())
        n_groups = tier.warps * m
        assert 32 * n_groups <= self.n_hap
        lo = 0 if first is None else first
        groups = {}
        for g in range(n_groups):
            w, i = g % tier.warps, g // tier.warps
            n = loads.get(w)
            n = 1 if n is None else (32 if i < m - 1 else n - 32 * (m - 1))
            if n <= 0:
                raise ValueError("warp %d: %s items in %d groups" % (w, loads.get(w), m))
            a = max(n.bit_length(), int(rs.randint(1, 33)))
            if n < 32 and rs.rand() < 0.5:
                a = max(n.bit_length(), min(a, 5))        # straight-line patterns
            a = min(a, n_obs - lo)
            if first is not None and g == min(loads):
                ks = [first] + sorted(rs.choice(np.arange(first + 1, n_obs), a - 1, replace=False))
            else:
                ks = sorted(rs.choice(np.arange(lo, n_obs), a, replace=False))
            groups[g] = group_entries([int(k) for k in ks], n, rs)
        self.group_row(n_obs, groups, **want)

    def build(self, n_inf=1, n_hit_inf=0):
        """The Case; n_inf positions get miss = -inf and n_hit_inf get hit = -inf, chosen among
        the positions that only the first non-empty row observes, so that the others stay finite."""
        rs = self.rs
        n_pos = max(1, len(self.cols))
        exp = np.zeros((self.n_hap, n_pos), np.uint8)
        for p, col in enumerate(self.cols):
            exp[:, p] = col
        perm = rs.permutation(n_pos)                  # position p becomes perm[p]
        exp_t = np.empty_like(exp)
        exp_t[:, perm] = exp
        hit = -10.0 ** rs.uniform(-10, 2, n_pos)
        miss = -10.0 ** rs.uniform(-10, 2, n_pos)
        n_rows_of = np.zeros(n_pos, np.int64)
        for pos, _ in self.rows:
            n_rows_of[np.unique(np.asarray(pos, np.int64))] += 1
        first = next((pos for pos, _ in self.rows if pos), [])
        private = rs.permutation(np.array([p for p in sorted(set(first)) if n_rows_of[p] == 1],
                                          dtype=np.int64))
        miss[perm[private[:n_inf]]] = -np.inf            # log(0) of a zero probability
        hit[perm[private[n_inf:n_inf + n_hit_inf]]] = -np.inf
        row_ptr = np.zeros(len(self.rows) + 1, np.int64)
        row_ptr[1:] = np.cumsum([len(pos) for pos, _ in self.rows])
        pos_idx = np.array([perm[p] for pos, _ in self.rows for p in pos], np.int32)
        codes = np.array([c for _, cs in self.rows for c in cs], np.uint8)
        tables = make_tables(exp_t, np.zeros(n_pos, np.uint8), hit, miss)
        return Case(self.name, tables, SignatureCSR(row_ptr, pos_idx, codes), self.want)


# ---- the cases ---------------------------------------------------------------------------------
def _k_cases():
    out = []
    b = Builder("K_0_to_33", 100, 1)
    for k in (0, 1, 7, 8, 9, 31, 32, 33):
        b.dev_row(b.random_row(k), K=k, route=0)
    out.append(b.build())
    b = Builder("K_255_256_257", 64, 2)
    for k, r in ((255, 0), (256, 0), (257, 1)):
        b.dev_row(b.random_row(k, 0.05, 2), K=k, route=r)
    out.append(b.build())
    b = Builder("K_511_512_513", 96, 3)
    for k, r in ((511, 1), (512, 1), (513, 2), (1024, 2), (1025, 2)):
        b.dev_row(b.random_row(k, 0.02, 2), K=k, route=r)
    out.append(b.build())
    b = Builder("K_1024_1025_dense_kernel", 8193, 4)
    for k in (1024, 1025, 3):
        b.dev_row(b.random_row(k, 0.2, 40), K=k, route=3)
    out.append(b.build())
    return out


def _entry_cases():
    out = []
    # tier 1: 1536 = 5 dense groups x 256 + 8 groups x 32; one more entry defers the row
    b = Builder("entries_1536_1537", 32 * 14, 5)
    rs = b.rs
    for extra in (0, 1):
        groups = {g: dense_entries(range(256), rs) for g in range(5)}
        for g in range(5, 13):
            groups[g] = group_entries(sorted(rs.choice(256, 32, replace=False)),
                                      int(rs.randint(1, 33)), rs)
        if extra:
            groups[13] = group_entries([int(rs.randint(256))], 1, rs)
        b.group_row(256, groups, K=256, carry=1536 + extra, n_dense=5, route=[20, 21][extra])
    out.append(b.build())
    # the same limit without dense groups: 48 groups x 32 deviating observations
    b = Builder("entries_1536_1537_no_dense", 32 * 49, 6)
    rs = b.rs
    for extra in (0, 1):
        groups = {g: group_entries(sorted(rs.choice(256, 32, replace=False)),
                                   int(rs.randint(1, 6)), rs) for g in range(48)}
        if extra:
            groups[48] = group_entries([int(rs.randint(256))], 1, rs)
        b.group_row(256, groups, K=256, carry=1536 + extra, n_dense=0, route=extra)
    out.append(b.build())
    # tier 2: 8064 = 15 dense groups x 512 + 12 groups x 32; one more goes to build_dense_row
    b = Builder("entries_8064_8065", 32 * 28, 7)
    rs = b.rs
    for extra in (0, 1):
        groups = {g: dense_entries(range(512), rs) for g in range(15)}
        for g in range(15, 27):
            groups[g] = group_entries(sorted(rs.choice(512, 32, replace=False)),
                                      int(rs.randint(1, 33)), rs)
        if extra:
            groups[27] = group_entries([int(rs.randint(512))], 1, rs)
        b.group_row(512, groups, K=512, carry=8064 + extra, route=[61, 2][extra])
    out.append(b.build())
    return out


def _pool_cases():
    out = []
    for tier, t, k in ((TIER1, "t1", 203), (TIER2, "t2", 300)):
        lim = tier.pool
        for w in (0, tier.warps - 1):
            n_hap = 32 * tier.warps * -(-(lim + 1) // 32) + 5
            b = Builder("pool_%d_%d_warp%d" % (lim, lim + 1, w), n_hap, 10 + w + lim)
            for extra in (0, 1):
                b.warp_row(k, tier, {w: lim + extra}, route=tier.path + extra,
                           items=(t, w, lim + extra))
            out.append(b.build())
    # single and dual chain runs on one warp
    b = Builder("items_on_one_warp", 32 * 28 + 12, 20)
    for n in (1, 31, 32, 33, 63, 64, 65, 97):
        b.warp_row(203, TIER1, {0: n}, items=("t1", 0, n), route=0)
    out.append(b.build())
    return out


def _group_cases():
    out = []
    for n_hap in (32 * 9 + 7, 32 * 9 + 4):
        b = Builder("group_sizes_H%d" % n_hap, n_hap, n_hap)
        rs = b.rs
        k = 100
        pick = (lambda a: sorted(rs.choice(k, a, replace=False)))
        # a = 1, 2, 5, 6, 31, 32 (classes), 33 (dense, next to class groups), 32 patterns with
        # no lane on the baseline, and the partial last group (n_hap % 32 valid lanes)
        last = n_hap % 32
        groups = {0: group_entries(pick(1), 1, rs), 1: group_entries(pick(2), 3, rs),
                  2: group_entries(pick(5), 31, rs), 3: group_entries(pick(6), 20, rs),
                  4: group_entries(pick(31), 32, rs), 5: dense_entries(pick(33), rs),
                  6: group_entries(pick(32), 17, rs), 7: group_entries(pick(6), 32, rs),
                  9: group_entries(pick(5), last, rs, lanes=last)}
        b.group_row(k, groups, n_dense=1, route=4, a_of=[1, 2, 5, 6, 31, 33, 32, 6, 0, 5])
        # a dense group in the partial last group, next to a class group
        groups = {8: group_entries(pick(4), 9, rs), 9: dense_entries(pick(40), rs, lanes=last)}
        b.group_row(k, groups, n_dense=1, route=4)
        # the partial last group with every valid lane deviating, the rest empty
        groups = {9: group_entries(pick(6), last, rs, lanes=last)}
        b.group_row(k, groups, n_dense=0, route=0)
        out.append(b.build())
    return out


def _first_dev_cases():
    """The lock step of run_chains starts at the 8-aligned block of the earliest first deviation
    among a warp's items and ends with a partial last eight when K mod 8 != 0."""
    out = []
    b = Builder("first_deviation", 32 * 14, 30)
    for r in range(1, 8):
        k = 40 + r
        for k0 in (0, 7, 8, 31, 32, k - 1):
            for n in ((1,) if k0 == k - 1 else (3, 40)):   # single and dual run_chains
                b.warp_row(k, TIER1, {0: n}, first=k0, K=k, first_dev=k0, items=("t1", 0, n),
                           route=0)
    out.append(b.build())
    return out


def _repeat_and_plane_cases():
    out = []
    b = Builder("repeated_positions", 64, 40)
    rs = b.rs
    pos = []
    for _ in range(20):
        col = np.zeros(64, np.uint8)
        for c in (1, 2, 3):
            col[rs.choice(64, rs.randint(0, 6), replace=False)] = c
        pos.append(b.position(col))
    for _ in range(4):
        seq = list(rs.choice(pos, 30))
        seq += [seq[3], seq[3], seq[10]]                 # the same plane twice (and three times)
        codes = list(rs.randint(0, 4, len(seq)))
        codes[-2] = codes[3]
        codes[-3] = codes[3]
        codes[-1] = (codes[10] + 1) % 4                  # the same position, another plane
        order = rs.permutation(len(seq))
        b.row([seq[i] for i in order], [codes[i] for i in order], route=0)
    out.append(b.build())

    b = Builder("planes", 64, 41)
    rs = b.rs
    half = np.zeros(64, np.uint8)
    half[rs.choice(64, 32, replace=False)] = 1           # exactly half carry 1: a tie is "no match"
    major = np.zeros(64, np.uint8)
    major[rs.choice(64, 40, replace=False)] = 2          # the derived allele is the majority
    major[np.nonzero(major == 0)[0][:5]] = 3
    p_half, p_major = b.position(half), b.position(major)
    p_plain = [b.position() for _ in range(60)]
    for _ in range(4):
        pos = [p_half] * 3 + [p_major] * 4 + list(rs.choice(p_plain, 20, replace=False))
        codes = [0, 1, 2, 2, 0, 3, 1] + list(rs.choice([0, 1, 4, 255], 20))
        order = rs.permutation(len(pos))
        b.row([pos[i] for i in order], [codes[i] for i in order], route=0)
    out.append(b.build())
    return out


def _width_cases():
    out = []
    for n_hap in (1, 4, 31, 32, 33, 5404, 5406, 5632, 5633, 8191, 8192, 8193, 10241):
        b = Builder("width_%d" % n_hap, n_hap, n_hap)
        rs = b.rs
        # clades: contiguous runs of columns carrying a derived base, some of them the majority
        pos = []
        for _ in range(150):
            col = np.zeros(n_hap, np.uint8)
            size = min(n_hap, int(rs.geometric(0.02)))
            if rs.rand() < 0.05:
                size = n_hap - size // 4
            j0 = rs.randint(0, n_hap - size + 1)
            col[j0:j0 + size] = rs.randint(1, 4)
            pos.append(b.position(col))
        for k in (90, 150, 260):
            seq = list(rs.choice(pos, k - 8)) + [b.position(b.cols[p]) for p in rs.choice(pos, 8)]
            codes = list(rs.choice([0, 0, 0, 1, 2, 3, 4, 255], k))
            order = rs.permutation(k)
            b.row([seq[i] for i in order], [codes[i] for i in order])
        out.append(b.build(n_inf=2, n_hit_inf=1))
    return out


def all_cases():
    return (_k_cases() + _entry_cases() + _pool_cases() + _group_cases() + _first_dev_cases() +
            _repeat_and_plane_cases() + _width_cases())


_CASES = None


def cases():
    global _CASES
    if _CASES is None:
        _CASES = all_cases()
    return _CASES


CASE_NAMES = ["K_0_to_33", "K_255_256_257", "K_511_512_513", "K_1024_1025_dense_kernel",
              "entries_1536_1537", "entries_1536_1537_no_dense", "entries_8064_8065",
              "pool_146_147_warp0", "pool_146_147_warp6", "pool_273_274_warp0",
              "pool_273_274_warp14", "items_on_one_warp", "group_sizes_H295",
              "group_sizes_H292", "first_deviation", "repeated_positions", "planes"] + \
    ["width_%d" % h for h in (1, 4, 31, 32, 33, 5404, 5406, 5632, 5633, 8191, 8192, 8193, 10241)]


def case(name):
    return {c.name: c for c in cases()}[name]
