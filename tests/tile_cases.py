"""Matrices with a chosen number of column classes per 128-row batch, and long-double references,
for the tests of the class-tile kernels (csrc/em_tiles.cuh; CPU side in test_tile_cases.py, GPU
side in test_tile_kernels_gpu.py).

The batch's class count C decides how tile_pass_kernel runs a row (2^lg threads, tile_plan.h:
tile_layout), how many double2 chunks a row has ((C + 1) >> 1, the last one carries the weight),
the ring geometry (the widest row of the matrix) and whether the end-of-batch scratch alternates
halves (lg <= 4).  H decides how many entries of the sorted columns a thread of tile_pi_kernel
sums (PER = 4, 8, 12 or 16).  class_matrix builds a matrix whose batches have exactly the class
counts asked for, with class sizes that put runs across the chunk and warp borders of the class
sums; CASES lists the matrices the tests share."""
import numpy as np

from test_tile_model import column_classes
from test_tile_plan import plan, ROWS

NUM_SMS = 148                   # B200
BOOT_SMS = NUM_SMS // 16        # the plan of a bootstrap session with 16 replicate slots
SPREAD = 600.0                  # every finite cell lies within this many log units of its row max
DYING_GAP = 200.0               # the dying column: this far below every row's best, or further

_MASK = (1 << 64) - 1
_SEED = 0x243F6A8885A308D3


def per_of(h):
    """Entries of the sorted columns one thread of tile_pi_kernel sums (em_tiles.cu:
    launch_tile_class and the class-sum launch take ITEMS = 4, 8, 12 or 16 from ceil(H / 512))."""
    items = -(-h // 512)
    return 4 if items <= 4 else 8 if items <= 8 else 12 if items <= 12 else 16


def _class_sizes(c, h, want, first):
    """c sizes that sum to h: `first` fixed sizes, then want(k) as far as the columns left allow
    (every later class keeps at least one column); the last class takes the rest."""
    sizes = list(first)
    left = h - sum(sizes)
    for k in range(len(sizes), c - 1):
        s = max(1, min(want(k), left - (c - 1 - k)))
        sizes.append(s)
        left -= s
    if len(sizes) < c:
        sizes.append(left)
    assert len(sizes) == c and min(sizes) >= 1 and sum(sizes) == h, (c, h)
    return sizes


def class_matrix(ncls, h, n_rows, sizes, seed, dead=False, dying=False):
    """(matrix N x H, weights, dead column or None, dying column or None).

    Batch b has exactly ncls[b] classes of bit-identical columns.  Values are drawn per (row,
    class) within SPREAD log units of the row maximum, with ties at the maximum in some rows;
    weights include zeros and values up to 1e6.  sizes picks the class sizes of every batch:
    "giant" = one class of all the remaining columns (spanning every warp of the class sums)
    plus singletons, "per" = PER - 1, PER, PER + 1, 32 PER - 1, 32 PER + 1 in turn, "random" =
    1 .. 3 PER.  dead: one column is -inf in every row, and in one batch its class takes further
    columns (a class that is -inf in every row of that batch).  dying: one column lies DYING_GAP
    to DYING_GAP + 20 below the row maximum in every row (a singleton class everywhere)."""
    rs = np.random.RandomState(seed)
    nb = -(-n_rows // ROWS)
    ncls = [int(c) for c in ncls]
    assert len(ncls) == nb and max(ncls) <= h
    per = per_of(h)
    cycle = [per - 1, per, per + 1, 32 * per - 1, 32 * per + 1]
    n_fixed = int(dead) + int(dying)
    assert min(ncls) >= n_fixed + 1, "every batch needs a finite class besides the fixed ones"
    cols = rs.permutation(h)
    j_dead = int(cols[0]) if dead else None
    j_dying = int(cols[int(dead)]) if dying else None
    free_cols = cols[n_fixed:]
    dead_batch = int(rs.randint(nb)) if dead else -1
    mat = np.empty((n_rows, h))
    w = rs.randint(1, 50, size=n_rows).astype(np.float64)
    w[rs.rand(n_rows) < 0.1] = 0.0
    w[rs.rand(n_rows) < 0.03] = 1e6
    if not w.any():
        w[0] = 1.0
    for b in range(nb):
        c = ncls[b]
        r0, r1 = b * ROWS, min(n_rows, (b + 1) * ROWS)
        nr = r1 - r0
        if sizes == "giant":
            want = lambda k: 1          # singletons; the last class takes the rest
        elif sizes == "per":
            want = lambda k: cycle[k % len(cycle)]
        else:
            want = lambda k: int(rs.randint(1, 3 * per + 1))
        first = [1] * n_fixed
        # the dead batch: its -inf class takes PER + 1 more columns, if the others can spare them
        extra = min(per + 1, h - c) if b == dead_batch else 0
        if extra:
            first[0] += extra
        body = _class_sizes(c - n_fixed, h - n_fixed - extra, want, [])
        if sizes == "giant":   # the giant class (the rest) first
            body = [body[-1]] + body[:-1]
        all_sizes = first + body
        assert len(all_sizes) == c and sum(all_sizes) == h
        # column -> class; the fixed columns head the classes they belong to
        label = np.empty(h, dtype=np.int64)
        order = rs.permutation(free_cols)
        pos = 0
        for k, s in enumerate(all_sizes):
            members = []
            if k == 0 and dead:
                members.append(j_dead)
            elif k == int(dead) and dying:
                members.append(j_dying)
            take = s - len(members)
            members.extend(order[pos:pos + take].tolist())
            pos += take
            label[members] = k
        assert pos == len(order)
        # values per (row, class): an offset per row, then up to SPREAD - 20 below it
        off = rs.uniform(-50.0, 30.0, size=(nr, 1))
        val = off - (SPREAD - 20.0) * rs.beta(0.7, 2.5, size=(nr, c))
        finite0 = n_fixed
        tied = rs.rand(nr) < 0.2
        if c - finite0 >= 2:      # rows tied at their maximum: two classes share it
            k2 = finite0 + 1
            val[tied, k2] = val[tied, finite0:].max(axis=1)
        if dead:
            val[:, 0] = -np.inf
        if dying:
            best = val[:, finite0:].max(axis=1)
            val[:, int(dead)] = best - DYING_GAP - rs.uniform(0.0, 20.0, size=nr)
        mat[r0:r1] = val[:, label]
        # the classes are exactly the intended ones
        cm, reps = column_classes(mat[r0:r1])
        assert len(reps) == c, (b, len(reps), c)
        assert np.array_equal(np.unique(np.stack([cm, label]), axis=1).shape, (2, c))
    return mat, w, j_dead, j_dying


def predicted_pass_bytes(ncls, n_rows, h, num_sms=NUM_SMS):
    """What mxb_em_pass_bytes reports for a session over class tiles (em_tiles.cu: tile_pass_bytes):
    the tiles, perm + cmap for the class sums and cmap for the gather, and the class vectors Pi
    and U, each written and read.  A segment that starts inside its batch has a U vector of its
    own."""
    seg, _, _, _, errors = plan(ncls, n_rows, num_sms)
    assert errors == 0
    nb = len(ncls)
    hs = -(-h // 8) * 8
    r_pad = [(int(c) + 1 + 3) // 4 * 4 for c in ncls]
    v_cells = sum(min(ROWS, n_rows - b * ROWS) * r_pad[b] for b in range(nb))
    p_cells = sum(r_pad)
    u_cells = p_cells + sum(int(rp) for _, _, r0, _, _, _, _, rp in seg.tolist() if r0 > 0)
    return v_cells * 8 + 3 * nb * hs * 2 + 2 * (p_cells + u_cells) * 8


def fp64_pass_bytes(n_rows, h):
    return n_rows * (-(-h // 16) * 16) * 8


def _ld_lse(a, axis, b=None):
    """log sum (b) exp(a) along axis in long double, max-shifted; -inf where every term is 0."""
    a = np.asarray(a, dtype=np.longdouble)
    live = np.isfinite(a) if b is None else np.isfinite(a) & (b > 0)
    m = np.where(live, a, -np.inf).max(axis=axis, keepdims=True)
    shift = np.where(np.isfinite(m), m, 0)
    with np.errstate(invalid="ignore", divide="ignore", under="ignore"):
        e = np.where(live, np.exp(a - shift), 0)
        if b is not None:
            e = e * np.asarray(b, dtype=np.longdouble)
        return (np.log(e.sum(axis=axis, keepdims=True)) + shift).squeeze(axis)


def ld_read_mix(mat, lnp):
    """em.py:80-82 in long double: log responsibilities Z = ln pi + M - logsumexp_row."""
    z = np.asarray(lnp, dtype=np.longdouble) + np.asarray(mat, dtype=np.longdouble)
    return z - _ld_lse(z, 1)[:, None]


def ld_iterate(mat, w, lnp, k):
    """k iterations of em.py:80-89 in long double, the plain log-space formula (oracle_np works
    in float64).  Returns the k + 1 log-proportions of the trajectory, start first."""
    out = [np.asarray(lnp, dtype=np.longdouble)]
    wl = np.asarray(w, dtype=np.longdouble)[:, None]
    for _ in range(k):
        z = ld_read_mix(mat, out[-1])
        new = _ld_lse(z, 0, np.broadcast_to(wl, z.shape))
        out.append(new - _ld_lse(new, 0))
    return np.array(out)


def _mix(h, v):
    """tile_mix (em_tiles.cuh) in Python integers."""
    h = ((h ^ v) * 0xFF51AFD7ED558CCD) & _MASK
    h ^= h >> 29
    h = (h * 0xC4CEB9FE1A85EC53) & _MASK
    return h ^ (h >> 32)


def _bits(x):
    return int(np.float64(x).view(np.uint64))


def tile_hash(col):
    """tile_hash_kernel for one column of one batch (its values over the batch's rows)."""
    h = _SEED
    for x in np.asarray(col, dtype=np.float64):
        h = _mix(h, _bits(x))
    return _MASK - 1 if h == _MASK else h


def colliding_column(col, seed):
    """A column that differs from col in rows 0 and 1 and hashes to the same value: with b0
    drawn, b1 = a1 ^ mix(h0, a0) ^ mix(h0, b0) makes the states equal after row 1 (tile_mix is a
    bijection of h ^ v), so the rows after it keep them equal.  b0 is redrawn until b1 is a
    normal double in (-60, 0)."""
    rs = np.random.RandomState(seed)
    col = np.asarray(col, dtype=np.float64)
    a0, a1 = _bits(col[0]), _bits(col[1])
    for _ in range(10000):
        b0 = rs.uniform(-60.0, 0.0)
        if b0 == col[0]:
            continue
        b1_bits = a1 ^ _mix(_SEED, a0) ^ _mix(_SEED, _bits(b0))
        b1 = float(np.uint64(b1_bits).view(np.float64))
        if -60.0 < b1 < 0.0 and abs(b1) >= np.finfo(np.float64).tiny:
            out = col.copy()
            out[0], out[1] = b0, b1
            return out
    raise AssertionError("no colliding column found")


# The shared cases: (name, H, rows, class counts per batch, sizes, dead, dying).  Together they
# cover every lg (3..9), the class counts around every power of two from 128 to 4096, the ring
# geometry changes at C = 6656 (longer slots) and 6784 (two slots), every PER, short last
# batches of 1, 31 and 127 rows, and the plans' segment patterns test_tile_cases.py asserts.
def _n(nb, last):
    return (nb - 1) * ROWS + last


CASES = [
    ("tiny_classes", 2048, _n(5, 127), [1, 2, 3, 1, 2], "giant", False, False),
    ("lg3_to_6", 2049, _n(16, 31),
     [127, 128, 129, 130, 3, 255, 256, 257, 258, 5, 511, 512, 513, 514, 9, 4], "per", True, True),
    ("lg6_to_8", 4097, _n(12, 1),
     [1023, 1024, 1025, 1026, 4, 2047, 2048, 2049, 2050, 3, 7, 3], "random", True, True),
    ("lg8_to_9", 6145, _n(10, 128),
     [4095, 4096, 4097, 4098, 3, 5, 3, 60, 3, 3], "per", True, False),
    ("slot_6655", 6784, _n(3, 127), [4, 6655, 3], "giant", True, True),
    ("slot_6656", 6784, _n(4, 31), [6656, 3, 5, 3], "random", True, False),
    ("slot_6783", 6784, _n(4, 1), [3, 6783, 4, 3], "per", True, True),
    ("slot_6784", 6784, _n(3, 127), [5, 3, 6784], "giant", False, False),
    ("widest", 8192, _n(7, 31), [8191, 3, 3, 8192, 4, 3, 3], "random", True, False),
    ("narrow_wide_narrow", 2048, _n(24, 128),
     [3, 40, 300, 5, 3, 1500, 4, 3, 90, 400, 3, 3, 3, 700, 3, 120, 3, 3, 260, 3, 6, 3, 3, 3],
     "random", True, True),
    ("h130", 130, _n(4, 31), [3, 130, 66, 2], "per", False, False),
]


def case_matrix(case, seed=None):
    name, h, n, ncls, sizes, dead, dying = case
    if seed is None:
        seed = sum(map(ord, name))
    return class_matrix(ncls, h, n, sizes, seed, dead=dead, dying=dying)
