"""The generator and references of tile_cases.py (no GPU): the shared cases reach every row width
and class layout of the class-tile pass, read back from the plan mxb_tile_plan makes for the
full GPU and for a bootstrap session; the long-double iteration equals the numpy oracle; the
constructed colliding column collides under the restated column hash."""
import numpy as np
import pytest

from oracle import oracle_np
from test_tile_plan import plan, ROWS
from tile_cases import (BOOT_SMS, CASES, NUM_SMS, SPREAD, case_matrix, colliding_column,
                        fp64_pass_bytes, ld_iterate, per_of, predicted_pass_bytes, tile_hash)

C_WANTED = {1, 2, 3, 6655, 6656, 6783, 6784, 8191, 8192}
for _k in range(7, 13):
    C_WANTED |= {2 ** _k - 1, 2 ** _k, 2 ** _k + 1, 2 ** _k + 2}


@pytest.fixture(scope="module")
def matrices():
    return {case[0]: case_matrix(case) for case in CASES}


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_case_matrix_has_the_intended_classes(case, matrices):
    """class_matrix asserts the classes itself; here: the spread of the values, the fixed
    columns, short last batches, weights, and that a session over tiles pays off."""
    name, h, n, ncls, sizes, dead, dying = case
    mat, w, j_dead, j_dying = matrices[name]
    assert mat.shape == (n, h) and w.shape == (n,)
    fin = np.isfinite(mat)
    row_max = mat.max(axis=1)
    assert np.isfinite(row_max).all()
    assert (row_max[:, None] - mat)[fin].max() < SPREAD
    assert (w == 0).any() and w.max() == 1e6
    assert ((mat == row_max[:, None]).sum(axis=1) > 1).any()          # ties at the maximum
    if dead:
        assert np.isneginf(mat[:, j_dead]).all()
        assert (~fin).sum() > n                                         # the dead batch's class
    if dying:
        others = np.delete(mat, j_dying, axis=1).max(axis=1)
        assert (others - mat[:, j_dying] >= 200.0).all()
    if h >= 1024:     # the fast path (ld >= 1024) takes tiles when they save half the bytes
        for sms in (NUM_SMS, BOOT_SMS):
            assert predicted_pass_bytes(ncls, n, h, sms) < 0.5 * fp64_pass_bytes(n, h)


def test_cases_reach_every_boundary():
    lgs, cls, geometry, pers = set(), set(), {}, set()
    narrow_wide_narrow = two_narrow = split_wide = 0
    for name, h, n, ncls, *_ in CASES:
        cls |= set(ncls)
        pers.add(per_of(h))
        for sms in (NUM_SMS, BOOT_SMS):
            seg, n_cta, n_slots, slot_bytes, errors = plan(ncls, n, sms)
            assert errors == 0
            lgs |= set(seg[:, 6].tolist())
            geometry[max(ncls)] = (slot_bytes, n_slots)
            for c in range(n_cta):
                wide = (seg[seg[:, 0] == c, 6] >= 5).tolist()
                narrow_wide_narrow += any(not a and b and not d
                                          for a, b, d in zip(wide, wide[1:], wide[2:]))
                two_narrow += any(not a and not b for a, b in zip(wide, wide[1:]))
            for cta, b, r0, rows, fit, copies, lg, r_pad in seg.tolist():
                batch_rows = min(ROWS, n - b * ROWS)
                if lg >= 5 and rows < batch_rows and rows % (512 >> lg):
                    split_wide += 1
    assert lgs == set(range(3, 10))
    assert C_WANTED <= cls, sorted(C_WANTED - cls)
    assert pers == {4, 8, 12, 16}
    assert {(n - 1) % ROWS + 1 for _, _, n, *_ in CASES} >= {1, 31, 127, 128}
    # the ring: longer slots from C = 6656 on, two slots from C = 6784 on
    assert geometry[6655] == (53248, 3) and geometry[6656] == (54272, 3)
    assert geometry[6783] == (54272, 3) and geometry[6784][1] == 2
    assert narrow_wide_narrow >= 1 and two_narrow >= 1 and split_wide >= 1


@pytest.mark.parametrize("case", CASES[:3] + CASES[-2:], ids=lambda c: c[0])
def test_ld_iterate_equals_numpy_oracle(case, matrices):
    name, h, *_ = case
    mat, w, j_dead, j_dying = matrices[name]
    rs = np.random.RandomState(4)
    p = rs.dirichlet([1.0] * h)
    if j_dying is not None:
        p[j_dying] = 1e-3
    lnp = np.log(p / p.sum())
    traj = ld_iterate(mat, w, lnp, 3)
    assert np.array_equal(traj[0], lnp)
    for k in range(3):
        _, want = oracle_np.em_step(mat, w, np.asarray(traj[k], dtype=np.float64))
        got = traj[k + 1]
        assert np.array_equal(np.isneginf(got), np.isneginf(want))
        fin = np.isfinite(want)
        err = np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))
        assert err.max() < 1e-13, (k, err.max())


@pytest.mark.parametrize("seed", range(3))
def test_colliding_column(seed, matrices):
    mat = matrices["lg3_to_6"][0]
    b = 2
    a = mat[b * ROWS:(b + 1) * ROWS, 7 + seed]
    c = colliding_column(a, seed)
    assert tile_hash(c) == tile_hash(a)
    diff = np.flatnonzero(c.view(np.uint64) != a.view(np.uint64))
    assert diff.tolist() == [0, 1]
    assert np.isfinite(c).all() and -60.0 < c[1] < 0.0
    moved = c.copy()
    moved[1] = np.nextafter(c[1], 0.0)
    assert tile_hash(moved) != tile_hash(a)
