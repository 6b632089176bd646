"""The class-tile form of an EM iteration (csrc/em_tiles.cuh, DESIGN.md 3.2) restated in numpy on
top of the plan the library makes for the pass (``mxb_tile_plan``; no GPU): per 128-row batch the
bit-identical columns collapse into classes, ``Pi_b[c]`` sums the proportions of a class, every
*segment* of the plan (the rows of a batch inside one CTA's range) forms ``s_i = V_b[i] . Pi_b``
and its own vector ``U[c] = sum_i (w_i / s_i) V_b[i][c]``, and the gather adds the segments'
vectors back to columns.  The result must be the iteration the reference computes
(em.py:80-89, here through the numpy oracle) to rounding: the regrouping adds the same
non-negative terms, and splitting a batch over two CTAs only splits a sum.
"""
import numpy as np
import pytest

from mixemt_b200 import synth
from mixemt_b200.preprocess import HapVarBaseMatrix
from oracle import oracle_c, oracle_np
from test_tile_plan import plan, ROWS


def column_classes(block):
    """(cmap[H], representatives[C]) of a row block: columns equal in every row, bit for bit;
    classes numbered by first column (the kernels number them by hash: any numbering works)."""
    cols = np.ascontiguousarray(block.T).view(np.dtype((np.void, block.shape[0] * 8))).ravel()
    _, first, inv = np.unique(cols, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    return rank[inv.ravel()], first[order]


def tile_iteration(mat, weights, ln_props, num_sms):
    """One iteration over class tiles, segment by segment as tile_pass_kernel walks them.
    Returns (new proportions, bytes of tiles, number of segments)."""
    n, h = mat.shape
    pi = np.exp(ln_props)
    nb = (n + ROWS - 1) // ROWS
    cmaps, reps = [], []
    for b in range(nb):
        cm, rp = column_classes(mat[b * ROWS:(b + 1) * ROWS])
        cmaps.append(cm)
        reps.append(rp)
    n_cls = np.array([len(r) for r in reps], dtype=np.int32)
    seg, n_cta, n_slots, slot_bytes, errors = plan(n_cls, n, num_sms)
    assert errors == 0
    t = np.zeros(h)
    tile_bytes = 0
    for cta, b, r0, rows, fit, copies, lg, r_pad in seg.tolist():
        assert r_pad >= n_cls[b] + 1                       # class values + the row's weight
        lo = b * ROWS + r0
        block = mat[lo:lo + rows]
        # tile_fill_kernel: exp(M - rowmax) of the class representatives (the row maximum is
        # over the representatives, which is the row maximum)
        rowmax = block[:, reps[b]].max(axis=1, keepdims=True)
        assert np.array_equal(rowmax.ravel(), block.max(axis=1))
        v = np.exp(block[:, reps[b]] - rowmax)
        pi_cls = np.bincount(cmaps[b], weights=pi, minlength=n_cls[b])      # tile_pi_kernel
        s = v @ pi_cls                                                      # tile_pass_kernel
        assert (s > 0).all()
        u = (weights[lo:lo + rows] / s) @ v
        t += u[cmaps[b]]                                                    # tile_gather_kernel
        tile_bytes += rows * r_pad * 8
    new = pi * t
    return new / new.sum(), tile_bytes, len(seg)                            # em_finish_kernel


@pytest.mark.parametrize("num_sms", [148, 5])
def test_tile_iteration_equals_reference_iteration(phylo17, num_sms):
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.6), ("L3e", 0.4)], 1500, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _ = oracle_c.build_matrix(tables, mix.csr(tables), want_counts=False)
    n, h = mat.shape
    assert n > 4 * ROWS
    wts = mix.weights.astype(np.float64)
    ln_props = np.log(np.random.RandomState(8).dirichlet([1.0] * h))
    for _ in range(3):
        got, tile_bytes, n_seg = tile_iteration(mat, wts, ln_props, num_sms)
        _, want_ln = oracle_np.em_step(mat, wts, ln_props)
        want = np.exp(want_ln)
        assert abs(got.sum() - 1.0) < 1e-12
        assert np.abs(got - want).max() < 1e-13
        ln_props = want_ln
    # string-sorted signatures compress: the tiles are a fraction of the fp64 rows; a batch is
    # split only where two CTAs' ranges meet (with 148 CTAs most of these few batches are)
    assert tile_bytes < 0.5 * mat.nbytes
    nb = (n + ROWS - 1) // ROWS
    assert nb <= n_seg <= nb + num_sms - 1
    if num_sms == 148:
        assert n_seg > nb


def test_rows_in_random_order_do_not_compress(phylo17):
    """The same rows shuffled: neighbouring rows no longer share column classes, which is why
    such a session keeps fp64 rows (em_tiles.cu: tiles must save at least half of the bytes)."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.6), ("L3e", 0.4)], 1500, seed=4)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    mat, _ = oracle_c.build_matrix(tables, mix.csr(tables), want_counts=False)
    perm = np.random.RandomState(1).permutation(mat.shape[0])
    sorted_cls = [len(column_classes(mat[b:b + ROWS])[1]) for b in range(0, mat.shape[0], ROWS)]
    shuffled = mat[perm]
    random_cls = [len(column_classes(shuffled[b:b + ROWS])[1])
                  for b in range(0, mat.shape[0], ROWS)]
    assert np.mean(random_cls) > 3 * np.mean(sorted_cls)
