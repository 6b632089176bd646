"""The log-space EM step of a row-sharded session, restated in numpy (no GPU).

When a row's mixture likelihood underflows in linear space, every rank of a row-sharded run
redoes that iteration in log space (em.cu: em_logspace_step).  Each rank holds whole rows, so
the row logsumexp is local; the column reduction new_lnp_j = logsumexp_i(Z_ij, b=w_i)
(em.py:87-88) spans the ranks.  It is formed the way scipy forms it: the global column maxima
(an all-reduce max), then per rank the weight m of the maximal terms and the sum s of
w_i exp(Z_ij - max) over the others, summed over the ranks (an all-reduce sum), and
log1p(s/m) + log(m) + max.  This pins that arithmetic against oracle_np.em_step, which holds
scipy's logsumexp bit for bit, for 2, 3 and 8 shards.
"""
import numpy as np
import pytest

from oracle import oracle_np


def _row_lse(z):
    """em_logspace_rows_kernel: max + log(sum exp(z - max)), -inf for a row without mass."""
    mx = np.max(z, axis=1, keepdims=True)
    with np.errstate(invalid="ignore", divide="ignore"):
        lse = mx + np.log(np.sum(np.exp(z - np.where(np.isfinite(mx), mx, 0.0)), axis=1,
                                 keepdims=True))
    return np.where(np.isfinite(mx), lse, -np.inf)


def sharded_lnprops(mat, w, lnp, n_shards):
    """One log-space EM step over row shards, in the kernels' order of operations."""
    n, h = mat.shape
    bounds = [n * r // n_shards for r in range(n_shards + 1)]
    zs, ws = [], []
    for r in range(n_shards):
        lo, hi = bounds[r], bounds[r + 1]
        z = (mat[lo:hi] + lnp) - _row_lse(mat[lo:hi] + lnp)   # local to the rank
        zs.append(z)
        ws.append(w[lo:hi])
    # em_logspace_cols_kernel + colreduce (max), then the all-reduce max
    colmax = np.full(h, -np.inf)
    for z, wr in zip(zs, ws):
        live = z[wr != 0]
        if len(live):
            colmax = np.maximum(colmax, live.max(axis=0))
    # em_logspace_cols_split_kernel per rank, then the all-reduce sum of [s][m]
    s = np.zeros(h)
    m = np.zeros(h)
    with np.errstate(invalid="ignore", over="ignore"):
        for z, wr in zip(zs, ws):
            keep = wr != 0
            z, wk = z[keep], wr[keep][:, None]
            is_max = z == colmax
            s += np.sum(np.where(is_max, 0.0, wk * np.exp(z - colmax)), axis=0)
            m += np.sum(np.where(is_max, wk, 0.0), axis=0)
    # em_logspace_update_kernel with colcnt
    finite = colmax > -np.inf
    with np.errstate(divide="ignore", invalid="ignore"):
        v = np.where(finite, np.log1p(s / m) + np.log(m) + colmax, -np.inf)
    mx = v.max()
    norm = mx + np.log(np.sum(np.exp(v - mx)))
    return v - norm


def _case(kind, seed):
    rs = np.random.RandomState(seed)
    n, h = 97, 41
    mat = -rs.gamma(2.0, 4.0, size=(n, h))
    w = rs.randint(1, 9, size=n).astype(np.float64)
    lnp = np.log(rs.dirichlet([1.0] * h))
    if kind == "inf_cells":
        mat[rs.rand(n, h) < 0.2] = -np.inf
        mat[:, 3] = 0.0                      # every row keeps a finite cell
    elif kind == "dead_columns":
        lnp[[2, 7]] = -np.inf                # haplotypes without mass
        mat[:, 11] = -np.inf                 # a haplotype no read supports
    elif kind == "zero_weights":
        w[rs.rand(n) < 0.3] = 0.0
        w[:12] = 0.0                         # the first of 8 shards carries no weight
    elif kind == "underflow":
        # the rows that trigger the log-space step: all their mass sits ~800 log units
        # below their best haplotype, which starts with almost no mass
        mat[:, 0] = 0.0
        mat[: n // 4, 1:] -= 800.0
        lnp = np.full(h, -np.log(h - 1.0))
        lnp[0] = -760.0
    elif kind == "ties":
        # repeated rows: a column's maximum is reached in several shards, m counts them all
        mat[n // 2:] = mat[:n - n // 2]
        w[n // 2:] = w[:n - n // 2]
    return mat, w, lnp


@pytest.mark.parametrize("n_shards", [2, 3, 8])
@pytest.mark.parametrize("kind", ["plain", "inf_cells", "dead_columns", "zero_weights",
                                  "underflow", "ties"])
def test_sharded_logspace_step_matches_reference(kind, n_shards):
    mat, w, lnp = _case(kind, seed=3)
    _, want = oracle_np.em_step(mat, w, lnp)
    got = sharded_lnprops(mat, w, lnp, n_shards)
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    assert np.isfinite(got[fin]).all()
    assert np.abs(got[fin] - want[fin]).max() < 1e-13


def test_sharding_does_not_change_the_step():
    """The step does not depend on how the rows are split (one shard is the whole matrix)."""
    mat, w, lnp = _case("underflow", seed=4)
    one = sharded_lnprops(mat, w, lnp, 1)
    for k in (2, 3, 8):
        assert np.abs(sharded_lnprops(mat, w, lnp, k) - one).max() < 1e-13
