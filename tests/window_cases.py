"""Matrices in which a quarter of the rows have a mixture likelihood t_i = sum_j L_ij pi_j of
about e^level, for the tests of the rule that sends a row to the log-space step
(csrc/em_kernels.cuh: row_needs_logspace; CPU side in test_row_likelihood_rule.py, GPU side in
test_row_likelihood_window_gpu.py).

The linear-space pass forms coef_i = w_i / t_i, which overflows to +inf once t_i < w_i / DBL_MAX:
every subnormal t_i, and with large weights normal t_i too.  The rows enter that window in one
of three ways (MODES):

- "pi": the row's only plausible column (0) has ln pi_0 = level, every other cell lies 800
  lower, so a subnormal or tiny pi carries the row;
- "L": the row's best column (1) has pi = 0 exactly (a -inf start); the columns that carry mass
  lie about -level below it, shifted so that ln t_i = level exactly, so L is subnormal or tiny;
- "product": column 1 as in "L", column 0 has L = e^-400 and ln pi_0 = level + 400, every other
  cell 800 below the row's best: both factors are normal, their product is not.

Weights are scaled by SCALES (coefficient overflow at normal t).  EM is invariant under a common
scale of the weights, so one long-double trajectory serves every scale.  Layouts (SHAPES): fp64
rows at H = 1100 and 8192, the general path's H = 3 and 9000, and class tiles (64-column blocks
at H = 5408, as test_logspace_rescue_gpu._underflowing_matrix("tiles") builds them)."""
import numpy as np

LN_THETA = -960.0 * np.log(2.0)      # ln kRowLikelihoodMin (2^-960)
LEVELS = (-760.0, -745.0, -744.0, -740.0, -730.0, -720.0, -709.0, -708.4, -705.0, -700.0, -690.0,
          LN_THETA - 0.5, LN_THETA + 0.5, -600.0)
# the wide matrices (long-double references cost ~10x more): exact 0 as the control, the
# subnormal range, the DBL_MIN boundary, normal t with coefficient overflow, both sides of theta
WIDE_LEVELS = (-760.0, -740.0, -708.4, -700.0, LN_THETA - 0.5, LN_THETA + 0.5)
MODES = ("pi", "L", "product")
SCALES = (1.0, 1e3, 1e6)
# layout -> (rows, H, class tiles)
SHAPES = {"rows": (300, 1100, False), "rows8": (128, 8192, False), "narrow": (300, 3, False),
          "wide": (128, 9000, False), "tiles": (256, 5408, True)}


def levels_of(layout):
    return LEVELS if SHAPES[layout][1] <= 1100 else WIDE_LEVELS


def _lse_rows(a):
    """Row logsumexp in long double (finite entries only)."""
    a = np.asarray(a, dtype=np.longdouble)
    m = a.max(axis=1, keepdims=True)
    return (np.log(np.exp(a - m).sum(axis=1, keepdims=True)) + m)[:, 0]


def window_case(layout, mode, level, scale=1.0):
    """(matrix N x H, weights, start ln pi, window rows).  Rows [0, N/4) are the window rows."""
    n, h, tiles = SHAPES[layout]
    rs = np.random.RandomState(5)
    if tiles:
        base = np.repeat(-rs.gamma(2.0, 3.0, size=(n, h // 64 + 1)), 64, axis=1)[:, :h].copy()
    else:
        base = -rs.gamma(2.0, 3.0, size=(n, h))
    base[:, 0] = 0.0
    w = rs.randint(1, 5, size=n).astype(np.float64) * scale
    q = n // 4
    mat = base.copy()
    lnp = np.full(h, -np.log(h - 1.0))
    if mode == "pi":
        mat[:q, 1:] -= 800.0
        lnp[0] = level
    elif mode == "L":
        lnp[1] = -np.inf
        others = np.arange(h) != 1
        shift = level - _lse_rows(base[:q][:, others] + lnp[others])
        mat[:q, others] = (base[:q][:, others] + shift[:, None]).astype(np.float64)
        mat[:q, 1] = 0.0
    elif mode == "product":
        lnp[1] = -np.inf
        lnp[0] = level + 400.0
        mat[:q, 2:] -= 800.0
        mat[:q, 0] = -400.0
        mat[:q, 1] = 0.0
    else:
        raise ValueError(mode)
    return mat, w, lnp, q


def plain_start(h):
    """A uniform start: no row of any window_case matrix comes near the window from it."""
    return np.full(h, -np.log(float(h)))


# ---- the pass arithmetic in numpy fp64 -------------------------------------------------------
THETA = 2.0 ** -960


def rule_new(t):
    """row_needs_logspace (csrc/em_kernels.cuh)."""
    return ~(t >= THETA)


def rule_old(t):
    """The test it replaced: only an exact zero went to the log-space step."""
    return t == 0.0


def model_pass(mat, w, lnp, rule):
    """One linear-space iteration as the fp64-row pass computes it: L = exp(M - rowmax),
    t = L pi, coef = w / t (rows of weight 0 skipped), T = coef^T L, then mstep_lnp.  Returns
    (whether `rule` flags a row of nonzero weight, the new ln pi)."""
    with np.errstate(all="ignore"):
        lin = np.exp(mat - mat.max(axis=1, keepdims=True))
        pi = np.exp(lnp)
        t = lin @ pi
        live = w != 0.0
        flagged = bool(np.any(live & rule(t)))
        coef = np.where(live, w / np.where(live, t, 1.0), 0.0)
        col = coef @ lin
        total = float((pi * col).sum())
        linear = (pi >= 1e-290) & (pi * col >= 1e-290)
        new = np.where(linear, np.log(pi * col / total), lnp + np.log(col / total))
    return flagged, new


def model_iterate(mat, w, lnp, k, rule, log_step):
    """k iterations: a flagged iteration is redone by log_step(lnp) -> ln pi' (the log-space
    step); returns the trajectory (start first) and the flags."""
    out, flags = [np.asarray(lnp, dtype=np.float64)], []
    for _ in range(k):
        flagged, new = model_pass(mat, w, out[-1], rule)
        flags.append(flagged)
        out.append(np.asarray(log_step(out[-1]), dtype=np.float64) if flagged else new)
    return np.array(out), flags
