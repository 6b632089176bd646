// Device code of kernel 2 (the EM fit) over fp64 rows: everything csrc/em.cu launches except
// the class-tile kernels (em_tiles.cuh).  See em.cu for the formulation and the host side.
#pragma once

#include <cooperative_groups.h>

#include "block_reduce.cuh"
#include "em_common.cuh"
#include "row_likelihood.cuh"
#define MXB_DYN_SHARED extern __shared__

#include <math.h>
#include <stdint.h>

#include <type_traits>

namespace mxb {

constexpr int kPassThreads = 512;
constexpr int kPassWarps = kPassThreads / 32;
constexpr int kPassGroup = 2;       // rows reduced together per block barrier
constexpr int kMaxNC = 8;           // column chunks (double2) per thread
constexpr int kLdAlign = 16;        // row stride of L in doubles (128 B)

// ---- M -> L ------------------------------------------------------------------
// L_ij = exp(M_ij - max_j M_ij); padding columns [n_cols, ld) are 0.
__global__ void __launch_bounds__(256)
to_linear_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols, int64_t ld,
                 double *__restrict__ lin) {
    __shared__ double scratch[8];
    for (int64_t r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const double *row = m + r * n_cols;
        double mx = -INFINITY;
        bool has_nan = false;
        for (int64_t j = threadIdx.x; j < n_cols; j += 256) {
            double v = row[j];
            has_nan |= (v != v);
            mx = fmax(mx, v);
        }
        mx = block_max<256>(mx, scratch);
        double *dst = lin + r * ld;
        for (int64_t j = threadIdx.x; j < ld; j += 256)
            dst[j] = (j < n_cols) ? exp(row[j] - mx) : 0.0;  // row re-read hits L1/L2
        (void)has_nan;
    }
}

// ---- fused E+M pass (fast path) ----------------------------------------------
// Rows are handled two at a time between block barriers.  The two partial dot
// products of a thread are reduced together: the first shuffle step hands row 0
// to lanes 0-15 and row 1 to lanes 16-31, so one 5-step butterfly serves both
// rows; lanes 0 and 16 publish the warp totals, and after the barrier every
// warp folds the 16 + 16 warp totals with a 4-step butterfly over its two
// half-warps, divides once per row and broadcasts the two coefficients.  All
// index arithmetic in the loop is 32-bit and incremental (no 64-bit division).
__device__ __forceinline__ double shfl_xor_f64(double v, int off) {
    return __shfl_xor_sync(0xffffffffu, v, off);
}

template <int NC>
__global__ void __launch_bounds__(kPassThreads, 1)
em_pass_fast_kernel(const unsigned char *__restrict__ rows, uint32_t row_bytes, int64_t ld,
                    int64_t n_rows, const double *__restrict__ weights,
                    const double *__restrict__ pi0, const double *__restrict__ pi1,
                    EmState *__restrict__ st, double *__restrict__ partials, int n_stages) {
    static_assert(kPassGroup == 2 && kPassWarps == 16, "reduction layout below");
    pdl_launch_dependents();  // the tail kernel may be scheduled as SMs drain

    MXB_DYN_SHARED __align__(128) unsigned char smem_raw[];
    double *scratch = reinterpret_cast<double *>(
        smem_raw + (((size_t)n_stages * row_bytes + 127) & ~(size_t)127));
    uint64_t *full = reinterpret_cast<uint64_t *>(scratch + 2 * kPassWarps * kPassGroup);

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int64_t r_begin = n_rows * (int64_t)blockIdx.x / gridDim.x;
    const int64_t r_end = n_rows * (int64_t)(blockIdx.x + 1) / gridDim.x;
    const int n_my = (int)(r_end - r_begin);
    const unsigned char *my_rows = rows + (size_t)r_begin * row_bytes;
    const double *my_w = weights + r_begin;
    const uint32_t stages_u32 = smem_u32(smem_raw);
    const uint32_t full_u32 = smem_u32(full);

    // Prologue: L and the weights do not depend on the previous iteration's tail, so the
    // ring is primed before waiting for it (the loads overlap the tail kernel).
    if (tid == 0) {
        for (int s = 0; s < n_stages; ++s) mbar_init(&full[s], 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (tid == 0) {
        for (int q = 0; q < n_my && q < n_stages; ++q) {
            mbar_expect_tx(&full[q], row_bytes);
            bulk_load(smem_raw + (size_t)q * row_bytes, my_rows + (size_t)q * row_bytes, row_bytes,
                      &full[q]);
        }
    }
    pdl_wait();  // proportions and control block of the previous iteration are final
    if (st->done) {
        // finished run: the primed loads must land before this CTA's shared memory is released
        for (int q = 0; q < n_my && q < n_stages; ++q) mbar_wait_u32(full_u32 + 8u * (uint32_t)q, 0u);
        return;
    }
    const double *__restrict__ pi = st->cur ? pi1 : pi0;

    // Thread-private column slice: chunk c = tid + k*512 covers doubles 2c, 2c+1.
    const int n_chunks = (int)(ld >> 1);
    double2 pr[NC], tr[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int c = tid + k * kPassThreads;
        pr[k] = (c < n_chunks) ? reinterpret_cast<const double2 *>(pi)[c] : make_double2(0.0, 0.0);
        tr[k] = make_double2(0.0, 0.0);
    }
    const bool last_live = tid + (NC - 1) * kPassThreads < n_chunks;  // only chunk NC-1 can be ragged

    int stage = 0;          // ring slot of row q0
    uint32_t phase = 0;     // its mbarrier parity
    int sbuf = 0;
    int bad = 0;
    const bool upper = lane >= 16;
    for (int q0 = 0; q0 < n_my; q0 += kPassGroup) {
        double2 lv[kPassGroup][NC];
        double dot[kPassGroup];
        const int q_mine = q0 + (upper ? 1 : 0);
        const double w_mine = (q_mine < n_my) ? my_w[q_mine] : 0.0;
        int s_of[kPassGroup];
        int s = stage;
        uint32_t ph = phase;
#pragma unroll
        for (int g = 0; g < kPassGroup; ++g) {
            s_of[g] = s;
            double dx = 0.0, dy = 0.0;
            if (q0 + g < n_my) {
                mbar_wait_u32(full_u32 + 8u * (uint32_t)s, ph);
                const double2 *srow = reinterpret_cast<const double2 *>(
                    smem_raw + (size_t)s * row_bytes) + tid;
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    if (k < NC - 1 || last_live) lv[g][k] = srow[k * kPassThreads];
                    else lv[g][k] = make_double2(0.0, 0.0);
                    dx = fma(lv[g][k].x, pr[k].x, dx);
                    dy = fma(lv[g][k].y, pr[k].y, dy);
                }
            } else {
#pragma unroll
                for (int k = 0; k < NC; ++k) lv[g][k] = make_double2(0.0, 0.0);
            }
            dot[g] = dx + dy;
            if (++s == n_stages) { s = 0; ph ^= 1u; }
        }
        // both rows in one butterfly: lanes 0-15 end up with row 0, lanes 16-31 with row 1
        double v = (upper ? dot[1] : dot[0]) + shfl_xor_f64(upper ? dot[0] : dot[1], 16);
        v += shfl_xor_f64(v, 8);
        v += shfl_xor_f64(v, 4);
        v += shfl_xor_f64(v, 2);
        v += shfl_xor_f64(v, 1);
        double *sc = scratch + sbuf * (kPassWarps * kPassGroup);
        if ((lane & 15) == 0) sc[(lane >> 4) * kPassWarps + warp] = v;
        __syncthreads();  // all reads of this group's stages are done; warp totals visible
        if (tid == 0) {
#pragma unroll
            for (int g = 0; g < kPassGroup; ++g) {
                const int q = q0 + g + n_stages;
                if (q < n_my) {
                    const uint32_t bar = full_u32 + 8u * (uint32_t)s_of[g];
                    mbar_expect_tx_u32(bar, row_bytes);
                    bulk_load_u32(stages_u32 + (uint32_t)s_of[g] * row_bytes,
                                  my_rows + (size_t)q * row_bytes, row_bytes, bar);
                }
            }
        }
        // 16 warp totals per row sit in sc[0..15] / sc[16..31]: one value per lane
        double t = sc[lane];
        t += shfl_xor_f64(t, 8);
        t += shfl_xor_f64(t, 4);
        t += shfl_xor_f64(t, 2);
        t += shfl_xor_f64(t, 1);
        double coef_mine = 0.0;
        if (w_mine != 0.0) {
            coef_mine = w_mine / t;
            bad |= row_needs_logspace(t);
        }
        const double coef0 = __shfl_sync(0xffffffffu, coef_mine, 0);
        const double coef1 = __shfl_sync(0xffffffffu, coef_mine, 16);
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            tr[k].x = fma(coef0, lv[0][k].x, tr[k].x);
            tr[k].y = fma(coef0, lv[0][k].y, tr[k].y);
        }
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            tr[k].x = fma(coef1, lv[1][k].x, tr[k].x);
            tr[k].y = fma(coef1, lv[1][k].y, tr[k].y);
        }
        stage = s;
        phase = ph;
        sbuf ^= 1;
    }

    double2 *out = reinterpret_cast<double2 *>(partials + (size_t)blockIdx.x * ld);
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int c = tid + k * kPassThreads;
        if (c < n_chunks) out[c] = tr[k];
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0 && warp == 0) atomicAdd(&st->bad, 1);
}

// ---- fused E+M pass for two restarts at once ---------------------------------------
// Restarts of one run_em call share the matrix (em.py:117-156), so two of them can
// share each read of L: the pass is HBM-bound and the fp64 pipe is ~20 % busy.  Same
// streaming structure as em_pass_fast_kernel; a thread keeps the proportions and the
// column sums of BOTH restarts in registers (96 of its 128), so a staged row is read
// from shared memory twice -- once for the two dot products, once for the two
// column-sum updates -- and a second block barrier per row pair releases the stages.
// The four (row, restart) dot products of a row pair ride one butterfly.
template <int NC>
__global__ void __launch_bounds__(kPassThreads, 1)
em_pass_pair_kernel(const double *__restrict__ lin, int64_t ld, int64_t n_rows,
                    const double *__restrict__ weights, const double *__restrict__ pi_a0,
                    const double *__restrict__ pi_a1, const double *__restrict__ pi_b0,
                    const double *__restrict__ pi_b1, EmState *__restrict__ st,
                    double *__restrict__ partials_a, double *__restrict__ partials_b,
                    int n_stages) {
    static_assert(kPassGroup == 2 && kPassWarps == 16, "reduction layout below");
    pdl_launch_dependents();

    MXB_DYN_SHARED __align__(128) unsigned char smem_raw[];
    const uint32_t row_bytes = (uint32_t)(ld * sizeof(double));
    double *scratch = reinterpret_cast<double *>(smem_raw + (size_t)n_stages * row_bytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(scratch + 2 * kPassWarps * kPassGroup);

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int64_t r_begin = n_rows * (int64_t)blockIdx.x / gridDim.x;
    const int64_t r_end = n_rows * (int64_t)(blockIdx.x + 1) / gridDim.x;
    const int n_my = (int)(r_end - r_begin);
    const unsigned char *my_rows = reinterpret_cast<const unsigned char *>(lin + r_begin * ld);
    const double *my_w = weights + r_begin;
    const uint32_t stages_u32 = smem_u32(smem_raw);
    const uint32_t full_u32 = smem_u32(full);

    if (tid == 0) {
        for (int s = 0; s < n_stages; ++s) mbar_init(&full[s], 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (tid == 0) {
        for (int q = 0; q < n_my && q < n_stages; ++q) {
            mbar_expect_tx(&full[q], row_bytes);
            bulk_load(smem_raw + (size_t)q * row_bytes, my_rows + (size_t)q * row_bytes, row_bytes,
                      &full[q]);
        }
    }

    pdl_wait();
    const int done_a = st[0].done, done_b = st[1].done;
    if (done_a && done_b) {
        for (int q = 0; q < n_my && q < n_stages; ++q) mbar_wait_u32(full_u32 + 8u * (uint32_t)q, 0u);
        return;
    }
    const double *__restrict__ pia = st[0].cur ? pi_a1 : pi_a0;
    const double *__restrict__ pib = st[1].cur ? pi_b1 : pi_b0;

    const int n_chunks = (int)(ld >> 1);
    double2 pa[NC], pb[NC], ta[NC], tb[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int c = tid + k * kPassThreads;
        const bool in = c < n_chunks;
        pa[k] = in ? reinterpret_cast<const double2 *>(pia)[c] : make_double2(0.0, 0.0);
        pb[k] = in ? reinterpret_cast<const double2 *>(pib)[c] : make_double2(0.0, 0.0);
        ta[k] = make_double2(0.0, 0.0);
        tb[k] = make_double2(0.0, 0.0);
    }
    const bool last_live = tid + (NC - 1) * kPassThreads < n_chunks;

    int stage = 0;
    uint32_t phase = 0;
    int bad = 0;
    // quarter q4 = lane >> 3 owns pair (row g = q4 >> 1, restart = q4 & 1) after the butterfly
    const int q4 = lane >> 3;
    const bool mine_done = (q4 & 1) ? done_b != 0 : done_a != 0;
    for (int q0 = 0; q0 < n_my; q0 += kPassGroup) {
        const int q_mine = q0 + (q4 >> 1);
        const double w_mine = (q_mine < n_my) ? my_w[q_mine] : 0.0;
        int s_of[kPassGroup];
        double d[4];  // [row][restart]
        int s = stage;
        uint32_t ph = phase;
#pragma unroll
        for (int g = 0; g < kPassGroup; ++g) {
            s_of[g] = s;
            double ax = 0.0, ay = 0.0, bx = 0.0, by = 0.0;
            if (q0 + g < n_my) {
                mbar_wait_u32(full_u32 + 8u * (uint32_t)s, ph);
                const double2 *srow = reinterpret_cast<const double2 *>(
                    smem_raw + (size_t)s * row_bytes) + tid;
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    if (k < NC - 1 || last_live) {
                        const double2 l = srow[k * kPassThreads];
                        ax = fma(l.x, pa[k].x, ax);
                        ay = fma(l.y, pa[k].y, ay);
                        bx = fma(l.x, pb[k].x, bx);
                        by = fma(l.y, pb[k].y, by);
                    }
                }
            }
            d[2 * g] = ax + ay;
            d[2 * g + 1] = bx + by;
            if (++s == n_stages) { s = 0; ph ^= 1u; }
        }
        // four sums in one butterfly: halves keep a row, quarters keep a restart
        const bool up16 = (lane & 16) != 0, up8 = (lane & 8) != 0;
        double e0 = (up16 ? d[2] : d[0]) + shfl_xor_f64(up16 ? d[0] : d[2], 16);
        double e1 = (up16 ? d[3] : d[1]) + shfl_xor_f64(up16 ? d[1] : d[3], 16);
        double v = (up8 ? e1 : e0) + shfl_xor_f64(up8 ? e0 : e1, 8);
        v += shfl_xor_f64(v, 4);
        v += shfl_xor_f64(v, 2);
        v += shfl_xor_f64(v, 1);
        // scratch[pair q4][warp]; the loop's second barrier separates consecutive groups
        if ((lane & 7) == 0) scratch[q4 * kPassWarps + warp] = v;
        __syncthreads();
        // 16 warp totals per pair: lane reads two of them, 3-step butterfly inside its quarter
        double t = scratch[q4 * kPassWarps + (lane & 7)] + scratch[q4 * kPassWarps + 8 + (lane & 7)];
        t += shfl_xor_f64(t, 4);
        t += shfl_xor_f64(t, 2);
        t += shfl_xor_f64(t, 1);
        double coef_mine = 0.0;
        if (w_mine != 0.0) {
            coef_mine = w_mine / t;
            bad |= (row_needs_logspace(t) && !mine_done);
        }
        const double c0a = __shfl_sync(0xffffffffu, coef_mine, 0);
        const double c0b = __shfl_sync(0xffffffffu, coef_mine, 8);
        const double c1a = __shfl_sync(0xffffffffu, coef_mine, 16);
        const double c1b = __shfl_sync(0xffffffffu, coef_mine, 24);
#pragma unroll
        for (int g = 0; g < kPassGroup; ++g) {
            if (q0 + g < n_my) {
                const double ca = g ? c1a : c0a, cb = g ? c1b : c0b;
                const double2 *srow = reinterpret_cast<const double2 *>(
                    smem_raw + (size_t)s_of[g] * row_bytes) + tid;
#pragma unroll
                for (int k = 0; k < NC; ++k) {
                    if (k < NC - 1 || last_live) {
                        const double2 l = srow[k * kPassThreads];
                        ta[k].x = fma(ca, l.x, ta[k].x);
                        ta[k].y = fma(ca, l.y, ta[k].y);
                        tb[k].x = fma(cb, l.x, tb[k].x);
                        tb[k].y = fma(cb, l.y, tb[k].y);
                    }
                }
            }
        }
        __syncthreads();  // both staged rows have been read twice: release them
        if (tid == 0) {
#pragma unroll
            for (int g = 0; g < kPassGroup; ++g) {
                const int q = q0 + g + n_stages;
                if (q < n_my) {
                    const uint32_t bar = full_u32 + 8u * (uint32_t)s_of[g];
                    mbar_expect_tx_u32(bar, row_bytes);
                    bulk_load_u32(stages_u32 + (uint32_t)s_of[g] * row_bytes,
                                  my_rows + (size_t)q * row_bytes, row_bytes, bar);
                }
            }
        }
        stage = s;
        phase = ph;
    }

    double2 *out_a = reinterpret_cast<double2 *>(partials_a + (size_t)blockIdx.x * ld);
    double2 *out_b = reinterpret_cast<double2 *>(partials_b + (size_t)blockIdx.x * ld);
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int c = tid + k * kPassThreads;
        if (c < n_chunks) {
            out_a[c] = ta[k];
            out_b[c] = tb[k];
        }
    }
    if (bad) atomicOr(&st[(q4 & 1)].bad, 1);
}

// ---- general path: any shape, two passes over L -------------------------------
// coef_i = w_i / sum_j L_ij pi_j, one warp per row.
__global__ void __launch_bounds__(256)
em_rowdot_kernel(const double *__restrict__ lin, int64_t ld, int64_t n_rows,
                 const double *__restrict__ weights, const double *__restrict__ pi0,
                 const double *__restrict__ pi1, EmState *__restrict__ st,
                 double *__restrict__ coef) {
    if (st->done) return;
    const double2 *__restrict__ pi = reinterpret_cast<const double2 *>(st->cur ? pi1 : pi0);
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int64_t n_warps = (int64_t)gridDim.x * 8;
    const int64_t n_chunks = ld >> 1;
    int bad = 0;
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        const double2 *row = reinterpret_cast<const double2 *>(lin + r * ld);
        double dot = 0.0;
        for (int64_t c = lane; c < n_chunks; c += 32) {
            const double2 l = row[c];
            const double2 p = pi[c];
            dot = fma(l.x, p.x, dot);
            dot = fma(l.y, p.y, dot);
        }
        dot = warp_sum(dot);
        if (lane == 0) {
            const double w = weights[r];
            double c = 0.0;
            if (w != 0.0) { c = w / dot; bad |= row_needs_logspace(dot); }
            coef[r] = c;
        }
    }
    if (bad) atomicAdd(&st->bad, 1);
}

// partial T_j over a row range; thread owns one double2 column chunk.
__global__ void __launch_bounds__(256)
em_colacc_kernel(const double *__restrict__ lin, int64_t ld, int64_t n_rows,
                 const double *__restrict__ coef, const EmState *__restrict__ st,
                 double *__restrict__ partials) {
    if (st->done) return;
    const int64_t c = (int64_t)blockIdx.y * 256 + threadIdx.x;
    if (c >= (ld >> 1)) return;
    const int64_t r_begin = n_rows * (int64_t)blockIdx.x / gridDim.x;
    const int64_t r_end = n_rows * (int64_t)(blockIdx.x + 1) / gridDim.x;
    double2 t = make_double2(0.0, 0.0);
    int64_t r = r_begin;
    for (; r + 4 <= r_end; r += 4) {
        double2 l[4];
        double cf[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            l[u] = reinterpret_cast<const double2 *>(lin + (r + u) * ld)[c];
            cf[u] = coef[r + u];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            t.x = fma(cf[u], l[u].x, t.x);
            t.y = fma(cf[u], l[u].y, t.y);
        }
    }
    for (; r < r_end; ++r) {
        const double2 l = reinterpret_cast<const double2 *>(lin + r * ld)[c];
        const double cf = coef[r];
        t.x = fma(cf, l.x, t.x);
        t.y = fma(cf, l.y, t.y);
    }
    reinterpret_cast<double2 *>(partials + (size_t)blockIdx.x * ld)[c] = t;
}

// T_j = sum over CTAs of partials, fixed order.  tsum[ld] carries the row-likelihood underflow
// flag, so that a row-sharded run sums it over the ranks together with the column sums and
// every rank takes the same decision in em_update_kernel.  Launch ceil_div(ld + 1, 256) CTAs.
__global__ void __launch_bounds__(256)
em_colreduce_kernel(const double *__restrict__ partials, int n_part, int64_t ld,
                    const EmState *__restrict__ st, double *__restrict__ tsum) {
    if (st->done) return;
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j == ld) tsum[ld] = st->bad ? 1.0 : 0.0;
    if (j >= ld) return;
    double t = 0.0;
    for (int b = 0; b < n_part; ++b) t += partials[(size_t)b * ld + j];
    tsum[j] = t;
}

// ln pi'_j of the M-step (em.py:89) from pi_j, its column sum t and the normaliser total.
// When pi or pi * T underflows (a column far worse than the mixture in every row, whose
// decay factor T / total is tiny) it stays in log space, else ln pi' would be -inf.
// lnp_old is read only then.
__device__ __forceinline__ double mstep_lnp(double p, double t, double total,
                                            const double *lnp_old) {
    if (p >= 1e-290 && p * t >= 1e-290) return log(p * t / total);
    return *lnp_old + log(t / total);
}

// Advances the control block after an iteration (em.py:39-54): one more iteration, then
// converged, max_iter reached, a peer that timed out, or the proportion buffers swapped.
__device__ __forceinline__ void advance_state(EmState *st, double delta, int cur,
                                              bool timeout = false) {
    st->delta = delta;
    const long long it = st->iters + 1;
    st->iters = it;
    if (timeout) st->done = 3;
    else if (delta < st->tol) st->done = 1;
    else if (it >= st->max_iter) st->done = 2;
    else st->cur = 1 - cur;
}

// M-step normalisation + convergence test (em.py:89 and :39-54), one CTA.
constexpr int kUpdThreads = 1024;
__global__ void __launch_bounds__(kUpdThreads)
em_update_kernel(const double *__restrict__ tsum, int64_t n_cols, int64_t ld,
                 double *__restrict__ lnp0, double *__restrict__ lnp1,
                 double *__restrict__ pi0, double *__restrict__ pi1,
                 EmState *__restrict__ st) {
    if (st->done) return;
    if (tsum[ld] != 0.0) {       // a row needs the log-space step (on some rank): see em_logspace_*
        if (threadIdx.x == 0) st->done = kDoneNeedsLogStep;
        return;
    }
    __shared__ double scratch[kUpdThreads / 32];
    const int cur = st->cur;
    const double *lnp_old = cur ? lnp1 : lnp0;
    const double *pi_old = cur ? pi1 : pi0;
    double *lnp_new = cur ? lnp0 : lnp1;
    double *pi_new = cur ? pi0 : pi1;

    double local = 0.0;
    for (int64_t j = threadIdx.x; j < n_cols; j += kUpdThreads) local += pi_old[j] * tsum[j];
    const double total = block_sum<kUpdThreads>(local, scratch);

    double dl = 0.0;
    for (int64_t j = threadIdx.x; j < n_cols; j += kUpdThreads) {
        const double p = pi_old[j];
        const double ln_new = mstep_lnp(p, tsum[j], total, lnp_old + j);
        const double p_new = exp(ln_new);
        lnp_new[j] = ln_new;
        pi_new[j] = p_new;
        dl += fabs(p_new - p);
    }
    const double delta = block_sum<kUpdThreads>(dl, scratch);
    if (threadIdx.x == 0) advance_state(st, delta, cur);
}

// ---- fused tail of an iteration (fast path) ------------------------------------
// One launch replaces em_colreduce_kernel + em_update_kernel: a single cluster of
// kFinCtas CTAs, one thread per column.  Each thread adds the per-CTA partial
// sums of its column in fixed order, the two scalars of the M-step (the
// normaliser sum_k pi_k T_k and the convergence distance sum_j |pi'_j - pi_j|,
// em.py:89 and :39-54) are reduced across the cluster through distributed shared
// memory, and CTA 0 advances the control block.  Deterministic: fixed summation
// orders, no atomics.
constexpr int kFinCtas = 8;
constexpr int kFinThreads = 1024;

// Sum of one double per thread over the whole cluster; every thread gets it.
// slots: kFinCtas doubles in *every* CTA's shared memory, wsum: kFinThreads/32.
__device__ __forceinline__ double cluster_sum(double v, double *wsum, double *slots) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    if (lane == 0) wsum[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double t = wsum[lane];  // kFinThreads / 32 == 32 warps
        t = warp_sum(t);
        if (lane < kFinCtas) {
            // lane r publishes this CTA's total in CTA r's slot array
            double *remote = cluster.map_shared_rank(slots, lane);
            remote[cluster.block_rank()] = t;
        }
    }
    cluster.sync();
    double total = 0.0;
#pragma unroll
    for (int r = 0; r < kFinCtas; ++r) total += slots[r];
    return total;
}

// Multi-GPU form of the tail (kP2P): the ranks' column sums are exchanged through
// peer memory instead of a separate collective.  Every rank stores its H sums
// into slot (seq & 1) of each peer's inbox (NVLink P2P stores), fences, and
// raises its flag there with the launch sequence number; it then waits until all
// `world` flags in its own block carry that number and adds the inbox rows in
// rank order, so that every rank forms bit-identical totals and takes the same
// convergence decision.  Two slots suffice: a rank can be at most one launch
// ahead of a peer, because it needs that peer's flag to finish a launch.  A rank
// whose pass flagged a row-likelihood underflow (st->bad) raises its flags with
// kP2PBadBit set; every rank then sees it in the same launch, sets
// done = kDoneNeedsLogStep instead of advancing, and the iteration is redone in log
// space by all ranks together (em_logspace_step).  The sequence number advances as
// in any other launch, so the mailboxes stay in step.
constexpr unsigned long long kP2PBadBit = 1ull << 63;
struct P2PArgs {
    int world, rank;
    unsigned char *block[kP2PMaxWorld];  // [r] = rank r's mailbox block (own block at [rank])
};
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
constexpr unsigned long long kP2PTimeoutNs = 120ull * 1000000000ull;

template <bool kP2P>
__global__ void __cluster_dims__(kFinCtas, 1, 1) __launch_bounds__(kFinThreads)
em_finish_kernel(const double *partials, int n_part, int64_t n_cols, int64_t ld,
                 double *lnp0, double *lnp1, double *pi0, double *pi1, EmState *st, P2PArgs pa) {
    static_assert(kFinThreads == 1024, "cluster_sum assumes 32 warps");
    pdl_wait();               // the pass kernel's partial sums are complete and visible
    pdl_launch_dependents();  // the next pass may prime its ring while this tail runs
    {   // blockIdx.y = restart slot of a batched session (one cluster per slot)
        const size_t slot = blockIdx.y;
        st += slot;
        partials += slot * (size_t)n_part * ld;
        lnp0 += slot * ld; lnp1 += slot * ld;
        pi0 += slot * ld; pi1 += slot * ld;
    }
    if (st->done) return;  // same answer in every CTA: the block below is the only writer
    if (!kP2P && st->bad) {
        // A row's mixture likelihood is too small for linear space: this iteration is redone in
        // log space by the host (em_logspace_* kernels), the queued launches become no-ops.
        // (st->bad was final before this launch began; the write below is seen by later
        // launches only.)  Row-sharded runs first tell the other ranks (kP2PBadBit below).
        cooperative_groups::this_cluster().sync();
        if (blockIdx.x == 0 && threadIdx.x == 0) st->done = kDoneNeedsLogStep;
        return;
    }
    __shared__ double wsum[2][kFinThreads / 32];
    __shared__ double slots[2][kFinCtas];
    __shared__ int s_timeout, s_bad;
    const int cur = st->cur;
    const double *lnp_old = cur ? lnp1 : lnp0;
    const double *pi_old = cur ? pi1 : pi0;
    double *lnp_new = cur ? lnp0 : lnp1;
    double *pi_new = cur ? pi0 : pi1;

    // Column sums.  A CTA owns ld/16 column pairs; its 1024 threads split the per-CTA
    // partials of a pair into n_grp contiguous ranges (three at H=5408) that are summed
    // concurrently and then added in range order: fixed order, a third of the latency.
    __shared__ double2 red[kFinThreads];
    const int ppc = (int)(ld >> 4);                       // column pairs per CTA
    const int n_grp = min(8, kFinThreads / ppc);
    const int pair_local = threadIdx.x % ppc, grp = threadIdx.x / ppc;
    const int64_t c = (int64_t)blockIdx.x * ppc + pair_local;   // columns 2c, 2c+1
    if (grp < n_grp) {
        const int b0 = (int)((int64_t)n_part * grp / n_grp), b1 = (int)((int64_t)n_part * (grp + 1) / n_grp);
        const double2 *col = reinterpret_cast<const double2 *>(partials) + c;
        const size_t stride = (size_t)(ld >> 1);
        double2 acc = make_double2(0.0, 0.0);
        int b = b0;
        for (; b + 4 <= b1; b += 4) {
            double2 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = col[(size_t)(b + u) * stride];
#pragma unroll
            for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; }
        }
        for (; b < b1; ++b) { const double2 v = col[(size_t)b * stride]; acc.x += v.x; acc.y += v.y; }
        red[grp * ppc + pair_local] = acc;
    }
    __syncthreads();
    const bool owner = grp == 0;                          // one thread per column pair from here on
    const bool live_x = owner && 2 * c < n_cols, live_y = owner && 2 * c + 1 < n_cols;
    double2 t = make_double2(0.0, 0.0);
    if (owner) {
        for (int g = 0; g < n_grp; ++g) { t.x += red[g * ppc + pair_local].x; t.y += red[g * ppc + pair_local].y; }
    }
    // a peer CTA's shared memory may only be written once that CTA is known to have
    // started: one cluster barrier before the first distributed-shared-memory store
    cooperative_groups::this_cluster().sync();
    unsigned long long seq = 0;
    if (kP2P) {
        namespace cg = cooperative_groups;
        cg::cluster_group cluster = cg::this_cluster();
        const int W = pa.world;
        unsigned long long *my_flags = reinterpret_cast<unsigned long long *>(pa.block[pa.rank]);
        unsigned long long *my_seq = my_flags + 2 * kP2PMaxWorld;
        if (threadIdx.x == 0) { s_timeout = 0; s_bad = 0; }
        seq = *my_seq + 1;  // advanced by CTA 0 at the very end of this launch
        const int slot = (int)(seq & 1ull);
        if (owner) {
            for (int r = 0; r < W; ++r) {
                double2 *inbox = reinterpret_cast<double2 *>(pa.block[r] + kP2PInboxOffset);
                inbox[((size_t)slot * kP2PMaxWorld + pa.rank) * (kP2PMaxLd / 2) + c] = t;
            }
        }
        __threadfence_system();
        cluster.sync();  // every store of this rank is fenced
        if (blockIdx.x == 0 && threadIdx.x < W) {
            const int r = threadIdx.x;
            unsigned long long *peer_flags = reinterpret_cast<unsigned long long *>(pa.block[r]);
            st_release_sys(&peer_flags[slot * kP2PMaxWorld + pa.rank],
                           seq | (st->bad ? kP2PBadBit : 0ull));
            const unsigned long long t0 = global_timer_ns();
            for (;;) {
                const unsigned long long f = ld_acquire_sys(&my_flags[slot * kP2PMaxWorld + r]);
                if ((f & ~kP2PBadBit) == seq) {
                    if (f & kP2PBadBit) s_bad = 1;
                    break;
                }
                if (global_timer_ns() - t0 > kP2PTimeoutNs) { s_timeout = 1; break; }
            }
        }
        cluster.sync();  // all ranks' sums have landed in this rank's inbox
        if (owner) {
            const double2 *inbox = reinterpret_cast<const double2 *>(pa.block[pa.rank] + kP2PInboxOffset);
            t = make_double2(0.0, 0.0);
            for (int r = 0; r < W; ++r) {
                const double2 v = __ldcg(&inbox[((size_t)slot * kP2PMaxWorld + r) * (kP2PMaxLd / 2) + c]);
                t.x += v.x;
                t.y += v.y;
            }
        }
    }
    double2 p = make_double2(0.0, 0.0);
    if (owner) p = reinterpret_cast<const double2 *>(pi_old)[c];
    if (!live_x) p.x = 0.0;
    if (!live_y) p.y = 0.0;
    const double total = cluster_sum((live_x ? p.x * t.x : 0.0) + (live_y ? p.y * t.y : 0.0),
                                     wsum[0], slots[0]);

    double dl = 0.0;
    if (owner) {
        double2 ln_new = make_double2(-INFINITY, -INFINITY), p_new = make_double2(0.0, 0.0);
        if (live_x) {
            ln_new.x = mstep_lnp(p.x, t.x, total, lnp_old + 2 * c);
            p_new.x = exp(ln_new.x);
            dl += fabs(p_new.x - p.x);
        }
        if (live_y) {
            ln_new.y = mstep_lnp(p.y, t.y, total, lnp_old + 2 * c + 1);
            p_new.y = exp(ln_new.y);
            dl += fabs(p_new.y - p.y);
        }
        reinterpret_cast<double2 *>(lnp_new)[c] = ln_new;   // padding columns: (-inf, 0) as set_props left them
        reinterpret_cast<double2 *>(pi_new)[c] = p_new;
    }
    const double delta = cluster_sum(dl, wsum[1], slots[1]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (kP2P) {
            unsigned long long *my_flags = reinterpret_cast<unsigned long long *>(pa.block[pa.rank]);
            my_flags[2 * kP2PMaxWorld] = seq;
        }
        if (kP2P && !s_timeout && s_bad) {
            st->done = kDoneNeedsLogStep;    // the proportions written above are discarded
            return;
        }
        advance_state(st, delta, cur, kP2P && s_timeout);   // timeout: a peer never showed up
    }
}

// ln pi -> (ln pi, pi) device buffers, padding zeroed.

__global__ void em_set_props_kernel(const double *__restrict__ src, int64_t n_cols, int64_t ld,
                                    double *__restrict__ lnp, double *__restrict__ pi,
                                    double *__restrict__ lnp_other, double *__restrict__ pi_other) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ld) return;
    const bool in = j < n_cols;
    const double v = in ? src[j] : -INFINITY;
    lnp[j] = v;
    pi[j] = in ? exp(v) : 0.0;
    lnp_other[j] = -INFINITY;
    pi_other[j] = 0.0;
}

// ---- read matrix: Z = (M + ln pi) - logsumexp_row(M + ln pi) -------------------
// (em.py:80-83).  mode 1 folds into dst with numpy.logaddexp (em.py:156).
__device__ __forceinline__ double np_logaddexp(double x, double y) {
    if (x == y) return x + 0.693147180559945309417232121458176568;
    const double tmp = x - y;
    if (tmp > 0) return x + log1p(exp(-tmp));
    if (tmp <= 0) return y + log1p(exp(tmp));
    return tmp;  // NaN
}

constexpr int kMixThreads = 256;
__global__ void __launch_bounds__(kMixThreads)
read_mix_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols,
                const double *__restrict__ lnp, double *__restrict__ dst, int mode,
                double sub_log) {
    __shared__ double scratch[kMixThreads / 32];
    for (int64_t r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const double *row = m + r * n_cols;
        double mx = -INFINITY;
        double nan_flag = 0.0;  // fmax drops NaN; numpy.max propagates it
        for (int64_t j = threadIdx.x; j < n_cols; j += kMixThreads) {
            const double z = row[j] + lnp[j];
            if (z != z) nan_flag = 1.0;
            mx = fmax(mx, z);
        }
        nan_flag = block_sum<kMixThreads>(nan_flag, scratch);
        mx = block_max<kMixThreads>(mx, scratch);
        double lse;
        if (nan_flag > 0.0) {
            lse = NAN;
        } else if (isinf(mx)) {
            lse = mx;  // all -inf -> log(0); any +inf -> +inf (scipy's out_inf branch)
        } else {
            // scipy _logsumexp: s over non-max terms, m = number of max terms
            double s = 0.0, cnt = 0.0;
            for (int64_t j = threadIdx.x; j < n_cols; j += kMixThreads) {
                const double z = row[j] + lnp[j];
                if (z == mx) cnt += 1.0;
                else s += exp(z - mx);
            }
            s = block_sum<kMixThreads>(s, scratch);
            cnt = block_sum<kMixThreads>(cnt, scratch);
            lse = log1p(s / cnt) + log(cnt) + mx;
        }
        double *out = dst + r * n_cols;
        for (int64_t j = threadIdx.x; j < n_cols; j += kMixThreads) {
            double z = (row[j] + lnp[j]) - lse;
            if (mode == 1) z = np_logaddexp(out[j], z);
            if (sub_log != 0.0) z -= sub_log;
            out[j] = z;
        }
    }
}

// ---- one EM iteration in log space (rescue path) -------------------------------------
// The linear-space pass needs s_i = sum_j L_ij pi_j >= kRowLikelihoodMin = 2^-960 (about
// e^-665; row_needs_logspace), or w_i / s_i may overflow.  When every haplotype that still has
// mass explains a row more than ~665 log units worse than the row's best one, s_i falls below
// that although the reference's log-space arithmetic (em.py:80-89, max-shifted logsumexp)
// stays finite.  The iteration is then redone exactly as the reference states it:
//   Z_ij = M_ij + ln pi_j - lse_i,  ln pi'_j = lse_i(Z_ij + ln w_i) - lse_j(...)
// in three sweeps over M (row lse; column maxima; column sums).  Rare and slow by design.
__global__ void __launch_bounds__(256)
em_logspace_rows_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols,
                        const double *__restrict__ lnp, double *__restrict__ lse) {
    __shared__ double scratch[8];
    for (int64_t r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const double *row = m + r * n_cols;
        double mx = -INFINITY;
        for (int64_t j = threadIdx.x; j < n_cols; j += 256) mx = fmax(mx, row[j] + lnp[j]);
        mx = block_max<256>(mx, scratch);
        double sum = 0.0;
        if (mx > -INFINITY)
            for (int64_t j = threadIdx.x; j < n_cols; j += 256) sum += exp(row[j] + lnp[j] - mx);
        sum = block_sum<256>(sum, scratch);
        if (threadIdx.x == 0) lse[r] = mx > -INFINITY ? mx + log(sum) : -INFINITY;
    }
}

// partial column maxima / sums over a block of rows; thread = column, blockIdx.y = row block
__global__ void __launch_bounds__(256)
em_logspace_cols_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols,
                        const double *__restrict__ lnp, const double *__restrict__ lse,
                        const double *__restrict__ w, const double *__restrict__ colmax,
                        double *__restrict__ part) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= n_cols) return;
    const int64_t r0 = n_rows * blockIdx.y / gridDim.y, r1 = n_rows * (blockIdx.y + 1) / gridDim.y;
    const double lp = lnp[j];
    double acc = colmax ? 0.0 : -INFINITY;
    const double cm = colmax ? colmax[j] : 0.0;
    for (int64_t r = r0; r < r1; ++r) {
        const double wr = w[r];
        if (wr == 0.0) continue;                       // scipy: a = -inf where b == 0
        const double z = (m[r * n_cols + j] + lp) - lse[r];
        if (colmax) { if (cm > -INFINITY) acc += wr * exp(z - cm); }
        else acc = fmax(acc, z);
    }
    part[(size_t)blockIdx.y * n_cols + j] = acc;
}

// Row-sharded form of the column sums: the maxima `colmax` are global (all-reduced over the
// ranks), and scipy's logsumexp terms are kept apart as its formula needs them,
// part[b][0][j] = s (sum of w_i exp(Z_ij - max) over the non-maximal terms) and
// part[b][1][j] = m (sum of w_i over the maximal terms), so that the ranks' sums of s and m
// can be added before ln pi'_j = log1p(s/m) + log(m) + max is formed.
__global__ void __launch_bounds__(256)
em_logspace_cols_split_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols,
                              const double *__restrict__ lnp, const double *__restrict__ lse,
                              const double *__restrict__ w, const double *__restrict__ colmax,
                              double *__restrict__ part) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= n_cols) return;
    const int64_t r0 = n_rows * blockIdx.y / gridDim.y, r1 = n_rows * (blockIdx.y + 1) / gridDim.y;
    const double lp = lnp[j], cm = colmax[j];
    double s = 0.0, cnt = 0.0;
    if (cm > -INFINITY) {
        for (int64_t r = r0; r < r1; ++r) {
            const double wr = w[r];
            if (wr == 0.0) continue;                   // scipy: a = -inf where b == 0
            const double z = (m[r * n_cols + j] + lp) - lse[r];
            if (z == cm) cnt += wr;
            else s += wr * exp(z - cm);
        }
    }
    part[(size_t)blockIdx.y * 2 * n_cols + j] = s;
    part[(size_t)blockIdx.y * 2 * n_cols + n_cols + j] = cnt;
}

__global__ void __launch_bounds__(256)
em_logspace_colreduce_kernel(const double *__restrict__ part, int n_part, int64_t n_cols,
                             int is_max, double *__restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= n_cols) return;
    double acc = is_max ? -INFINITY : 0.0;
    for (int b = 0; b < n_part; ++b) {
        const double v = part[(size_t)b * n_cols + j];
        acc = is_max ? fmax(acc, v) : acc + v;
    }
    out[j] = acc;
}

// ln pi' = colmax + log(colsum) - logsumexp(.), convergence test, control block (one CTA).
// With `colcnt` (row-sharded runs, em_logspace_cols_split_kernel) colsum holds scipy's s and
// colcnt its m: ln pi' = log1p(s/m) + log(m) + colmax - logsumexp(.).
__global__ void __launch_bounds__(kUpdThreads)
em_logspace_update_kernel(const double *__restrict__ colmax, const double *__restrict__ colsum,
                          const double *__restrict__ colcnt,
                          int64_t n_cols, int64_t ld, double *__restrict__ lnp0,
                          double *__restrict__ lnp1, double *__restrict__ pi0,
                          double *__restrict__ pi1, EmState *__restrict__ st) {
    __shared__ double scratch[kUpdThreads / 32];
    const int cur = st->cur;
    const double *pi_old = cur ? pi1 : pi0;
    double *lnp_new = cur ? lnp0 : lnp1;
    double *pi_new = cur ? pi0 : pi1;
    double mx = -INFINITY;
    for (int64_t j = threadIdx.x; j < n_cols; j += kUpdThreads) {
        double v = -INFINITY;
        if (colmax[j] > -INFINITY)
            v = colcnt ? log1p(colsum[j] / colcnt[j]) + log(colcnt[j]) + colmax[j]
                       : colmax[j] + log(colsum[j]);
        lnp_new[j] = v;
        mx = fmax(mx, v);
    }
    mx = block_max<kUpdThreads>(mx, scratch);
    double sum = 0.0;
    for (int64_t j = threadIdx.x; j < n_cols; j += kUpdThreads) sum += exp(lnp_new[j] - mx);
    sum = block_sum<kUpdThreads>(sum, scratch);
    const double norm = mx + log(sum);
    double dl = 0.0;
    for (int64_t j = threadIdx.x; j < ld; j += kUpdThreads) {
        const bool in = j < n_cols;
        const double v = in ? lnp_new[j] - norm : -INFINITY;
        const double p = in ? exp(v) : 0.0;
        lnp_new[j] = v;
        pi_new[j] = p;
        if (in) dl += fabs(p - pi_old[j]);
    }
    const double delta = block_sum<kUpdThreads>(dl, scratch);
    if (threadIdx.x == 0) {
        st->bad = 0;
        st->done = 0;
        advance_state(st, delta, cur);
    }
}

// Restart fan-out (mxb_matrix_fold_ranks): `own` is this rank's shard of its own fold of read
// matrices, recv[q] the same rows as folded by rank q.  numpy.logaddexp in rank order
// (em.py:156), then - log(n_multi) (em.py:161).
__global__ void fold_shards_kernel(double *__restrict__ own, const double *__restrict__ recv,
                                   int64_t slot, int64_t cells, int world, int me, double sub_log) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells;
         i += (int64_t)gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int q = 0; q < world; ++q) {
            const double v = q == me ? own[i] : recv[(int64_t)q * slot + i];
            acc = q == 0 ? v : np_logaddexp(acc, v);
        }
        own[i] = acc - sub_log;
    }
}

__global__ void fold_shift_kernel(double *__restrict__ m, int64_t n, double sub_log) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x)
        m[i] -= sub_log;
}

}  // namespace mxb
