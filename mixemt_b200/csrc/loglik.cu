// Kernel 4: the log-likelihood of a fit, for up to kLlMaxVec proportion vectors per read of M.
//
//     l(pi) = sum_i w_i logsumexp_j(M_ij + ln pi_j)
//
// Fast path, per row: m_i = max_j M_ij and L_ij = exp(M_ij - m_i), one exp per cell shared by
// every vector of the launch; then s_ik = sum_j L_ij pi_kj (one FMA per cell and vector) and
// l_ik = m_i + log s_ik.  A (row, vector) whose s_ik fails the EM's own rule
// (row_likelihood.cuh: row_needs_logspace) is redone in log space with scipy's max-shifted form,
// as read_mix_kernel forms it.  -inf cells and zero proportions add nothing; a row without a
// finite term gives -inf; a row of weight 0 adds exactly 0, whatever its l_i (scipy's b == 0).
//
// Determinism: block b owns a contiguous row range that depends on N and the grid only, and
// thread k adds w_i l_ik of vector k in row order into the block's partial; the host adds the
// partials in block order.  No floating-point atomics; a vector's bits do not depend on which
// vectors share its launch or on how the host splits the vectors into launches.
#include <math.h>
#include <string.h>

#include <vector>

#include "block_reduce.cuh"
#include "common.cuh"
#include "row_likelihood.cuh"

namespace mxb {

constexpr int kLlThreads = 256;
constexpr int kLlMaxVec = 16;      // vectors per launch (more are split into launches)
constexpr int kLlBlocksPerSm = 4;  // the grid: a function of N and the SM count, never of K

// One row's logsumexp_j(row_j + lnp_j) in log space (scipy: the maximal terms counted apart);
// called by the whole block, every thread gets the result.
__device__ double row_lse_logspace(const double *__restrict__ row, const double *__restrict__ lnp,
                                   int64_t n_cols, double *scratch) {
    double mx = -INFINITY;
    for (int64_t j = threadIdx.x; j < n_cols; j += kLlThreads) mx = fmax(mx, row[j] + lnp[j]);
    mx = block_max<kLlThreads>(mx, scratch);
    if (mx == -INFINITY) return -INFINITY;
    double s = 0.0, cnt = 0.0;
    for (int64_t j = threadIdx.x; j < n_cols; j += kLlThreads) {
        const double z = row[j] + lnp[j];
        if (z == mx) cnt += 1.0;
        else s += exp(z - mx);
    }
    s = block_sum<kLlThreads>(s, scratch);
    cnt = block_sum<kLlThreads>(cnt, scratch);
    return log1p(s / cnt) + log(cnt) + mx;
}

// KV vectors (n_vec of them real) over RB rows at a time.  pi_t: [n_cols][KV] proportions,
// lnp: [KV][n_cols] log-proportions (the log-space redo), partials: [gridDim.x][KV].
template <int KV, int RB>
__global__ void __launch_bounds__(kLlThreads)
loglik_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols,
              const double *__restrict__ w, const double *__restrict__ pi_t,
              const double *__restrict__ lnp, int n_vec, double *__restrict__ partials) {
    constexpr int kWarps = kLlThreads / 32, kCells = RB * KV;
    __shared__ double scratch[kWarps];
    __shared__ double red[kWarps][kCells];
    __shared__ double ll[kCells];    // s_ik
    __shared__ double lik[kCells];   // l_ik
    __shared__ double rmax[RB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t r0 = n_rows * blockIdx.x / gridDim.x;
    const int64_t r1 = n_rows * (blockIdx.x + 1) / gridDim.x;
    double acc = 0.0;   // thread k < KV: the block's sum of w_i l_ik
    for (int64_t g = r0; g < r1; g += RB) {
        const int nr = (int)min((int64_t)RB, r1 - g);
        const double *row[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) row[r] = m + (g + min(r, nr - 1)) * n_cols;
        double mx[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) mx[r] = -INFINITY;
#pragma unroll 4
        for (int64_t j = tid; j < n_cols; j += kLlThreads) {
#pragma unroll
            for (int r = 0; r < RB; ++r) mx[r] = fmax(mx[r], row[r][j]);
        }
        double shift[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
            mx[r] = block_max<kLlThreads>(mx[r], scratch);
            shift[r] = mx[r] == -INFINITY ? 0.0 : mx[r];   // a row of -inf cells: L = 0
            if (tid == 0) rmax[r] = mx[r];
        }
        double s[RB][KV];
#pragma unroll
        for (int r = 0; r < RB; ++r)
#pragma unroll
            for (int k = 0; k < KV; ++k) s[r][k] = 0.0;
        for (int64_t j = tid; j < n_cols; j += kLlThreads) {
            double p[KV];
            if constexpr (KV == 1) {
                p[0] = __ldg(pi_t + j);
            } else {
                const double2 *pv = reinterpret_cast<const double2 *>(pi_t + j * KV);
#pragma unroll
                for (int k = 0; k < KV / 2; ++k) {
                    const double2 v = __ldg(pv + k);
                    p[2 * k] = v.x;
                    p[2 * k + 1] = v.y;
                }
            }
#pragma unroll
            for (int r = 0; r < RB; ++r) {
                const double l = exp(row[r][j] - shift[r]);
#pragma unroll
                for (int k = 0; k < KV; ++k) s[r][k] = fma(l, p[k], s[r][k]);
            }
        }
#pragma unroll
        for (int r = 0; r < RB; ++r)
#pragma unroll
            for (int k = 0; k < KV; ++k) {
                const double v = warp_sum(s[r][k]);
                if (lane == 0) red[warp][r * KV + k] = v;
            }
        __syncthreads();
        if (tid < kCells) {
            double t = 0.0;
#pragma unroll
            for (int q = 0; q < kWarps; ++q) t += red[q][tid];
            ll[tid] = t;
        }
        __syncthreads();
        // l_ik in the fast form; a pair that fails the rule is redone in log space by the whole
        // block (the decisions read shared sums: block-uniform)
        bool need = false;
        if (tid < nr * KV) {
            const int r = tid / KV, k = tid - r * KV;
            const double t = ll[tid], mr = rmax[r];
            lik[tid] = mr == -INFINITY ? -INFINITY : mr + log(t);
            need = k < n_vec && mr != -INFINITY && w[g + r] != 0.0 && row_needs_logspace(t);
        }
        if (__syncthreads_or(need)) {
            for (int c = 0; c < nr * KV; ++c) {
                const int r = c / KV, k = c - r * KV;
                if (k < n_vec && rmax[r] != -INFINITY && w[g + r] != 0.0 &&
                    row_needs_logspace(ll[c])) {
                    const double v = row_lse_logspace(m + (g + r) * n_cols,
                                                      lnp + (int64_t)k * n_cols, n_cols, scratch);
                    if (tid == 0) lik[c] = v;
                }
            }
            __syncthreads();
        }
        if (tid < n_vec) {
            for (int r = 0; r < nr; ++r) {
                const double wr = w[g + r];
                if (wr != 0.0) acc += wr * lik[r * KV + tid];
            }
        }
        __syncthreads();   // red, ll, lik and rmax free for the next rows
    }
    if (tid < KV) partials[(int64_t)blockIdx.x * KV + tid] = acc;
}

template <int KV>
static void launch_loglik(mxb_ctx *ctx, int grid, const mxb_matrix *m, const double *w,
                          const double *pi_t, const double *lnp, int n_vec, double *partials) {
    constexpr int RB = KV <= 4 ? 4 : 2;
    loglik_kernel<KV, RB><<<grid, kLlThreads, 0, ctx->stream>>>(m->data, m->n_rows, m->n_cols, w,
                                                                 pi_t, lnp, n_vec, partials);
}

}  // namespace mxb

using namespace mxb;

extern "C" int mxb_matrix_loglik(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                                 const double *lnprops, int64_t n_vec, double *out) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr && lnprops != nullptr && out != nullptr,
                "NULL argument");
    MXB_REQUIRE(n_vec >= 1 && m->n_cols >= 1, "need n_vec >= 1 and a matrix with columns");
    MXB_REQUIRE(weights != nullptr || m->n_rows == 0, "weights is NULL");
    const int64_t n = m->n_rows, h = m->n_cols;
    for (int64_t i = 0; i < n_vec * h; ++i) {
        if (isnan(lnprops[i])) {
            set_error("mxb_matrix_loglik: log-proportion %lld of vector %lld is NaN",
                      (long long)(i % h), (long long)(i / h));
            return MXB_ERR_VALUE;
        }
    }
    for (int64_t k = 0; k < n_vec; ++k) out[k] = 0.0;
    if (n == 0) return MXB_OK;   // a rank of a row-sharded run may hold no rows
    MXB_CUDA(cudaSetDevice(ctx->device));
    const int grid = (int)std::min<int64_t>(n, (int64_t)ctx->num_sms * kLlBlocksPerSm);
    DevBlock buf;   // [weights][pi_t][lnp][partials]
    double *d_w = nullptr, *d_pi = nullptr, *d_lnp = nullptr, *d_part = nullptr;
    MXB_TRY(buf.alloc_parts(ctx, "mxb_matrix_loglik", [&](Carve &c) {
        d_w = c.part<double>(n);
        d_pi = c.part<double>((size_t)h * kLlMaxVec);
        d_lnp = c.part<double>((size_t)h * kLlMaxVec);
        d_part = c.part<double>((size_t)grid * kLlMaxVec);
    }));
    MXB_TRY(copy_h2d(ctx, d_w, weights, (size_t)n * sizeof(double)));
    std::vector<double> pi_t, part;
    try {
        pi_t.resize((size_t)h * kLlMaxVec);
        part.resize((size_t)grid * kLlMaxVec);
    } catch (const std::bad_alloc &) {
        set_error("mxb_matrix_loglik: out of host memory");
        return MXB_ERR_NOMEM;
    }
    for (int64_t k0 = 0; k0 < n_vec; k0 += kLlMaxVec) {
        const int cnt = (int)std::min<int64_t>(kLlMaxVec, n_vec - k0);
        const int kv = cnt <= 1 ? 1 : cnt <= 2 ? 2 : cnt <= 4 ? 4 : cnt <= 8 ? 8 : 16;
        const double *src = lnprops + k0 * h;
        for (int64_t j = 0; j < h; ++j)
            for (int k = 0; k < kv; ++k)
                pi_t[(size_t)j * kv + k] = k < cnt ? exp(src[k * h + j]) : 0.0;
        MXB_TRY(copy_h2d(ctx, d_pi, pi_t.data(), (size_t)h * kv * sizeof(double)));
        MXB_TRY(copy_h2d(ctx, d_lnp, src, (size_t)h * cnt * sizeof(double)));
        switch (kv) {
            case 1: launch_loglik<1>(ctx, grid, m, d_w, d_pi, d_lnp, cnt, d_part); break;
            case 2: launch_loglik<2>(ctx, grid, m, d_w, d_pi, d_lnp, cnt, d_part); break;
            case 4: launch_loglik<4>(ctx, grid, m, d_w, d_pi, d_lnp, cnt, d_part); break;
            case 8: launch_loglik<8>(ctx, grid, m, d_w, d_pi, d_lnp, cnt, d_part); break;
            default: launch_loglik<16>(ctx, grid, m, d_w, d_pi, d_lnp, cnt, d_part); break;
        }
        ctx->launches++;
        MXB_CUDA(cudaGetLastError());
        MXB_TRY(copy_d2h(ctx, part.data(), d_part, (size_t)grid * kv * sizeof(double)));
        for (int k = 0; k < cnt; ++k) {
            double total = 0.0;
            for (int b = 0; b < grid; ++b) total += part[(size_t)b * kv + k];
            out[k0 + k] = total;
        }
    }
    return MXB_OK;
}
