// Kernel 3: the draws of the nonparametric bootstrap of the mixture proportions.
//
// Replicate b draws W = sum_i w_i fragments with replacement from the empirical distribution of
// the signature rows (row i carries w_i fragments).  The draw of fragment f is counter-based and
// fully specified, so that a host restatement reproduces it bit for bit and a replicate depends
// only on (w, seed, b):
//
//     (x0, x1, x2, x3) = Philox4x32-10(counter {f_lo, f_hi, b, 0}, key {seed_lo, seed_hi})
//     r = x0 | x1 << 32,  t = mulhi64(r, W)            (0 <= t < W; bias below W / 2^64)
//     row = first i with cumw[i] > t                   (cumw: inclusive prefix sums of w)
//
// A row of weight 0 is never drawn.  Counts are integer atomics: deterministic.
#include <math.h>

#include <curand_philox4x32_x.h>

#include "bootstrap.cuh"
#include "common.cuh"

namespace mxb {

constexpr int kBootThreads = 256;

__global__ void __launch_bounds__(kBootThreads)
boot_counts_kernel(const int64_t *__restrict__ cumw, int64_t n_rows, uint64_t total,
                   uint64_t seed, int64_t boot0, uint32_t *__restrict__ counts) {
    const uint64_t f = (uint64_t)blockIdx.x * kBootThreads + threadIdx.x;
    if (f >= total) return;
    const uint64_t b = (uint64_t)(boot0 + blockIdx.y);
    const uint4 x = curand_Philox4x32_10(
        make_uint4((uint32_t)f, (uint32_t)(f >> 32), (uint32_t)b, 0u),
        make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint64_t r = (uint64_t)x.x | ((uint64_t)x.y << 32);
    const int64_t t = (int64_t)__umul64hi(r, total);
    int64_t lo = 0, hi = n_rows - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(cumw + mid) > t) hi = mid;
        else lo = mid + 1;
    }
    atomicAdd(counts + (size_t)blockIdx.y * n_rows + lo, 1u);
}

__global__ void boot_take_counts_kernel(uint32_t *__restrict__ counts, int64_t n_rows,
                                        double *__restrict__ w) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows;
         i += (int64_t)gridDim.x * blockDim.x) {
        w[i] = (double)counts[i];
        counts[i] = 0u;
    }
}

int boot_prefix(const double *weights, int64_t n_rows, std::vector<int64_t> &cumw,
                uint64_t &total) {
    cumw.resize((size_t)n_rows);
    double sum = 0.0;
    int64_t acc = 0;
    for (int64_t i = 0; i < n_rows; ++i) {
        const double v = weights[i];
        if (!(v >= 0.0) || !isfinite(v) || floor(v) != v || v >= 4294967296.0) {
            set_error("bootstrap: weight %lld is %g; weights must be finite, non-negative "
                      "integers", (long long)i, v);
            return MXB_ERR_VALUE;
        }
        sum += v;
        if (sum >= 4294967296.0) {
            set_error("bootstrap: the weights sum to 2^32 or more");
            return MXB_ERR_VALUE;
        }
        acc += (int64_t)v;
        cumw[(size_t)i] = acc;
    }
    if (acc < 1) {
        set_error("bootstrap: the weights sum to 0");
        return MXB_ERR_VALUE;
    }
    total = (uint64_t)acc;
    return MXB_OK;
}

int boot_draw(mxb_ctx *ctx, const int64_t *cumw, int64_t n_rows, uint64_t total, uint64_t seed,
              int64_t boot0, int64_t n_boot, uint32_t *counts) {
    constexpr int64_t kMaxY = 65535;
    const unsigned gx = (unsigned)ceil_div((int64_t)total, kBootThreads);
    for (int64_t k = 0; k < n_boot; k += kMaxY) {
        const unsigned gy = (unsigned)std::min<int64_t>(kMaxY, n_boot - k);
        boot_counts_kernel<<<dim3(gx, gy), kBootThreads, 0, ctx->stream>>>(
            cumw, n_rows, total, seed, boot0 + k, counts + (size_t)k * n_rows);
        ctx->launches++;
    }
    MXB_CUDA(cudaGetLastError());
    return MXB_OK;
}

int boot_take_counts(mxb_ctx *ctx, uint32_t *counts, int64_t n_rows, double *w) {
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n_rows, 256),
                                                                 (int64_t)ctx->num_sms * 4));
    boot_take_counts_kernel<<<grid, 256, 0, ctx->stream>>>(counts, n_rows, w);
    ctx->launches++;
    MXB_CUDA(cudaGetLastError());
    return MXB_OK;
}

}  // namespace mxb

using namespace mxb;

extern "C" int mxb_boot_counts(mxb_ctx *ctx, const double *weights, int64_t n_rows, uint64_t seed,
                               int64_t boot0, int64_t n_boot, uint32_t *counts_out) {
    MXB_REQUIRE(ctx != nullptr && weights != nullptr && counts_out != nullptr, "NULL argument");
    MXB_REQUIRE(n_rows >= 1 && n_boot >= 1 && boot0 >= 0 && boot0 + n_boot <= (1ll << 32),
                "need n_rows >= 1, n_boot >= 1 and replicates below 2^32");
    std::vector<int64_t> cumw;
    uint64_t total = 0;
    MXB_TRY(boot_prefix(weights, n_rows, cumw, total));
    MXB_CUDA(cudaSetDevice(ctx->device));
    const size_t b_cnt = (size_t)n_boot * n_rows * sizeof(uint32_t);
    DevBlock buf;   // [prefix sums][counts]
    int64_t *d_cum = nullptr;
    uint32_t *d_cnt = nullptr;
    MXB_TRY(buf.alloc_parts(ctx, "mxb_boot_counts", [&](Carve &c) {
        d_cum = c.part<int64_t>(n_rows);
        d_cnt = c.part<uint32_t>((size_t)n_boot * n_rows);
    }));
    MXB_TRY(copy_h2d(ctx, d_cum, cumw.data(), (size_t)n_rows * sizeof(int64_t)));
    MXB_CUDA(cudaMemsetAsync(d_cnt, 0, b_cnt, ctx->stream));
    MXB_TRY(boot_draw(ctx, d_cum, n_rows, total, seed, boot0, n_boot, d_cnt));
    return copy_d2h(ctx, counts_out, d_cnt, b_cnt);
}
