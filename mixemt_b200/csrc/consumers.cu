// Device-side forms of the consumers that sit right after the EM fit in the
// reference's pipeline (SURVEY.md 8f, rows N2-N4).  They keep the N x H result
// in HBM instead of walking it on the host:
//
//   mxb_matrix_gather_cols   preprocess.reduce_em_matrix   (preprocess.py:230-251)
//   mxb_matrix_vote_count    assemble._find_contribs_from_reads (assemble.py:102-124),
//                            stats.report_read_votes        (stats.py:34-46)
//   mxb_matrix_vote_first    the same votes plus each column's first row, over a row shard
//   mxb_assign_reads         assemble.assign_read_indexes   (assemble.py:267-334)
//   mxb_matrix_{down,up}load_rows   row-range transfers for streaming .npy files
//                            (bin/mixemt:214-245 dump_all / :168-211 load_prev)
#include <math.h>

#include <algorithm>
#include <memory>

#include "common.cuh"

namespace mxb {

// dst[r][k] = src[r][cols[k]]
__global__ void __launch_bounds__(256)
gather_cols_kernel(const double *__restrict__ src, int64_t n_rows, int64_t src_cols,
                   const int64_t *__restrict__ cols, int64_t n_out, double *__restrict__ dst) {
    const int64_t total = n_rows * n_out;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / n_out, k = i - r * n_out;
        dst[i] = src[r * src_cols + cols[k]];
    }
}

// votes[argmax[r]] += weights[r]; with first != nullptr also first[argmax[r]] = min(row0 + r).
// Integer atomics: the result does not depend on the order the rows are visited in.
__global__ void __launch_bounds__(256)
vote_kernel(const int64_t *__restrict__ best, const int64_t *__restrict__ weights, int64_t n_rows,
            unsigned long long *__restrict__ votes, unsigned long long *__restrict__ first,
            int64_t row0) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows;
         r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = best[r];
        atomicAdd(&votes[j], (unsigned long long)weights[r]);
        if (first) atomicMin(&first[j], (unsigned long long)(row0 + r));
    }
}

// Per row: the two contributor columns with the highest read_mix - ln(props)
// (assemble.py:319-323) and the odds-ratio test (:325).  Ties are ordered as a
// reversed stable ascending sort would order them (the higher column first);
// with min_fold > 1 a tie between the top two is unassigned either way.
__global__ void __launch_bounds__(256)
assign_reads_kernel(const double *__restrict__ mix, int64_t n_rows, int64_t n_cols,
                    const int64_t *__restrict__ con_cols, const double *__restrict__ con_lnprops,
                    int n_con, double ln_min_fold, int32_t *__restrict__ out) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows;
         r += (int64_t)gridDim.x * blockDim.x) {
        const double *row = mix + r * n_cols;
        double best_v = 0.0, next_v = 0.0;
        int best_k = -1, next_k = -1;
        int64_t best_c = -1, next_c = -1;
        for (int k = 0; k < n_con; ++k) {
            const int64_t c = con_cols[k];
            const double v = row[c] - con_lnprops[k];
            const bool beats_best = best_k < 0 || v > best_v || (v == best_v && c > best_c);
            if (beats_best) {
                next_v = best_v; next_k = best_k; next_c = best_c;
                best_v = v; best_k = k; best_c = c;
            } else if (next_k < 0 || v > next_v || (v == next_v && c > next_c)) {
                next_v = v; next_k = k; next_c = c;
            }
        }
        int32_t res = -1;
        if (n_con == 1) res = 0;
        else if (best_k >= 0 && next_k >= 0 && best_v - next_v >= ln_min_fold) res = best_k;
        out[r] = res;
    }
}

// First maximum of every row (numpy.argmax semantics; NaN wins like numpy).
__global__ void argmax_rows_kernel(const double *__restrict__ m, int64_t n_rows,
                                   int64_t n_cols, int64_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        const double *row = m + r * n_cols;
        double best = 0.0;
        int64_t best_j = INT64_MAX;
        bool best_nan = false;
        for (int64_t j = lane; j < n_cols; j += 32) {
            double v = row[j];
            bool v_nan = (v != v);
            if (best_j == INT64_MAX || (!best_nan && (v_nan || v > best))) {
                best = v; best_j = j; best_nan = v_nan;
            }
        }
        for (int off = 16; off > 0; off >>= 1) {
            double ov = __shfl_xor_sync(0xffffffffu, best, off);
            long long oj = __shfl_xor_sync(0xffffffffu, (long long)best_j, off);
            int on = __shfl_xor_sync(0xffffffffu, (int)best_nan, off);
            if (oj == INT64_MAX) continue;
            bool take;
            if (best_j == INT64_MAX) take = true;
            else if (best_nan || on) take = on && (!best_nan || oj < best_j);
            else take = (ov > best) || (ov == best && oj < best_j);
            if (take) { best = ov; best_j = oj; best_nan = on; }
        }
        if (lane == 0) out[r] = best_j == INT64_MAX ? 0 : best_j;
    }
}


static int grid_for(mxb_ctx *ctx, int64_t items, int per_block) {
    return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(items, per_block),
                                                       (int64_t)ctx->num_sms * 16));
}

}  // namespace mxb

using namespace mxb;

extern "C" {

int mxb_matrix_gather_cols(mxb_ctx *ctx, const mxb_matrix *src, const int64_t *cols,
                           int64_t n_out, mxb_matrix **out) {
    MXB_REQUIRE(ctx != nullptr && src != nullptr && out != nullptr, "NULL argument");
    MXB_REQUIRE(n_out >= 0 && (n_out == 0 || cols != nullptr), "bad column list");
    *out = nullptr;
    for (int64_t k = 0; k < n_out; ++k) {
        if (cols[k] < 0 || cols[k] >= src->n_cols) {
            set_error("mxb_matrix_gather_cols: column %lld out of range (%lld columns)",
                      (long long)cols[k], (long long)src->n_cols);
            return MXB_ERR_ARG;
        }
    }
    MXB_CUDA(cudaSetDevice(ctx->device));
    mxb_matrix *m = nullptr;
    MXB_TRY(mxb_matrix_alloc(ctx, src->n_rows, n_out, &m));
    std::unique_ptr<mxb_matrix, decltype(&mxb_matrix_destroy)> dst(m, mxb_matrix_destroy);
    const int64_t total = src->n_rows * n_out;
    if (total > 0) {
        DevBlock d_cols;
        MXB_TRY(d_cols.alloc(ctx, n_out * sizeof(int64_t), __func__));
        MXB_CUDA(cudaMemcpyAsync(d_cols.get(), cols, n_out * sizeof(int64_t), cudaMemcpyHostToDevice,
                                 ctx->stream));
        gather_cols_kernel<<<grid_for(ctx, total, 256), 256, 0, ctx->stream>>>(
            src->data, src->n_rows, src->n_cols, d_cols.get<int64_t>(), n_out, m->data);
        ctx->launches++;
        MXB_CUDA(cudaGetLastError());
        MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    *out = dst.release();
    return MXB_OK;
}

}  // extern "C"

// Row argmax + weighted votes over m's rows; first_out (nullable) gets each column's smallest
// row0 + r (-1: no row votes for it), argmax_out (nullable) the row maxima positions.
static int vote_rows(mxb_ctx *ctx, const mxb_matrix *m, const int64_t *weights, int64_t row0,
                     int64_t *votes_out, int64_t *first_out, int64_t *argmax_out,
                     const char *what) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL argument");
    MXB_REQUIRE(m->n_cols > 0 || m->n_rows == 0, "vote count over empty rows");
    MXB_REQUIRE(votes_out != nullptr || m->n_cols == 0, "votes_out is NULL");
    MXB_REQUIRE(row0 >= 0, "negative first row");
    for (int64_t j = 0; j < m->n_cols; ++j) votes_out[j] = 0;
    if (first_out)
        for (int64_t j = 0; j < m->n_cols; ++j) first_out[j] = -1;
    if (m->n_rows == 0) return MXB_OK;
    MXB_REQUIRE(weights != nullptr, "weights is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    DevBlock buf;   // [row maxima][weights][votes][first rows]
    int64_t *d_best = nullptr, *d_w = nullptr;
    unsigned long long *d_votes = nullptr, *d_first = nullptr;
    MXB_TRY(buf.alloc_parts(ctx, what, [&](Carve &c) {
        d_best = c.part<int64_t>(m->n_rows);
        d_w = c.part<int64_t>(m->n_rows);
        d_votes = c.part<unsigned long long>(m->n_cols);
        if (first_out) d_first = c.part<unsigned long long>(m->n_cols);
    }));
    cudaStream_t s = ctx->stream;
    MXB_CUDA(cudaMemcpyAsync(d_w, weights, m->n_rows * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    MXB_CUDA(cudaMemsetAsync(d_votes, 0, m->n_cols * sizeof(unsigned long long), s));
    if (d_first)      // all bits set: UINT64_MAX, no row yet (-1 as int64_t)
        MXB_CUDA(cudaMemsetAsync(d_first, 0xff, m->n_cols * sizeof(unsigned long long), s));
    const int blocks = (int)std::min<int64_t>(ceil_div(m->n_rows, 8), (int64_t)ctx->num_sms * 8);
    argmax_rows_kernel<<<blocks, 256, 0, s>>>(m->data, m->n_rows, m->n_cols, d_best);
    vote_kernel<<<grid_for(ctx, m->n_rows, 256), 256, 0, s>>>(d_best, d_w, m->n_rows, d_votes,
                                                              d_first, row0);
    ctx->launches += 2;
    MXB_CUDA(cudaGetLastError());
    MXB_CUDA(cudaMemcpyAsync(votes_out, d_votes, m->n_cols * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    if (d_first)
        MXB_CUDA(cudaMemcpyAsync(first_out, d_first, m->n_cols * sizeof(int64_t),
                                 cudaMemcpyDeviceToHost, s));
    if (argmax_out)
        MXB_CUDA(cudaMemcpyAsync(argmax_out, d_best, m->n_rows * sizeof(int64_t),
                                 cudaMemcpyDeviceToHost, s));
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;     // an untouched first[j] (UINT64_MAX) reads back as int64_t -1
}

extern "C" {

int mxb_matrix_vote_count(mxb_ctx *ctx, const mxb_matrix *m, const int64_t *weights,
                          int64_t *votes_out, int64_t *argmax_out) {
    return vote_rows(ctx, m, weights, 0, votes_out, nullptr, argmax_out, "mxb_matrix_vote_count");
}

int mxb_matrix_vote_first(mxb_ctx *ctx, const mxb_matrix *m, const int64_t *weights,
                          int64_t row0, int64_t *votes_out, int64_t *first_out) {
    MXB_REQUIRE(first_out != nullptr || m == nullptr || m->n_cols == 0, "first_out is NULL");
    return vote_rows(ctx, m, weights, row0, votes_out, first_out, nullptr, "mxb_matrix_vote_first");
}

int mxb_assign_reads(mxb_ctx *ctx, const mxb_matrix *read_mix, const int64_t *con_cols,
                     const double *con_lnprops, int32_t n_con, double ln_min_fold,
                     int32_t *assign_out) {
    MXB_REQUIRE(ctx != nullptr && read_mix != nullptr, "NULL argument");
    MXB_REQUIRE(n_con >= 1 && con_cols != nullptr && con_lnprops != nullptr,
                "need at least one contributor");
    for (int k = 0; k < n_con; ++k) {
        if (con_cols[k] < 0 || con_cols[k] >= read_mix->n_cols) {
            set_error("mxb_assign_reads: contributor column %lld out of range",
                      (long long)con_cols[k]);
            return MXB_ERR_ARG;
        }
    }
    if (read_mix->n_rows == 0) return MXB_OK;
    MXB_REQUIRE(assign_out != nullptr, "assign_out is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    DevBlock buf;   // [contributor columns][their log-proportions][assignments]
    int64_t *d_cols = nullptr;
    double *d_ln = nullptr;
    int32_t *d_out = nullptr;
    MXB_TRY(buf.alloc_parts(ctx, __func__, [&](Carve &c) {
        d_cols = c.part<int64_t>(n_con);
        d_ln = c.part<double>(n_con);
        d_out = c.part<int32_t>(read_mix->n_rows);
    }));
    cudaStream_t s = ctx->stream;
    MXB_CUDA(cudaMemcpyAsync(d_cols, con_cols, n_con * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    MXB_CUDA(cudaMemcpyAsync(d_ln, con_lnprops, n_con * sizeof(double), cudaMemcpyHostToDevice, s));
    assign_reads_kernel<<<grid_for(ctx, read_mix->n_rows, 256), 256, 0, s>>>(
        read_mix->data, read_mix->n_rows, read_mix->n_cols, d_cols, d_ln, n_con, ln_min_fold, d_out);
    ctx->launches++;
    MXB_CUDA(cudaGetLastError());
    MXB_CUDA(cudaMemcpyAsync(assign_out, d_out, read_mix->n_rows * sizeof(int32_t),
                             cudaMemcpyDeviceToHost, s));
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

int mxb_matrix_argmax_rows(mxb_ctx *ctx, const mxb_matrix *m, int64_t *out_host) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL argument");
    if (m->n_rows == 0) return MXB_OK;
    MXB_REQUIRE(out_host != nullptr, "out_host is NULL");
    MXB_REQUIRE(m->n_cols > 0, "argmax of empty rows");
    MXB_CUDA(cudaSetDevice(ctx->device));
    DevBlock d;
    MXB_TRY(d.alloc(ctx, m->n_rows * sizeof(int64_t), __func__));
    int blocks = (int)std::min<int64_t>(ceil_div(m->n_rows, 8), (int64_t)ctx->num_sms * 8);
    argmax_rows_kernel<<<blocks, 256, 0, ctx->stream>>>(m->data, m->n_rows, m->n_cols, d.get<int64_t>());
    ctx->launches++;
    MXB_CUDA(cudaGetLastError());
    MXB_CUDA(cudaMemcpyAsync(out_host, d.get(), m->n_rows * sizeof(int64_t), cudaMemcpyDeviceToHost,
                             ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXB_OK;
}

int mxb_matrix_download_rows(mxb_ctx *ctx, const mxb_matrix *m, int64_t row0, int64_t n_rows,
                             double *host) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL argument");
    MXB_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= m->n_rows, "row range out of bounds");
    const size_t bytes = (size_t)n_rows * (size_t)m->n_cols * sizeof(double);
    if (!bytes) return MXB_OK;
    MXB_REQUIRE(host != nullptr, "host is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    return copy_d2h(ctx, host, m->data + row0 * m->n_cols, bytes);
}

int mxb_matrix_upload_rows(mxb_ctx *ctx, mxb_matrix *m, int64_t row0, int64_t n_rows,
                           const double *host) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL argument");
    MXB_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= m->n_rows, "row range out of bounds");
    const size_t bytes = (size_t)n_rows * (size_t)m->n_cols * sizeof(double);
    if (!bytes) return MXB_OK;
    MXB_REQUIRE(host != nullptr, "host is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    return copy_h2d(ctx, m->data + row0 * m->n_cols, host, bytes);
}

}  // extern "C"
