// Shared internals of libmixemt_b200 (not part of the C-ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <vector>

#include "block_pool.h"
#include "mixemt_b200.h"

namespace mxb {

void set_error(const char *fmt, ...);

#define MXB_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t err__ = (call);                                           \
        if (err__ != cudaSuccess) {                                           \
            mxb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,      \
                           cudaGetErrorString(err__));                        \
            return MXB_ERR_CUDA;                                              \
        }                                                                     \
    } while (0)

#define MXB_REQUIRE(cond, msg)                                                \
    do {                                                                      \
        if (!(cond)) {                                                        \
            mxb::set_error("%s: %s", __func__, msg);                          \
            return MXB_ERR_ARG;                                               \
        }                                                                     \
    } while (0)

#define MXB_TRY(call)                                                         \
    do {                                                                      \
        int rc__ = (call);                                                    \
        if (rc__ != MXB_OK) return rc__;                                      \
    } while (0)

// Minimal NCCL surface, resolved with dlopen so that the library loads (and
// single-GPU runs work) without libnccl on the link line.
struct NcclApi;

constexpr int kNumSMsFallback = 148;  // B200
constexpr int kP2PMaxWorld = 8;       // one NVSwitch domain
constexpr int kP2PMaxLd = 8192;       // widest row of the fused EM tail
constexpr size_t kP2PInboxOffset = 256;
constexpr size_t kP2PBlockBytes = kP2PInboxOffset + (size_t)2 * kP2PMaxWorld * kP2PMaxLd * 8;

// Device memory for matrix-sized buffers comes from the context's pool (api.cu).  cudaMalloc /
// cudaFree of multi-GB blocks cost 1-10 ms each and now and then 0.1-1 s (measured on the B200
// boxes), which is visible next to a 1.4 s run_em call; freed blocks of >= 1 MiB are therefore
// kept per context (up to MXB_CACHE_MB, default a quarter of the device memory) and handed out
// again to requests of about the same size (1/8 slack).  An allocation that fails releases the
// cache and retries.  dev_alloc gives nullptr on failure; code outside api.cu holds its blocks
// in a DevBlock.
constexpr size_t kCacheMinBlock = (size_t)1 << 20;   // smallest block the cache keeps
void *dev_alloc(mxb_ctx *ctx, size_t bytes);
void dev_free(mxb_ctx *ctx, void *ptr);
void *cuda_block_new(size_t bytes);   // the pool's cudaMalloc (nullptr on failure) and cudaFree
void cuda_block_delete(void *ptr);

// The parts of a device block, each starting 256-byte aligned.  The same calls size the block
// (no base: every part is nullptr and bytes() is the block's size) and point the parts into it.
class Carve {
public:
    explicit Carve(void *base = nullptr) : base_((unsigned char *)base) {}
    template <typename T> T *part(size_t count) { return parts<T>(count, 1); }
    // n parts of `count` T each; *stride (optional) gets the distance between them in T
    template <typename T> T *parts(size_t count, size_t n, int64_t *stride = nullptr) {
        const size_t b = (count * sizeof(T) + 255) & ~(size_t)255;
        T *p = base_ ? reinterpret_cast<T *>(base_ + off_) : nullptr;
        off_ += n * b;
        if (stride) *stride = (int64_t)(b / sizeof(T));
        return p;
    }
    size_t bytes() const { return off_; }

private:
    unsigned char *base_;
    size_t off_ = 0;
};

// One block of a context's device pool, given back (dev_free) when its owner goes out of scope.
class DevBlock {
public:
    DevBlock() = default;
    DevBlock(DevBlock &&o) noexcept { *this = std::move(o); }
    DevBlock &operator=(DevBlock &&o) noexcept {   // our old block leaves with `o`
        std::swap(ctx_, o.ctx_);
        std::swap(p_, o.p_);
        return *this;
    }
    DevBlock(const DevBlock &) = delete;
    DevBlock &operator=(const DevBlock &) = delete;
    ~DevBlock() { reset(); }

    // MXB_OK, or MXB_ERR_NOMEM with an error naming `who` and the byte count.  0 bytes give a
    // null block and succeed (a rank of a row-sharded run may hold no rows).
    int alloc(mxb_ctx *ctx, size_t bytes, const char *who);
    // A block of the parts layout(Carve &) lays out (at least min_bytes), and the parts pointed
    // into it by a second call of layout.
    template <typename Layout>
    int alloc_parts(mxb_ctx *ctx, const char *who, Layout layout, size_t min_bytes = 0) {
        Carve size;
        layout(size);
        MXB_TRY(alloc(ctx, std::max(size.bytes(), min_bytes), who));
        Carve parts(p_);
        layout(parts);
        return MXB_OK;
    }
    void reset();
    template <typename T = unsigned char> T *get() const { return static_cast<T *>(p_); }

private:
    mxb_ctx *ctx_ = nullptr;
    void *p_ = nullptr;
};

// CUDA events, destroyed with their owner.
class Events {
public:
    Events() = default;
    Events(const Events &) = delete;
    Events &operator=(const Events &) = delete;
    ~Events() { for (cudaEvent_t e : ev_) cudaEventDestroy(e); }
    // MXB_OK, MXB_ERR_NOMEM or MXB_ERR_CUDA (the error names `who`)
    int create(size_t n, unsigned flags, const char *who);
    cudaEvent_t operator[](size_t i) const { return ev_[i]; }
    cudaEvent_t *data() { return ev_.data(); }

private:
    std::vector<cudaEvent_t> ev_;
};

}  // namespace mxb

struct mxb_ctx {
    int device = 0;
    int num_sms = mxb::kNumSMsFallback;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int64_t launches = 0;
    // pinned staging ring of the host<->device copy engine (api.cu), lazily allocated
    void *stage_buf[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t stage_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t stage_chunk = 0;
    // device memory of the context (api.cu: dev_alloc / dev_free); MXB_DEBUG_FAIL_ALLOC=k makes
    // allocation number k fail as out of memory would
    mxb::BlockPool pool{mxb::cuda_block_new, mxb::cuda_block_delete, 8, mxb::kCacheMinBlock};
    int64_t fail_alloc_at = 0;
    std::atomic<int64_t> n_allocs{0};
    void *pinned = nullptr;  // small pinned host scratch (control-block polling), lazily allocated
    // NCCL (optional)
    void *nccl_comm = nullptr;
    int rank = 0;
    int world = 1;
    // Peer-memory mailboxes of the fused EM tail (api.cu: p2p_setup).  Every rank owns one
    // cudaMalloc'ed block [flags: 2 x world u64][seq u64][inbox: 2 x world x kP2PMaxLd doubles]
    // and maps the blocks of its peers through CUDA IPC over NVLink.
    bool p2p_ready = false;
    mxb::DevBlock p2p_vote;       // one device double for the barriers of p2p_resync
    unsigned char *p2p_block[mxb::kP2PMaxWorld] = {};  // [r] = rank r's block as seen from here
};

struct mxb_matrix {
    mxb_ctx *ctx = nullptr;
    mxb::DevBlock mem;
    double *data = nullptr;  // row-major, stride n_cols (in mem)
    int64_t n_rows = 0;
    int64_t n_cols = 0;
};

struct mxb_phylo {
    mxb_ctx *ctx = nullptr;
    int32_t n_pos = 0;
    int32_t n_hap = 0;
    int32_t n_sym = 0;     // planes 0..n_sym-1, plane n_sym is all-zero ("other")
    int32_t n_words = 0;   // 32-bit words per plane (padded to a multiple of 4)
    mxb::DevBlock mem;     // the tables below
    uint32_t *bits = nullptr;   // [n_pos][n_sym+1][n_words]
    double2 *hitmiss = nullptr; // [n_pos] (hit, miss)
    // sparse deviation form of `bits` (see build.cu)
    uint8_t *plane_base = nullptr;  // [n_pos * (n_sym+1)] baseline outcome of the plane
    int32_t *dev_ptr = nullptr;   // [n_pos * (n_sym+1) + 1]
    uint2 *dev_ent = nullptr;     // {word index, D}
    int64_t n_dev = 0;
};

namespace mxb {

int nccl_allreduce_sum_f64(mxb_ctx *ctx, double *dev_buf, int64_t n);
int nccl_allreduce_f64(mxb_ctx *ctx, double *dev_buf, int64_t n, int op_is_max);
int nccl_alltoall_rows(mxb_ctx *ctx, const double *src, double *recv, int64_t n_rows,
                       int64_t n_cols, int64_t slot_doubles);
int nccl_allgather_rows(mxb_ctx *ctx, double *m, int64_t n_rows, int64_t n_cols);
int p2p_resync(mxb_ctx *ctx);   // zero the peer mailboxes behind a barrier (start of a sharded session)

// Host <-> device copies of matrix-sized buffers (api.cu).  Pageable host memory
// goes through a pinned staging ring filled/drained by several host threads
// (~43 GB/s instead of 11-19 GB/s for a plain pageable cudaMemcpy); pinned or
// registered host memory is copied directly.  Both return after completion.
int copy_h2d(mxb_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int copy_d2h(mxb_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
constexpr size_t kPinnedScratchBytes = 4096;
void *pinned_scratch(mxb_ctx *ctx);  // kPinnedScratchBytes of pinned host memory, NULL on failure

// Touch every page of a caller-owned *output* buffer from background threads
// while the GPU works, so that the final copy does not pay first-touch faults.
struct Prefault {
    void *impl = nullptr;
    void start(void *buf, size_t bytes);
    void join();
    ~Prefault() { join(); }
};

// Wall-clock stage times of the one-call entry points (upload, session set-up, iterations,
// read-matrix kernel, download), collected when mxb_stage_timing(1) is on (or MXB_TIMING=1,
// which also prints them): bench.py's e2e breakdown.  Index = Stage.
enum Stage { kStageH2D = 0, kStageSetup, kStageIterate, kStageReadMix, kStageD2H, kStageOther,
             kNumStages };
extern bool g_stage_on;
extern double g_stage_ms[kNumStages];

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

}  // namespace mxb
