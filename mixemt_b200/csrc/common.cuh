// Shared internals of libmixemt_b200 (not part of the C-ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

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
    // cache of large freed device blocks (api.cu: dev_alloc / dev_free)
    void *block_cache = nullptr;
    void *pinned = nullptr;  // small pinned host scratch (control-block polling), lazily allocated
    // NCCL (optional)
    void *nccl_comm = nullptr;
    int rank = 0;
    int world = 1;
    // Peer-memory mailboxes of the fused EM tail (api.cu: p2p_setup).  Every rank owns one
    // cudaMalloc'ed block [flags: 2 x world u64][seq u64][inbox: 2 x world x kP2PMaxLd doubles]
    // and maps the blocks of its peers through CUDA IPC over NVLink.
    bool p2p_ready = false;
    double *p2p_vote = nullptr;   // one device double for the barriers of p2p_resync
    unsigned char *p2p_block[mxb::kP2PMaxWorld] = {};  // [r] = rank r's block as seen from here
};

struct mxb_matrix {
    mxb_ctx *ctx = nullptr;
    double *data = nullptr;  // row-major, stride n_cols
    int64_t n_rows = 0;
    int64_t n_cols = 0;
};

struct mxb_phylo {
    mxb_ctx *ctx = nullptr;
    int32_t n_pos = 0;
    int32_t n_hap = 0;
    int32_t n_sym = 0;     // planes 0..n_sym-1, plane n_sym is all-zero ("other")
    int32_t n_words = 0;   // 32-bit words per plane (padded to a multiple of 4)
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
// Device memory for matrix-sized buffers.  cudaMalloc / cudaFree of multi-GB blocks
// cost 1-10 ms each and now and then 0.1-1 s (measured on the B200 boxes), which is
// visible next to a 1.4 s run_em call; freed blocks of >= 1 MiB are therefore kept
// per context (up to MXB_CACHE_MB, default a quarter of the device memory) and
// handed out again to requests of about the same size.  An allocation that fails
// releases the cache and retries.  The cache is guarded by a mutex (a Python GC may free a
// matrix from any thread).
constexpr size_t kPinnedScratchBytes = 4096;
void *pinned_scratch(mxb_ctx *ctx);  // kPinnedScratchBytes of pinned host memory, NULL on failure
constexpr size_t kCacheMinBlock = (size_t)1 << 20;   // smallest block the cache keeps
cudaError_t dev_alloc(mxb_ctx *ctx, void **out, size_t bytes);
void dev_free(mxb_ctx *ctx, void *ptr);
void dev_cache_release(mxb_ctx *ctx);

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
// Byte size of one part of a device block whose parts each start 256-byte aligned.
inline size_t align256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

}  // namespace mxb
