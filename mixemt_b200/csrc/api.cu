// Context, device matrices, NCCL plumbing and error reporting of libmixemt_b200.
#include <dlfcn.h>
#include <omp.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <new>
#include <thread>
#include <utility>
#include <vector>

#include "common.cuh"

namespace mxb {

static thread_local char g_error[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

// ---------------------------------------------------------------------------
// NCCL through dlopen: only the five calls the EM loop needs.
// ---------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid_t;
typedef int (*fn_get_uid)(nccl_uid_t *);
typedef int (*fn_comm_init_rank)(void **, int, nccl_uid_t, int);
typedef int (*fn_comm_destroy)(void *);
typedef int (*fn_allreduce)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_allgather)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef const char *(*fn_error_string)(int);
typedef int (*fn_send)(const void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_recv)(void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_bcast)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_group)(void);

struct NcclApi {
    void *handle = nullptr;
    fn_get_uid get_uid = nullptr;
    fn_comm_init_rank init_rank = nullptr;
    fn_comm_destroy destroy = nullptr;
    fn_allreduce allreduce = nullptr;
    fn_allgather allgather = nullptr;
    fn_error_string error_string = nullptr;
    fn_send send = nullptr;
    fn_recv recv = nullptr;
    fn_bcast bcast = nullptr;
    fn_group group_start = nullptr, group_end = nullptr;
};

static NcclApi g_nccl;

static int load_nccl() {
    if (g_nccl.handle) return MXB_OK;
    const char *names[] = {getenv("MXB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *n : names) {
        if (!n || !*n) continue;
        h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) {
        set_error("cannot dlopen libnccl.so.2 (set MXB_NCCL_LIB): %s", dlerror());
        return MXB_ERR_CUDA;
    }
    g_nccl.get_uid = (fn_get_uid)dlsym(h, "ncclGetUniqueId");
    g_nccl.init_rank = (fn_comm_init_rank)dlsym(h, "ncclCommInitRank");
    g_nccl.destroy = (fn_comm_destroy)dlsym(h, "ncclCommDestroy");
    g_nccl.allreduce = (fn_allreduce)dlsym(h, "ncclAllReduce");
    g_nccl.allgather = (fn_allgather)dlsym(h, "ncclAllGather");
    g_nccl.error_string = (fn_error_string)dlsym(h, "ncclGetErrorString");
    g_nccl.send = (fn_send)dlsym(h, "ncclSend");
    g_nccl.recv = (fn_recv)dlsym(h, "ncclRecv");
    g_nccl.bcast = (fn_bcast)dlsym(h, "ncclBroadcast");
    g_nccl.group_start = (fn_group)dlsym(h, "ncclGroupStart");
    g_nccl.group_end = (fn_group)dlsym(h, "ncclGroupEnd");
    if (!g_nccl.get_uid || !g_nccl.init_rank || !g_nccl.destroy || !g_nccl.allreduce) {
        set_error("libnccl is missing a required symbol");
        dlclose(h);
        return MXB_ERR_CUDA;
    }
    g_nccl.handle = h;
    return MXB_OK;
}

#define MXB_NCCL(call)                                                        \
    do {                                                                      \
        int r__ = (call);                                                     \
        if (r__ != 0) {                                                       \
            set_error("%s:%d: %s -> nccl error %d (%s)", __FILE__, __LINE__,  \
                      #call, r__,                                             \
                      g_nccl.error_string ? g_nccl.error_string(r__) : "?");  \
            return MXB_ERR_CUDA;                                              \
        }                                                                     \
    } while (0)

// ncclDouble = 8, ncclSum = 0, ncclMax = 2 (nccl.h, stable since 2.0).
int nccl_allreduce_f64(mxb_ctx *ctx, double *dev_buf, int64_t n, int op_is_max) {
    if (!ctx->nccl_comm || ctx->world <= 1) return MXB_OK;
    MXB_NCCL(g_nccl.allreduce(dev_buf, dev_buf, (size_t)n, 8, op_is_max ? 2 : 0,
                              ctx->nccl_comm, ctx->stream));
    return MXB_OK;
}

// Row shards of an N x H matrix (rank q owns rows [N q / W, N (q + 1) / W)): every rank sends
// shard q of its matrix `src` to rank q and receives the W versions of its own shard into
// `recv` (W slots of max_rows x n_cols doubles; the own slot is not filled: read `src`).
int nccl_alltoall_rows(mxb_ctx *ctx, const double *src, double *recv, int64_t n_rows,
                       int64_t n_cols, int64_t slot_doubles) {
    if (!ctx->nccl_comm || ctx->world <= 1) return MXB_OK;
    if (!g_nccl.send || !g_nccl.recv || !g_nccl.group_start || !g_nccl.group_end) {
        set_error("libnccl lacks ncclSend/ncclRecv");
        return MXB_ERR_CUDA;
    }
    const int W = ctx->world, me = ctx->rank;
    const int64_t my_lo = n_rows * me / W, my_hi = n_rows * (me + 1) / W;
    MXB_NCCL(g_nccl.group_start());
    for (int q = 0; q < W; ++q) {
        if (q == me) continue;
        const int64_t lo = n_rows * q / W, hi = n_rows * (q + 1) / W;
        if (hi > lo)
            MXB_NCCL(g_nccl.send(src + lo * n_cols, (size_t)((hi - lo) * n_cols), 8, q,
                                 ctx->nccl_comm, ctx->stream));
        if (my_hi > my_lo)
            MXB_NCCL(g_nccl.recv(recv + (int64_t)q * slot_doubles, (size_t)((my_hi - my_lo) * n_cols),
                                 8, q, ctx->nccl_comm, ctx->stream));
    }
    MXB_NCCL(g_nccl.group_end());
    return MXB_OK;
}

// Every rank broadcasts its row shard of `m` (in place): afterwards all ranks hold all rows.
int nccl_allgather_rows(mxb_ctx *ctx, double *m, int64_t n_rows, int64_t n_cols) {
    if (!ctx->nccl_comm || ctx->world <= 1) return MXB_OK;
    if (!g_nccl.bcast || !g_nccl.group_start || !g_nccl.group_end) {
        set_error("libnccl lacks ncclBroadcast");
        return MXB_ERR_CUDA;
    }
    const int W = ctx->world;
    MXB_NCCL(g_nccl.group_start());
    for (int q = 0; q < W; ++q) {
        const int64_t lo = n_rows * q / W, hi = n_rows * (q + 1) / W;
        if (hi > lo)
            MXB_NCCL(g_nccl.bcast(m + lo * n_cols, m + lo * n_cols, (size_t)((hi - lo) * n_cols), 8,
                                  q, ctx->nccl_comm, ctx->stream));
    }
    MXB_NCCL(g_nccl.group_end());
    return MXB_OK;
}

int nccl_allreduce_sum_f64(mxb_ctx *ctx, double *dev_buf, int64_t n) {
    return nccl_allreduce_f64(ctx, dev_buf, n, 0);
}

// ---------------------------------------------------------------------------
// Host <-> device copy engine.
//
// The drop-in entry points take and return ordinary numpy arrays, i.e. pageable
// host memory.  A plain cudaMemcpy of pageable memory runs at 11 GB/s (H2D) /
// 19 GB/s (D2H, 4.8 GB/s into never-touched pages) on the B200 boxes, pinning
// a 6 GB buffer on the fly costs 0.7-2.5 s.  Instead a small pinned ring
// (kStageSlots x 32 MiB, allocated once per context) is filled or drained by
// all host threads while the DMA engine works on the neighbouring slot:
// 43 GB/s both ways, measured with scripts/micro/hostmem.cu.
// ---------------------------------------------------------------------------
constexpr int kStageSlots = 4;
constexpr size_t kStageChunk = (size_t)32 << 20;
constexpr size_t kDirectCopyBytes = (size_t)8 << 20;  // below this a plain copy wins

static int copy_threads() {
    static int n = 0;
    if (n == 0) {
        const char *env = getenv("MXB_COPY_THREADS");
        int v = env ? atoi(env) : 0;
        if (v <= 0) {
            // one process per GPU: share the host cores between the local ranks
            const char *lw = getenv("LOCAL_WORLD_SIZE");
            const int ranks = std::max(1, lw ? atoi(lw) : 1);
            v = std::min(16, std::max(2, omp_get_num_procs() / ranks));
        }
        n = std::max(1, v);
    }
    return n;
}

static int ensure_stage(mxb_ctx *ctx) {
    if (ctx->stage_chunk) return MXB_OK;
    for (int i = 0; i < kStageSlots; ++i) {
        MXB_CUDA(cudaHostAlloc(&ctx->stage_buf[i], kStageChunk, cudaHostAllocDefault));
        MXB_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
    }
    ctx->stage_chunk = kStageChunk;
    return MXB_OK;
}

static void free_stage(mxb_ctx *ctx) {
    for (int i = 0; i < kStageSlots; ++i) {
        if (ctx->stage_buf[i]) cudaFreeHost(ctx->stage_buf[i]);
        if (ctx->stage_ev[i]) cudaEventDestroy(ctx->stage_ev[i]);
        ctx->stage_buf[i] = nullptr;
        ctx->stage_ev[i] = nullptr;
    }
    ctx->stage_chunk = 0;
}

static bool host_is_pinned(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

static void parallel_memcpy(void *dst, const void *src, size_t n) {
    const int T = copy_threads();
    if (T == 1 || n < ((size_t)1 << 20)) {
        memcpy(dst, src, n);
        return;
    }
#pragma omp parallel num_threads(T)
    {
        const size_t t = (size_t)omp_get_thread_num(), nt = (size_t)omp_get_num_threads();
        // 4 KiB-aligned slices so that two threads never share a page
        const size_t per = (((n + nt - 1) / nt) + 4095) & ~(size_t)4095;
        const size_t a = per * t;
        if (a < n) memcpy((char *)dst + a, (const char *)src + a, std::min(per, n - a));
    }
}

int copy_h2d(mxb_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes) {
    if (!bytes) return MXB_OK;
    cudaStream_t s = ctx->stream;
    if (bytes < kDirectCopyBytes || host_is_pinned(src_host) || getenv("MXB_COPY_DIRECT")) {
        MXB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, s));
        MXB_CUDA(cudaStreamSynchronize(s));
        return MXB_OK;
    }
    MXB_TRY(ensure_stage(ctx));
    const size_t cb = ctx->stage_chunk;
    const size_t n_chunks = (bytes + cb - 1) / cb;
    for (size_t c = 0; c < n_chunks; ++c) {
        const int slot = (int)(c % kStageSlots);
        const size_t off = c * cb, n = std::min(cb, bytes - off);
        if (c >= (size_t)kStageSlots) MXB_CUDA(cudaEventSynchronize(ctx->stage_ev[slot]));
        parallel_memcpy(ctx->stage_buf[slot], (const char *)src_host + off, n);
        MXB_CUDA(cudaMemcpyAsync((char *)dst_dev + off, ctx->stage_buf[slot], n,
                                 cudaMemcpyHostToDevice, s));
        MXB_CUDA(cudaEventRecord(ctx->stage_ev[slot], s));
    }
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

int copy_d2h(mxb_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes) {
    if (!bytes) return MXB_OK;
    cudaStream_t s = ctx->stream;
    if (bytes < kDirectCopyBytes || host_is_pinned(dst_host) || getenv("MXB_COPY_DIRECT")) {
        MXB_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, s));
        MXB_CUDA(cudaStreamSynchronize(s));
        return MXB_OK;
    }
    MXB_TRY(ensure_stage(ctx));
    const size_t cb = ctx->stage_chunk;
    const size_t n_chunks = (bytes + cb - 1) / cb;
    size_t issued = 0;
    for (size_t c = 0; c < n_chunks; ++c) {
        // keep the DMA engine kStageSlots - 1 chunks ahead of the host threads
        while (issued < n_chunks && issued < c + kStageSlots) {
            const int slot = (int)(issued % kStageSlots);
            const size_t off = issued * cb, n = std::min(cb, bytes - off);
            MXB_CUDA(cudaMemcpyAsync(ctx->stage_buf[slot], (const char *)src_dev + off, n,
                                     cudaMemcpyDeviceToHost, s));
            MXB_CUDA(cudaEventRecord(ctx->stage_ev[slot], s));
            ++issued;
        }
        const int slot = (int)(c % kStageSlots);
        const size_t off = c * cb, n = std::min(cb, bytes - off);
        MXB_CUDA(cudaEventSynchronize(ctx->stage_ev[slot]));
        parallel_memcpy((char *)dst_host + off, ctx->stage_buf[slot], n);
    }
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

// ---------------------------------------------------------------------------
// Device memory: the context's block pool (see common.cuh) and its owners.
// ---------------------------------------------------------------------------
void *pinned_scratch(mxb_ctx *ctx) {
    if (!ctx->pinned && cudaHostAlloc(&ctx->pinned, kPinnedScratchBytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        ctx->pinned = nullptr;
    }
    return ctx->pinned;
}

void *cuda_block_new(size_t bytes) {
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void cuda_block_delete(void *ptr) { cudaFree(ptr); }

void *dev_alloc(mxb_ctx *ctx, size_t bytes) {
    if (bytes == 0) return nullptr;
    if (++ctx->n_allocs == ctx->fail_alloc_at) return nullptr;   // MXB_DEBUG_FAIL_ALLOC
    void *p = ctx->pool.take(bytes);
    if (!p) {   // the cached blocks may be what is missing
        ctx->pool.trim();
        p = ctx->pool.take(bytes);
    }
    return p;
}

void dev_free(mxb_ctx *ctx, void *ptr) {
    if (!ptr) return;
    // a block that is cached may still be read by work queued on the context's stream
    ctx->pool.give(ptr, [ctx]() { cudaStreamSynchronize(ctx->stream); });
}

int DevBlock::alloc(mxb_ctx *ctx, size_t bytes, const char *who) {
    reset();
    ctx_ = ctx;
    p_ = dev_alloc(ctx, bytes);
    if (bytes && !p_) {
        set_error("%s: out of device memory for %zu bytes", who, bytes);
        return MXB_ERR_NOMEM;
    }
    return MXB_OK;
}

void DevBlock::reset() {
    if (p_) dev_free(ctx_, p_);
    p_ = nullptr;
}

int Events::create(size_t n, unsigned flags, const char *who) {
    try {
        ev_.reserve(ev_.size() + n);
    } catch (const std::bad_alloc &) {
        set_error("%s: out of host memory", who);
        return MXB_ERR_NOMEM;
    }
    for (size_t i = 0; i < n; ++i) {
        cudaEvent_t e = nullptr;
        const cudaError_t err = cudaEventCreateWithFlags(&e, flags);
        if (err != cudaSuccess) {
            set_error("%s: cudaEventCreate: %s", who, cudaGetErrorString(err));
            return MXB_ERR_CUDA;
        }
        ev_.push_back(e);
    }
    return MXB_OK;
}

// ---------------------------------------------------------------------------
// Pool of pinned host blocks for matrix-sized *results* (process-wide; pinned memory is
// allocated portable).  The drop-in calls hand N x H arrays back to Python; when such an
// array lives in a pooled pinned block the device->host copy is one DMA at PCIe speed with no
// staging memcpy and no first-touch page faults -- which is what limits eight ranks sharing
// the host cores of one box.  Pinning is slow (about a second per 6 GB), so blocks are kept
// when their arrays die and handed out again (mxb_host_trim releases them).
// ---------------------------------------------------------------------------
bool g_stage_on = false;
double g_stage_ms[kNumStages] = {};

static size_t host_pool_limit() {
    const char *env = getenv("MXB_PINNED_CACHE_MB");
    if (env) return ((size_t)atoll(env) << 20) + 1;
    const long pages = sysconf(_SC_PHYS_PAGES), psz = sysconf(_SC_PAGE_SIZE);
    return pages > 0 && psz > 0 ? (size_t)pages * (size_t)psz / 4 : ((size_t)16 << 30);
}

static BlockPool &host_pool() {
    static BlockPool pool(
        [](size_t bytes) -> void * {
            void *p = nullptr;
            if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
            return p;
        },
        [](void *p) { cudaFreeHost(p); }, 4, 0, host_pool_limit());
    return pool;
}

struct PrefaultImpl {
    std::vector<std::thread> threads;
};

void Prefault::start(void *buf, size_t bytes) {
    join();
    if (!buf || bytes < kDirectCopyBytes || host_is_pinned(buf) || getenv("MXB_NO_PREFAULT")) return;
    const size_t page = (size_t)sysconf(_SC_PAGESIZE);
    char *lo = (char *)(((uintptr_t)buf + page - 1) & ~(uintptr_t)(page - 1));
    char *hi = (char *)(((uintptr_t)buf + bytes) & ~(uintptr_t)(page - 1));
    if (hi <= lo) return;
    // transparent huge pages halve the fault time on an idle box but stall for compaction
    // on a fragmented one (seen as 0.2-0.4 s outliers): opt-in only
    if (getenv("MXB_PREFAULT_HUGEPAGE")) madvise(lo, (size_t)(hi - lo), MADV_HUGEPAGE);
    PrefaultImpl *pi = new (std::nothrow) PrefaultImpl();
    if (!pi) return;
    const char *env = getenv("MXB_PREFAULT_THREADS");
    const int T = std::max(1, env ? atoi(env) : copy_threads() / 2);
    const size_t n_pages = (size_t)(hi - lo) / page;
    try {
        for (int t = 0; t < T; ++t) {
            const size_t a = n_pages * t / T, b = n_pages * (t + 1) / T;
            pi->threads.emplace_back([lo, page, a, b]() {
                // output buffer: its contents are overwritten by the copy that follows
                for (size_t i = a; i < b; ++i) *(volatile char *)(lo + i * page) = 0;
            });
        }
    } catch (...) {
    }
    impl = pi;
}

void Prefault::join() {
    PrefaultImpl *pi = (PrefaultImpl *)impl;
    if (!pi) return;
    for (auto &t : pi->threads) if (t.joinable()) t.join();
    delete pi;
    impl = nullptr;
}

// ---------------------------------------------------------------------------
// Peer mailboxes for the fused EM tail.  NCCL carries the 64-byte IPC handles
// once (ncclAllGather) and the vote on whether every rank could map every peer;
// after that the per-iteration exchange of the H column sums is plain stores
// into peer memory from inside em_finish_kernel (em.cu).
// ---------------------------------------------------------------------------
static void p2p_teardown(mxb_ctx *ctx) {
    for (int r = 0; r < kP2PMaxWorld; ++r) {
        if (!ctx->p2p_block[r]) continue;
        if (r == ctx->rank) cudaFree(ctx->p2p_block[r]);
        else cudaIpcCloseMemHandle(ctx->p2p_block[r]);
        ctx->p2p_block[r] = nullptr;
    }
    ctx->p2p_vote.reset();
    ctx->p2p_ready = false;
}

static int p2p_setup(mxb_ctx *ctx) {
    ctx->p2p_ready = false;
    if (ctx->world <= 1 || ctx->world > kP2PMaxWorld || !g_nccl.allgather || getenv("MXB_NO_P2P"))
        return MXB_OK;
    const int W = ctx->world;
    cudaStream_t s = ctx->stream;
    unsigned char *mine = nullptr;
    MXB_CUDA(cudaMalloc(&mine, kP2PBlockBytes));
    ctx->p2p_block[ctx->rank] = mine;
    MXB_CUDA(cudaMemsetAsync(mine, 0, kP2PBlockBytes, s));
    cudaIpcMemHandle_t handles[kP2PMaxWorld];
    memset(handles, 0, sizeof(handles));
    int ok = cudaIpcGetMemHandle(&handles[ctx->rank], mine) == cudaSuccess;
    if (!ok) cudaGetLastError();
    DevBlock dh_block, vote_block;
    MXB_TRY(dh_block.alloc(ctx, sizeof(handles), "mxb_comm_init"));
    MXB_TRY(vote_block.alloc(ctx, sizeof(double), "mxb_comm_init"));
    unsigned char *dh = dh_block.get();
    double *vote = vote_block.get<double>();
    MXB_CUDA(cudaMemcpyAsync(dh, handles, sizeof(handles), cudaMemcpyHostToDevice, s));
    MXB_NCCL(g_nccl.allgather(dh + (size_t)ctx->rank * sizeof(cudaIpcMemHandle_t), dh,
                              sizeof(cudaIpcMemHandle_t), 1 /* ncclUint8 */, ctx->nccl_comm, s));
    MXB_CUDA(cudaMemcpyAsync(handles, dh, sizeof(handles), cudaMemcpyDeviceToHost, s));
    MXB_CUDA(cudaStreamSynchronize(s));
    for (int r = 0; r < W && ok; ++r) {
        if (r == ctx->rank) continue;
        void *peer = nullptr;
        if (cudaIpcOpenMemHandle(&peer, handles[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            ok = 0;
        } else {
            ctx->p2p_block[r] = (unsigned char *)peer;
        }
    }
    // unanimous or not at all: a rank that fell back to NCCL would wait forever
    double v = ok ? 0.0 : 1.0;
    MXB_CUDA(cudaMemcpyAsync(vote, &v, sizeof(v), cudaMemcpyHostToDevice, s));
    MXB_CUDA(cudaStreamSynchronize(s));
    MXB_TRY(nccl_allreduce_f64(ctx, vote, 1, 0));
    MXB_CUDA(cudaMemcpyAsync(&v, vote, sizeof(v), cudaMemcpyDeviceToHost, s));
    MXB_CUDA(cudaStreamSynchronize(s));
    if (v != 0.0) {
        p2p_teardown(ctx);
        return MXB_OK;  // NCCL all-reduce path stays in use
    }
    ctx->p2p_vote = std::move(vote_block);
    ctx->p2p_ready = true;
    return MXB_OK;
}

// Start of a row-sharded session: put every rank's mailbox flags and launch sequence number
// back to zero behind a barrier.  A rank that timed out, failed, or ran a different number of
// tail launches than its peers in an earlier session would otherwise leave the sequence
// numbers out of step for good (every later session would wait for a number that never comes).
int p2p_resync(mxb_ctx *ctx) {
    if (!ctx->p2p_ready || ctx->world <= 1) return MXB_OK;
    cudaStream_t s = ctx->stream;
    MXB_CUDA(cudaStreamSynchronize(s));                 // my own tail launches are done
    double *vote = ctx->p2p_vote.get<double>();
    MXB_CUDA(cudaMemsetAsync(vote, 0, sizeof(double), s));
    MXB_TRY(nccl_allreduce_f64(ctx, vote, 1, 0));   // ... and so are everybody else's
    MXB_CUDA(cudaMemsetAsync(ctx->p2p_block[ctx->rank], 0, kP2PInboxOffset, s));
    MXB_TRY(nccl_allreduce_f64(ctx, vote, 1, 0));   // nobody stores before all are zeroed
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

}  // namespace mxb

using namespace mxb;

extern "C" {

int mxb_abi_version(void) { return MXB_ABI_VERSION; }

const char *mxb_last_error(void) { return g_error; }

int mxb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int mxb_ctx_create(int device, mxb_ctx **out) {
    MXB_REQUIRE(out != nullptr, "out is NULL");
    *out = nullptr;
    int n = 0;
    MXB_CUDA(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) {
        set_error("mxb_ctx_create: device %d out of range (%d visible)", device, n);
        return MXB_ERR_ARG;
    }
    MXB_CUDA(cudaSetDevice(device));
    mxb_ctx *ctx = new (std::nothrow) mxb_ctx();
    if (!ctx) { set_error("out of host memory"); return MXB_ERR_NOMEM; }
    ctx->device = device;
    cudaDeviceProp prop;
    MXB_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx->num_sms = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    MXB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
    const char *env = getenv("MXB_CACHE_MB");
    if (env) {
        ctx->pool.set_limit((size_t)atoll(env) << 20);
    } else {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) ctx->pool.set_limit(total_b / 4);
        else cudaGetLastError();
    }
    env = getenv("MXB_DEBUG_FAIL_ALLOC");
    ctx->fail_alloc_at = env ? atoll(env) : 0;
    *out = ctx;
    return MXB_OK;
}

int mxb_ctx_destroy(mxb_ctx *ctx) {
    if (!ctx) return MXB_OK;
    cudaSetDevice(ctx->device);
    if (ctx->nccl_comm) mxb_comm_destroy(ctx);
    free_stage(ctx);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pool.trim();
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return MXB_OK;
}

int mxb_ctx_set_stream(mxb_ctx *ctx, void *cuda_stream) {
    MXB_REQUIRE(ctx != nullptr, "ctx is NULL");
    if (ctx->own_stream && ctx->stream) {
        MXB_CUDA(cudaStreamSynchronize(ctx->stream));
        MXB_CUDA(cudaStreamDestroy(ctx->stream));
    }
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return MXB_OK;
}

int mxb_ctx_synchronize(mxb_ctx *ctx) {
    MXB_REQUIRE(ctx != nullptr, "ctx is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXB_OK;
}

int mxb_ctx_trim(mxb_ctx *ctx) {
    MXB_REQUIRE(ctx != nullptr, "ctx is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->pool.trim();
    return MXB_OK;
}

int mxb_ctx_mem_stats(const mxb_ctx *ctx, int64_t *live_bytes, int64_t *cached_bytes) {
    MXB_REQUIRE(ctx != nullptr, "ctx is NULL");
    size_t live = 0, cached = 0;
    ctx->pool.stats(&live, &cached);
    if (live_bytes) *live_bytes = (int64_t)live;
    if (cached_bytes) *cached_bytes = (int64_t)cached;
    return MXB_OK;
}

int mxb_host_alloc(size_t bytes, int only_if_cached, void **out) {
    MXB_REQUIRE(out != nullptr && bytes > 0, "bad argument");
    // NULL when nothing fits or pinning fails: not an error, the caller uses pageable memory
    *out = host_pool().take(bytes, only_if_cached != 0);
    return MXB_OK;
}

int mxb_host_free(void *ptr) {
    if (!ptr) return MXB_OK;
    MXB_REQUIRE(host_pool().give(ptr), "not a block of mxb_host_alloc");
    return MXB_OK;
}

int mxb_host_reserve(size_t bytes, int count) {
    MXB_REQUIRE(bytes > 0 && count >= 1 && count <= 16, "bad argument");
    std::vector<void *> got;
    int rc = MXB_OK;
    for (int i = 0; i < count && rc == MXB_OK; ++i) {
        void *p = nullptr;
        rc = mxb_host_alloc(bytes, 0, &p);
        if (rc == MXB_OK && !p) {
            set_error("mxb_host_reserve: could not pin %zu bytes", bytes);
            rc = MXB_ERR_NOMEM;
        }
        if (p) got.push_back(p);
    }
    for (void *p : got) mxb_host_free(p);
    return rc;
}

int mxb_stage_timing(int on) {
    g_stage_on = on != 0 || getenv("MXB_TIMING") != nullptr;
    for (int i = 0; i < kNumStages; ++i) g_stage_ms[i] = 0.0;
    return MXB_OK;
}

int mxb_stage_times(double *ms_out, int n) {
    MXB_REQUIRE(ms_out != nullptr && n >= 0, "bad argument");
    for (int i = 0; i < n; ++i) ms_out[i] = i < kNumStages ? g_stage_ms[i] : 0.0;
    return MXB_OK;
}

int mxb_host_trim(void) {
    host_pool().trim();
    return MXB_OK;
}

int64_t mxb_ctx_launch_count(const mxb_ctx *ctx) { return ctx ? ctx->launches : 0; }

int mxb_comm_unique_id(void *id128) {
    MXB_REQUIRE(id128 != nullptr, "id128 is NULL");
    MXB_TRY(load_nccl());
    nccl_uid_t uid;
    MXB_NCCL(g_nccl.get_uid(&uid));
    memcpy(id128, &uid, sizeof(uid));
    return MXB_OK;
}

int mxb_comm_init(mxb_ctx *ctx, const void *id128, int rank, int world) {
    MXB_REQUIRE(ctx != nullptr && id128 != nullptr, "NULL argument");
    MXB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
    MXB_REQUIRE(ctx->nccl_comm == nullptr, "comm already initialised");
    MXB_TRY(load_nccl());
    MXB_CUDA(cudaSetDevice(ctx->device));
    nccl_uid_t uid;
    memcpy(&uid, id128, sizeof(uid));
    void *comm = nullptr;
    MXB_NCCL(g_nccl.init_rank(&comm, world, uid, rank));
    ctx->nccl_comm = comm;
    ctx->rank = rank;
    ctx->world = world;
    return p2p_setup(ctx);
}

int mxb_comm_destroy(mxb_ctx *ctx) {
    MXB_REQUIRE(ctx != nullptr, "ctx is NULL");
    if (ctx->nccl_comm) {
        cudaStreamSynchronize(ctx->stream);
        p2p_teardown(ctx);
        g_nccl.destroy(ctx->nccl_comm);
        ctx->nccl_comm = nullptr;
    }
    ctx->rank = 0;
    ctx->world = 1;
    return MXB_OK;
}

int mxb_comm_p2p_enabled(const mxb_ctx *ctx) { return ctx && ctx->p2p_ready ? 1 : 0; }

int mxb_comm_allreduce_host(mxb_ctx *ctx, double *buf, int64_t n, int op_is_max) {
    MXB_REQUIRE(ctx != nullptr && (buf != nullptr || n == 0) && n >= 0, "bad argument");
    if (!ctx->nccl_comm || ctx->world <= 1 || n == 0) return MXB_OK;
    MXB_CUDA(cudaSetDevice(ctx->device));
    DevBlock d_block;
    MXB_TRY(d_block.alloc(ctx, n * sizeof(double), "mxb_comm_allreduce_host"));
    double *d = d_block.get<double>();
    MXB_CUDA(cudaMemcpyAsync(d, buf, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    MXB_TRY(nccl_allreduce_f64(ctx, d, n, op_is_max));
    MXB_CUDA(cudaMemcpyAsync(buf, d, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXB_OK;
}

// ---- matrices ---------------------------------------------------------------

int mxb_matrix_alloc(mxb_ctx *ctx, int64_t n_rows, int64_t n_cols, mxb_matrix **out) {
    MXB_REQUIRE(ctx != nullptr && out != nullptr, "NULL argument");
    MXB_REQUIRE(n_rows >= 0 && n_cols >= 0, "negative shape");
    *out = nullptr;
    MXB_CUDA(cudaSetDevice(ctx->device));
    mxb_matrix *m = new (std::nothrow) mxb_matrix();
    if (!m) { set_error("out of host memory"); return MXB_ERR_NOMEM; }
    m->ctx = ctx;
    m->n_rows = n_rows;
    m->n_cols = n_cols;
    const int rc = m->mem.alloc(ctx, (size_t)n_rows * (size_t)n_cols * sizeof(double),
                                "mxb_matrix_alloc");
    if (rc != MXB_OK) {
        delete m;
        return rc;
    }
    m->data = m->mem.get<double>();
    *out = m;
    return MXB_OK;
}

int mxb_matrix_upload(mxb_ctx *ctx, const double *host, int64_t n_rows,
                      int64_t n_cols, mxb_matrix **out) {
    MXB_REQUIRE(host != nullptr || n_rows * n_cols == 0, "host is NULL");
    MXB_TRY(mxb_matrix_alloc(ctx, n_rows, n_cols, out));
    size_t bytes = (size_t)n_rows * (size_t)n_cols * sizeof(double);
    if (bytes) {
        const auto t0 = std::chrono::steady_clock::now();
        const int rc = copy_h2d(ctx, (*out)->data, host, bytes);
        if (g_stage_on)
            g_stage_ms[kStageH2D] += std::chrono::duration<double, std::milli>(
                std::chrono::steady_clock::now() - t0).count();
        if (rc != MXB_OK) {
            mxb_matrix_destroy(*out);
            *out = nullptr;
            return rc;
        }
    }
    return MXB_OK;
}

int mxb_matrix_download(mxb_ctx *ctx, const mxb_matrix *m, double *host) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL argument");
    size_t bytes = (size_t)m->n_rows * (size_t)m->n_cols * sizeof(double);
    if (!bytes) return MXB_OK;
    MXB_REQUIRE(host != nullptr, "host is NULL");
    MXB_CUDA(cudaSetDevice(ctx->device));
    return copy_d2h(ctx, host, m->data, bytes);
}

int mxb_matrix_shape(const mxb_matrix *m, int64_t *n_rows, int64_t *n_cols) {
    MXB_REQUIRE(m != nullptr, "matrix is NULL");
    if (n_rows) *n_rows = m->n_rows;
    if (n_cols) *n_cols = m->n_cols;
    return MXB_OK;
}

void *mxb_matrix_data(const mxb_matrix *m) { return m ? (void *)m->data : nullptr; }

int mxb_matrix_destroy(mxb_matrix *m) {
    if (!m) return MXB_OK;
    if (m->data) cudaSetDevice(m->ctx->device);
    delete m;   // (gives its block back)
    return MXB_OK;
}

}  // extern "C"
