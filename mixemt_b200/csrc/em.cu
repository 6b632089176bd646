// Kernel 2: the EM mixture-proportion fit.
//
// Replaces em_step / converged / run_em (reference mixemt/em.py:39-165) and the
// scipy.special.logsumexp calls inside them (em.py:82, :87-89).
//
// Formulation.  The reference works on Z_ij = M_ij + ln pi_j - lse_i in log
// space and makes ~30 passes over the N x H matrix per iteration (two
// max-shifted logsumexp reductions).  With m_i = max_j M_ij and
// L_ij = exp(M_ij - m_i) (computed once per run_em call, shared by all
// restarts), one iteration is
//
//     s_i   = sum_j L_ij pi_j                      (row dot product)
//     T_j   = sum_i (w_i / s_i) L_ij               (weighted column sum)
//     pi'_j = pi_j T_j / sum_k pi_k T_k            (M-step; == em.py:87-89)
//
// i.e. exactly two fp64 FMAs per cell and ONE read of L per iteration: the pass
// is bound by HBM bandwidth (8 B/cell), not by exp throughput.  ln pi is
// carried in log space next to pi (ln pi'_j = ln pi_j + log(T_j / total) once
// pi_j leaves the normal range), so dying components keep following the
// reference's trajectory after exp() underflows.  The read matrix the reference
// returns (em.py:130-136: responsibilities at the *previous* proportions) is
// produced in log space straight from M by read_mix_kernel, with scipy's
// logsumexp formula (log1p(s/m) + log(m) + max).
//
// The fused pass (em_pass_fast_kernel) is a persistent kernel, one CTA per SM,
// that streams its contiguous row range through a shared-memory ring filled by
// 1-D bulk async copies (TMA engine, cp.async.bulk + mbarrier complete_tx).
// Thread t owns the same 2*NC columns of every row: it reads each staged cell
// once into registers, contributes to the row's dot product, and after a
// block-wide reduction adds (w_i/s_i) * L_ij into its private column sums.
// Per-CTA column sums are written once at the end and reduced in a fixed order
// (deterministic: no floating-point atomics anywhere).
#include <math.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <memory>
#include <new>
#include <vector>

#include "bootstrap.cuh"
#include "common.cuh"
#include "em_kernels.cuh"
#include "em_tiles.cuh"
#include "tile_plan.h"


using namespace mxb;

namespace mxb {
// What an iteration runs (decide_form): its pass over class tiles, over fp64 rows (streamed,
// or streamed with two restarts per read of L) or the general path; its tail in one cluster
// launch (em_finish_kernel), the same with the ranks' sums exchanged through peer memory, or
// split (em_colreduce_kernel, NCCL all-reduce across ranks, em_update_kernel).
enum class EmForm { kTiles, kRows, kRowPairs, kGeneral };
enum class EmTail { kFused, kPeer, kSplit };
}  // namespace mxb

struct mxb_em {
    mxb_ctx *ctx = nullptr;
    const mxb_matrix *mat = nullptr;
    int64_t n_rows = 0, n_cols = 0, ld = 0;
    bool sharded = false;
    DevBlock lin;                 // [n_rows][ld] doubles
    double *weights = nullptr;    // [n_rows]
    double *coef = nullptr;       // [n_rows] (general path)
    double *lnp[2] = {nullptr, nullptr};
    double *pi[2] = {nullptr, nullptr};
    double *partials = nullptr;   // [n_part][ld]
    double *tsum = nullptr;       // [ld]
    double *props_in = nullptr;   // [n_cols] staging for set_lnprops
    EmState *state = nullptr;     // device
    EmState *host_state = nullptr;  // pinned, 2 slots
    Events poll_ev;               // 2
    int n_part = 0;
    // decide_form
    EmForm form = EmForm::kGeneral;
    EmTail tail = EmTail::kSplit;
    // Restart slots: a batched session (run_em with n_multi > 1) iterates two restarts per read
    // of L, a bootstrap session R replicates per iteration.  Slot s lives at lnp[b] + s*ld,
    // pi[b] + s*ld, partials + s*n_part*ld, state + s (slot_block).
    int n_slots = 1;
    // streaming pass (n_stages > 0 when the rows fit its ring)
    int nc = 0;
    int n_stages = 0;
    size_t smem_bytes = 0;
    int grid_fast = 0;
    // general path
    int row_blocks = 0, col_blocks = 0;
    // Class tiles (em_tiles.cuh): form kTiles reads `tile_v` instead of `lin`.
    int n_batches = 0, tile_hs = 0, tile_grid = 0;   // (the gather's blocks: n_part)
    DevBlock tile_block;   // [perm][cmap][cword][desc]
    DevBlock tile_vecs;    // [pi_cls][u_sum][ctas][segs][gather entries]
    unsigned short *tile_perm = nullptr, *tile_cmap = nullptr;
    unsigned int *tile_cword = nullptr;
    TileDesc *tile_desc = nullptr;
    TileCta *tile_ctas = nullptr;           // plan of the pass (em_tiles.cuh)
    TileSeg *tile_segs = nullptr;
    int *tile_ent_batch = nullptr;          // gather entries: batch and offset of every U vector
    int64_t *tile_ent_off = nullptr;
    int tile_n_ent = 0, tile_n_slots = 0;
    uint32_t tile_slot_bytes = 0;
    double *tile_pi = nullptr, *tile_usum = nullptr;
    DevBlock tile_v;                       // the tiles (doubles)
    int64_t tile_cells = 0;                // doubles in tile_v
    int64_t tile_bytes_per_pass = 0;
    DevBlock small;   // one device block behind weights ... props_in (fewer driver calls)
    DevBlock slots;   // the slot block (slot_block)
    bool zero_iter = false;  // last iterate() ran no iteration
    // Bootstrap session (run_bootstrap): n_slots replicates per launch, each with its own weight
    // vector (slot_weights); over class tiles the slots' Pi and U vectors lie tile_pi_stride and
    // tile_u_stride doubles apart.
    bool boot = false;
    double *slot_w = nullptr;
    int64_t tile_pi_stride = 0, tile_u_stride = 0;
};

namespace mxb {

static decltype(&em_pass_fast_kernel<1>) pick_pass(int nc) {
    switch (nc) {
        case 1: return em_pass_fast_kernel<1>;
        case 2: return em_pass_fast_kernel<2>;
        case 3: return em_pass_fast_kernel<3>;
        case 4: return em_pass_fast_kernel<4>;
        case 5: return em_pass_fast_kernel<5>;
        case 6: return em_pass_fast_kernel<6>;
        case 7: return em_pass_fast_kernel<7>;
        case 8: return em_pass_fast_kernel<8>;
    }
    return nullptr;
}
static decltype(&em_pass_pair_kernel<1>) pick_pair(int nc) {
    switch (nc) {
        case 1: return em_pass_pair_kernel<1>;
        case 2: return em_pass_pair_kernel<2>;
        case 3: return em_pass_pair_kernel<3>;
        case 4: return em_pass_pair_kernel<4>;
        case 5: return em_pass_pair_kernel<5>;
        case 6: return em_pass_pair_kernel<6>;
    }
    return nullptr;
}
constexpr int kMaxPairNC = 6;   // 2 restarts x (pi + T) x NC double2 must fit 128 registers
constexpr int kMaxSlots = kBootMaxSlots;

// Launch with the programmatic-stream-serialization attribute (see pdl_wait): the kernel may
// be scheduled before its predecessor in the stream has finished.  MXB_EM_NO_PDL=1 turns the
// attribute off (plain stream order).
// (set before a call to launch that kernel in plain stream order)
static thread_local bool g_plain_launch = false;
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t s, Args... args) {
    static const bool pdl_on = getenv("MXB_EM_NO_PDL") == nullptr;
    const bool use_pdl = pdl_on && !g_plain_launch;
    g_plain_launch = false;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = use_pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// The weights slot `slot` iterates on: its resampled counts in a bootstrap session.
static double *slot_weights(mxb_em *em, int slot) {
    return em->boot ? em->slot_w + slot * em->n_rows : em->weights;
}

// The class-sum kernel of a tiled iteration for `per` = ceil(H / kTileThreads) columns a thread.
template <bool kSlots>
static auto pick_tile_pi(int64_t n_cols) {
    const int per = (int)ceil_div(n_cols, kTileThreads);
    return per <= 4 ? tile_pi_kernel<4, kSlots> : per <= 8 ? tile_pi_kernel<8, kSlots>
           : per <= 12 ? tile_pi_kernel<12, kSlots> : tile_pi_kernel<16, kSlots>;
}

// The pass of a tiled iteration: class sums, pass and gather.  kSlots: the R replicate slots of
// a bootstrap session side by side, the slot in blockIdx.y (z for the gather), all on one plan
// of num_sms / R CTAs; a slot whose control block says done costs nothing.
template <bool kSlots>
static int enqueue_tile_pass(mxb_em *em, unsigned R, cudaEvent_t *marks) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const int64_t pi_stride = kSlots ? em->tile_pi_stride : 0;
    const int64_t u_stride = kSlots ? em->tile_u_stride : 0;
    MXB_CUDA(launch_pdl(pick_tile_pi<kSlots>(em->n_cols),
                        dim3(std::min(em->n_batches, std::max(1, 2 * ctx->num_sms / (int)R)), R),
                        dim3(kTileThreads), (size_t)em->ld * sizeof(double), s,
                        (const unsigned short *)em->tile_perm, (const unsigned int *)em->tile_cword,
                        em->tile_hs, (int)em->n_cols, (const TileDesc *)em->tile_desc,
                        em->n_batches, (const double *)em->pi[0], (const double *)em->pi[1],
                        (const EmState *)em->state, em->tile_pi, kSlots ? em->ld : (int64_t)0,
                        pi_stride));
    if (marks) MXB_CUDA(cudaEventRecord(marks[0], s));
    MXB_CUDA(launch_pdl(tile_pass_kernel<kSlots>, dim3(em->tile_grid, R), dim3(kTilePassThreads),
                        kSlots ? kTilePassSlotSmem : kTilePassSmem, s, (const TileCta *)em->tile_ctas,
                        (const TileSeg *)em->tile_segs, em->tile_v.get<const double>(),
                        (const double *)em->tile_pi, em->state, em->tile_usum,
                        em->tile_slot_bytes, em->tile_n_slots,
                        (const double *)(kSlots ? slot_weights(em, 0) : nullptr),
                        kSlots ? em->n_rows : (int64_t)0, pi_stride, u_stride));
    if (marks) MXB_CUDA(cudaEventRecord(marks[1], s));
    // The gather waits in plain stream order: launched early it would sit on the SMs the
    // first CTAs of the pass leave and keep them from nothing, but measured it costs 27 us
    // per iteration (B200, config 2), while the other three launches gain from the overlap.
    g_plain_launch = true;
    MXB_CUDA(launch_pdl(tile_gather_kernel<kSlots>,
                        dim3((unsigned)ceil_div(em->ld, kGatherThreads), em->n_part, R),
                        dim3(kGatherThreads), 0, s, (const unsigned short *)em->tile_cmap,
                        em->tile_hs, (int)em->n_cols, em->ld, (const int *)em->tile_ent_batch,
                        (const int64_t *)em->tile_ent_off, em->tile_n_ent,
                        (const double *)em->tile_usum, (const EmState *)em->state, em->partials,
                        u_stride));
    if (marks) MXB_CUDA(cudaEventRecord(marks[2], s));
    ctx->launches += 3;
    return MXB_OK;
}

// Shared memory of the pass and of the class sums, set once per session.
template <bool kSlots>
static cudaError_t tile_pass_attrs(int64_t n_cols) {
    cudaError_t e = cudaFuncSetAttribute((const void *)tile_pass_kernel<kSlots>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(kSlots ? kTilePassSlotSmem : kTilePassSmem));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute((const void *)pick_tile_pi<kSlots>(n_cols),
                                cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)(kTileMaxCols * sizeof(double)));
}

// Blocks of the gather over n_ent U vectors: the partial column sums the tail adds (n_part).
static int tile_gather_parts(int n_ent) { return std::max(1, std::min(32, n_ent / 8)); }

// The tail of an iteration of R slots (em->tail): column sums, M-step, control block.
static int enqueue_tail(mxb_em *em, unsigned R) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    if (em->tail == EmTail::kSplit) {
        em_colreduce_kernel<<<(int)ceil_div(em->ld + 1, 256), 256, 0, s>>>(
            em->partials, em->n_part, em->ld, em->state, em->tsum);
        ctx->launches += 1;
        // the column sums and the underflow flag behind them (tsum[ld])
        if (em->sharded && ctx->world > 1) MXB_TRY(nccl_allreduce_sum_f64(ctx, em->tsum, em->ld + 1));
        em_update_kernel<<<1, kUpdThreads, 0, s>>>(em->tsum, em->n_cols, em->ld, em->lnp[0],
                                                   em->lnp[1], em->pi[0], em->pi[1], em->state);
        ctx->launches += 1;
        MXB_CUDA(cudaGetLastError());
        return MXB_OK;
    }
    P2PArgs pa;
    memset(&pa, 0, sizeof(pa));
    if (em->tail == EmTail::kPeer) {
        pa.world = ctx->world;
        pa.rank = ctx->rank;
        for (int r = 0; r < ctx->world; ++r) pa.block[r] = ctx->p2p_block[r];
    }
    MXB_CUDA(launch_pdl(em->tail == EmTail::kPeer ? em_finish_kernel<true> : em_finish_kernel<false>,
                        dim3(kFinCtas, R), dim3(kFinThreads), 0, s, em->partials, em->n_part,
                        em->n_cols, em->ld, em->lnp[0], em->lnp[1], em->pi[0], em->pi[1],
                        em->state, pa));
    ctx->launches += 1;
    return MXB_OK;
}

// One EM iteration on em->ctx->stream (no host sync): the pass of the session's form, then its
// tail.  `marks` (optional, 3 events) are recorded after the class sums, after the pass and
// after the gather of a tiled iteration (after the pass only for fp64 rows): per-kernel
// attribution.
static int enqueue_iteration(mxb_em *em, cudaEvent_t pass_begin = nullptr,
                             cudaEvent_t pass_end = nullptr, cudaEvent_t *marks = nullptr) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const unsigned R = (unsigned)em->n_slots;
    // fp64 rows of a bootstrap session: one replicate at a time, with the slot's weights
    const double *weights = slot_weights(em, 0);
    if (pass_begin) MXB_CUDA(cudaEventRecord(pass_begin, s));
    switch (em->form) {
    case EmForm::kTiles:
        MXB_TRY(em->boot ? enqueue_tile_pass<true>(em, R, marks)
                         : enqueue_tile_pass<false>(em, R, marks));
        break;
    case EmForm::kRowPairs:
        MXB_CUDA(launch_pdl(pick_pair(em->nc), dim3(em->grid_fast), dim3(kPassThreads),
                            em->smem_bytes, s, em->lin.get<const double>(), em->ld, em->n_rows, em->weights,
                            em->pi[0], em->pi[1], em->pi[0] + em->ld, em->pi[1] + em->ld,
                            em->state, em->partials,
                            em->partials + (size_t)em->n_part * em->ld, em->n_stages));
        ctx->launches += 1;
        break;
    case EmForm::kRows:
        MXB_CUDA(launch_pdl(pick_pass(em->nc), dim3(em->grid_fast), dim3(kPassThreads),
                            em->smem_bytes, s, em->lin.get<const unsigned char>(),
                            (uint32_t)(em->ld * sizeof(double)), em->ld, em->n_rows, weights,
                            em->pi[0], em->pi[1], em->state, em->partials, em->n_stages));
        ctx->launches += 1;
        break;
    case EmForm::kGeneral: {
        const int rd_blocks = (int)std::max<int64_t>(
            1, std::min<int64_t>(ceil_div(em->n_rows, 8), (int64_t)ctx->num_sms * 8));
        em_rowdot_kernel<<<rd_blocks, 256, 0, s>>>(em->lin.get<double>(), em->ld, em->n_rows, weights,
                                                   em->pi[0], em->pi[1], em->state, em->coef);
        dim3 grid(em->row_blocks, em->col_blocks);
        em_colacc_kernel<<<grid, 256, 0, s>>>(em->lin.get<double>(), em->ld, em->n_rows, em->coef, em->state,
                                              em->partials);
        ctx->launches += 2;
        break;
    }
    }
    if (pass_end) MXB_CUDA(cudaEventRecord(pass_end, s));
    if (marks && em->form != EmForm::kTiles)
        for (int i = 0; i < 3; ++i) MXB_CUDA(cudaEventRecord(marks[i], s));
    return enqueue_tail(em, R);
}

// Wall-clock stage times of the one-call entry points: collected into g_stage_ms when
// mxb_stage_timing(1) is on, printed on stderr as well with MXB_TIMING=1.
struct StageTimer {
    bool on, print;
    cudaStream_t stream;
    std::chrono::steady_clock::time_point t;
    explicit StageTimer(cudaStream_t s)
        : on(g_stage_on || getenv("MXB_TIMING") != nullptr), print(getenv("MXB_TIMING") != nullptr),
          stream(s) {
        if (on) t = std::chrono::steady_clock::now();
    }
    void mark(const char *what, int stage) {
        if (!on) return;
        cudaStreamSynchronize(stream);
        auto now = std::chrono::steady_clock::now();
        const double ms = std::chrono::duration<double, std::milli>(now - t).count();
        g_stage_ms[stage] += ms;
        if (print) fprintf(stderr, "[mxb timing] %-28s %9.3f ms\n", what, ms);
        t = now;
    }
};

static int reset_state(mxb_em *em, long long max_iter, double tol, int slot = 0, int done = 0) {
    EmState st;
    memset(&st, 0, sizeof(st));
    st.max_iter = max_iter;
    st.tol = tol;
    st.done = done;
    // synchronous w.r.t. the host buffer: pageable copy of a stack struct
    MXB_CUDA(cudaMemcpyAsync(em->state + slot, &st, sizeof(st), cudaMemcpyHostToDevice,
                             em->ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(em->ctx->stream));
    return MXB_OK;
}

}  // namespace mxb

extern "C" {

int mxb_em_destroy(mxb_em *em) {
    if (!em) return MXB_OK;
    cudaSetDevice(em->ctx->device);
    cudaStreamSynchronize(em->ctx->stream);
    delete em;  // (its blocks and events go with it; host_state is the context's pinned scratch)
    return MXB_OK;
}

}  // extern "C"

namespace mxb {

__global__ void em_reset_state_kernel(EmState *st, long long max_iter, double tol) {
    st->done = 0;
    st->cur = 0;
    st->bad = 0;
    st->iters = 0;
    st->max_iter = max_iter;
    st->tol = tol;
    st->delta = 0.0;
}

// The slot block of a session with R slots: [slot weights (bootstrap sessions) R x n_rows]
// [lnp 2 x R x ld][pi 2 x R x ld][partials R x n_part x ld][control blocks R], laid out on `c`
// and the session's slot buffers pointed into it; R = 1 gives the bytes of one slot.
static void slot_block(mxb_em *em, int R, int n_part, Carve &c) {
    const size_t ns = (size_t)R, ld = (size_t)em->ld;
    if (em->boot) em->slot_w = c.part<double>(ns * em->n_rows);
    for (double *&p : em->lnp) p = c.part<double>(ns * ld);
    for (double *&p : em->pi) p = c.part<double>(ns * ld);
    em->partials = c.part<double>(ns * n_part * ld);
    em->state = c.part<EmState>(ns);
}

// Layout of the batches and ring of the pass for the class counts of n rows (tile_plan.h).
struct TileShape {
    std::vector<TileDesc> desc;
    int64_t v_cells = 0, p_cells = 0;
    uint32_t ring_bytes = 0;   // ring slots of the pass and their count (tile_ring)
    int ring_slots = 0;
    bool ring_ok = false;      // false: rows too long for the ring
};
static void tile_shape(const int32_t *n_cls, int nb, int64_t n, TileShape &t) {
    int max_r_pad = 4;
    tile_layout(n_cls, nb, n, t.desc, t.v_cells, t.p_cells, max_r_pad);
    t.ring_ok = tile_ring(max_r_pad, t.ring_bytes, t.ring_slots);
}
// The same for class counts handed in from outside (mxb_tile_plan, mxb_boot_slots), checked
// first; an error names the entry point `who`.
static int tile_shape_checked(const char *who, const int32_t *n_cls, int64_t n_batches,
                              int64_t n_rows, int32_t num_sms, TileShape &t) {
    const char *bad = nullptr;
    if (!(n_cls != nullptr && n_batches > 0 && n_rows > (n_batches - 1) * kTileRows &&
          n_rows <= n_batches * kTileRows && num_sms > 0))
        bad = "bad arguments";
    for (int64_t b = 0; !bad && b < n_batches; ++b)
        if (n_cls[b] < 1 || n_cls[b] > kTileMaxCols) bad = "class counts must be in 1..8192";
    if (bad) {
        set_error("%s: %s", who, bad);
        return MXB_ERR_ARG;
    }
    tile_shape(n_cls, (int)n_batches, n_rows, t);
    return MXB_OK;
}

// The session's form, slot count and tail (EmForm, EmTail, n_slots): decided here and nowhere
// else.  `tiles`: the session iterates over class tiles (em_pack_tiles, once their class counts
// are known; `plan` is their plan on all SMs).  A session whose tiles do not pay off is decided
// again without them.
static void decide_form(mxb_em *em, int want_slots, const TileShape *tiles = nullptr,
                        const TilePlanOut *plan = nullptr) {
    mxb_ctx *ctx = em->ctx;
    const bool streams = em->n_stages > 0;
    const bool across = em->sharded && ctx->world > 1;
    const bool fused = streams && em->ld <= (int64_t)kFinCtas * kFinThreads &&
                       (!across || ctx->p2p_ready) && getenv("MXB_EM_SPLIT_TAIL") == nullptr;
    em->tail = !fused ? EmTail::kSplit : across ? EmTail::kPeer : EmTail::kFused;
    em->n_slots = 1;
    if (tiles) {
        em->form = EmForm::kTiles;   // restarts run one at a time over the tiles
        if (!em->boot) return;
        // the slotted tile kernels exist for the fused tail only
        em->tail = EmTail::kFused;
        if (!fused) return;
        Carve one;   // one slot and its class vectors (Pi, U)
        slot_block(em, 1, tile_gather_parts((int)plan->ent_batch.size()), one);
        one.part<double>(tiles->p_cells);
        one.part<double>(tiles->p_cells + plan->extra_cells);
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = 0; }
        em->n_slots = boot_slots(tiles->desc, em->n_rows, ctx->num_sms, tiles->ring_bytes,
                                 tiles->p_cells, (double)one.bytes(),
                                 (double)free_b);
    } else if (!streams) {
        em->form = EmForm::kGeneral;
    } else if (want_slots == 2 && fused && em->nc <= kMaxPairNC && !em->sharded) {
        em->form = EmForm::kRowPairs;
        em->n_slots = 2;
    } else {
        em->form = EmForm::kRows;
    }
}

template <int ITEMS>
static cudaError_t launch_tile_class(mxb_ctx *ctx, int grid, const unsigned long long *hash, int hs,
                                     int n_cols, int n_batches, unsigned short *perm,
                                     unsigned int *cword, unsigned short *cmap,
                                     unsigned short *rep, int *n_cls) {
    using Sort = cub::BlockRadixSort<unsigned long long, kTileThreads, ITEMS, unsigned short>;
    using Scan = cub::BlockScan<int, kTileThreads>;
    const size_t smem = std::max(sizeof(typename Sort::TempStorage), sizeof(typename Scan::TempStorage));
    cudaError_t e = cudaFuncSetAttribute((const void *)tile_class_kernel<ITEMS>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    tile_class_kernel<ITEMS><<<grid, kTileThreads, smem, ctx->stream>>>(hash, hs, n_cols, n_batches,
                                                                        perm, cword, cmap, rep, n_cls);
    return cudaGetLastError();
}
// The class kernel for `items` = ceil(H / kTileThreads) columns a thread.
static auto pick_tile_class(int64_t n_cols) {
    const int items = (int)ceil_div(n_cols, kTileThreads);
    return items <= 4 ? launch_tile_class<4> : items <= 8 ? launch_tile_class<8>
           : items <= 12 ? launch_tile_class<12> : launch_tile_class<16>;
}

// Class tiles of the session's matrix (em_tiles.cuh), built straight from M: no N x ld copy of
// L is ever allocated when this succeeds (`built`).  The session's form is decided once the
// class counts are known (decide_form).  Falls through (MXB_OK, built == false) when the matrix
// does not compress to less than half of its fp64 rows, when memory is short, or when a batch
// fails the exact class check; the caller then decides the form without tiles and sets up the
// fp64 rows.  MXB_EM_NO_PACK=1 keeps the fp64 rows (cross-check).
static int em_pack_tiles(mxb_em *em, int want_slots, bool &built) {
    mxb_ctx *ctx = em->ctx;
    built = false;
    if (em->n_stages == 0 || em->n_rows == 0 || em->n_cols > kTileMaxCols ||
        getenv("MXB_EM_NO_PACK"))
        return MXB_OK;
    const int64_t n = em->n_rows, h = em->n_cols;
    const int nb = (int)ceil_div(n, kTileRows);
    const int hs = (int)round_up(h, 8);
    const bool verbose = getenv("MXB_TIMING") != nullptr;
    auto give_up = [&](const char *what) {
        if (verbose) fprintf(stderr, "[mxb tiles] not used: %s\n", what);
        return MXB_OK;
    };
    auto fail = [&](const char *what, cudaError_t e) {
        cudaGetLastError();
        set_error("em_pack_tiles (%s): %s", what, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? MXB_ERR_NOMEM : MXB_ERR_CUDA;
    };
    // scratch: [hash][rep][n_cls][bad]
    DevBlock scratch;
    unsigned long long *hash = nullptr;
    unsigned short *rep = nullptr;
    int *d_ncls = nullptr, *d_bad = nullptr;
    if (scratch.alloc_parts(ctx, __func__, [&](Carve &c) {
            hash = c.part<unsigned long long>((size_t)nb * hs);
            rep = c.part<unsigned short>((size_t)nb * hs);
            d_ncls = c.part<int>(nb);
            d_bad = c.part<int>(nb);
        }) != MXB_OK)
        return give_up("scratch");
    // persistent: [perm][cmap][cword][desc]; the class vectors and the plan of the pass follow in
    // a second block once the class counts are known
    DevBlock maps;
    unsigned short *perm = nullptr, *cmap = nullptr;
    unsigned int *cword = nullptr;
    TileDesc *d_desc = nullptr;
    if (maps.alloc_parts(ctx, __func__, [&](Carve &c) {
            perm = c.part<unsigned short>((size_t)nb * hs);
            cmap = c.part<unsigned short>((size_t)nb * hs);
            cword = c.part<unsigned int>((size_t)nb * kTileThreads);
            d_desc = c.part<TileDesc>(nb);
        }) != MXB_OK)
        return give_up("maps");

    const int grid = std::min(nb, ctx->num_sms * 2);
    tile_hash_kernel<<<std::min(nb, ctx->num_sms * 4), kTileThreads, 0, ctx->stream>>>(
        em->mat->data, n, h, nb, hash, hs);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = pick_tile_class(h)(ctx, grid, hash, hs, (int)h, nb, perm, cword, cmap, rep, d_ncls);
    ctx->launches += 2;
    std::vector<int> ncls((size_t)nb);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(ncls.data(), d_ncls, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost,
                            ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail("classes", e);

    // layout of the batches, ring geometry and plan of the pass (tile_plan.h)
    TileShape shape;
    tile_shape(ncls.data(), nb, n, shape);
    if (!shape.ring_ok) return give_up("rows too long for the ring");
    const std::vector<TileDesc> &desc = shape.desc;
    const int64_t v_cells = shape.v_cells, p_cells = shape.p_cells;
    const uint32_t slot_bytes = shape.ring_bytes;
    const int n_slots = shape.ring_slots;
    TilePlanOut plan;
    tile_plan(desc, n, ctx->num_sms, slot_bytes, p_cells, plan);
    decide_form(em, want_slots, &shape, &plan);
    const int n_rep = em->n_slots;   // replicate slots of a bootstrap session
    if (n_rep > 1) {
        plan = TilePlanOut();
        tile_plan(desc, n, ctx->num_sms / n_rep, slot_bytes, p_cells, plan);
    }
    const std::vector<TileCta> &ctas = plan.ctas;
    const std::vector<TileSeg> &segs = plan.segs;
    const std::vector<int> &ent_batch = plan.ent_batch;
    const std::vector<int64_t> &ent_off = plan.ent_off;
    const int64_t extra_cells = plan.extra_cells;
    const int n_copy = plan.n_copy;
    const int n_cta = (int)ctas.size(), n_seg = (int)segs.size();
    const int n_ent = (int)ent_batch.size();
    const int64_t u_cells = p_cells + extra_cells;
    const double tile_bytes = (double)v_cells * 8 + 3.0 * (double)nb * hs * 2 +
                              ((double)p_cells + (double)u_cells) * 8 * 2;
    const double fp64_bytes = (double)n * (double)em->ld * 8;
    if (verbose) {
        fprintf(stderr, "[mxb tiles] plan check: %d errors\n", tile_plan_check(desc, plan));
        int64_t c_sum = 0, c_max = 0, wide = 0;
        for (int b = 0; b < nb; ++b) {
            c_sum += desc[(size_t)b].n_cls;
            c_max = std::max<int64_t>(c_max, desc[(size_t)b].n_cls);
            wide += desc[(size_t)b].lg > 5;
        }
        {
            double mx = 0, mn = 1e30; int smx = 0, cmx = 0;
            for (const TileCta &c : ctas) {
                double by = 0;
                for (int q = 0; q < c.n_segs; ++q) by += (double)segs[(size_t)(c.seg0 + q)].n_rows * segs[(size_t)(c.seg0 + q)].r_pad * 8;
                mx = std::max(mx, by); mn = std::min(mn, by); smx = std::max(smx, c.n_segs); cmx = std::max(cmx, c.n_copies);
            }
            fprintf(stderr, "[mxb tiles] per CTA: bytes min %.0f max %.0f, segments max %d, copies max %d\n", mn, mx, smx, cmx);
        }
        fprintf(stderr, "[mxb tiles] %d batches of %d rows: classes mean %.1f max %lld, %lld wide "
                "batches, tiles %.3f GB (+ maps and vectors: %.3f GB) vs fp64 rows %.3f GB; %d CTAs, "
                "%d segments, %d copies, %d slots of %u B\n",
                nb, kTileRows, (double)c_sum / nb, (long long)c_max, (long long)wide,
                (double)v_cells * 8 / 1e9, tile_bytes / 1e9, fp64_bytes / 1e9, n_cta, n_seg, n_copy,
                n_slots, slot_bytes);
    }
    if (tile_bytes > 0.5 * fp64_bytes) return give_up("not worth it");

    // [Pi x n_rep][U x n_rep][plan]
    DevBlock v, vecs;
    double *pi_cls = nullptr, *u_sum = nullptr;
    TileCta *d_ctas = nullptr;
    TileSeg *d_segs = nullptr;
    int *d_entb = nullptr;
    int64_t *d_ento = nullptr;
    int64_t pi_stride = 0, u_stride = 0;
    size_t b_vecs = 0;
    if (v.alloc(ctx, (size_t)v_cells * sizeof(double), __func__) != MXB_OK ||
        vecs.alloc_parts(ctx, __func__, [&](Carve &c) {
            pi_cls = c.parts<double>(p_cells, n_rep, &pi_stride);
            u_sum = c.parts<double>(u_cells, n_rep, &u_stride);
            b_vecs = c.bytes();
            d_ctas = c.part<TileCta>(n_cta);
            d_segs = c.part<TileSeg>(n_seg);
            d_entb = c.part<int>(n_ent);
            d_ento = c.part<int64_t>(n_ent);
        }) != MXB_OK)
        return give_up("tiles");
    e = cudaMemcpyAsync(d_desc, desc.data(), (size_t)nb * sizeof(TileDesc), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_ctas, ctas.data(), (size_t)n_cta * sizeof(TileCta), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_segs, segs.data(), (size_t)n_seg * sizeof(TileSeg), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_entb, ent_batch.data(), (size_t)n_ent * sizeof(int), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_ento, ent_off.data(), (size_t)n_ent * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(pi_cls, 0, b_vecs, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_bad, 0, (size_t)nb * sizeof(int), ctx->stream);
    if (e == cudaSuccess) {
        tile_fill_kernel<<<std::min(nb, ctx->num_sms * 4), kTileThreads, 0, ctx->stream>>>(
            em->mat->data, h, d_desc, nb, cmap, rep, hs, (const double *)em->weights,
            v.get<double>(), d_bad);
        ctx->launches += 1;
        e = cudaGetLastError();
    }
    std::vector<int> bad((size_t)nb);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(bad.data(), d_bad, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = em->boot ? tile_pass_attrs<true>(h) : tile_pass_attrs<false>(h);
    if (e != cudaSuccess) return fail("fill", e);
    for (int b = 0; b < nb; ++b)
        if (bad[(size_t)b] != 0) return give_up("hash collision");

    built = true;
    em->n_batches = nb;
    em->tile_hs = hs;
    em->tile_block = std::move(maps);
    em->tile_vecs = std::move(vecs);
    em->tile_v = std::move(v);
    em->tile_perm = perm;
    em->tile_cmap = cmap;
    em->tile_cword = cword;
    em->tile_desc = d_desc;
    em->tile_ctas = d_ctas;
    em->tile_segs = d_segs;
    em->tile_ent_batch = d_entb;
    em->tile_ent_off = d_ento;
    em->tile_n_ent = n_ent;
    em->tile_slot_bytes = slot_bytes;
    em->tile_n_slots = n_slots;
    em->tile_usum = u_sum;
    em->tile_pi = pi_cls;
    em->tile_cells = v_cells;
    em->tile_grid = n_cta;
    em->n_part = tile_gather_parts(n_ent);
    em->tile_pi_stride = pi_stride;
    em->tile_u_stride = u_stride;
    // what an iteration reads and writes: the tiles, perm + cmap (Pi), cmap (gather), the class
    // vectors (Pi written and read, U written and read)
    em->tile_bytes_per_pass = v_cells * 8 + 3 * (int64_t)nb * hs * 2 + 2 * (p_cells + u_cells) * 8;
    return MXB_OK;
}

static int em_create_impl(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, int sharded,
                          int want_slots, mxb_em **out, bool boot = false) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr && out != nullptr, "NULL argument");
    // a rank of a row-sharded run may hold no rows at all (fewer signatures than GPUs)
    MXB_REQUIRE((m->n_rows > 0 || sharded) && m->n_cols > 0, "EM needs a non-empty matrix");
    MXB_REQUIRE(weights != nullptr || m->n_rows == 0, "weights is NULL");
    *out = nullptr;
    MXB_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<mxb_em> em(new (std::nothrow) mxb_em());
    if (!em) { set_error("out of host memory"); return MXB_ERR_NOMEM; }
    em->ctx = ctx;
    em->mat = m;
    em->n_rows = m->n_rows;
    em->n_cols = m->n_cols;
    em->ld = round_up(m->n_cols, kLdAlign);
    em->sharded = sharded != 0;
    em->boot = boot;

    // launch geometry
    const size_t row_bytes = (size_t)em->ld * sizeof(double);
    const size_t fixed = 2 * kPassWarps * kPassGroup * sizeof(double) + 8 * sizeof(uint64_t) + 128;
    const bool force_general = getenv("MXB_EM_FORCE_GENERAL") != nullptr;
    em->nc = (int)ceil_div(em->ld / 2, kPassThreads);
    if (!force_general && em->ld >= 1024 && em->nc <= kMaxNC && ctx->smem_optin > fixed) {
        int stages = (int)std::min<size_t>(8, (ctx->smem_optin - fixed) / row_bytes);
        if (stages >= kPassGroup + 1) {
            em->n_stages = stages;
            em->smem_bytes = (size_t)stages * row_bytes + fixed;
            em->grid_fast = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->num_sms, em->n_rows));
            em->n_part = em->grid_fast;
        }
    }
    const bool streams = em->n_stages > 0;
    if (!streams) {
        em->col_blocks = (int)ceil_div(em->ld / 2, 256);
        int64_t rb = std::max<int64_t>(1, (int64_t)ctx->num_sms * 4 / em->col_blocks);
        rb = std::min<int64_t>(rb, ceil_div(em->n_rows, 16));
        em->row_blocks = (int)std::max<int64_t>(1, rb);
        em->n_part = em->row_blocks;
    }

    // both blocks >= kCacheMinBlock: reused from the pool's cache, no cudaMalloc/cudaFree per session
    const char *who = "mxb_em_create";
    // the session-wide buffers in one block: [weights][coef (general path)][tsum + underflow
    // flag][props_in]
    MXB_TRY(em->small.alloc_parts(ctx, who, [&](Carve &c) {
        em->weights = c.part<double>(em->n_rows);
        if (!streams) em->coef = c.part<double>(em->n_rows);
        em->tsum = c.part<double>(em->ld + 1);
        em->props_in = c.part<double>(em->n_cols);
    }, kCacheMinBlock));
    MXB_TRY(em->poll_ev.create(2, cudaEventDisableTiming, who));
    static_assert(2 * kMaxSlots * sizeof(EmState) <= kPinnedScratchBytes, "pinned scratch");
    em->host_state = (EmState *)pinned_scratch(ctx);
    if (!em->host_state) {
        set_error("%s: cannot pin %zu bytes of host memory", who, kPinnedScratchBytes);
        return MXB_ERR_NOMEM;
    }
    if (em->n_rows > 0)   // (tile_fill_kernel reads them)
        MXB_CUDA(cudaMemcpyAsync(em->weights, weights, em->n_rows * sizeof(double),
                                 cudaMemcpyHostToDevice, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    // class tiles straight from M; only a matrix that does not compress gets fp64 rows of L
    bool tiled = false;
    MXB_TRY(em_pack_tiles(em.get(), want_slots, tiled));
    if (!tiled) decide_form(em.get(), want_slots);
    if (streams)
        MXB_CUDA(cudaFuncSetAttribute((const void *)pick_pass(em->nc),
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)em->smem_bytes));
    if (em->form == EmForm::kRowPairs)
        MXB_CUDA(cudaFuncSetAttribute((const void *)pick_pair(em->nc),
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)em->smem_bytes));
    MXB_TRY(em->slots.alloc_parts(ctx, who, [&](Carve &c) {
        slot_block(em.get(), em->n_slots, em->n_part, c);
    }, kCacheMinBlock));
    MXB_CUDA(cudaMemsetAsync(em->state, 0, em->n_slots * sizeof(EmState), ctx->stream));
    if (!tiled) {
        MXB_TRY(em->lin.alloc(ctx, (size_t)em->n_rows * row_bytes, who));
        if (em->n_rows > 0) {
            const int grid = (int)std::min<int64_t>(em->n_rows, (int64_t)ctx->num_sms * 8);
            to_linear_kernel<<<grid, 256, 0, ctx->stream>>>(m->data, em->n_rows, em->n_cols, em->ld,
                                                            em->lin.get<double>());
            ctx->launches++;
            MXB_CUDA(cudaGetLastError());
        }
    }
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    // a sharded session starts from zeroed peer mailboxes on every rank (collective)
    if (em->tail == EmTail::kPeer) MXB_TRY(p2p_resync(ctx));
    *out = em.release();
    return MXB_OK;
}

}  // namespace mxb

extern "C" {

int mxb_em_create(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, int sharded,
                  mxb_em **out) {
    return em_create_impl(ctx, m, weights, sharded, 1, out);
}

int mxb_em_pass_bytes(const mxb_em *em, int64_t *bytes_per_pass, int64_t *n_dense_rows) {
    MXB_REQUIRE(em != nullptr, "NULL argument");
    const int64_t row_bytes = em->ld * (int64_t)sizeof(double);
    if (bytes_per_pass && em->form == EmForm::kTiles) {
        *bytes_per_pass = em->tile_bytes_per_pass;
        if (n_dense_rows) *n_dense_rows = 0;
        return MXB_OK;
    }
    if (bytes_per_pass) *bytes_per_pass = em->n_rows * row_bytes;
    if (n_dense_rows) *n_dense_rows = -1;
    return MXB_OK;
}

// One iteration in log space on the proportions lnp[cur] of restart slot `slot` (see
// em_logspace_*): called when the tail flagged done = kDoneNeedsLogStep.  Leaves the control
// block as a normal tail would (iters + 1, convergence / max_iter decision, buffers swapped).
// In a row-sharded session every rank calls it for the same iteration (the tails agree on
// the flag): the row lse is local, the column reduction spans the ranks as scipy's
// logsumexp forms it, global maxima first (all-reduce max), then the non-maximal sum s and
// the weight m of the maximal terms per column (all-reduce sum), so every rank forms the
// same ln pi' and takes the same decision.
static int em_logspace_step(mxb_em *em, int cur, int slot, const double *weights) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const int64_t n = em->n_rows, h = em->n_cols, ld = em->ld;
    const bool across = em->sharded && ctx->world > 1;
    const int64_t n_sums = across ? 2 * h : h;      // [s][m] or the plain column sums
    constexpr int kRowBlocks = 64;
    DevBlock tmp;
    double *lse = nullptr, *colmax = nullptr, *colsum = nullptr, *part = nullptr;
    MXB_TRY(tmp.alloc_parts(ctx, "EM log-space step", [&](Carve &c) {
        lse = c.part<double>(n);
        colmax = c.part<double>(h);
        colsum = c.part<double>(n_sums);
        part = c.part<double>((size_t)kRowBlocks * n_sums);
    }));
    const double *lnp = em->lnp[cur] + slot * ld;
    const int col_blocks = (int)ceil_div(h, 256);
    const dim3 col_grid(col_blocks, kRowBlocks);
    if (n > 0) {   // a rank of a row-sharded run may hold no rows
        const int row_grid = (int)std::min<int64_t>(n, (int64_t)ctx->num_sms * 8);
        em_logspace_rows_kernel<<<row_grid, 256, 0, s>>>(em->mat->data, n, h, lnp, lse);
        ctx->launches += 1;
    }
    em_logspace_cols_kernel<<<col_grid, 256, 0, s>>>(em->mat->data, n, h, lnp, lse, weights,
                                                     nullptr, part);
    em_logspace_colreduce_kernel<<<col_blocks, 256, 0, s>>>(part, kRowBlocks, h, 1, colmax);
    ctx->launches += 2;
    if (across) {
        MXB_TRY(nccl_allreduce_f64(ctx, colmax, h, 1));
        em_logspace_cols_split_kernel<<<col_grid, 256, 0, s>>>(
            em->mat->data, n, h, lnp, lse, weights, colmax, part);
        em_logspace_colreduce_kernel<<<(int)ceil_div(n_sums, 256), 256, 0, s>>>(
            part, kRowBlocks, n_sums, 0, colsum);
        ctx->launches += 2;
        MXB_TRY(nccl_allreduce_sum_f64(ctx, colsum, n_sums));
    } else {
        em_logspace_cols_kernel<<<col_grid, 256, 0, s>>>(em->mat->data, n, h, lnp, lse,
                                                         weights, colmax, part);
        em_logspace_colreduce_kernel<<<col_blocks, 256, 0, s>>>(part, kRowBlocks, h, 0, colsum);
        ctx->launches += 2;
    }
    em_logspace_update_kernel<<<1, kUpdThreads, 0, s>>>(
        colmax, colsum, across ? colsum + h : nullptr, h, ld, em->lnp[0] + slot * ld,
        em->lnp[1] + slot * ld, em->pi[0] + slot * ld, em->pi[1] + slot * ld, em->state + slot);
    ctx->launches += 1;
    MXB_CUDA(cudaGetLastError());
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

}  // extern "C"

namespace mxb {

// The host side of every EM run that stops on convergence (mxb_em_iterate, run_em's restarts).
// Iterations are enqueued in chunks ahead of the device for the restart slots that are live, and
// the host polls the control blocks of all slots two chunks behind; a finished restart turns
// the launches queued after it into early-exit no-ops.  No more iterations are enqueued than a
// live restart may still run (max_iter minus those already enqueued for it), so a run of one
// iteration launches one iteration's kernels.  Every decision depends only on the polled
// control blocks and the arguments: in a row-sharded session the control blocks are identical
// on every rank, so every rank enqueues the same launches (the NCCL tail and the peer-mailbox
// sequence numbers rely on it).
// An iteration flagged kDoneNeedsLogStep is redone in log space on its slot, and the run goes
// on from the state the step leaves; the other slots' runs are not touched.  Polls taken
// before a slot was redone or handed a new restart are ignored for that slot (generation
// counters).  finish(slot, state, again) is called for every restart that converged or reached
// max_iter; it sets `again` when it has put a new restart on the slot.
template <typename Finish>
static int em_poll_loop(mxb_em *em, int64_t max_iter, int n_live, Finish finish) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    constexpr int64_t kChunk = 16;
    bool live[kMaxSlots] = {};
    int gen[kMaxSlots] = {}, poll_gen[2][kMaxSlots] = {};
    int64_t enq[kMaxSlots] = {}, poll_enq[2][kMaxSlots] = {};   // iterations enqueued per restart
    bool pending[2] = {false, false};
    for (int sl = 0; sl < n_live; ++sl) live[sl] = true;
    auto room = [&]() {   // iterations the live restarts may still run
        int64_t r = 0;
        for (int sl = 0; sl < kMaxSlots; ++sl)
            if (live[sl]) r = std::max(r, max_iter - enq[sl]);
        return r;
    };
    for (int which = 0; n_live > 0; which ^= 1) {
        const int64_t n = std::min(kChunk, room());
        for (int64_t i = 0; i < n; ++i) MXB_TRY(enqueue_iteration(em));
        for (int sl = 0; sl < kMaxSlots; ++sl) enq[sl] += n;
        MXB_CUDA(cudaMemcpyAsync(em->host_state + which * kMaxSlots, em->state,
                                 em->n_slots * sizeof(EmState), cudaMemcpyDeviceToHost, s));
        MXB_CUDA(cudaEventRecord(em->poll_ev[which], s));
        std::copy(gen, gen + kMaxSlots, poll_gen[which]);
        std::copy(enq, enq + kMaxSlots, poll_enq[which]);
        pending[which] = true;
        // wait for the older poll, or for this one when nothing more can be enqueued
        const int w = pending[which ^ 1] ? which ^ 1 : room() == 0 ? which : -1;
        if (w < 0) continue;
        MXB_CUDA(cudaEventSynchronize(em->poll_ev[w]));
        pending[w] = false;
        for (int sl = 0; sl < em->n_slots; ++sl) {
            if (!live[sl] || poll_gen[w][sl] != gen[sl]) continue;
            EmState &st = em->host_state[w * kMaxSlots + sl];
            if (st.done == kDoneNeedsLogStep) {
                MXB_TRY(em_logspace_step(em, st.cur, sl, slot_weights(em, sl)));   // returns with the stream drained
                ++gen[sl];
                MXB_CUDA(cudaMemcpyAsync(&st, em->state + sl, sizeof(EmState),
                                         cudaMemcpyDeviceToHost, s));
                MXB_CUDA(cudaStreamSynchronize(s));
                enq[sl] = st.iters;
            } else if (!st.done && poll_enq[w][sl] >= max_iter) {
                // cannot happen: max_iter iterations always set done
                set_error("EM: run did not terminate");
                return MXB_ERR_CUDA;
            }
            if (!st.done) continue;
            if (st.done == 3) {
                set_error("EM: a peer rank did not deliver its column sums within %llu s",
                          (unsigned long long)(kP2PTimeoutNs / 1000000000ull));
                return MXB_ERR_CUDA;
            }
            if (st.bad) {
                set_error("EM: the mixture likelihood of %d row group(s) fell below 2^-960 or was NaN "
                          "(proportions left the fp64 range)", st.bad);
                return MXB_ERR_RANGE;
            }
            bool again = false;
            MXB_TRY(finish(sl, st, again));
            if (again) {
                ++gen[sl];
                enq[sl] = 0;
            } else {
                live[sl] = false;
                --n_live;
            }
        }
    }
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

// What a finished slot hands back (em.py:137-143): its final log-proportions are lnp[1 - cur],
// the ones before its last step (the read matrix's, SURVEY F5) lnp[cur].
struct SlotResult {
    const double *fin, *prev;
    int64_t iters;
    int32_t converged;
};
static SlotResult slot_result(const mxb_em *em, int sl, const EmState &st) {
    return {em->lnp[1 - st.cur] + sl * em->ld, em->lnp[st.cur] + sl * em->ld, st.iters,
            st.done == 1 ? 1 : 0};
}

// Read matrix of the log-proportions lnp (em.py:80-83) stored into dst (mode 0) or folded into
// it with numpy.logaddexp (mode 1, em.py:156); sub_log is subtracted afterwards (em.py:161).
static int launch_read_mix(mxb_em *em, const double *lnp, mxb_matrix *dst, int mode,
                           double sub_log) {
    if (em->n_rows == 0) return MXB_OK;   // a rank of a row-sharded run may hold no rows
    mxb_ctx *ctx = em->ctx;
    const int grid = (int)std::min<int64_t>(em->n_rows, (int64_t)ctx->num_sms * 8);
    read_mix_kernel<<<grid, kMixThreads, 0, ctx->stream>>>(em->mat->data, em->n_rows, em->n_cols,
                                                           lnp, dst->data, mode, sub_log);
    ctx->launches++;
    MXB_CUDA(cudaGetLastError());
    return MXB_OK;
}

}  // namespace mxb

extern "C" {

int mxb_em_set_lnprops(mxb_em *em, const double *lnprops) {
    MXB_REQUIRE(em != nullptr && lnprops != nullptr, "NULL argument");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    MXB_CUDA(cudaMemcpyAsync(em->props_in, lnprops, em->n_cols * sizeof(double),
                             cudaMemcpyHostToDevice, ctx->stream));
    em_set_props_kernel<<<(int)ceil_div(em->ld, 256), 256, 0, ctx->stream>>>(
        em->props_in, em->n_cols, em->ld, em->lnp[0], em->pi[0], em->lnp[1], em->pi[1]);
    ctx->launches++;
    MXB_CUDA(cudaGetLastError());
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));  // lnprops may be a temporary
    MXB_TRY(reset_state(em, 0, 0.0));
    em->zero_iter = true;
    return MXB_OK;
}

int mxb_em_iterate(mxb_em *em, int64_t max_iter, double tol, int64_t *iters_out,
                   int32_t *converged_out) {
    MXB_REQUIRE(em != nullptr, "em is NULL");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    if (iters_out) *iters_out = 0;
    if (converged_out) *converged_out = 0;
    em->zero_iter = max_iter <= 0;
    if (em->zero_iter) return MXB_OK;  // em.py:126 loop body never runs; :141-143 hands back the init
    // keep `cur` as set_lnprops left it (0), restart counters
    MXB_TRY(reset_state(em, max_iter, tol));
    return em_poll_loop(em, max_iter, 1, [&](int, const EmState &st, bool &) {
        if (iters_out) *iters_out = st.iters;
        if (converged_out) *converged_out = (st.done == 1);
        return MXB_OK;
    });
}

int mxb_em_iterate_fixed(mxb_em *em, int64_t n_iter, float *elapsed_ms, float *pass_ms) {
    MXB_REQUIRE(em != nullptr && n_iter >= 1 && n_iter <= 100000, "bad argument");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    em->zero_iter = false;
    MXB_TRY(reset_state(em, (long long)1 << 60, -1.0));
    // [start][end] of the run, then [begin][end] of every pass (pass_ms)
    Events evs;
    MXB_TRY(evs.create(2 + (pass_ms ? 2 * (size_t)n_iter : 0), cudaEventDefault, __func__));
    MXB_CUDA(cudaEventRecord(evs[0], ctx->stream));
    for (int64_t i = 0; i < n_iter; ++i) {
        if (pass_ms) MXB_TRY(enqueue_iteration(em, evs[2 + 2 * i], evs[3 + 2 * i]));
        else MXB_TRY(enqueue_iteration(em));
    }
    MXB_CUDA(cudaEventRecord(evs[1], ctx->stream));
    MXB_CUDA(cudaMemcpyAsync(&em->host_state[0], em->state, sizeof(EmState),
                             cudaMemcpyDeviceToHost, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (em->host_state[0].done == 3) {
        set_error("EM: a peer rank did not deliver its column sums in time");
        return MXB_ERR_CUDA;
    }
    // a tail that set done (kDoneNeedsLogStep after a row-likelihood underflow) turned the
    // remaining launches into no-ops: neither the time nor the proportions are those of n_iter
    // iterations
    if (em->host_state[0].done != 0 || em->host_state[0].iters != n_iter) {
        set_error("mxb_em_iterate_fixed: stopped after %lld of %lld iterations (done = %d)",
                  (long long)em->host_state[0].iters, (long long)n_iter,
                  (int)em->host_state[0].done);
        return MXB_ERR_RANGE;
    }
    if (elapsed_ms) MXB_CUDA(cudaEventElapsedTime(elapsed_ms, evs[0], evs[1]));
    if (pass_ms) {
        double total = 0.0;
        for (int64_t i = 0; i < n_iter; ++i) {
            float ms = 0.f;
            MXB_CUDA(cudaEventElapsedTime(&ms, evs[2 + 2 * i], evs[3 + 2 * i]));
            total += ms;
        }
        *pass_ms = (float)total;
    }
    return MXB_OK;
}

#ifdef MXB_TILE_TRACE
extern "C" int mxb_debug_tile_trace(unsigned long long *out, size_t n_words) {
    cudaDeviceSynchronize();
    return (int)cudaMemcpyFromSymbol(out, mxb::g_tile_trace, std::min(n_words * 8, sizeof(mxb::g_tile_trace)));
}
#endif

int mxb_tile_plan(const int32_t *n_cls, int64_t n_batches, int64_t n_rows, int32_t num_sms,
                  int32_t *seg_out, int64_t seg_cap, int32_t *n_cta, int32_t *n_seg,
                  int32_t *n_slots_out, int32_t *slot_bytes_out, int32_t *errors) {
    TileShape t;
    MXB_TRY(tile_shape_checked(__func__, n_cls, n_batches, n_rows, num_sms, t));
    const std::vector<TileDesc> &desc = t.desc;
    if (n_slots_out) *n_slots_out = t.ring_slots;
    if (slot_bytes_out) *slot_bytes_out = (int32_t)t.ring_bytes;
    MXB_REQUIRE(t.ring_ok, "rows too long for the ring");
    TilePlanOut plan;
    tile_plan(desc, n_rows, num_sms, t.ring_bytes, t.p_cells, plan);
    if (n_cta) *n_cta = (int32_t)plan.ctas.size();
    if (n_seg) *n_seg = (int32_t)plan.segs.size();
    if (errors) *errors = tile_plan_check(desc, plan);
    if (seg_out) {
        int64_t k = 0;
        for (size_t c = 0; c < plan.ctas.size(); ++c) {
            for (int q = 0; q < plan.ctas[c].n_segs && k < seg_cap; ++q, ++k) {
                const TileSeg &g = plan.segs[(size_t)(plan.ctas[c].seg0 + q)];
                const TileDesc &d = desc[(size_t)g.batch];
                int32_t *o = seg_out + 8 * k;
                o[0] = (int32_t)c;
                o[1] = g.batch;
                o[2] = (int32_t)((g.v_off - d.v_off) / d.r_pad);     // first row inside the batch
                o[3] = g.n_rows;
                o[4] = g.fit;
                o[5] = g.n_copies;
                o[6] = g.lg;
                o[7] = g.r_pad;
            }
        }
    }
    return MXB_OK;
}

int mxb_em_profile(mxb_em *em, int64_t n_iter, float *ms_out) {
    MXB_REQUIRE(em != nullptr && ms_out != nullptr && n_iter >= 1 && n_iter <= 10000, "bad argument");
    MXB_REQUIRE(em->n_slots == 1, "single-restart sessions only");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    em->zero_iter = false;
    MXB_TRY(reset_state(em, (long long)1 << 60, -1.0));
    Events evs;
    MXB_TRY(evs.create((size_t)n_iter * 5, cudaEventDefault, __func__));
    for (int64_t i = 0; i < n_iter; ++i) {
        cudaEvent_t *e = evs.data() + (size_t)i * 5;
        MXB_TRY(enqueue_iteration(em, e[0], nullptr, e + 1));
        MXB_CUDA(cudaEventRecord(e[4], ctx->stream));
    }
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    double tot[4] = {0, 0, 0, 0};
    for (int64_t i = 0; i < n_iter; ++i) {
        for (int k = 0; k < 4; ++k) {
            float ms = 0.f;
            MXB_CUDA(cudaEventElapsedTime(&ms, evs[(size_t)i * 5 + k], evs[(size_t)i * 5 + k + 1]));
            tot[k] += ms;
        }
    }
    // fp64 rows: the three marks coincide after the pass, so [0] holds the pass
    if (em->form != EmForm::kTiles) { tot[1] = tot[0]; tot[0] = 0.0; }
    for (int k = 0; k < 4; ++k) ms_out[k] = (float)(tot[k] / (double)n_iter);
    return MXB_OK;
}

int mxb_em_get_lnprops(mxb_em *em, int which, double *out) {
    MXB_REQUIRE(em != nullptr && out != nullptr && (which == 0 || which == 1), "bad argument");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    EmState st;
    MXB_CUDA(cudaMemcpyAsync(&st, em->state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    // after a finished run: lnp[cur] = previous, lnp[1-cur] = latest.
    int idx = (which == 0) ? 1 - st.cur : st.cur;
    if (st.done == 0) idx = 1 - idx;  // iterate_fixed: buffers were swapped after the last step
    if (em->zero_iter) idx = st.cur;  // no iteration ran: only the init exists
    MXB_CUDA(cudaMemcpyAsync(out, em->lnp[idx], em->n_cols * sizeof(double),
                             cudaMemcpyDeviceToHost, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXB_OK;
}

int mxb_em_read_mix(mxb_em *em, mxb_matrix *dst, int mode, double sub_log) {
    MXB_REQUIRE(em != nullptr && dst != nullptr && (mode == 0 || mode == 1), "bad argument");
    MXB_REQUIRE(dst->n_rows == em->n_rows && dst->n_cols == em->n_cols, "shape mismatch");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    EmState st;
    MXB_CUDA(cudaMemcpyAsync(&st, em->state, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return launch_read_mix(em, em->lnp[st.cur], dst, mode, sub_log);
}

int mxb_matrix_fold_ranks(mxb_ctx *ctx, mxb_matrix *m, double sub_log) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL argument");
    MXB_CUDA(cudaSetDevice(ctx->device));
    const int64_t n = m->n_rows * m->n_cols;
    if (n == 0) return MXB_OK;
    const int W = ctx->world, me = ctx->rank;
    cudaStream_t s = ctx->stream;
    if (W <= 1 || !ctx->nccl_comm) {
        if (sub_log != 0.0) {
            const int grid = (int)std::min<int64_t>(ceil_div(n, 256), (int64_t)ctx->num_sms * 16);
            fold_shift_kernel<<<grid, 256, 0, s>>>(m->data, n, sub_log);
            ctx->launches++;
            MXB_CUDA(cudaGetLastError());
        }
        MXB_CUDA(cudaStreamSynchronize(s));
        return MXB_OK;
    }
    // SURVEY 8(e): all-to-all of row shards, local logaddexp fold in rank order (restarts are
    // dealt in contiguous blocks, so rank order is restart order), shards gathered back.
    const int64_t lo = m->n_rows * me / W, hi = m->n_rows * (me + 1) / W;
    const int64_t max_rows = ceil_div(m->n_rows, W);
    const int64_t slot = max_rows * m->n_cols;
    DevBlock recv_block;   // the W receive slots
    MXB_TRY(recv_block.alloc(ctx, (size_t)W * (size_t)slot * sizeof(double), __func__));
    double *recv = recv_block.get<double>();
    MXB_TRY(nccl_alltoall_rows(ctx, m->data, recv, m->n_rows, m->n_cols, slot));
    if (hi > lo) {
        const int64_t cells = (hi - lo) * m->n_cols;
        const int grid = (int)std::min<int64_t>(ceil_div(cells, 256), (int64_t)ctx->num_sms * 16);
        fold_shards_kernel<<<grid, 256, 0, s>>>(m->data + lo * m->n_cols, recv, slot, cells, W, me,
                                                 sub_log);
        ctx->launches++;
        MXB_CUDA(cudaGetLastError());
    }
    MXB_TRY(nccl_allgather_rows(ctx, m->data, m->n_rows, m->n_cols));
    MXB_CUDA(cudaStreamSynchronize(s));
    return MXB_OK;
}

}  // extern "C"

namespace mxb {

// run_em's restart loop (em.py:117-163) on a session with one or two restart slots: restart i
// starts on the device from init_lnprops[i] as soon as a slot is free (two slots iterate two
// restarts per read of L), and em_poll_loop drives all of them.  Results are combined as the
// reference combines them: final log-proportions summed in restart order (em.py:145-155), then
// averaged and exponentiated unless `raw` (em.py:158-163); read matrices folded with logaddexp
// in restart order (em.py:156, :161).  A restart that finishes before an earlier one parks the
// proportions its read matrix is formed from until its turn.
static int run_restarts(mxb_em *em, const double *init_lnprops, int32_t n_multi, int64_t max_iter,
                        double tol, bool raw, mxb_matrix *mix, StageTimer &tm, double *props_out,
                        int64_t *iters_out, int32_t *converged_out) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const int64_t h = em->n_cols, ld = em->ld;
    // device: [inits n_multi x h][final log-proportions n_multi x h][the proportions before
    // the last step n_multi x h]; the finals are read back in one copy at the end (no pinned
    // host buffer, no blocking copy mid-run)
    const size_t vec_bytes = (size_t)n_multi * h * sizeof(double);
    DevBlock vecs;
    MXB_TRY(vecs.alloc(ctx, 3 * vec_bytes, "run_em"));
    double *d_inits = vecs.get<double>();
    double *d_fin = d_inits + (size_t)n_multi * h;
    double *d_prev = d_fin + (size_t)n_multi * h;
    std::vector<double> h_fin;
    std::vector<char> done_restart;       // finished, read matrix not folded yet (or folded)
    try {
        h_fin.resize((size_t)n_multi * h);
        done_restart.assign((size_t)n_multi, 0);
    } catch (const std::bad_alloc &) {
        set_error("run_em: out of host memory");
        return MXB_ERR_NOMEM;
    }
    MXB_TRY(copy_h2d(ctx, d_inits, init_lnprops, vec_bytes));

    int32_t next = 0, folded = 0;
    int slot_restart[kMaxSlots] = {-1, -1};
    auto start_slot = [&](int sl) {
        const int32_t idx = next++;
        slot_restart[sl] = idx;
        em_set_props_kernel<<<(int)ceil_div(ld, 256), 256, 0, s>>>(
            d_inits + (size_t)idx * h, h, ld, em->lnp[0] + sl * ld, em->pi[0] + sl * ld,
            em->lnp[1] + sl * ld, em->pi[1] + sl * ld);
        em_reset_state_kernel<<<1, 1, 0, s>>>(em->state + sl, (long long)max_iter, tol);
        ctx->launches += 2;
    };
    // fin, prev: the restart's final log-proportions and the ones before its last step
    auto finish_restart = [&](int32_t idx, const SlotResult &res) -> int {
        if (iters_out) iters_out[idx] = res.iters;
        if (converged_out) converged_out[idx] = res.converged;
        MXB_CUDA(cudaMemcpyAsync(d_fin + (size_t)idx * h, res.fin, h * sizeof(double),
                                 cudaMemcpyDeviceToDevice, s));
        if (!mix) return MXB_OK;
        // the read matrix comes from the proportions before the last step (SURVEY F5)
        MXB_CUDA(cudaMemcpyAsync(d_prev + (size_t)idx * h, res.prev, h * sizeof(double),
                                 cudaMemcpyDeviceToDevice, s));
        done_restart[(size_t)idx] = 1;
        if (!done_restart[(size_t)folded]) return MXB_OK;
        tm.mark("iterate", kStageIterate);
        for (; folded < n_multi && done_restart[(size_t)folded]; ++folded) {
            const bool last = folded == n_multi - 1;
            const double sub = (last && n_multi > 1 && !raw) ? log((double)n_multi) : 0.0;
            MXB_TRY(launch_read_mix(em, d_prev + (size_t)folded * h, mix, folded == 0 ? 0 : 1, sub));
        }
        tm.mark("read_mix kernel", kStageReadMix);
        return MXB_OK;
    };
    if (max_iter <= 0) {
        // em.py:126's loop body never runs: every restart hands back its init (em.py:141-143)
        for (int32_t i = 0; i < n_multi; ++i)
            MXB_TRY(finish_restart(i, {d_inits + (size_t)i * h, d_inits + (size_t)i * h, 0, 0}));
    } else {
        int n_live = 0;
        for (; n_live < em->n_slots && n_live < n_multi; ++n_live) start_slot(n_live);
        MXB_TRY(em_poll_loop(em, max_iter, n_live, [&](int sl, const EmState &st, bool &again) -> int {
            MXB_TRY(finish_restart(slot_restart[sl], slot_result(em, sl, st)));
            again = next < n_multi;
            if (again) start_slot(sl);
            return MXB_OK;
        }));
    }
    MXB_CUDA(cudaStreamSynchronize(s));
    tm.mark("iterate", kStageIterate);
    MXB_TRY(copy_d2h(ctx, h_fin.data(), d_fin, vec_bytes));
    for (int64_t j = 0; j < h; ++j) {
        double v = h_fin[j];
        for (int32_t i = 1; i < n_multi; ++i) v += h_fin[(size_t)i * h + j];  // em.py:155
        if (!raw) {
            if (n_multi > 1) v /= (double)n_multi;  // em.py:158-160
            v = exp(v);                             // em.py:163
        }
        props_out[j] = v;
    }
    return MXB_OK;
}

// Replicates whose results are kept on the device at a time: the output is downloaded in
// windows of this many rows (at most 177 MB at H = 5408), whatever n_boot is.
constexpr int64_t kBootOutRows = 4096;

// The bootstrap (bootstrap.cu for the draw): replicates boot0 .. boot0 + n_boot - 1 are put on
// the session's slots in order, each resampled on the device when its slot is handed it, started
// from `start` and iterated by em_poll_loop as one restart of run_em on its counts; a finished
// slot's final log-proportions go to row b - boot0 of the output and the slot takes the next
// replicate of the window.  Over class tiles the slots iterate side by side
// (enqueue_tile_pass<true>), over fp64 rows one at a time.
static int run_bootstrap(mxb_em *em, const double *start, const int64_t *d_cumw, uint64_t total,
                         uint64_t seed, int64_t boot0, int64_t n_boot, int64_t max_iter,
                         double tol, double *lnprops_out, int64_t *iters_out,
                         int32_t *converged_out) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const int64_t n = em->n_rows, h = em->n_cols, ld = em->ld;
    const size_t ns = (size_t)em->n_slots;
    const int64_t win = std::min(n_boot, kBootOutRows);
    // [counts n][start h][results win x h]
    DevBlock work;
    uint32_t *counts = nullptr;
    double *d_start = nullptr, *d_out = nullptr;
    MXB_TRY(work.alloc_parts(ctx, "bootstrap", [&](Carve &c) {
        counts = c.part<uint32_t>(n);
        d_start = c.part<double>(h);
        d_out = c.part<double>((size_t)win * h);
    }));
    MXB_CUDA(cudaMemsetAsync(counts, 0, (size_t)n * sizeof(uint32_t), s));
    // slots that get no replicate (n_boot < n_slots) stay done: their CTAs exit at once
    std::vector<EmState> idle(ns);
    for (EmState &st : idle) {
        memset(&st, 0, sizeof(st));
        st.done = 1;
    }
    MXB_TRY(copy_h2d(ctx, em->state, idle.data(), ns * sizeof(EmState)));
    MXB_TRY(copy_h2d(ctx, d_start, start, (size_t)h * sizeof(double)));

    int64_t next = 0, w_end = 0;
    int64_t slot_rep[kMaxSlots] = {};
    auto start_slot = [&](int sl) -> int {
        const int64_t k = next++;
        slot_rep[sl] = k;
        double *w = slot_weights(em, sl);
        MXB_TRY(boot_draw(ctx, d_cumw, n, total, seed, boot0 + k, 1, counts));
        MXB_TRY(boot_take_counts(ctx, counts, n, w));
        em_set_props_kernel<<<(int)ceil_div(ld, 256), 256, 0, s>>>(
            d_start, h, ld, em->lnp[0] + sl * ld, em->pi[0] + sl * ld, em->lnp[1] + sl * ld,
            em->pi[1] + sl * ld);
        em_reset_state_kernel<<<1, 1, 0, s>>>(em->state + sl, (long long)max_iter, tol);
        ctx->launches += 2;
        MXB_CUDA(cudaGetLastError());
        return MXB_OK;
    };
    for (int64_t w0 = 0; w0 < n_boot; w0 = w_end) {
        w_end = std::min(n_boot, w0 + win);
        int n_live = 0;
        for (; n_live < em->n_slots && next < w_end; ++n_live) MXB_TRY(start_slot(n_live));
        MXB_TRY(em_poll_loop(em, max_iter, n_live, [&](int sl, const EmState &st, bool &again) -> int {
                const SlotResult res = slot_result(em, sl, st);
                const int64_t k = slot_rep[sl];
                iters_out[k] = res.iters;
                converged_out[k] = res.converged;
                MXB_CUDA(cudaMemcpyAsync(d_out + (size_t)(k - w0) * h, res.fin,
                                         h * sizeof(double), cudaMemcpyDeviceToDevice, s));
            again = next < w_end;
            if (again) MXB_TRY(start_slot(sl));
            return MXB_OK;
        }));
        MXB_TRY(copy_d2h(ctx, lnprops_out + (size_t)w0 * h, d_out,
                         (size_t)(w_end - w0) * h * sizeof(double)));
    }
    return MXB_OK;
}

}  // namespace mxb

extern "C" {

int mxb_boot_slots(const int32_t *n_cls, int64_t n_batches, int64_t n_rows, int32_t num_sms,
                   double bytes_per_slot, double free_bytes, int32_t *slots_out) {
    MXB_REQUIRE(slots_out != nullptr, "bad arguments");
    TileShape t;
    MXB_TRY(tile_shape_checked(__func__, n_cls, n_batches, n_rows, num_sms, t));
    MXB_REQUIRE(t.ring_ok, "rows too long for the ring");
    *slots_out = boot_slots(t.desc, n_rows, num_sms, t.ring_bytes, t.p_cells, bytes_per_slot,
                            free_bytes);
    return MXB_OK;
}

int mxb_em_bootstrap(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                     const double *start_lnprops, int64_t boot0, int64_t n_boot, uint64_t seed,
                     int64_t max_iter, double tol, double *lnprops_out, int64_t *iters_out,
                     int32_t *converged_out, int32_t *slots_out) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr && weights != nullptr && start_lnprops != nullptr,
                "NULL argument");
    MXB_REQUIRE(lnprops_out != nullptr && iters_out != nullptr && converged_out != nullptr,
                "NULL buffer");
    const int64_t n = m->n_rows, h = m->n_cols;
    if (n_boot < 1 || boot0 < 0 || boot0 + n_boot > (1ll << 32)) {
        set_error("bootstrap: need n_boot >= 1 and replicate numbers in [0, 2^32)");
        return MXB_ERR_VALUE;
    }
    double mass = 0.0;
    for (int64_t j = 0; j < h; ++j) {
        if (isnan(start_lnprops[j])) {
            set_error("bootstrap: start log-proportion %lld is NaN", (long long)j);
            return MXB_ERR_VALUE;
        }
        mass += exp(start_lnprops[j]);
    }
    if (!(mass > 0.0)) {
        set_error("bootstrap: the start proportions sum to 0");
        return MXB_ERR_VALUE;
    }
    std::vector<int64_t> cumw;
    uint64_t total = 0;
    MXB_TRY(boot_prefix(weights, n, cumw, total));
    if (slots_out) *slots_out = 1;
    if (max_iter <= 0) {
        // em.py:126's loop body never runs: every replicate hands back the start (em.py:141-143)
        for (int64_t k = 0; k < n_boot; ++k) {
            memcpy(lnprops_out + k * h, start_lnprops, (size_t)h * sizeof(double));
            iters_out[k] = 0;
            converged_out[k] = 0;
        }
        return MXB_OK;
    }
    MXB_CUDA(cudaSetDevice(ctx->device));
    mxb_em *em = nullptr;
    MXB_TRY(em_create_impl(ctx, m, weights, 0, 1, &em, true));
    std::unique_ptr<mxb_em, decltype(&mxb_em_destroy)> session(em, mxb_em_destroy);
    DevBlock cumw_block;
    MXB_TRY(cumw_block.alloc(ctx, (size_t)n * sizeof(int64_t), "bootstrap"));
    int64_t *d_cumw = cumw_block.get<int64_t>();
    MXB_TRY(copy_h2d(ctx, d_cumw, cumw.data(), (size_t)n * sizeof(int64_t)));
    if (slots_out) *slots_out = em->n_slots;
    MXB_TRY(run_bootstrap(em, start_lnprops, d_cumw, total, seed, boot0, n_boot, max_iter, tol,
                          lnprops_out, iters_out, converged_out));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXB_OK;
}

int mxb_run_em_dev(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                   const double *init_lnprops, int32_t n_multi, int64_t max_iter, double tol,
                   int32_t flags, double *props_out, double *read_mix_out,
                   mxb_matrix **read_mix_dev, int64_t *iters_out, int32_t *converged_out) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr, "NULL handle");
    MXB_REQUIRE(init_lnprops != nullptr && props_out != nullptr, "NULL buffer");
    MXB_REQUIRE(n_multi >= 1, "n_multi must be >= 1");
    if (read_mix_dev) *read_mix_dev = nullptr;
    const int64_t h = m->n_cols;
    const bool raw = (flags & MXB_EM_RAW) != 0;
    const bool want_mix = read_mix_out != nullptr || read_mix_dev != nullptr;

    mxb_em *em = nullptr;
    mxb_matrix *mix = nullptr;
    StageTimer tm(ctx->stream);
    // the caller's result buffer is usually fresh pageable memory: fault its pages in
    // from background threads while the GPU iterates
    Prefault fault_mix;
    const bool sharded = (flags & MXB_EM_SHARDED) != 0;
    const int want_slots = (n_multi >= 2 && max_iter > 0 && !sharded &&
                            getenv("MXB_EM_NO_BATCH") == nullptr) ? 2 : 1;
    int rc = em_create_impl(ctx, m, weights, sharded, want_slots, &em);
    tm.mark("em_create (tiles or fp64 rows)", kStageSetup);
    if (rc == MXB_OK && want_mix) rc = mxb_matrix_alloc(ctx, m->n_rows, h, &mix);
    tm.mark("alloc read_mix", kStageSetup);
    // (started after the device allocations: page faults and cudaMalloc contend for the
    // process's mmap lock)
    if (rc == MXB_OK && read_mix_out)
        fault_mix.start(read_mix_out, (size_t)m->n_rows * (size_t)h * sizeof(double));
    if (rc == MXB_OK)
        rc = run_restarts(em, init_lnprops, n_multi, max_iter, tol, raw, mix, tm, props_out,
                          iters_out, converged_out);
    if (rc == MXB_OK && read_mix_out) {
        fault_mix.join();
        rc = mxb_matrix_download(ctx, mix, read_mix_out);
        tm.mark("download read_mix", kStageD2H);
    }
    mxb_em_destroy(em);
    if (rc == MXB_OK && read_mix_dev) *read_mix_dev = mix;
    else mxb_matrix_destroy(mix);
    tm.mark("free", kStageOther);
    return rc;
}

int mxb_run_em(mxb_ctx *ctx, const double *read_hap_mat, const double *weights, int64_t n_rows,
               int64_t n_cols, const double *init_lnprops, int32_t n_multi, int64_t max_iter,
               double tol, int32_t flags, double *props_out, double *read_mix_out,
               int64_t *iters_out, int32_t *converged_out) {
    mxb_matrix *m = nullptr;
    MXB_TRY(mxb_matrix_upload(ctx, read_hap_mat, n_rows, n_cols, &m));
    int rc = mxb_run_em_dev(ctx, m, weights, init_lnprops, n_multi, max_iter, tol, flags,
                            props_out, read_mix_out, nullptr, iters_out, converged_out);
    mxb_matrix_destroy(m);
    return rc;
}

int mxb_em_step(mxb_ctx *ctx, const double *read_hap_mat, const double *weights,
                const double *ln_props, int64_t n_rows, int64_t n_cols, double *read_mix_out,
                double *new_props_out) {
    MXB_REQUIRE(read_mix_out != nullptr && new_props_out != nullptr && ln_props != nullptr,
                "NULL buffer");
    // one restart, one iteration that never converges (tol -1), not averaged: the result is
    // its new log-proportions, the read matrix is stored from the previous ones (= ln_props)
    return mxb_run_em(ctx, read_hap_mat, weights, n_rows, n_cols, ln_props, 1, 1, -1.0,
                      MXB_EM_RAW, new_props_out, read_mix_out, nullptr, nullptr);
}

}  // extern "C"
