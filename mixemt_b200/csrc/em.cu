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
#include "em_tiles.h"


using namespace mxb;

namespace mxb {
// What an iteration runs (decide_form): its pass over class tiles, over fp64 rows (streamed,
// or streamed with two restarts per read of L) or the general path; its tail in one cluster
// launch (em_finish_kernel), the same with the ranks' sums exchanged through peer memory, or
// split (em_colreduce_kernel, NCCL all-reduce across ranks, em_update_kernel).
enum class EmForm { kTiles, kRows, kRowPairs, kGeneral };
enum class EmTail { kFused, kPeer, kSplit };
// What a session is created for: run_em's restarts (and mxb_em_create's sessions), or a slotted
// session of constrained refits (the slots share one weight vector) or of bootstrap replicates
// (every slot iterates on its own resampled counts).
enum class EmKind { kRestarts, kRefit, kBootstrap };

// The fp64-row form: L and the launch geometry of its passes (row_form).  The streaming pass
// (em_pass_fast_kernel, em_pass_pair_kernel) runs when the rows fit its ring (n_stages > 0);
// otherwise the general path (em_rowdot_kernel, em_colacc_kernel).
struct RowForm {
    DevBlock lin;              // [n_rows][ld] doubles; not allocated over class tiles
    double *coef = nullptr;    // [n_rows] (general path)
    int nc = 0;                // double2 column chunks per thread of the streaming pass
    int n_stages = 0;
    size_t smem_bytes = 0;
    int grid = 0;
    int row_blocks = 0, col_blocks = 0;   // general path
};
}  // namespace mxb

struct mxb_em {
    mxb_ctx *ctx = nullptr;
    const mxb_matrix *mat = nullptr;
    int64_t n_rows = 0, n_cols = 0, ld = 0;
    bool sharded = false;
    double *weights = nullptr;    // [n_rows]
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
    // of L, a slotted session R restarts per iteration.  Slot s lives at lnp[b] + s*ld,
    // pi[b] + s*ld, partials + s*n_part*ld, state + s (slot_block).
    int n_slots = 1;
    RowForm rows;     // the fp64 rows (geometry set for every session)
    TileForm tiles;   // form kTiles: class tiles (em_tiles.h) instead of rows.lin
    DevBlock small;   // one device block behind weights ... props_in (fewer driver calls)
    DevBlock slots;   // the slot block (slot_block)
    bool zero_iter = false;  // last iterate() ran no iteration
    // Slotted session (EmKind::kRefit, kBootstrap): n_slots restarts per launch, side by side
    // over class tiles.  A bootstrap session gives every slot its own weight vector (own_weights:
    // slot_w, the resampled counts); the slots of a refit session share `weights`.
    bool slotted = false, own_weights = false;
    double *slot_w = nullptr;
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

// The weights slot `slot` iterates on: its resampled counts in a bootstrap session.
static double *slot_weights(mxb_em *em, int slot) {
    return em->own_weights ? em->slot_w + slot * em->n_rows : em->weights;
}

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
    MXB_CUDA(launch_kernel(true, em->tail == EmTail::kPeer ? em_finish_kernel<true>
                                                           : em_finish_kernel<false>,
                           dim3(kFinCtas, R), dim3(kFinThreads), 0, s, em->partials, em->n_part,
                           em->n_cols, em->ld, em->lnp[0], em->lnp[1], em->pi[0], em->pi[1],
                           em->state, pa));
    ctx->launches += 1;
    return MXB_OK;
}

// One EM iteration on em->ctx->stream (no host sync): the pass of the session's form, then its
// tail.  `marks` (optional, kMarks events) are recorded before the pass, after the class sums,
// after the pass and after the gather of a tiled iteration (the three coincide after the pass
// of fp64 rows), and after the tail: per-kernel attribution.
constexpr int kMarks = 5;
static int enqueue_iteration(mxb_em *em, const cudaEvent_t *marks = nullptr) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const unsigned R = (unsigned)em->n_slots;
    const RowForm &rf = em->rows;
    // fp64 rows of a slotted session: one restart at a time, with the slot's weights
    const double *weights = slot_weights(em, 0);
    if (marks) MXB_CUDA(cudaEventRecord(marks[0], s));
    switch (em->form) {
    case EmForm::kTiles:
        MXB_TRY(tile_pass(ctx, em->tiles, R, em->n_cols, em->ld, em->pi, em->state, em->partials,
                          weights, em->own_weights ? em->n_rows : (int64_t)0,
                          marks ? marks + 1 : nullptr));
        break;
    case EmForm::kRowPairs:
        MXB_CUDA(launch_kernel(true, pick_pair(rf.nc), dim3(rf.grid), dim3(kPassThreads),
                               rf.smem_bytes, s, rf.lin.get<const double>(), em->ld, em->n_rows,
                               em->weights, em->pi[0], em->pi[1], em->pi[0] + em->ld,
                               em->pi[1] + em->ld, em->state, em->partials,
                               em->partials + (size_t)em->n_part * em->ld, rf.n_stages));
        ctx->launches += 1;
        break;
    case EmForm::kRows:
        MXB_CUDA(launch_kernel(true, pick_pass(rf.nc), dim3(rf.grid), dim3(kPassThreads),
                               rf.smem_bytes, s, rf.lin.get<const unsigned char>(),
                               (uint32_t)(em->ld * sizeof(double)), em->ld, em->n_rows, weights,
                               em->pi[0], em->pi[1], em->state, em->partials, rf.n_stages));
        ctx->launches += 1;
        break;
    case EmForm::kGeneral: {
        const int rd_blocks = (int)std::max<int64_t>(
            1, std::min<int64_t>(ceil_div(em->n_rows, 8), (int64_t)ctx->num_sms * 8));
        em_rowdot_kernel<<<rd_blocks, 256, 0, s>>>(rf.lin.get<double>(), em->ld, em->n_rows, weights,
                                                   em->pi[0], em->pi[1], em->state, rf.coef);
        dim3 grid(rf.row_blocks, rf.col_blocks);
        em_colacc_kernel<<<grid, 256, 0, s>>>(rf.lin.get<double>(), em->ld, em->n_rows, rf.coef, em->state,
                                              em->partials);
        ctx->launches += 2;
        break;
    }
    }
    if (marks && em->form != EmForm::kTiles)
        for (int i = 1; i < 4; ++i) MXB_CUDA(cudaEventRecord(marks[i], s));
    MXB_TRY(enqueue_tail(em, R));
    if (marks) MXB_CUDA(cudaEventRecord(marks[4], s));
    return MXB_OK;
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

// The slot block of a session with R slots: [slot weights (own_weights) R x n_rows]
// [lnp 2 x R x ld][pi 2 x R x ld][partials R x n_part x ld][control blocks R], laid out on `c`
// and the session's slot buffers pointed into it; R = 1 gives the bytes of one slot.
static void slot_block(mxb_em *em, int R, int n_part, Carve &c) {
    const size_t ns = (size_t)R, ld = (size_t)em->ld;
    if (em->own_weights) em->slot_w = c.part<double>(ns * em->n_rows);
    for (double *&p : em->lnp) p = c.part<double>(ns * ld);
    for (double *&p : em->pi) p = c.part<double>(ns * ld);
    em->partials = c.part<double>(ns * n_part * ld);
    em->state = c.part<EmState>(ns);
}

// The session's form, slot count and tail (EmForm, EmTail, n_slots): decided here and nowhere
// else.  `tiles`: the session iterates over class tiles (tile_classify, once their class counts
// are known; `plan` is their plan on all SMs).  A session whose tiles do not pay off is decided
// again without them.
static void decide_form(mxb_em *em, int want_slots, const TileShape *tiles = nullptr,
                        const TilePlanOut *plan = nullptr) {
    mxb_ctx *ctx = em->ctx;
    const bool streams = em->rows.n_stages > 0;
    const bool across = em->sharded && ctx->world > 1;
    const bool fused = streams && em->ld <= (int64_t)kFinCtas * kFinThreads &&
                       (!across || ctx->p2p_ready) && getenv("MXB_EM_SPLIT_TAIL") == nullptr;
    em->tail = !fused ? EmTail::kSplit : across ? EmTail::kPeer : EmTail::kFused;
    em->n_slots = 1;
    if (tiles) {
        em->form = EmForm::kTiles;   // restarts run one at a time over the tiles
        if (!em->slotted) return;
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
    } else if (want_slots == 2 && fused && em->rows.nc <= kMaxPairNC && !em->sharded) {
        em->form = EmForm::kRowPairs;
        em->n_slots = 2;
    } else {
        em->form = EmForm::kRows;
    }
}

// Launch geometry of the fp64-row passes of an n_rows x ld session: the streaming pass when a
// ring of at least kPassGroup + 1 rows fits the shared memory (and MXB_EM_FORCE_GENERAL is not
// set), else the general path.  Returns the blocks of column-sum partials of the pass (n_part).
static int row_form(const mxb_ctx *ctx, int64_t n_rows, int64_t ld, RowForm &r) {
    const size_t row_bytes = (size_t)ld * sizeof(double);
    const size_t fixed = 2 * kPassWarps * kPassGroup * sizeof(double) + 8 * sizeof(uint64_t) + 128;
    const bool force_general = getenv("MXB_EM_FORCE_GENERAL") != nullptr;
    r.nc = (int)ceil_div(ld / 2, kPassThreads);
    if (!force_general && ld >= 1024 && r.nc <= kMaxNC && ctx->smem_optin > fixed) {
        int stages = (int)std::min<size_t>(8, (ctx->smem_optin - fixed) / row_bytes);
        if (stages >= kPassGroup + 1) {
            r.n_stages = stages;
            r.smem_bytes = (size_t)stages * row_bytes + fixed;
            r.grid = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->num_sms, n_rows));
            return r.grid;
        }
    }
    r.col_blocks = (int)ceil_div(ld / 2, 256);
    int64_t rb = std::max<int64_t>(1, (int64_t)ctx->num_sms * 4 / r.col_blocks);
    rb = std::min<int64_t>(rb, ceil_div(n_rows, 16));
    r.row_blocks = (int)std::max<int64_t>(1, rb);
    return r.row_blocks;
}

static int em_create_impl(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, int sharded,
                          int want_slots, EmKind kind, mxb_em **out) {
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
    em->slotted = kind != EmKind::kRestarts;
    em->own_weights = kind == EmKind::kBootstrap;

    em->n_part = row_form(ctx, em->n_rows, em->ld, em->rows);
    RowForm &rf = em->rows;
    const bool streams = rf.n_stages > 0;

    // both blocks >= kCacheMinBlock: reused from the pool's cache, no cudaMalloc/cudaFree per session
    const char *who = "mxb_em_create";
    // the session-wide buffers in one block: [weights][coef (general path)][tsum + underflow
    // flag][props_in]
    MXB_TRY(em->small.alloc_parts(ctx, who, [&](Carve &c) {
        em->weights = c.part<double>(em->n_rows);
        if (!streams) rf.coef = c.part<double>(em->n_rows);
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
    if (em->n_rows > 0)   // (tile_fill reads them)
        MXB_CUDA(cudaMemcpyAsync(em->weights, weights, em->n_rows * sizeof(double),
                                 cudaMemcpyHostToDevice, ctx->stream));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    // class tiles straight from M in a session whose rows stream (not the general path); only a
    // matrix that does not compress gets fp64 rows of L
    bool tiled = false;
    {
        TileClasses classes;
        if (streams) MXB_TRY(tile_classify(ctx, m, classes, tiled));
        if (tiled) {
            decide_form(em.get(), want_slots, &classes.shape, &classes.plan);
            MXB_TRY(tile_fill(ctx, m, em->weights, em->ld, em->n_slots, em->slotted, classes,
                              tiled));
        }
        if (tiled) {
            em->tiles = std::move(classes.form);
            em->n_part = tile_gather_parts(em->tiles.n_ent);
        }
    }
    if (!tiled) decide_form(em.get(), want_slots);
    if (streams)
        MXB_CUDA(cudaFuncSetAttribute((const void *)pick_pass(rf.nc),
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rf.smem_bytes));
    if (em->form == EmForm::kRowPairs)
        MXB_CUDA(cudaFuncSetAttribute((const void *)pick_pair(rf.nc),
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rf.smem_bytes));
    MXB_TRY(em->slots.alloc_parts(ctx, who, [&](Carve &c) {
        slot_block(em.get(), em->n_slots, em->n_part, c);
    }, kCacheMinBlock));
    MXB_CUDA(cudaMemsetAsync(em->state, 0, em->n_slots * sizeof(EmState), ctx->stream));
    if (!tiled) {
        MXB_TRY(rf.lin.alloc(ctx, (size_t)em->n_rows * em->ld * sizeof(double), who));
        if (em->n_rows > 0) {
            const int grid = (int)std::min<int64_t>(em->n_rows, (int64_t)ctx->num_sms * 8);
            to_linear_kernel<<<grid, 256, 0, ctx->stream>>>(m->data, em->n_rows, em->n_cols, em->ld,
                                                            rf.lin.get<double>());
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
    return em_create_impl(ctx, m, weights, sharded, 1, EmKind::kRestarts, out);
}

int mxb_em_pass_bytes(const mxb_em *em, int64_t *bytes_per_pass, int64_t *n_dense_rows) {
    MXB_REQUIRE(em != nullptr, "NULL argument");
    const int64_t row_bytes = em->ld * (int64_t)sizeof(double);
    if (bytes_per_pass && em->form == EmForm::kTiles) {
        *bytes_per_pass = em->tiles.bytes_per_pass;
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

// The host side of every EM run that stops on convergence (mxb_em_iterate, run_tasks).
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

// The timed runs of mxb_em_iterate_fixed and mxb_em_profile: n_iter iterations from the
// session's proportions that never converge, enqueued without a host sync.  `evs` (created
// here; event errors name `who`) gets the start and the end of the run, then with `marked` the
// kMarks marks of every iteration (enqueue_iteration).
static int enqueue_fixed(mxb_em *em, int64_t n_iter, bool marked, Events &evs, const char *who) {
    cudaStream_t s = em->ctx->stream;
    em->zero_iter = false;
    MXB_TRY(reset_state(em, (long long)1 << 60, -1.0));
    MXB_TRY(evs.create(2 + (marked ? kMarks * (size_t)n_iter : 0), cudaEventDefault, who));
    MXB_CUDA(cudaEventRecord(evs[0], s));
    for (int64_t i = 0; i < n_iter; ++i)
        MXB_TRY(enqueue_iteration(em, marked ? evs.data() + 2 + kMarks * i : nullptr));
    MXB_CUDA(cudaEventRecord(evs[1], s));
    return MXB_OK;
}
// Milliseconds from mark a to mark b of every iteration of enqueue_fixed, summed.
static int marks_ms(Events &evs, int64_t n_iter, int a, int b, double &total) {
    total = 0.0;
    for (int64_t i = 0; i < n_iter; ++i) {
        float ms = 0.f;
        MXB_CUDA(cudaEventElapsedTime(&ms, evs[2 + kMarks * i + a], evs[2 + kMarks * i + b]));
        total += ms;
    }
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
    Events evs;
    MXB_TRY(enqueue_fixed(em, n_iter, pass_ms != nullptr, evs, __func__));
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
        MXB_TRY(marks_ms(evs, n_iter, 0, 3, total));   // the pass: before it to after the gather
        *pass_ms = (float)total;
    }
    return MXB_OK;
}

int mxb_em_profile(mxb_em *em, int64_t n_iter, float *ms_out) {
    MXB_REQUIRE(em != nullptr && ms_out != nullptr && n_iter >= 1 && n_iter <= 10000, "bad argument");
    MXB_REQUIRE(em->n_slots == 1, "single-restart sessions only");
    mxb_ctx *ctx = em->ctx;
    MXB_CUDA(cudaSetDevice(ctx->device));
    Events evs;
    MXB_TRY(enqueue_fixed(em, n_iter, true, evs, __func__));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    double tot[4] = {0, 0, 0, 0};   // class sums, pass, gather, tail
    for (int k = 0; k < 4; ++k) MXB_TRY(marks_ms(evs, n_iter, k, k + 1, tot[k]));
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

// Tasks whose final log-proportions are kept on the device at a time: they are downloaded in
// windows of this many rows (at most 177 MB at H = 5408), whatever the number of tasks.
constexpr int64_t kOutRows = 4096;

// The driver of every run of restarts on a session's slots (run_em's restarts, bootstrap
// replicates, constrained refits): tasks 0 .. n_tasks - 1 are put on the slots in order.  When a
// slot is handed task k, set_up(slot, k, start) does what the task needs first and names the
// device log-proportions it starts from; the slot then runs one run_em restart from there
// (em.py:117-143) under em_poll_loop.  A finished task's iterations and converged flag go to
// iters_out[k] and converged_out[k] (either may be NULL), its final log-proportions to row k of
// lnprops_out (host; downloaded one window of kOutRows tasks at a time), and finish(k, result)
// is called.  With max_iter <= 0 em.py:126's loop body never runs: every task hands back its
// start (em.py:141-143) and nothing is launched on the slots.  Over class tiles the slots of a
// slotted session iterate side by side (tile_pass), over fp64 rows one at a time;
// the two slots of a run_em session iterate two restarts per read of L.
template <typename SetUp, typename Finish>
static int run_tasks(mxb_em *em, int64_t n_tasks, int64_t max_iter, double tol,
                     double *lnprops_out, int64_t *iters_out, int32_t *converged_out,
                     SetUp set_up, Finish finish) {
    mxb_ctx *ctx = em->ctx;
    cudaStream_t s = ctx->stream;
    const int64_t h = em->n_cols, ld = em->ld;
    const int64_t win = std::min(n_tasks, kOutRows);
    DevBlock out_block;   // [final log-proportions win x h]
    MXB_TRY(out_block.alloc(ctx, (size_t)win * h * sizeof(double), "EM tasks"));
    double *d_out = out_block.get<double>();
    if (max_iter > 0 && n_tasks < em->n_slots) {
        // slots that get no task stay done: their CTAs exit at once
        std::vector<EmState> idle((size_t)(em->n_slots - n_tasks));
        for (EmState &st : idle) {
            memset(&st, 0, sizeof(st));
            st.done = 1;
        }
        MXB_TRY(copy_h2d(ctx, em->state + n_tasks, idle.data(), idle.size() * sizeof(EmState)));
    }

    int64_t next = 0, w0 = 0, w_end = 0;
    int64_t slot_task[kMaxSlots] = {};
    auto task_done = [&](int64_t k, const SlotResult &res) -> int {
        if (iters_out) iters_out[k] = res.iters;
        if (converged_out) converged_out[k] = res.converged;
        MXB_CUDA(cudaMemcpyAsync(d_out + (size_t)(k - w0) * h, res.fin, h * sizeof(double),
                                 cudaMemcpyDeviceToDevice, s));
        return finish(k, res);
    };
    auto start_slot = [&](int sl) -> int {
        const int64_t k = next++;
        slot_task[sl] = k;
        const double *start = nullptr;
        MXB_TRY(set_up(sl, k, start));
        em_set_props_kernel<<<(int)ceil_div(ld, 256), 256, 0, s>>>(
            start, h, ld, em->lnp[0] + sl * ld, em->pi[0] + sl * ld, em->lnp[1] + sl * ld,
            em->pi[1] + sl * ld);
        em_reset_state_kernel<<<1, 1, 0, s>>>(em->state + sl, (long long)max_iter, tol);
        ctx->launches += 2;
        MXB_CUDA(cudaGetLastError());
        return MXB_OK;
    };
    for (; w0 < n_tasks; w0 = w_end) {
        w_end = std::min(n_tasks, w0 + win);
        if (max_iter <= 0) {
            for (; next < w_end; ++next) {
                const double *start = nullptr;
                MXB_TRY(set_up(0, next, start));
                MXB_TRY(task_done(next, {start, start, 0, 0}));
            }
        } else {
            int n_live = 0;
            for (; n_live < em->n_slots && next < w_end; ++n_live) MXB_TRY(start_slot(n_live));
            MXB_TRY(em_poll_loop(em, max_iter, n_live, [&](int sl, const EmState &st,
                                                           bool &again) -> int {
                MXB_TRY(task_done(slot_task[sl], slot_result(em, sl, st)));
                again = next < w_end;
                if (again) MXB_TRY(start_slot(sl));
                return MXB_OK;
            }));
        }
        MXB_TRY(copy_d2h(ctx, lnprops_out + (size_t)w0 * h, d_out,
                         (size_t)(w_end - w0) * h * sizeof(double)));
    }
    return MXB_OK;
}

// run_em (em.py:117-163) on a session with one or two restart slots: restart i starts from
// init_lnprops[i] (run_tasks).  Results are combined as the reference combines them: final
// log-proportions summed in restart order (em.py:145-155), then averaged and exponentiated
// unless `raw` (em.py:158-163); read matrices folded with logaddexp in restart order (em.py:156,
// :161).  A restart that finishes before an earlier one parks the proportions its read matrix
// is formed from until its turn.
static int run_em_session(mxb_em *em, const double *init_lnprops, int32_t n_multi,
                          int64_t max_iter, double tol, bool raw, mxb_matrix *mix, StageTimer &tm,
                          double *props_out, int64_t *iters_out, int32_t *converged_out) {
    mxb_ctx *ctx = em->ctx;
    const int64_t h = em->n_cols;
    // device: [inits n_multi x h][the proportions before the last step n_multi x h]
    const size_t vec_bytes = (size_t)n_multi * h * sizeof(double);
    DevBlock vecs;
    MXB_TRY(vecs.alloc(ctx, 2 * vec_bytes, "run_em"));
    double *d_inits = vecs.get<double>();
    double *d_prev = d_inits + (size_t)n_multi * h;
    std::vector<double> h_fin;            // final log-proportions, restart by restart
    std::vector<char> done_restart;       // finished, read matrix not folded yet (or folded)
    try {
        h_fin.resize((size_t)n_multi * h);
        done_restart.assign((size_t)n_multi, 0);
    } catch (const std::bad_alloc &) {
        set_error("run_em: out of host memory");
        return MXB_ERR_NOMEM;
    }
    MXB_TRY(copy_h2d(ctx, d_inits, init_lnprops, vec_bytes));

    int32_t folded = 0;
    MXB_TRY(run_tasks(em, n_multi, max_iter, tol, h_fin.data(), iters_out, converged_out,
                      [&](int, int64_t i, const double *&start) -> int {
        start = d_inits + (size_t)i * h;
        return MXB_OK;
    }, [&](int64_t i, const SlotResult &res) -> int {
        if (!mix) return MXB_OK;
        // the read matrix comes from the proportions before the last step (SURVEY F5)
        MXB_CUDA(cudaMemcpyAsync(d_prev + (size_t)i * h, res.prev, h * sizeof(double),
                                 cudaMemcpyDeviceToDevice, ctx->stream));
        done_restart[(size_t)i] = 1;
        if (!done_restart[(size_t)folded]) return MXB_OK;
        tm.mark("iterate", kStageIterate);
        for (; folded < n_multi && done_restart[(size_t)folded]; ++folded) {
            const bool last = folded == n_multi - 1;
            const double sub = (last && n_multi > 1 && !raw) ? log((double)n_multi) : 0.0;
            MXB_TRY(launch_read_mix(em, d_prev + (size_t)folded * h, mix, folded == 0 ? 0 : 1, sub));
        }
        tm.mark("read_mix kernel", kStageReadMix);
        return MXB_OK;
    }));
    tm.mark("iterate", kStageIterate);
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

// Start log-proportions (K x H, host): no NaN, and proportions that sum to more than 0; an error
// names the entry point `who` and the vector.
static int check_starts(const char *who, const double *starts, int64_t n_vec, int64_t h) {
    for (int64_t k = 0; k < n_vec; ++k) {
        double mass = 0.0;
        for (int64_t j = 0; j < h; ++j) {
            if (isnan(starts[k * h + j])) {
                set_error("%s: start log-proportion %lld of vector %lld is NaN", who,
                          (long long)j, (long long)k);
                return MXB_ERR_VALUE;
            }
            mass += exp(starts[k * h + j]);
        }
        if (!(mass > 0.0)) {
            set_error("%s: the start proportions of vector %lld sum to 0", who, (long long)k);
            return MXB_ERR_VALUE;
        }
    }
    return MXB_OK;
}

// The body of the slotted entry points (mxb_em_bootstrap, mxb_em_refit) once their arguments
// are checked: n_tasks tasks on a session of `kind`, task k started from the host vector
// starts + k * stride (stride 0: one start for all) after prepare(em, slot, k) has done what
// else it needs.  With max_iter <= 0 em.py:126's loop body never runs: no session is created,
// nothing is launched, and every task hands back its start (em.py:141-143).
template <typename Prepare>
static int run_slotted(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, EmKind kind,
                       const double *starts, int64_t stride, int64_t n_tasks, int64_t max_iter,
                       double tol, double *lnprops_out, int64_t *iters_out,
                       int32_t *converged_out, int32_t *slots_out, Prepare prepare) {
    const int64_t h = m->n_cols;
    if (slots_out) *slots_out = 1;
    if (max_iter <= 0) {
        for (int64_t k = 0; k < n_tasks; ++k) {
            memcpy(lnprops_out + k * h, starts + k * stride, (size_t)h * sizeof(double));
            iters_out[k] = 0;
            converged_out[k] = 0;
        }
        return MXB_OK;
    }
    MXB_CUDA(cudaSetDevice(ctx->device));
    mxb_em *em = nullptr;
    MXB_TRY(em_create_impl(ctx, m, weights, 0, 1, kind, &em));
    std::unique_ptr<mxb_em, decltype(&mxb_em_destroy)> session(em, mxb_em_destroy);
    const size_t start_bytes = (size_t)(stride ? n_tasks : 1) * h * sizeof(double);
    DevBlock starts_block;
    MXB_TRY(starts_block.alloc(ctx, start_bytes, "slotted EM"));
    const double *d_starts = starts_block.get<double>();
    MXB_TRY(copy_h2d(ctx, starts_block.get(), starts, start_bytes));
    if (slots_out) *slots_out = em->n_slots;
    MXB_TRY(run_tasks(em, n_tasks, max_iter, tol, lnprops_out, iters_out, converged_out,
                      [&](int sl, int64_t k, const double *&start) -> int {
        MXB_TRY(prepare(em, sl, k));
        start = d_starts + k * stride;
        return MXB_OK;
    }, [](int64_t, const SlotResult &) { return MXB_OK; }));
    MXB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXB_OK;
}

}  // namespace mxb

extern "C" {

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
    MXB_TRY(check_starts("bootstrap", start_lnprops, 1, h));
    std::vector<int64_t> cumw;
    uint64_t total = 0;
    MXB_TRY(boot_prefix(weights, n, cumw, total));
    DevBlock work;   // [prefix sums n][counts n]
    int64_t *d_cumw = nullptr;
    uint32_t *counts = nullptr;
    // task k is replicate boot0 + k (bootstrap.cu for the draw), resampled on the device into
    // its slot's weights; all start from start_lnprops
    return run_slotted(ctx, m, weights, EmKind::kBootstrap, start_lnprops, 0, n_boot, max_iter,
                       tol, lnprops_out, iters_out, converged_out, slots_out,
                       [&](mxb_em *em, int sl, int64_t k) -> int {
        if (k == 0) {   // the first replicate takes the prefix sums to the device
            MXB_TRY(work.alloc_parts(ctx, "bootstrap", [&](Carve &c) {
                d_cumw = c.part<int64_t>(n);
                counts = c.part<uint32_t>(n);
            }));
            MXB_TRY(copy_h2d(ctx, d_cumw, cumw.data(), (size_t)n * sizeof(int64_t)));
            MXB_CUDA(cudaMemsetAsync(counts, 0, (size_t)n * sizeof(uint32_t), ctx->stream));
        }
        MXB_TRY(boot_draw(ctx, d_cumw, n, total, seed, boot0 + k, 1, counts));
        return boot_take_counts(ctx, counts, n, slot_weights(em, sl));
    });
}

int mxb_em_refit(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, const double *starts,
                 int64_t n_starts, int64_t max_iter, double tol, double *lnprops_out,
                 int64_t *iters_out, int32_t *converged_out, int32_t *slots_out) {
    MXB_REQUIRE(ctx != nullptr && m != nullptr && weights != nullptr && starts != nullptr,
                "NULL argument");
    MXB_REQUIRE(lnprops_out != nullptr && iters_out != nullptr && converged_out != nullptr,
                "NULL buffer");
    MXB_REQUIRE(n_starts >= 1, "need at least one start");
    MXB_TRY(check_starts("refit", starts, n_starts, m->n_cols));
    // refit k starts from starts[k]
    return run_slotted(ctx, m, weights, EmKind::kRefit, starts, m->n_cols, n_starts, max_iter,
                       tol, lnprops_out, iters_out, converged_out, slots_out,
                       [](mxb_em *, int, int64_t) { return MXB_OK; });
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
    int rc = em_create_impl(ctx, m, weights, sharded, want_slots, EmKind::kRestarts, &em);
    tm.mark("em_create (tiles or fp64 rows)", kStageSetup);
    if (rc == MXB_OK && want_mix) rc = mxb_matrix_alloc(ctx, m->n_rows, h, &mix);
    tm.mark("alloc read_mix", kStageSetup);
    // (started after the device allocations: page faults and cudaMalloc contend for the
    // process's mmap lock)
    if (rc == MXB_OK && read_mix_out)
        fault_mix.start(read_mix_out, (size_t)m->n_rows * (size_t)h * sizeof(double));
    if (rc == MXB_OK)
        rc = run_em_session(em, init_lnprops, n_multi, max_iter, tol, raw, mix, tm, props_out,
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
