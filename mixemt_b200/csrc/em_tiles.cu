// Host side of the class tiles (em_tiles.cuh): the set-up of a session's tiles, the three
// launches of a tiled pass, and the plan and slot count exposed to the CPU tests (mxb_tile_plan,
// mxb_boot_slots).
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "em_tiles.cuh"
#include "em_tiles.h"

namespace mxb {

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

// What an iteration reads and writes: the tiles, perm + cmap (Pi), cmap (gather), the class
// vectors (Pi written and read, U written and read).
static int64_t tile_pass_bytes(const TileShape &s, const TilePlanOut &plan, int nb, int hs) {
    const int64_t u_cells = s.p_cells + plan.extra_cells;
    return s.v_cells * 8 + 3 * (int64_t)nb * hs * 2 + 2 * (s.p_cells + u_cells) * 8;
}

int tile_gather_parts(int n_ent) { return std::max(1, std::min(32, n_ent / 8)); }

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

// The class-sum kernel of a tiled iteration for `per` = ceil(H / kTileThreads) columns a thread.
template <bool kSlots>
static auto pick_tile_pi(int64_t n_cols) {
    const int per = (int)ceil_div(n_cols, kTileThreads);
    return per <= 4 ? tile_pi_kernel<4, kSlots> : per <= 8 ? tile_pi_kernel<8, kSlots>
           : per <= 12 ? tile_pi_kernel<12, kSlots> : tile_pi_kernel<16, kSlots>;
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

// The set-up's name in error texts and allocation failures.
static const char kWho[] = "em_pack_tiles";

static int give_up(const char *what) {
    if (getenv("MXB_TIMING") != nullptr) fprintf(stderr, "[mxb tiles] not used: %s\n", what);
    return MXB_OK;
}
static int fail(const char *what, cudaError_t e) {
    cudaGetLastError();
    set_error("%s (%s): %s", kWho, what, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? MXB_ERR_NOMEM : MXB_ERR_CUDA;
}

int tile_classify(mxb_ctx *ctx, const mxb_matrix *m, TileClasses &c, bool &used) {
    used = false;
    if (m->n_rows == 0 || m->n_cols > kTileMaxCols || getenv("MXB_EM_NO_PACK")) return MXB_OK;
    const int64_t n = m->n_rows, h = m->n_cols;
    const int nb = (int)ceil_div(n, kTileRows);
    const int hs = (int)round_up(h, 8);
    unsigned long long *hash = nullptr;
    int *d_ncls = nullptr;
    if (c.scratch.alloc_parts(ctx, kWho, [&](Carve &p) {
            hash = p.part<unsigned long long>((size_t)nb * hs);
            c.rep = p.part<unsigned short>((size_t)nb * hs);
            d_ncls = p.part<int>(nb);
            c.bad = p.part<int>(nb);
        }) != MXB_OK)
        return give_up("scratch");
    // persistent: the maps; the class vectors and the plan of the pass follow in a second block
    // once the class counts are known
    TileForm &t = c.form;
    if (t.maps.alloc_parts(ctx, kWho, [&](Carve &p) {
            t.perm = p.part<unsigned short>((size_t)nb * hs);
            t.cmap = p.part<unsigned short>((size_t)nb * hs);
            t.cword = p.part<unsigned int>((size_t)nb * kTileThreads);
            t.desc = p.part<TileDesc>(nb);
        }) != MXB_OK)
        return give_up("maps");

    const int grid = std::min(nb, ctx->num_sms * 2);
    tile_hash_kernel<<<std::min(nb, ctx->num_sms * 4), kTileThreads, 0, ctx->stream>>>(
        m->data, n, h, nb, hash, hs);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = pick_tile_class(h)(ctx, grid, hash, hs, (int)h, nb, t.perm, t.cword, t.cmap, c.rep,
                               d_ncls);
    ctx->launches += 2;
    std::vector<int> ncls((size_t)nb);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(ncls.data(), d_ncls, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost,
                            ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail("classes", e);

    // layout of the batches, ring geometry and plan of the pass (tile_plan.h)
    tile_shape(ncls.data(), nb, n, c.shape);
    if (!c.shape.ring_ok) return give_up("rows too long for the ring");
    tile_plan(c.shape.desc, n, ctx->num_sms, c.shape.ring_bytes, c.shape.p_cells, c.plan);
    t.n_batches = nb;
    t.hs = hs;
    used = true;
    return MXB_OK;
}

int tile_fill(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, int64_t ld, int n_slots,
              bool slotted, TileClasses &c, bool &used) {
    used = false;
    const int64_t n = m->n_rows, h = m->n_cols;
    TileForm &t = c.form;
    const int nb = t.n_batches, hs = t.hs;
    const std::vector<TileDesc> &desc = c.shape.desc;
    const int64_t v_cells = c.shape.v_cells, p_cells = c.shape.p_cells;
    TilePlanOut &plan = c.plan;
    if (n_slots > 1) {
        plan = TilePlanOut();
        tile_plan(desc, n, ctx->num_sms / n_slots, c.shape.ring_bytes, p_cells, plan);
    }
    const std::vector<TileCta> &ctas = plan.ctas;
    const std::vector<TileSeg> &segs = plan.segs;
    const int n_cta = (int)ctas.size(), n_seg = (int)segs.size();
    const int n_ent = (int)plan.ent_batch.size();
    const int64_t u_cells = p_cells + plan.extra_cells;
    const int64_t tile_bytes = tile_pass_bytes(c.shape, plan, nb, hs);
    const double fp64_bytes = (double)n * (double)ld * 8;
    if (getenv("MXB_TIMING") != nullptr) {
        fprintf(stderr, "[mxb tiles] plan check: %d errors\n", tile_plan_check(desc, plan));
        int64_t c_sum = 0, c_max = 0, wide = 0;
        for (int b = 0; b < nb; ++b) {
            c_sum += desc[(size_t)b].n_cls;
            c_max = std::max<int64_t>(c_max, desc[(size_t)b].n_cls);
            wide += desc[(size_t)b].lg > 5;
        }
        {
            double mx = 0, mn = 1e30; int smx = 0, cmx = 0;
            for (const TileCta &cta : ctas) {
                double by = 0;
                for (int q = 0; q < cta.n_segs; ++q) by += (double)segs[(size_t)(cta.seg0 + q)].n_rows * segs[(size_t)(cta.seg0 + q)].r_pad * 8;
                mx = std::max(mx, by); mn = std::min(mn, by); smx = std::max(smx, cta.n_segs); cmx = std::max(cmx, cta.n_copies);
            }
            fprintf(stderr, "[mxb tiles] per CTA: bytes min %.0f max %.0f, segments max %d, copies max %d\n", mn, mx, smx, cmx);
        }
        fprintf(stderr, "[mxb tiles] %d batches of %d rows: classes mean %.1f max %lld, %lld wide "
                "batches, tiles %.3f GB (+ maps and vectors: %.3f GB) vs fp64 rows %.3f GB; %d CTAs, "
                "%d segments, %d copies, %d slots of %u B\n",
                nb, kTileRows, (double)c_sum / nb, (long long)c_max, (long long)wide,
                (double)v_cells * 8 / 1e9, (double)tile_bytes / 1e9, fp64_bytes / 1e9, n_cta, n_seg,
                plan.n_copy, c.shape.ring_slots, c.shape.ring_bytes);
    }
    if ((double)tile_bytes > 0.5 * fp64_bytes) return give_up("not worth it");

    // [Pi x n_slots][U x n_slots][plan]
    size_t b_vecs = 0;
    if (t.v.alloc(ctx, (size_t)v_cells * sizeof(double), kWho) != MXB_OK ||
        t.vecs.alloc_parts(ctx, kWho, [&](Carve &p) {
            t.pi = p.parts<double>(p_cells, n_slots, &t.pi_stride);
            t.usum = p.parts<double>(u_cells, n_slots, &t.u_stride);
            b_vecs = p.bytes();
            t.ctas = p.part<TileCta>(n_cta);
            t.segs = p.part<TileSeg>(n_seg);
            t.ent_batch = p.part<int>(n_ent);
            t.ent_off = p.part<int64_t>(n_ent);
        }) != MXB_OK)
        return give_up("tiles");
    cudaError_t e = cudaMemcpyAsync(t.desc, desc.data(), (size_t)nb * sizeof(TileDesc), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(t.ctas, ctas.data(), (size_t)n_cta * sizeof(TileCta), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(t.segs, segs.data(), (size_t)n_seg * sizeof(TileSeg), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(t.ent_batch, plan.ent_batch.data(), (size_t)n_ent * sizeof(int), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(t.ent_off, plan.ent_off.data(), (size_t)n_ent * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(t.pi, 0, b_vecs, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c.bad, 0, (size_t)nb * sizeof(int), ctx->stream);
    if (e == cudaSuccess) {
        tile_fill_kernel<<<std::min(nb, ctx->num_sms * 4), kTileThreads, 0, ctx->stream>>>(
            m->data, h, t.desc, nb, t.cmap, c.rep, hs, weights, t.v.get<double>(), c.bad);
        ctx->launches += 1;
        e = cudaGetLastError();
    }
    std::vector<int> bad((size_t)nb);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(bad.data(), c.bad, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = slotted ? tile_pass_attrs<true>(h) : tile_pass_attrs<false>(h);
    if (e != cudaSuccess) return fail("fill", e);
    for (int b = 0; b < nb; ++b)
        if (bad[(size_t)b] != 0) return give_up("hash collision");

    t.n_ctas = n_cta;
    t.n_ent = n_ent;
    t.ring_slots = c.shape.ring_slots;
    t.slot_bytes = c.shape.ring_bytes;
    t.bytes_per_pass = tile_bytes;
    t.slotted = slotted;
    used = true;
    return MXB_OK;
}

// kSlots: the R slots of a slotted session side by side (weights w_stride apart, or shared), the
// slot in blockIdx.y (z for the gather), all on one plan of num_sms / R CTAs; a slot whose
// control block says done costs nothing.
template <bool kSlots>
static int tile_pass_slots(mxb_ctx *ctx, const TileForm &t, unsigned R, int64_t n_cols,
                           int64_t ld, double *const pi[2], EmState *state, double *partials,
                           const double *weights, int64_t w_stride, const cudaEvent_t *marks) {
    cudaStream_t s = ctx->stream;
    const int64_t pi_stride = kSlots ? t.pi_stride : 0;
    const int64_t u_stride = kSlots ? t.u_stride : 0;
    MXB_CUDA(launch_kernel(true, pick_tile_pi<kSlots>(n_cols),
                           dim3(std::min(t.n_batches, std::max(1, 2 * ctx->num_sms / (int)R)), R),
                           dim3(kTileThreads), (size_t)ld * sizeof(double), s,
                           (const unsigned short *)t.perm, (const unsigned int *)t.cword, t.hs,
                           (int)n_cols, (const TileDesc *)t.desc, t.n_batches,
                           (const double *)pi[0], (const double *)pi[1], (const EmState *)state,
                           t.pi, kSlots ? ld : (int64_t)0, pi_stride));
    if (marks) MXB_CUDA(cudaEventRecord(marks[0], s));
    MXB_CUDA(launch_kernel(true, tile_pass_kernel<kSlots>, dim3(t.n_ctas, R), dim3(kTilePassThreads),
                           kSlots ? kTilePassSlotSmem : kTilePassSmem, s, (const TileCta *)t.ctas,
                           (const TileSeg *)t.segs, t.v.get<const double>(), (const double *)t.pi,
                           state, t.usum, t.slot_bytes, t.ring_slots,
                           (const double *)(kSlots ? weights : nullptr), w_stride, pi_stride,
                           u_stride));
    if (marks) MXB_CUDA(cudaEventRecord(marks[1], s));
    // The gather waits in plain stream order: launched early it would sit on the SMs the
    // first CTAs of the pass leave and keep them from nothing, but measured it costs 27 us
    // per iteration (B200, config 2), while the other three launches gain from the overlap.
    MXB_CUDA(launch_kernel(false, tile_gather_kernel<kSlots>,
                           dim3((unsigned)ceil_div(ld, kGatherThreads), tile_gather_parts(t.n_ent), R),
                           dim3(kGatherThreads), 0, s, (const unsigned short *)t.cmap, t.hs,
                           (int)n_cols, ld, (const int *)t.ent_batch, (const int64_t *)t.ent_off,
                           t.n_ent, (const double *)t.usum, (const EmState *)state, partials,
                           u_stride));
    if (marks) MXB_CUDA(cudaEventRecord(marks[2], s));
    ctx->launches += 3;
    return MXB_OK;
}

int tile_pass(mxb_ctx *ctx, const TileForm &t, unsigned R, int64_t n_cols, int64_t ld,
              double *const pi[2], EmState *state, double *partials, const double *weights,
              int64_t w_stride, const cudaEvent_t *marks) {
    return t.slotted ? tile_pass_slots<true>(ctx, t, R, n_cols, ld, pi, state, partials, weights,
                                             w_stride, marks)
                     : tile_pass_slots<false>(ctx, t, R, n_cols, ld, pi, state, partials, weights,
                                              w_stride, marks);
}

}  // namespace mxb

using namespace mxb;

extern "C" {

#ifdef MXB_TILE_TRACE
// g_tile_trace (em_tiles.cuh) exists once per translation unit that includes it: the one read
// here must be the one the kernels launched from here write.
int mxb_debug_tile_trace(unsigned long long *out, size_t n_words) {
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

}  // extern "C"
