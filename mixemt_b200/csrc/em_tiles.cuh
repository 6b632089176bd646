// Class tiles: the EM pass over column classes instead of columns (host side: em_tiles.cu).
//
// A fragment covers ~78 of the 4070 variant positions, so over a batch of neighbouring
// signature rows (the rows arrive string-sorted, preprocess.py:219: neighbours start at the
// same or a nearby position) most of the 5408 haplotypes are indistinguishable: the columns of
// a 128-row batch of the config-2 matrix fall into a median of ~150 classes of bit-identical
// columns (mean ~250; ~2000 in the hypervariable regions).  With cmap_b[j] the class of column
// j in batch b and V_b[i][c] = L_i,rep(c) the value of class c in row i, an EM iteration
// (em.py:80-89 in the linear form of em.cu)
//
//     s_i = sum_j L_ij pi_j           T_j = sum_i (w_i / s_i) L_ij
//
// is evaluated exactly as
//
//     Pi_b[c] = sum_{j in class c} pi_j        (tile_pi_kernel, H adds per batch)
//     s_i     = sum_c V_b[i][c] Pi_b[c]        (tile_pass_kernel, C_b instead of H terms per row)
//     U_b[c]  = sum_{i in b} (w_i / s_i) V_b[i][c]
//     T_j     = sum_b U_b[cmap_b[j]]           (tile_gather_kernel, H adds per batch)
//
// Every sum adds non-negative terms, so regrouping them costs rounding in the last bits only
// (no cancellation); the trajectory equals that of the fp64-row pass to ~1e-13 with identical
// iteration counts (tests/test_em_gpu.py).  The pass reads N x C_b instead of N x H cells:
// 0.3 GB instead of 6.0 GB per iteration at config 2.  All orders of summation are fixed:
// results are run-to-run deterministic and identical on every rank.
//
// Classes are found from the matrix alone (the drop-in run_em sees no positions): a 64-bit
// hash of every column over the batch's rows (tile_hash_kernel), a block radix sort of
// (hash, column) per batch (tile_class_kernel; stable, so a class is a run of equal hashes
// with ascending columns), and an exact bitwise check of every cell against its class
// representative while the tiles are written (tile_fill_kernel); a batch that fails the check
// (a hash collision) sends the session back to the fp64 rows.
#pragma once

#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include "block_reduce.cuh"
#include "em_common.cuh"
#include "row_likelihood.cuh"
#include "tile_plan.h"

namespace mxb {

constexpr int kTileThreads = 512;
constexpr int kTileWarps = kTileThreads / 32;
constexpr int kTileMaxNK = 8;        // double2 per thread and row
constexpr int kTileMaxCols = 8192;   // widest matrix (the fast path's limit on ld)

__device__ __forceinline__ uint64_t tile_mix(uint64_t h, uint64_t v) {
    h = (h ^ v) * 0xFF51AFD7ED558CCDull;
    h ^= h >> 29;
    h *= 0xC4CEB9FE1A85EC53ull;
    return h ^ (h >> 32);
}

// hash[b][j] over the rows of batch b, column j of M (row stride n_cols).
__global__ void __launch_bounds__(kTileThreads)
tile_hash_kernel(const double *__restrict__ m, int64_t n_rows, int64_t n_cols, int n_batches,
                 unsigned long long *__restrict__ hash, int hs) {
    for (int b = blockIdx.x; b < n_batches; b += gridDim.x) {
        const int64_t r0 = (int64_t)b * kTileRows;
        const int nr = (int)min((int64_t)kTileRows, n_rows - r0);
        const double *base = m + r0 * n_cols;
        for (int64_t j = threadIdx.x; j < n_cols; j += kTileThreads) {
            uint64_t h = 0x243F6A8885A308D3ull;
            const double *p = base + j;
            int r = 0;
            for (; r + 4 <= nr; r += 4) {
                const double v0 = p[(int64_t)r * n_cols], v1 = p[(int64_t)(r + 1) * n_cols];
                const double v2 = p[(int64_t)(r + 2) * n_cols], v3 = p[(int64_t)(r + 3) * n_cols];
                h = tile_mix(h, (uint64_t)__double_as_longlong(v0));
                h = tile_mix(h, (uint64_t)__double_as_longlong(v1));
                h = tile_mix(h, (uint64_t)__double_as_longlong(v2));
                h = tile_mix(h, (uint64_t)__double_as_longlong(v3));
            }
            for (; r < nr; ++r) h = tile_mix(h, (uint64_t)__double_as_longlong(p[(int64_t)r * n_cols]));
            if (h == ~0ull) h = ~0ull - 1;   // ~0 pads the sort
            hash[(size_t)b * hs + j] = h;
        }
    }
}

// Classes of one batch: sort (hash, column), number the runs of equal hashes.
//   perm[b][e]  column at sorted position e (classes are contiguous, columns ascending inside)
//   cword[b][t] run structure of entries [ITEMS t, ITEMS (t + 1)) for the class-sum kernel
//   cmap[b][j]  class of column j
//   rep[b][c]   first (smallest) column of class c
template <int ITEMS>
__global__ void __launch_bounds__(kTileThreads)
tile_class_kernel(const unsigned long long *__restrict__ hash, int hs, int n_cols, int n_batches,
                  unsigned short *__restrict__ perm, unsigned int *__restrict__ cword,
                  unsigned short *__restrict__ cmap, unsigned short *__restrict__ rep,
                  int *__restrict__ n_cls) {
    using Sort = cub::BlockRadixSort<unsigned long long, kTileThreads, ITEMS, unsigned short>;
    using Scan = cub::BlockScan<int, kTileThreads>;
    extern __shared__ __align__(128) unsigned char tile_smem[];
    typename Sort::TempStorage &sort_tmp = *reinterpret_cast<typename Sort::TempStorage *>(tile_smem);
    typename Scan::TempStorage &scan_tmp = *reinterpret_cast<typename Scan::TempStorage *>(tile_smem);
    __shared__ unsigned long long last_key[kTileThreads];
    __shared__ int first_start[kTileThreads + 1];
    const int tid = threadIdx.x;
    for (int b = blockIdx.x; b < n_batches; b += gridDim.x) {
        unsigned long long keys[ITEMS];
        unsigned short vals[ITEMS];
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            const int j = tid * ITEMS + i;
            keys[i] = j < n_cols ? hash[(size_t)b * hs + j] : ~0ull;
            vals[i] = (unsigned short)j;
        }
        Sort(sort_tmp).Sort(keys, vals);
        __syncthreads();
        last_key[tid] = keys[ITEMS - 1];
        __syncthreads();
        int heads = 0;
        bool head[ITEMS];
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            const int e = tid * ITEMS + i;
            const unsigned long long prev = i ? keys[i - 1] : (tid ? last_key[tid - 1] : ~keys[0]);
            head[i] = e < n_cols && keys[i] != prev;   // padding (~0) sorts behind every column
            heads += head[i] ? 1 : 0;
        }
        int before = 0, total = 0;
        Scan(scan_tmp).ExclusiveSum(heads, before, total);
        int cls = before - 1;
        unsigned int starts = 0;             // bit i: a class begins at entry i of this chunk
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            const int e = tid * ITEMS + i;
            if (e < n_cols) {
                if (head[i]) {
                    ++cls;
                    rep[(size_t)b * hs + cls] = vals[i];
                    starts |= 1u << i;
                }
                perm[(size_t)b * hs + e] = vals[i];
                cmap[(size_t)b * hs + vals[i]] = (unsigned short)cls;
            } else {
                starts |= 1u << i;           // past the last column: every run has ended
            }
        }
        // chunk word of the class-sum kernel: bits 0..ITEMS = run starts (bit ITEMS: at the first
        // entry of the next chunk), bits 17.. = class of the chunk's first entry
        first_start[tid] = (int)(starts & 1u);
        if (tid == 0) first_start[kTileThreads] = 1;
        __syncthreads();
        starts |= (unsigned int)first_start[tid + 1] << ITEMS;
        const int first_cls = head[0] ? before : before - 1;
        cword[(size_t)b * kTileThreads + tid] = starts | ((unsigned int)max(first_cls, 0) << 17);
        if (tid == 0) n_cls[b] = total;
        __syncthreads();   // temp storage and last_key are reused by the next batch
    }
}

// Tiles V_b[r][c] = exp(M[row0 + r][rep_b[c]] - rowmax) (the value to_linear_kernel gives
// every member of the class), then the row's weight, zero padded to r_pad, with the exact check that makes the
// hashing safe: every cell of M must equal the cell of its class representative bit for bit.
// One warp per row.
__global__ void __launch_bounds__(kTileThreads)
tile_fill_kernel(const double *__restrict__ m, int64_t n_cols, const TileDesc *__restrict__ desc,
                 int n_batches, const unsigned short *__restrict__ cmap,
                 const unsigned short *__restrict__ rep, int hs,
                 const double *__restrict__ weights, double *__restrict__ v,
                 int *__restrict__ bad) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = blockIdx.x; b < n_batches; b += gridDim.x) {
        const TileDesc d = desc[b];
        const unsigned short *cm = cmap + (size_t)b * hs;
        const unsigned short *rp = rep + (size_t)b * hs;
        int mismatch = 0;
        for (int r = warp; r < d.n_rows; r += kTileWarps) {
            const double *row = m + (int64_t)(d.row0 + r) * n_cols;
            double mx = -INFINITY;
            for (int c = lane; c < d.n_cls; c += 32) mx = fmax(mx, row[rp[c]]);
            mx = warp_max(mx);
            for (int64_t j = lane; j < n_cols; j += 32)
                mismatch |= __double_as_longlong(row[j]) != __double_as_longlong(row[rp[cm[j]]]);
            double *dst = v + d.v_off + (int64_t)r * d.r_pad;
            const double w_row = weights[d.row0 + r];
            for (int c = lane; c < d.r_pad; c += 32)
                dst[c] = c < d.n_cls ? exp(row[rp[c]] - mx) : c == d.n_cls ? w_row : 0.0;
        }
        if (__any_sync(0xffffffffu, mismatch) && lane == 0) bad[b] = 1;
    }
}

// Pi_b[c] = sum of pi_j over the members of class c.  `perm` lists the columns of a batch class
// by class (ckey = class of every entry, non-decreasing), so a class is a run of entries and
// the sums are a segmented reduction: every thread adds the entries of its chunk run by run
// in order (branch-free: the run structure is data, not control flow), stores the runs that
// begin and end inside the chunk, and the runs that cross chunk borders are completed by a
// segmented scan over the threads (shuffles in the warp, one more shuffle scan over the 16
// warp totals).  Fixed order of additions: deterministic.
constexpr int kPiPer = 16;       // entries per thread, at most (512 x 16 = 8192 columns)

struct SegItem {
    int flag;      // 1: a new class starts at (or inside) this item
    double val;    // sum of the trailing run
};
__device__ __forceinline__ SegItem seg_combine(const SegItem &a, const SegItem &b) {
    SegItem r;
    r.flag = a.flag | b.flag;
    r.val = b.flag ? b.val : a.val + b.val;
    return r;
}
__device__ __forceinline__ SegItem seg_shfl_up(const SegItem &v, int off) {
    SegItem o;
    o.flag = __shfl_up_sync(0xffffffffu, v.flag, off);
    o.val = __shfl_up_sync(0xffffffffu, v.val, off);
    return o;
}

// kSlots (slotted sessions, em.cu: run_tasks): blockIdx.y is a replicate slot; its
// proportions, control block and class sums lie pi_stride, one EmState and cls_stride further.
template <int PER, bool kSlots = false>
__global__ void __launch_bounds__(kTileThreads)
tile_pi_kernel(const unsigned short *__restrict__ perm, const unsigned int *__restrict__ cword,
               int hs, int n_cols, const TileDesc *__restrict__ desc, int n_batches,
               const double *__restrict__ pi0, const double *__restrict__ pi1,
               const EmState *__restrict__ st, double *__restrict__ pi_cls,
               int64_t pi_stride, int64_t cls_stride) {
    static_assert(PER % 4 == 0 && PER <= 16, "chunks are read as 8-byte words");
    extern __shared__ __align__(128) unsigned char tile_smem[];
    double *pi = reinterpret_cast<double *>(tile_smem);     // [n_cols]: the gathers below are
    // random 8-byte reads, cheaper from shared memory than through L1 tags
    pdl_wait();
    pdl_launch_dependents();
    if (kSlots) {
        st += blockIdx.y;
        pi0 += blockIdx.y * pi_stride;
        pi1 += blockIdx.y * pi_stride;
        pi_cls += blockIdx.y * cls_stride;
    }
    if (st->done) return;
    const double *__restrict__ pi_g = st->cur ? pi1 : pi0;
    __shared__ int s_flag[kTileWarps];
    __shared__ double s_val[kTileWarps];
    __shared__ double s_carry[kTileWarps];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int j = tid; j < n_cols; j += kTileThreads) pi[j] = pi_g[j];
    __syncthreads();
    const int e0 = min(n_cols, tid * PER), cnt = min(n_cols, e0 + PER) - e0;
    const bool live = cnt > 0;
    for (int b = blockIdx.x; b < n_batches; b += gridDim.x) {
        double *out = pi_cls + desc[b].p_off;
        // the chunk's columns (PER 16-bit entries as 8-byte words) and its run structure
        const uint2 *pm = reinterpret_cast<const uint2 *>(perm + (size_t)b * hs + (size_t)tid * PER);
        uint2 words[PER / 4];
#pragma unroll
        for (int i = 0; i < PER / 4; ++i) words[i] = live ? pm[i] : make_uint2(0u, 0u);
        const unsigned int cw = cword[(size_t)b * kTileThreads + tid];
        const unsigned int starts = cw & 0x1FFFFu;
        int cls = (int)(cw >> 17);                  // class of the current run
        const int f_head = live ? (int)(starts & 1u) : 1;
        double s = 0.0, head_sum = 0.0;
        int head_open = 1;                           // the chunk's first run has not ended yet
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const unsigned int w = (q & 2) ? words[q >> 2].y : words[q >> 2].x;
            const int col = q < cnt ? (int)((q & 1) ? (w >> 16) : (w & 0xFFFFu)) : 0;
            const double v = pi[col];
            const bool start = q > 0 && ((starts >> q) & 1u);
            const bool ends = (starts >> (q + 1)) & 1u;
            if (q < cnt) {
                cls += start ? 1 : 0;
                s = (q == 0 || start) ? v : s + v;
                if (start) head_open = 0;
                // a run that ends here and did not come in from the previous thread is final
                if (ends && (!head_open || f_head)) out[cls] = s;
                if (head_open && ends) head_sum = s;
                if (ends) head_open = 0;
            }
        }
        const int started = (starts & ((1u << PER) - 1u)) != 0;     // a run began in this chunk
        const int head_cls = (int)(cw >> 17);
        if (live && head_open) head_sum = s;          // one run fills the chunk and goes on
        // aggregate of the chunk: trailing-run sum, and whether a run began here
        SegItem agg;
        agg.flag = live ? started : 1;
        agg.val = live ? s : 0.0;
        SegItem inc = agg;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const SegItem o = seg_shfl_up(inc, off);
            if (lane >= off) inc = seg_combine(o, inc);
        }
        __syncthreads();                       // the scratch of the previous batch has been read
        if (lane == 31) { s_flag[warp] = inc.flag; s_val[warp] = inc.val; }
        __syncthreads();
        if (warp == 0) {
            SegItem wv;
            wv.flag = lane < kTileWarps ? s_flag[lane] : 1;
            wv.val = lane < kTileWarps ? s_val[lane] : 0.0;
#pragma unroll
            for (int off = 1; off < kTileWarps; off <<= 1) {
                const SegItem o = seg_shfl_up(wv, off);
                if (lane >= off) wv = seg_combine(o, wv);
            }
            // exclusive: what is open at the end of the warps before this one
            const SegItem ex = seg_shfl_up(wv, 1);
            if (lane < kTileWarps) s_carry[lane] = lane == 0 ? 0.0 : ex.val;
        }
        __syncthreads();
        SegItem exc = seg_shfl_up(inc, 1);      // open run at the end of the previous thread
        if (lane == 0) { exc.flag = 0; exc.val = s_carry[warp]; }
        else if (!exc.flag) exc.val += s_carry[warp];
        if (live && !f_head) {
            // the first run came in from the previous thread(s): it is final here if it ended
            // inside the chunk or at its very end
            const bool ended = (starts >> 1) != 0;          // some later start bit, incl. bit PER
            if (ended) out[head_cls] = exc.val + head_sum;
        }
    }
}

// ---- the pass ------------------------------------------------------------------------------
// Every CTA owns one contiguous range of rows (ranges of equal cost, fixed when the tiles are
// built: em_tiles.cu) and streams it through a CTA-wide shared-memory ring of 1-D bulk async copies
// (cp.async.bulk + mbarrier complete_tx) of whole rows, up to a slot per copy, in row order;
// the warp that is the last to finish with a slot issues the copy that takes it next from a
// cursor every warp keeps.  The 16 warps work on the rows of one batch (segment) at a time.
// A row is handled by L = 2^lg threads (8 or 16 lanes for rows of at most 64 / 128 double2
// chunks -- four or two rows per warp step --, a warp, or 2..16 warps for more than 512
// classes); thread t owns the chunks (t mod L) + L k (k < 8) of the rows (t div L) + (512 / L) i
// of the batch, so Pi_b and its share of U_b stay in registers for the whole batch.  A row step
// costs 8 16-byte shared loads, 32 DFMA, a shuffle butterfly of lg levels (plus one named
// barrier across the warps of a wide row) and one division; the weight of a row travels with
// the row (column n_cls of the tile).  At the end of a batch the consumers add their shares in
// fixed order through shared memory and store U_b; the class sums of the next batch are already
// on their way into the registers.  No global atomics, fences or queues: the only global
// traffic of the pass is the tile stream (contiguous per CTA), Pi_b in and U_b out.
// A batch that straddles two CTAs' ranges is two segments with a U vector each; the gather
// kernel adds them like two batches.
constexpr int kTileConsumers = kTileWarps;
constexpr int kTilePassThreads = kTileThreads;
constexpr int kTileScratchBytes = 64 * 1024;                     // [row slices][class vector]
constexpr int kTileSlotBarrier0 = 10;
constexpr size_t kTilePassSmem = kTileRingBytes + kTileScratchBytes +
                                 2 * kTileMaxSlots * sizeof(uint64_t) +
                                 2 * kTileWarps * sizeof(double) + 128;
// the slotted pass (bootstrap) also stages the weights of two segments: [2][kTileRows] doubles
// behind `red`
constexpr size_t kTileWeightsOff = kTileRingBytes + kTileScratchBytes +
                                   2 * kTileMaxSlots * sizeof(uint64_t) +
                                   2 * kTileWarps * sizeof(double);
constexpr size_t kTilePassSlotSmem = kTilePassSmem + 2 * kTileRows * sizeof(double);

struct TileCursor {        // the copy that takes a freed slot: n_slots copies ahead of the warps
    int64_t v_off;
    int32_t r_pad, n_rows, fit, n_copies;
};
__device__ __forceinline__ TileCursor tile_cursor(const TileSeg *sg) {
    TileCursor c;
    c.v_off = sg->v_off;
    c.r_pad = sg->r_pad;
    c.n_rows = sg->n_rows;
    c.fit = sg->fit;
    c.n_copies = sg->n_copies;
    return c;
}

__device__ __forceinline__ void named_barrier(int id, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
#ifdef MXB_TILE_TRACE
// development aid (never in the product build): per CTA and warp: cycles blocked on the ring,
// in row steps, in the end-of-batch exchange; total
__device__ long long g_tile_trace[160 * kTileWarps * 8];
#endif

// kSlots: blockIdx.y is a bootstrap replicate slot (see tile_pi_kernel); the weight of a row is
// the slot's (n_rows doubles per slot) instead of column n_cls of the tile.  The weights of a
// segment are staged in shared memory (two buffers, segment si in buffer si & 1): the next
// segment's are stored before the barrier of the end-of-batch exchange, after which nobody reads
// the buffer they replace.
template <bool kSlots = false>
__global__ void __launch_bounds__(kTilePassThreads, 1)
tile_pass_kernel(const TileCta *__restrict__ ctas, const TileSeg *__restrict__ segs,
                 const double *__restrict__ v,
                 const double *__restrict__ pi_cls, EmState *__restrict__ st,
                 double *__restrict__ u_sum, uint32_t slot_bytes, int n_slots,
                 const double *__restrict__ slot_w, int64_t n_rows, int64_t cls_stride,
                 int64_t u_stride) {
    extern __shared__ __align__(128) unsigned char tile_smem[];
    double *scratch = reinterpret_cast<double *>(tile_smem + kTileRingBytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(tile_smem + kTileRingBytes + kTileScratchBytes);
    int *freed = reinterpret_cast<int *>(full + kTileMaxSlots);   // warps done with a slot ([16], padded)
    double *red = reinterpret_cast<double *>(full + 2 * kTileMaxSlots);  // [2][16]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int q = 0; q < n_slots; ++q) {
            mbar_init(full + q, 1);
            freed[q] = 0;
        }
        mbar_init_fence();
    }
    __syncthreads();
    pdl_wait();               // the class sums of this iteration are complete
    pdl_launch_dependents();
    // slot offsets are formed where a pointer is used, from the kernel parameters: registers are
    // short, and the parameters can be read again at no register cost
#define MXB_SLOT(stride) (kSlots ? (int64_t)blockIdx.y * (stride) : (int64_t)0)
    if (st[MXB_SLOT(1)].done) return;
    const TileCta cta = ctas[blockIdx.x];
    double *w_stage = reinterpret_cast<double *>(tile_smem + kTileWeightsOff);
    if (kSlots) {
        const TileSeg *s0 = segs + cta.seg0;
        if (tid < s0->n_rows) w_stage[tid] = slot_w[MXB_SLOT(n_rows) + s0->row0 + tid];
        __syncthreads();
    }
    const uint32_t ring_u32 = smem_u32(tile_smem);
    const uint32_t full_u32 = smem_u32(full);
    const TileSeg *my_segs = segs + cta.seg0;
    // The copy cursor (kept by every warp: any of them may be the one that fills a slot): primed
    // n_slots copies ahead by thread 0, then moved one copy per copy consumed.
    int ps = 0, pc = 0;
    TileCursor cur_p = tile_cursor(my_segs), next_p = cur_p;
    if (cta.n_segs > 1) next_p = tile_cursor(my_segs + 1);
    auto cursor_issue = [&](int q) {       // copy (ps, pc) -> slot q
        const int row0 = pc * cur_p.fit;
        const uint32_t bytes = (uint32_t)(min(cur_p.fit, cur_p.n_rows - row0) * cur_p.r_pad) * 8u;
        mbar_expect_tx_u32(full_u32 + 8u * q, bytes);
        bulk_load_u32(ring_u32 + (uint32_t)q * slot_bytes, v + cur_p.v_off + (size_t)row0 * cur_p.r_pad,
                      bytes, full_u32 + 8u * q);
    };
    auto cursor_advance = [&]() {
        if (++pc == cur_p.n_copies) {
            pc = 0;
            ++ps;
            cur_p = next_p;
            if (ps + 1 < cta.n_segs) next_p = tile_cursor(my_segs + ps + 1);
        }
    };
    for (int q = 0; q < n_slots && q < cta.n_copies; ++q) {
        if (tid == 0) cursor_issue(q);
        cursor_advance();
    }

#ifdef MXB_TILE_TRACE
    long long t_wait = 0, t_step = 0, t_red = 0, t_fill = 0;
    const long long t_begin = clock64();
#endif
    constexpr int K = 8;
    int j = 0, slot = 0, bad = 0, parity = 0;
    bool prev_small = true;
    uint32_t phase = 0;
    double2 p[K], u[K];
    TileSeg sg = segs[cta.seg0];
    int L = 1 << sg.lg, idx = tid & (L - 1);
    int kl = min(K, max(0, (((sg.n_cls + 1) >> 1) - idx + L - 1) >> sg.lg));
    {
        const double2 *pcls = reinterpret_cast<const double2 *>(pi_cls + MXB_SLOT(cls_stride) + sg.p_off) + idx;
#pragma unroll
        for (int k = 0; k < K; ++k) p[k] = k < kl ? pcls[k << sg.lg] : make_double2(0.0, 0.0);
    }
    for (int si = 0; si < cta.n_segs; ++si) {
        // the record of the next segment is on its way while this one is worked on
        TileSeg sg_next = sg;
        if (si + 1 < cta.n_segs) sg_next = my_segs[si + 1];
#pragma unroll
        for (int k = 0; k < K; ++k) u[k] = make_double2(0.0, 0.0);
        const int lg = sg.lg;
        const int tw = lg > 5 ? 1 << (lg - 5) : 1;                 // warps per row
        const int rows_per_sweep = (32 * kTileConsumers) >> lg;
        const uint32_t row_bytes = (uint32_t)sg.r_pad * 8u;
        const uint32_t chunk0 = (uint32_t)min(idx, ((sg.n_cls + 1) >> 1) - 1) * 16u;   // see the loads below
        const uint32_t chunk_stride = 16u << lg;
        const int k_last = max(kl, 1) - 1;
        int row = tid >> lg;                                       // this thread's next row
        const int warp_row = (lg >= 5 ? tid >> lg : (warp << (5 - lg)));   // first row of the warp's step
        const int warp0 = warp & ~(tw - 1);
        // (the warps of a row agree on the buffer of their partial dot products: the teams of
        // the previous batch may have taken different numbers of steps; every thread has passed
        // the barrier of the exchange since its last read of `red`)
        parity = 0;
        for (int c = 0; c < sg.n_copies; ++c, ++j) {
            const int copy_row0 = c * sg.fit;
            const int row_end = min(copy_row0 + sg.fit, sg.n_rows);
            // rows of this warp (or team of warps) inside the copy: warp-uniform test
            int wrow = warp_row + (row - (tid >> lg));
            // (every warp waits for every copy, also for one that holds none of its rows: its
            // count below must not land in the slot's previous round)
#ifdef MXB_TILE_TRACE
            const long long tw0 = clock64();
#endif
            mbar_wait_u32(full_u32 + 8u * slot, phase);
#ifdef MXB_TILE_TRACE
            const long long tw1 = clock64();
            t_wait += tw1 - tw0;
#endif
            if (wrow < row_end) {
                do {
                    const bool have = row < row_end;
                    // Branch-free loads: a chunk this thread does not own (k >= kl) or a row past
                    // the end of the batch reads a cell that exists (finite) instead; its class
                    // sum p[k] is zero and the weight of a missing row is zero, so neither
                    // reaches a result.
                    const uint32_t src = ring_u32 + (uint32_t)slot * slot_bytes +
                                         (uint32_t)((have ? row : wrow) - copy_row0) * row_bytes;
                    double2 x[K];
                    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        x[k] = lds_v2_f64(src + chunk0 + (uint32_t)min(k, k_last) * chunk_stride);
                    double wr;
                    if (kSlots) {
                        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(wr)
                                     : "r"(ring_u32 + (uint32_t)kTileWeightsOff +
                                           (uint32_t)(((si & 1) * kTileRows + (have ? row : 0)) * 8))
                                     : "memory");
                        if (!have) wr = 0.0;
                    } else {
                        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(wr) : "r"(src + (uint32_t)sg.n_cls * 8u) : "memory");
                        if (!have) wr = 0.0;
                    }
#pragma unroll
                    for (int k = 0; k < K; k += 2) {
                        d0 = fma(x[k].x, p[k].x, d0);
                        d1 = fma(x[k].y, p[k].y, d1);
                        d2 = fma(x[k + 1].x, p[k + 1].x, d2);
                        d3 = fma(x[k + 1].y, p[k + 1].y, d3);
                    }
                    double dot = (d0 + d1) + (d2 + d3);
                    if (lg >= 5) {
                        dot = warp_sum(dot);
                        if (tw > 1) {
                            // warp totals -> red[parity][warp]; after the barrier of the row's
                            // warps every thread adds them in warp order
                            if (lane == 0) red[parity * kTileWarps + warp] = dot;
                            named_barrier(1 + (warp0 >> 1), 32 * tw);
                            double t = lane < tw ? red[parity * kTileWarps + warp0 + lane] : 0.0;
                            for (int o = tw >> 1; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
                            dot = __shfl_sync(0xffffffffu, t, 0);
                            parity ^= 1;
                        }
                    } else if (lg == 4) {
#pragma unroll
                        for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
                    } else {
#pragma unroll
                        for (int o = 4; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
                    }
                    double coef = 0.0;
                    if (wr != 0.0) {
                        coef = wr / dot;
                        bad |= row_needs_logspace(dot);
                    }
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        u[k].x = fma(coef, x[k].x, u[k].x);
                        u[k].y = fma(coef, x[k].y, u[k].y);
                    }
                    row += rows_per_sweep;
                    wrow += rows_per_sweep;
                } while (wrow < row_end);
            }
#ifdef MXB_TILE_TRACE
            const long long tw2 = clock64();
            t_step += tw2 - tw1;
#endif
            // done with the slot (every lane's reads of it have been consumed by now): the warp
            // that is the last one to say so fills it again
            // A counter tells which warp is the last one (nobody waits to find out); a named
            // barrier per slot, on which the others only arrive, orders every warp's reads
            // before the copy that overwrites them.
            __syncwarp();
            int last = 0;
            if (lane == 0) {
                __threadfence_block();
                last = atomicAdd(freed + slot, 1) == kTileConsumers - 1;
            }
            last = __shfl_sync(0xffffffffu, last, 0);
            if (last) {
                named_barrier(kTileSlotBarrier0 + slot, 32 * kTileConsumers);
                if (lane == 0) {
                    freed[slot] = 0;
                    __threadfence_block();
                    if (j + n_slots < cta.n_copies) cursor_issue(slot);
                }
            } else {
                asm volatile("bar.arrive %0, %1;" ::"r"(kTileSlotBarrier0 + slot), "r"(32 * kTileConsumers) : "memory");
            }
            if (j + n_slots < cta.n_copies) cursor_advance();
#ifdef MXB_TILE_TRACE
            t_fill += clock64() - tw2;
#endif
            if (++slot == n_slots) { slot = 0; phase ^= 1u; }
        }
#ifdef MXB_TILE_TRACE
        const long long tr0 = clock64();
#endif
        // ---- end of the batch (segment): add the consumers' shares in fixed order ----
        const int chunks = (sg.n_cls + 1) >> 1;     // double2 chunks that hold class values
        const int slice = lg >= 5 ? tid >> lg : warp;              // of the scratch: [slices][chunks]
        const int n_slices = lg >= 5 ? (32 * kTileConsumers) >> lg : kTileConsumers;
        // the class sums of the next batch start their way into the registers now
        const int kl_cur = kl;
        const int idx_cur = idx;
        L = 1 << sg_next.lg;
        idx = tid & (L - 1);
        kl = min(K, max(0, (((sg_next.n_cls + 1) >> 1) - idx + L - 1) >> sg_next.lg));
        if (si + 1 < cta.n_segs) {
            const double2 *pcls = reinterpret_cast<const double2 *>(pi_cls + MXB_SLOT(cls_stride) + sg_next.p_off) + idx;
#pragma unroll
            for (int k = 0; k < K; ++k) p[k] = k < kl ? pcls[k << sg_next.lg] : make_double2(0.0, 0.0);
        }
        if (lg < 5) {
            // the groups of a warp first (pairwise, fixed)
#pragma unroll
            for (int k = 0; k < K; ++k) {
                for (int o = 1 << lg; o < 32; o <<= 1) {
                    u[k].x += __shfl_xor_sync(0xffffffffu, u[k].x, o);
                    u[k].y += __shfl_xor_sync(0xffffffffu, u[k].y, o);
                }
            }
        }
        // Shares that fit into half of the scratch alternate between its halves: the barrier
        // below then also says that the half written two batches ago has been read.  Otherwise
        // one more barrier: the scratch of the previous batch has been read.
        const bool small = n_slices * chunks * (int)sizeof(double2) <= kTileScratchBytes / 2;
        if (!(small && prev_small)) named_barrier(9, 32 * kTileConsumers);
        prev_small = small;
        double2 *sc_base = reinterpret_cast<double2 *>(scratch) +
                           (small && (si & 1) ? kTileScratchBytes / 2 / sizeof(double2) : 0);
        if (lg >= 5 || lane < (1 << lg)) {
            double2 *dst = sc_base + (size_t)slice * chunks + idx_cur;
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (k < kl_cur) dst[k << lg] = u[k];
        }
        if (kSlots && si + 1 < cta.n_segs && tid < sg_next.n_rows)
            w_stage[((si + 1) & 1) * kTileRows + tid] = slot_w[MXB_SLOT(n_rows) + sg_next.row0 + tid];
        named_barrier(9, 32 * kTileConsumers);
        {
            const double2 *sc = sc_base;
            double2 *out = reinterpret_cast<double2 *>(u_sum + MXB_SLOT(u_stride) + sg.u_dst);
            for (int c = tid; c < chunks; c += 32 * kTileConsumers) {
                double2 acc = sc[c];
                for (int t = 1; t < n_slices; ++t) {
                    const double2 o = sc[(size_t)t * chunks + c];
                    acc.x += o.x;
                    acc.y += o.y;
                }
                out[c] = acc;
            }
        }
        sg = sg_next;
#ifdef MXB_TILE_TRACE
        t_red += clock64() - tr0;
#endif
    }
#ifdef MXB_TILE_TRACE
    if (lane == 0) {
        long long *tr = g_tile_trace + ((size_t)blockIdx.x * kTileWarps + warp) * 8;
        tr[0] = clock64() - t_begin; tr[1] = t_wait; tr[2] = t_step; tr[3] = t_fill; tr[4] = t_red;
        tr[5] = cta.n_segs; tr[6] = cta.n_copies; tr[7] = 1;
    }
#endif
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicAdd(&st[MXB_SLOT(1)].bad, 1);
#undef MXB_SLOT
}

// T_j = sum over batches of U_b[cmap_b[j]], batches in ascending order; the batches are split
// into gridDim.y contiguous ranges whose partial sums the tail kernel adds in range order (its
// `partials` input).  One thread per column, eight batches in flight per thread.
constexpr int kGatherThreads = 256;
constexpr int kGatherUnroll = 8;

// kSlots: blockIdx.z is a bootstrap replicate slot (U vectors u_stride apart, partials of
// gridDim.y ranges per slot).
template <bool kSlots = false>
__global__ void __launch_bounds__(kGatherThreads)
tile_gather_kernel(const unsigned short *__restrict__ cmap, int hs, int n_cols, int64_t ld,
                   const int *__restrict__ ent_batch, const int64_t *__restrict__ ent_off,
                   int n_ent, const double *__restrict__ u_sum, const EmState *__restrict__ st,
                   double *__restrict__ partials, int64_t u_stride) {
    pdl_wait();
    pdl_launch_dependents();
    if (kSlots) {
        st += blockIdx.z;
        u_sum += blockIdx.z * u_stride;
        partials += (size_t)blockIdx.z * gridDim.y * ld;
    }
    if (st->done) return;
    const int j = blockIdx.x * kGatherThreads + threadIdx.x;
    if (j >= ld) return;
    const int part = blockIdx.y, n_part = gridDim.y;
    const int e0 = (int)((int64_t)n_ent * part / n_part);
    const int e1 = (int)((int64_t)n_ent * (part + 1) / n_part);
    double t = 0.0;
    if (j < n_cols) {
        int e = e0;
        for (; e + kGatherUnroll <= e1; e += kGatherUnroll) {
            double x[kGatherUnroll];
#pragma unroll
            for (int q = 0; q < kGatherUnroll; ++q)
                x[q] = u_sum[ent_off[e + q] + cmap[(size_t)ent_batch[e + q] * hs + j]];
#pragma unroll
            for (int q = 0; q < kGatherUnroll; ++q) t += x[q];
        }
        for (; e < e1; ++e) t += u_sum[ent_off[e] + cmap[(size_t)ent_batch[e] * hs + j]];
    }
    partials[(size_t)part * ld + j] = t;
}

}  // namespace mxb
