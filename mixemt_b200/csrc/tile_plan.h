// Host side of the class tiles (em_tiles.cuh): layout of the batches and plan of the pass.
// Plain C++ over the records the kernels read; em.cu calls it from em_pack_tiles, and
// mxb_tile_plan (include/mixemt_b200.h) exposes it to the CPU tests.
#pragma once

#include <algorithm>
#include <cstring>
#include <vector>

#include "em_tiles.cuh"

namespace mxb {

struct TilePlanOut {
    std::vector<TileCta> ctas;
    std::vector<TileSeg> segs;
    std::vector<int> ent_batch;           // gather entries: (batch, offset of a U vector)
    std::vector<int64_t> ent_off;
    int64_t extra_cells = 0;              // U vectors of the second, third.. segment of a batch
    int n_copy = 0;
    double time = 0.0;                    // modelled time of the pass: its slowest CTA (cycles)
};

// Layout: threads per row, tile and class-vector offsets of every batch.
inline void tile_layout(const int *ncls, int nb, int64_t n, std::vector<TileDesc> &desc,
                        int64_t &v_cells, int64_t &p_cells, int &max_r_pad) {
    desc.assign((size_t)nb, TileDesc());
    v_cells = 0;
    p_cells = 0;
    max_r_pad = 4;
    for (int b = 0; b < nb; ++b) {
        TileDesc &d = desc[(size_t)b];
        d.row0 = b * kTileRows;
        d.n_rows = (int)std::min<int64_t>(kTileRows, n - (int64_t)b * kTileRows);
        d.n_cls = ncls[b];
        d.r_pad = (int)round_up(d.n_cls + 1, 4);      // + the weight column
        // a row is handled by 2^lg threads, each with at most 8 double2 chunks of its class
        // values (the weight behind them is read apart): up to 8192 classes with 16 warps
        d.lg = 3;
        while (((d.n_cls + 1) >> 1) > (8 << d.lg)) ++d.lg;
        d.pad0 = d.pad1 = d.pad2 = 0;
        d.v_off = v_cells;
        d.p_off = p_cells;
        v_cells += (int64_t)d.n_rows * d.r_pad;
        p_cells += d.r_pad;
        max_r_pad = std::max(max_r_pad, d.r_pad);
    }
}

// The ring of the pass: three slots of 52 KB, fewer and longer ones if a row is longer than
// that (a copy costs every warp ~650 cycles: large copies, measured 24 to 78 KB).  False when
// not even two rows of the longest kind fit.
inline bool tile_ring(int max_r_pad, uint32_t &slot_bytes, int &n_slots) {
    slot_bytes = (uint32_t)round_up(std::max<int64_t>(kTileSlotBytes, (int64_t)max_r_pad * 8), 1024);
    n_slots = std::min(kTileMaxSlots, kTileRingBytes / (int)slot_bytes);
    return n_slots >= 2;
}

// Plan of the pass.  The rows are dealt to the CTAs in order, every CTA one contiguous range;
// the part of a batch inside a CTA's range is a segment, cut at copy boundaries.  A CTA takes
// rows until either of its two clocks reaches the target T: its bytes at the SM's share of
// HBM (22 B per cycle) or its warps' time (cycle counters of the kernel at config 2: ~4200
// cycles per segment for the exchange at its end and the wait for the next class sums, ~500
// per copy for waiting, handing back and refilling, and a row step of 440 .. 1900 cycles for
// every 512 >> lg rows of a copy); the smallest T that needs no more CTAs than there are SMs
// is found by bisection.
inline void tile_plan(const std::vector<TileDesc> &desc, int64_t n, int num_sms,
                      uint32_t slot_bytes, int64_t p_cells, TilePlanOut &out) {
    const int nb = (int)desc.size();
    static const double step_cycles[10] = {440, 440, 440, 440, 440, 600, 1000, 1300, 1626, 1900};
    const double seg_cycles = 4200.0, copy_cycles = 500.0, bytes_per_cycle = 22.0;
    auto rows_per_copy = [&](const TileDesc &d) {
        const int per_step = d.lg < 5 ? 32 >> d.lg : 1;
        return std::max(per_step, (int)(slot_bytes / (uint32_t)(d.r_pad * 8)) / per_step * per_step);
    };
    auto copy_cost = [&](const TileDesc &d, int rows) {      // warps' time for a copy of `rows`
        return copy_cycles + ceil_div(rows, 512 >> d.lg) * step_cycles[d.lg];
    };
    const int max_cta = (int)std::max<int64_t>(1, std::min<int64_t>(num_sms, ceil_div(n, 32)));
    // deal the rows for target T; with `emit` the segments are written down
    auto deal = [&](double T, bool emit) {
        int used_ctas = 0;
        double warp_t = 0.0, mem_t = 0.0;
        TileCta cur{(int)out.segs.size(), 0, 0, 0};
        auto close_cta = [&]() {
            if (warp_t > 0.0) {
                ++used_ctas;
                if (emit) {
                    out.ctas.push_back(cur);
                    out.time = std::max(out.time, std::max(warp_t, mem_t));
                }
            }
            cur.seg0 = (int)out.segs.size();
            cur.n_segs = cur.n_copies = 0;
            warp_t = mem_t = 0.0;
        };
        for (int b = 0; b < nb; ++b) {
            const TileDesc &d = desc[(size_t)b];
            const int fit = rows_per_copy(d);
            const double row_mem = (double)d.r_pad * 8 / bytes_per_cycle;
            int r = 0, seg_no = 0;
            while (r < d.n_rows) {
                const int left = d.n_rows - r;
                // whole copies of this batch that still fit under T on both clocks
                int take = 0;
                double w = warp_t + seg_cycles, m = mem_t;
                while (take < left) {
                    const int rows = std::min(fit, left - take);
                    if (std::max(w + copy_cost(d, rows), m + rows * row_mem) > T) break;
                    w += copy_cost(d, rows);
                    m += rows * row_mem;
                    take += rows;
                }
                if (take < left && left - take < 8) {         // no crumbs for the next CTA
                    w += copy_cost(d, left - take);
                    m += (left - take) * row_mem;
                    take = left;
                }
                if (take == 0) {
                    if (warp_t > 0.0) { close_cta(); continue; }
                    take = std::min(fit, left);               // a CTA takes at least one copy
                    w += copy_cost(d, take);
                    m += take * row_mem;
                }
                if (emit) {
                    TileSeg sg;
                    memset(&sg, 0, sizeof(sg));
                    sg.p_off = d.p_off;
                    sg.u_dst = seg_no == 0 ? d.p_off : p_cells + out.extra_cells;
                    if (seg_no > 0) out.extra_cells += d.r_pad;
                    sg.r_pad = d.r_pad;
                    sg.n_cls = d.n_cls;
                    sg.lg = d.lg;
                    sg.n_rows = take;
                    sg.batch = b;
                    sg.fit = fit;
                    sg.n_copies = (int)ceil_div(take, fit);
                    sg.v_off = d.v_off + (int64_t)r * d.r_pad;
                    sg.row0 = d.row0 + r;
                    out.ent_batch.push_back(b);
                    out.ent_off.push_back(sg.u_dst);
                    cur.n_copies += sg.n_copies;
                    out.n_copy += sg.n_copies;
                    out.segs.push_back(sg);
                    ++cur.n_segs;
                }
                warp_t = w;
                mem_t = m;
                r += take;
                ++seg_no;
            }
        }
        close_cta();
        return used_ctas;
    };
    double lo = 0.0, hi = 1.0;
    while (deal(hi, false) > max_cta) hi *= 2.0;
    for (int it = 0; it < 30; ++it) {
        const double mid = 0.5 * (lo + hi);
        if (deal(mid, false) > max_cta) lo = mid; else hi = mid;
    }
    deal(hi, true);
}

// Invariants of a plan: the CTAs' segments are consecutive, the segments of a batch cover its
// rows in order without gaps, copy counts agree.  Returns the number of violations.
inline int tile_plan_check(const std::vector<TileDesc> &desc, const TilePlanOut &plan) {
    const int nb = (int)desc.size();
    std::vector<int> rows_of((size_t)nb, 0);
    int errs = 0, next_seg = 0, copies_sum = 0;
    for (const TileCta &c : plan.ctas) {
        if (c.seg0 != next_seg) ++errs;
        int cc = 0;
        for (int q = 0; q < c.n_segs; ++q) {
            const TileSeg &g = plan.segs[(size_t)(c.seg0 + q)];
            const TileDesc &d = desc[(size_t)g.batch];
            if (g.v_off != d.v_off + (int64_t)rows_of[(size_t)g.batch] * d.r_pad) ++errs;
            rows_of[(size_t)g.batch] += g.n_rows;
            if (g.n_copies != (int)ceil_div(g.n_rows, g.fit)) ++errs;
            cc += g.n_copies;
        }
        if (cc != c.n_copies) ++errs;
        copies_sum += cc;
        next_seg += c.n_segs;
    }
    for (int b = 0; b < nb; ++b) if (rows_of[(size_t)b] != desc[(size_t)b].n_rows) ++errs;
    if (copies_sum != plan.n_copy || next_seg != (int)plan.segs.size()) ++errs;
    return errs;
}

// Replicate slots of a bootstrap session (em.cu: run_bootstrap): the pass of R slots runs on
// num_sms / R CTAs per slot, all R in one wave on one plan.  R is the largest power of two up to
// kBootMaxSlots whose plan models at most R times the time of the full-budget plan (R replicates
// then cost no more than R iterations one after another; launch and tail costs, which the model
// leaves out, only favour a larger R), and whose slot buffers (bytes_per_slot each) take at most
// an eighth of the free device memory.  From the matrix alone: a replicate's arithmetic does not
// depend on how many replicates are asked for.
constexpr int kBootMaxSlots = 16;
inline int boot_slots(const std::vector<TileDesc> &desc, int64_t n, int num_sms,
                      uint32_t slot_bytes, int64_t p_cells, double bytes_per_slot,
                      double free_bytes) {
    TilePlanOut full;
    tile_plan(desc, n, num_sms, slot_bytes, p_cells, full);
    int best = 1;
    for (int r = 2; r <= kBootMaxSlots && num_sms / r >= 1; r *= 2) {
        if ((double)r * bytes_per_slot > free_bytes / 8) break;
        TilePlanOut p;
        tile_plan(desc, n, num_sms / r, slot_bytes, p_cells, p);
        if (p.time <= r * full.time) best = r;
    }
    return best;
}

}  // namespace mxb
