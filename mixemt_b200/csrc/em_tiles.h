// Host side of the class-tile form of an EM session (em_tiles.cu): what em.cu calls.  The
// kernels are in em_tiles.cuh, the records they read and the plan of the pass in tile_plan.h.
#pragma once

#include <vector>

#include "em_common.cuh"
#include "tile_plan.h"

namespace mxb {

// Layout of the batches and ring of the pass for the class counts of n rows (tile_plan.h).
struct TileShape {
    std::vector<TileDesc> desc;
    int64_t v_cells = 0, p_cells = 0;
    uint32_t ring_bytes = 0;   // ring slots of the pass and their count (tile_ring)
    int ring_slots = 0;
    bool ring_ok = false;      // false: rows too long for the ring
};

// The class tiles of a session and what their launches need.  The R slots of a slotted session
// iterate side by side (the kSlots kernels); their class vectors Pi and U lie pi_stride and
// u_stride doubles apart.
struct TileForm {
    DevBlock maps;   // [perm][cmap][cword][desc]
    DevBlock v;      // the tiles (doubles)
    DevBlock vecs;   // [Pi x R][U x R][ctas][segs][gather entries]
    unsigned short *perm = nullptr, *cmap = nullptr;
    unsigned int *cword = nullptr;
    TileDesc *desc = nullptr;
    double *pi = nullptr, *usum = nullptr;
    TileCta *ctas = nullptr;       // plan of the pass
    TileSeg *segs = nullptr;
    int *ent_batch = nullptr;      // gather entries: batch and offset of every U vector
    int64_t *ent_off = nullptr;
    int n_batches = 0, hs = 0, n_ctas = 0, n_ent = 0;
    int ring_slots = 0;
    uint32_t slot_bytes = 0;
    int64_t pi_stride = 0, u_stride = 0;
    int64_t bytes_per_pass = 0;    // what an iteration reads and writes (mxb_em_pass_bytes)
    bool slotted = false;
};

// A session's tiles between the two steps of their set-up.
struct TileClasses {
    DevBlock scratch;     // [hash][rep][n_cls][bad]
    unsigned short *rep = nullptr;
    int *bad = nullptr;
    TileForm form;        // its maps (tile_classify), then the rest (tile_fill)
    TileShape shape;
    TilePlanOut plan;     // on all SMs (tile_classify), then on the slots' share (tile_fill)
};

// Class tiles of a session's matrix are built straight from M in two steps; the caller decides
// the session's form between them (decide_form, which needs the shape and the plan on all SMs).
// Either step sets `used` to false (with a "[mxb tiles] not used: ..." line under MXB_TIMING)
// when the tiles cannot serve: rows too long for the ring, memory short, tiles that do not save
// at least half of the fp64 rows' bytes, or a batch that fails the exact class check.
// MXB_EM_NO_PACK=1 keeps the fp64 rows (cross-check).
//   tile_classify: the column classes of every batch, the layout of their tiles and the plan.
//   tile_fill: for a session of n_slots slots (`slotted`: side by side), the plan on
//   num_sms / n_slots CTAs, the tiles, and the kernel attributes.
int tile_classify(mxb_ctx *ctx, const mxb_matrix *m, TileClasses &c, bool &used);
int tile_fill(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, int64_t ld, int n_slots,
              bool slotted, TileClasses &c, bool &used);

// Blocks of the gather over n_ent U vectors: the partial column sums the tail adds (n_part).
int tile_gather_parts(int n_ent);

// The pass of a tiled iteration of R slots on ctx's stream: class sums, pass and gather, reading
// the proportions pi[cur] of every slot (ld doubles apart) and the control blocks `state`, and
// writing tile_gather_parts(n_ent) x ld column sums per slot to `partials`.  A slotted pass
// reads slot s's weights at weights + s * w_stride.  `marks` (optional, 3 events) are recorded
// after the class sums, the pass and the gather.
int tile_pass(mxb_ctx *ctx, const TileForm &t, unsigned R, int64_t n_cols, int64_t ld,
              double *const pi[2], EmState *state, double *partials, const double *weights,
              int64_t w_stride, const cudaEvent_t *marks);

}  // namespace mxb
