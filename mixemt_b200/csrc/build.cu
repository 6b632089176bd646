// Kernel 1: read-signature x haplotype log-likelihood matrix.
//
// Replaces the N x H x K Python loop of build_em_matrix
// (reference mixemt/preprocess.py:177-198) and the per-cell dictionary walk of
// HapVarBaseMatrix._prob / prob_for_vars (preprocess.py:69-96).
//
// Haplotype tables.  For every variant position p and symbol code a the dense
// table bits[p][a][w] holds one bit per haplotype column: bit (j & 31) of word
// (j >> 5) is set iff haplotype j *expects* symbol a at p (its marker there,
// or the reference base when it carries none: preprocess.py:75-83).  A 32-bit
// word is a ready-made ballot over 32 haplotypes for one observed
// (position, base); plane n_sym is all zero and serves bases that can never
// match.  Nearly all haplotypes agree on the outcome of a plane, so the table is
// also kept in *sparse deviation* form: for plane (p, a) the list of
// (word index g, D) with D = bits[p][a][g] XOR (baseline ? all ones : 0) != 0,
// where the baseline outcome of the plane is the one the majority of the
// haplotypes has (the marker-free outcome a == ref[p], except for the few dozen
// planes whose derived allele is carried by more than half of the tree).
// Build 17: 4070 x 5 x 172 dense words (14 MB) against ~0.3 M sparse entries.
//
// Bit-exactness.  A cell is the fp64 sum, in signature order, of hit[p] on a
// match and miss[p] on a mismatch -- the same values in the same order as the
// reference's `total += math.log(...)` (preprocess.py:92-95).  fp64 addition is
// not associative, so the K terms of a cell cannot be re-grouped; what can be
// shared is whole chains: two haplotypes with the same match pattern over the
// row's K positions get the same sum, and a chain whose first deviation from
// the baseline pattern is at k0 may start from the baseline prefix sum P[k0]
// (the same additions in the same order).  A 300 bp fragment separates the 5408
// Build-17 haplotypes into only ~300 (32-column group, pattern) classes, so the
// class kernel evaluates ~15x fewer dependent-add chains than cells.
//
// build_matrix_kernel (class kernel), one CTA per row at a time, rows handed
// out by a device-wide counter (they cost 0.2x .. 10x the average):
//   0. stage the row: per observation k the (baseline, deviating) term pair,
//      its (position, symbol) plane and whether the baseline outcome matches;
//   1. the last warp forms the baseline prefix sums P[0..K] (one dependent
//      chain) while the other warps collect the row's deviation entries per
//      32-column group: a first walk over the sparse lists sets bit k in the
//      group's observation bitmap (shared-memory atomicOr), a scan of the
//      popcounts sizes the groups and lists the non-empty ones, and a second
//      walk drops every (k, D) at offset[group] + rank of k in the bitmap --
//      sorted by k without a sort;
//   2. one warp per non-empty group: every lane reads its pattern over the
//      group's entries (bit e = "deviates at the e-th deviating observation";
//      straight-line code for up to four entries, no cross-lane work for one),
//      match.any finds the distinct patterns and one chain item is taken from
//      the warp's own item pool per distinct non-empty pattern (no atomics); a
//      cell remembers its class within the group;
//   3. the same warp evaluates its items (run_chains): 32 or 64 items walk k in
//      lock step from the earliest first deviation among them -- a lane that has
//      not deviated yet retraces P[] -- with the deviations of each 32-observation
//      block gathered into a mask word up front, so a step is (shared load, bit
//      test, select, add), and two chains per lane share every load;
//   4. every cell looks up the value of its class and the row is written with
//      coalesced 16-byte stores, four cells per thread.
// The shared-memory layout is a compile-time constant (BuildSmem: group arrays
// sized for 176 or 256 groups), so addresses are immediates.  Two launches share
// the code: tier 1 (256 threads, 38 KB of shared memory, 5 CTAs per SM) takes rows
// with <= 256 observations, <= 1536 deviation entries and <= 146 chains per warp
// (93 % of the config-2 rows); rows beyond that are queued on the device and
// re-run by tier 2 (512 threads, 8064 entries, 273 chains per warp).
// What exceeds tier 2 as well (K > 512, or a group with more than 32 deviating
// observations) walks the dense bitset table cell by cell: build_dense_row /
// the per-group dense loop, the same arithmetic as build_matrix_dense_kernel,
// the plain kernel that is also used when H > 8192 (or MXB_BUILD_DENSE=1 is set).
#include <algorithm>
#include <memory>
#include <new>
#include <string.h>
#include <vector>

#include "common.cuh"

namespace mxb {

constexpr int kBuildThreads = 512;   // dense kernel
constexpr int kBuildCols = 4;        // dense path: haplotype columns per thread and group
constexpr int kBuildObsChunk = 512;  // observations staged per pass (dense path)

// ---- dense path ---------------------------------------------------------------
// One CTA walks one row; a thread owns 4 haplotype columns per 2048-column
// group (same bit lane, 4 different words), so every bitset load is
// warp-uniform and the four accumulation chains are independent.
template <int kThreads>
__device__ __noinline__ void build_dense_row(
        const uint32_t *__restrict__ bits, const double2 *__restrict__ hitmiss, int n_planes,
        int n_words, int n_hap, int64_t k0, int64_t k1, const int32_t *__restrict__ pos_idx,
        const uint8_t *__restrict__ base_code, double *__restrict__ out_row,
        int32_t *__restrict__ match_row, double2 *s_hm, uint32_t *s_off) {
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    constexpr int kGroup = kThreads * kBuildCols;
    constexpr int kWordsPerSlot = kThreads / 32;

    for (int64_t kc = k0; kc < k1 || kc == k0; kc += kBuildObsChunk) {
        const int n_obs = (int)min((int64_t)kBuildObsChunk, k1 - kc);
        __syncthreads();  // previous users of s_hm / s_off are done
        for (int k = tid; k < n_obs; k += kThreads) {
            const int p = pos_idx[kc + k];
            int c = base_code[kc + k];
            if (c >= n_planes - 1) c = n_planes - 1;  // "other": all-zero plane
            s_off[k] = (uint32_t)((p * n_planes + c) * n_words);
            s_hm[k] = hitmiss[p];
        }
        __syncthreads();
        const bool first = (kc == k0);

        for (int g0 = 0; g0 < n_hap; g0 += kGroup) {
            double acc[kBuildCols];
            int cnt[kBuildCols];
            const int word0 = (g0 >> 5) + warp;
#pragma unroll
            for (int u = 0; u < kBuildCols; ++u) {
                const int j = g0 + u * kThreads + tid;
                acc[u] = 0.0;
                cnt[u] = 0;
                if (!first && j < n_hap) {
                    acc[u] = out_row[j];
                    if (match_row) cnt[u] = match_row[j];
                }
            }
            for (int k = 0; k < n_obs; ++k) {
                const uint32_t *plane = bits + s_off[k] + word0;
                const double2 hm = s_hm[k];
                uint32_t w[kBuildCols];
#pragma unroll
                for (int u = 0; u < kBuildCols; ++u) {
                    // words past the table end belong to columns >= n_hap
                    w[u] = (word0 + u * kWordsPerSlot < n_words)
                               ? __ldg(plane + u * kWordsPerSlot) : 0u;
                }
#pragma unroll
                for (int u = 0; u < kBuildCols; ++u) {
                    const bool hit = (w[u] >> lane) & 1u;
                    acc[u] += hit ? hm.x : hm.y;
                    cnt[u] += hit ? 1 : 0;
                }
            }
#pragma unroll
            for (int u = 0; u < kBuildCols; ++u) {
                const int j = g0 + u * kThreads + tid;
                if (j < n_hap) {
                    out_row[j] = acc[u];
                    if (match_row) match_row[j] = cnt[u];
                }
            }
        }
        if (k1 == k0) break;  // empty row: cells are 0.0 (never produced by the reference)
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kBuildThreads)
build_matrix_dense_kernel(const uint32_t *__restrict__ bits, const double2 *__restrict__ hitmiss,
                          int n_planes, int n_words, int n_hap, int64_t n_rows,
                          const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ pos_idx,
                          const uint8_t *__restrict__ base_code, double *__restrict__ out,
                          int32_t *__restrict__ match_out) {
    __shared__ double2 s_hm[kBuildObsChunk];
    __shared__ uint32_t s_off[kBuildObsChunk];
    for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        build_dense_row<kBuildThreads>(bits, hitmiss, n_planes, n_words, n_hap, row_ptr[row], row_ptr[row + 1],
                        pos_idx, base_code, out + row * (int64_t)n_hap,
                        match_out ? match_out + row * (int64_t)n_hap : nullptr, s_hm, s_off);
    }
}

// ---- class kernel ---------------------------------------------------------------
struct BuildTables {
    const uint32_t *bits;      // dense [n_pos][n_planes][n_words]
    const double2 *hitmiss;    // [n_pos]
    const uint8_t *plane_base; // [n_pos * n_planes] outcome of the baseline pattern: 1 = match
    const int32_t *dev_ptr;    // [n_pos * n_planes + 1]
    const uint2 *dev_ent;      // {word index, D}
    int n_planes, n_words, n_hap, n_groups;
};

constexpr int kMaxObs = 512;         // observations per row (longer rows: dense path)
constexpr unsigned kDenseGroup = 0xFFFFu;   // s_gbase marker: group walked densely
constexpr unsigned kEmptyGroup = 0xFFFEu;   // s_gbase marker: no deviation, every cell in class 0
static_assert(kMaxObs == kBuildObsChunk, "the dense row path reuses the class kernel's staging area");

// Pool sizes of the launches: tier 1 serves the common rows at 5 CTAs/SM, tier 2 re-runs
// the few rows that overflowed tier 1's pools with larger ones.  kObsWords * 32 =
// observations per row the tier accepts.
struct Tier1 {
    static constexpr int kThreads = 256, kEntries = 1536, kItems = 1024, kObsWords = 8, kMinBlocks = 5;
};
struct Tier2 {
    static constexpr int kThreads = 512, kEntries = 8064, kItems = 4096, kObsWords = 16, kMinBlocks = 2;
};
static_assert(Tier2::kObsWords * 32 == kMaxObs, "tier 2 takes every row the staging area holds");

// Shared-memory layout of the class kernel (bytes).  Every offset is a compile-time
// constant (the group arrays are sized for kMaxGroups 32-column groups), so shared-memory
// addresses are immediates instead of values recomputed around every loop.
template <class Tier, int kMaxGroups, bool kCounts>
struct BuildSmem {
    static constexpr int kObs = Tier::kObsWords * 32;
    static constexpr size_t term = 0;                                    // (baseline, deviating) terms
    static constexpr size_t prefix = term + sizeof(double2) * kObs;      // baseline prefix sums
    static constexpr size_t item = prefix + sizeof(double) * (kObs + 1); // (pattern, group) -> value
    static constexpr size_t ew = item + sizeof(uint2) * Tier::kItems;    // entry pool: D words
    static constexpr size_t plane = ew + sizeof(uint32_t) * (Tier::kEntries > kObs ? Tier::kEntries : kObs);
    static constexpr size_t gmap = plane + sizeof(int) * kObs;           // deviating k per group
    static constexpr size_t gcnt = gmap + sizeof(uint32_t) * kMaxGroups * Tier::kObsWords;
    static constexpr size_t goff = gcnt + sizeof(int) * kMaxGroups;      // pool offset of the group
    static constexpr size_t icnt = goff + sizeof(int) * kMaxGroups;      // match count per item
    static constexpr size_t ek = icnt + (kCounts ? sizeof(int) * Tier::kItems : 0);  // entry pool: k
    static constexpr size_t pcnt = ek + sizeof(uint16_t) * Tier::kEntries;  // baseline match prefix
    static constexpr size_t gbase = pcnt + sizeof(uint16_t) * (kObs + 2);   // first item of the group
    static constexpr size_t glist = gbase + sizeof(uint16_t) * kMaxGroups;  // groups with entries
    static constexpr size_t cell = (glist + sizeof(uint16_t) * kMaxGroups + 3) & ~(size_t)3;  // class of the cell in its group
    static constexpr size_t total = (cell + (size_t)kMaxGroups * 32 + 15) & ~(size_t)15;
};

// Barrier among the scatter/classify warps only (all but the last warp, which
// runs the prefix chain meanwhile).
template <int kWorkThreads>
__device__ __forceinline__ void work_warps_sync() {
    asm volatile("bar.sync 1, %0;" ::"n"(kWorkThreads) : "memory");
}

// mbarrier through which the prefix warp releases P[] to the warps that evaluate chains
// (one arrival per row; the waiters track the phase parity).
__device__ __forceinline__ uint32_t bar_addr(const uint64_t *bar) {
    return (uint32_t)__cvta_generic_to_shared(bar);
}
__device__ __forceinline__ void bar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_addr(bar)), "r"(count));
}
__device__ __forceinline__ void bar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(bar_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void bar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar_addr(bar)), "r"(parity)
        : "memory");
}

// Dependent-add chains of up to 32 (64 with kDual) chain items starting at s_item[first]:
// lane l evaluates item first + l (and first + 32 + l).  The warp walks k in lock step from
// the 8-aligned block of the earliest first deviation among its items: a lane that has not
// deviated yet adds the baseline terms, i.e. it retraces P[] exactly, so starting every
// lane at P[k_start] is the same chain as starting it at P[its own first deviation].  The
// deviations of an item inside the current 32-observation block are gathered into one mask
// word up front, which leaves (shared load, bit test, select, add) per step.
template <bool kCounts, bool kDual>
__device__ __forceinline__ void run_chains(int first, int n_left, int lane, int n_obs,
                                           uint2 *s_item, double *s_val, int *s_icnt,
                                           const uint16_t *s_ek, const int *s_goff,
                                           const double2 *s_term, const double *s_prefix,
                                           const uint16_t *s_pcnt) {
    constexpr int kNoDev = 0x7FFFFFFF;
    constexpr int kChains = kDual ? 2 : 1;
    uint32_t rem[kChains];   // bit e: deviates at the group's e-th deviating observation
    int ek[kChains];         // pool offset of the group's entries
    int nk[kChains];         // next deviating observation
    bool valid[kChains];
#pragma unroll
    for (int c = 0; c < kChains; ++c) {
        valid[c] = c * 32 + lane < n_left;
        rem[c] = 0u;
        ek[c] = 0;
        nk[c] = kNoDev;
        if (valid[c]) {
            const uint2 item = s_item[first + c * 32 + lane];
            rem[c] = item.x;
            ek[c] = s_goff[item.y];
            nk[c] = s_ek[ek[c] + __ffs(rem[c]) - 1];
            rem[c] &= rem[c] - 1;
        }
    }
    int k = __reduce_min_sync(0xffffffffu, kDual ? min(nk[0], nk[kChains - 1]) : nk[0]) & ~7;
    double acc[kChains];
    int cnt[kChains];
#pragma unroll
    for (int c = 0; c < kChains; ++c) {
        acc[c] = s_prefix[k];
        cnt[c] = kCounts ? (int)s_pcnt[k] : 0;
    }
    while (k < n_obs) {   // warp-uniform
        const int kb = k & ~31;
        uint32_t word[kChains];   // bit (k' - kb): the item deviates at observation k'
#pragma unroll
        for (int c = 0; c < kChains; ++c) {
            word[c] = 0u;
            while (nk[c] < kb + 32) {
                word[c] |= 1u << (nk[c] - kb);
                nk[c] = rem[c] ? (int)s_ek[ek[c] + __ffs(rem[c]) - 1] : kNoDev;
                rem[c] &= rem[c] - 1;
            }
        }
        const int k_end = min(kb + 32, n_obs);
#pragma unroll 1
        for (; k + 8 <= k_end; k += 8) {
            uint32_t w8[kChains];
#pragma unroll
            for (int c = 0; c < kChains; ++c) w8[c] = word[c] >> (k - kb);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const double2 t = s_term[k + u];
#pragma unroll
                for (int c = 0; c < kChains; ++c) {
                    const bool dev = (w8[c] >> u) & 1u;
                    acc[c] += dev ? t.y : t.x;
                    if (kCounts) {
                        const int bm = (int)s_pcnt[k + u + 1] - (int)s_pcnt[k + u];
                        cnt[c] += dev ? 1 - bm : bm;
                    }
                }
            }
        }
        if (k_end == n_obs) {   // the last, partial group of eight
#pragma unroll 1
            for (; k < k_end; ++k) {
                const double2 t = s_term[k];
#pragma unroll
                for (int c = 0; c < kChains; ++c) {
                    const bool dev = (word[c] >> (k - kb)) & 1u;
                    acc[c] += dev ? t.y : t.x;
                    if (kCounts) {
                        const int bm = (int)s_pcnt[k + 1] - (int)s_pcnt[k];
                        cnt[c] += dev ? 1 - bm : bm;
                    }
                }
            }
        }
    }
    __syncwarp();   // every lane has read its items before the slots become values
#pragma unroll
    for (int c = 0; c < kChains; ++c) {
        if (valid[c]) {
            s_val[first + c * 32 + lane] = acc[c];
            if (kCounts) s_icnt[first + c * 32 + lane] = cnt[c];
        }
    }
}

// Rows come from row_list[0 .. *n_list) when row_list != NULL, else 0 .. n_rows.
// Rows that do not fit the pools are appended to overflow_list when there is
// one (tier 1), else they take the dense path (tier 2).
// route_out (nullable, zeroed by the host): route_out[row] = path + 4 * (groups walked by the
// per-group dense loop), path 0 = tier 1, 1 = tier 2, 2 = build_dense_row (mxb_build_matrix).
// Tier 1 writes only rows with dense groups, tier 2 every row it finishes.
template <bool kCounts, class Tier, int kMaxGroups>
__global__ void __launch_bounds__(Tier::kThreads, kCounts ? 1 : Tier::kMinBlocks)
build_matrix_kernel(BuildTables tb, int64_t n_rows, const int32_t *__restrict__ row_list,
                    const int *__restrict__ n_list, int32_t *__restrict__ overflow_list,
                    int *__restrict__ overflow_count, int *__restrict__ work_counter,
                    const int64_t *__restrict__ row_ptr,
                    const int32_t *__restrict__ pos_idx, const uint8_t *__restrict__ base_code,
                    double *__restrict__ out, int32_t *__restrict__ match_out,
                    int32_t *__restrict__ route_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_next[2];
    __shared__ int s_overflow;
    __shared__ int s_ndense;
    __shared__ __align__(8) uint64_t s_prefix_bar;   // completes once per row: P[] is written
    __shared__ int s_nlist;
    using L = BuildSmem<Tier, kMaxGroups, kCounts>;
    constexpr int W = Tier::kObsWords;
    constexpr bool kLastTier = W * 32 == kMaxObs;   // only the last tier has the staging room
    constexpr int kClassThreads = Tier::kThreads;
    constexpr int kClassWarps = kClassThreads / 32;
    constexpr int kWorkWarps = kClassWarps - 1;  // the last warp runs the prefix chain
    // every work warp allocates chain items from its own pool: no atomics, and the warp
    // that found a class also evaluates it (item 0 is the baseline class)
    constexpr int kPool = (Tier::kItems - 1) / kWorkWarps;
    double2 *s_term = reinterpret_cast<double2 *>(smem + L::term);
    double *s_prefix = reinterpret_cast<double *>(smem + L::prefix);
    uint2 *s_item = reinterpret_cast<uint2 *>(smem + L::item);
    double *s_val = reinterpret_cast<double *>(smem + L::item);  // overwrites the item
    uint32_t *s_ew = reinterpret_cast<uint32_t *>(smem + L::ew);
    int *s_plane = reinterpret_cast<int *>(smem + L::plane);
    uint32_t *s_gmap = reinterpret_cast<uint32_t *>(smem + L::gmap);
    int *s_gcnt = reinterpret_cast<int *>(smem + L::gcnt);
    int *s_goff = reinterpret_cast<int *>(smem + L::goff);
    int *s_icnt = reinterpret_cast<int *>(smem + L::icnt);
    uint16_t *s_ek = reinterpret_cast<uint16_t *>(smem + L::ek);
    uint16_t *s_pcnt = reinterpret_cast<uint16_t *>(smem + L::pcnt);
    uint16_t *s_gbase = reinterpret_cast<uint16_t *>(smem + L::gbase);
    uint16_t *s_glist = reinterpret_cast<uint16_t *>(smem + L::glist);
    uint8_t *s_cell = reinterpret_cast<uint8_t *>(smem + L::cell);
    // the dense row path reuses the staging areas: (hit, miss) and plane offsets
    uint32_t *s_off = reinterpret_cast<uint32_t *>(smem + L::ew);

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int n_hap = tb.n_hap;
    const int n_groups = tb.n_groups;
    const int64_t n_work = row_list ? (int64_t)*n_list : n_rows;
    if (tid == 0) {
        bar_init(&s_prefix_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    uint32_t prefix_parity = 0;   // block-uniform: phase of s_prefix_bar the current row completes
    __syncthreads();

    // Rows cost between 0.2x and 10x the average: after its first row a CTA takes rows from
    // a device-wide counter.  The next index is fetched while the current row is processed
    // and handed over through s_next[parity] behind the row's closing barrier.
    int parity = 0;
    for (int64_t wi = blockIdx.x; wi < n_work; wi = s_next[parity], parity ^= 1) {
        if (tid == 0) s_next[parity] = (int)gridDim.x + atomicAdd(work_counter, 1);
        const int64_t row = row_list ? (int64_t)row_list[wi] : wi;
        const int64_t k0 = row_ptr[row];
        const int64_t k1 = row_ptr[row + 1];
        double *out_row = out + row * (int64_t)n_hap;
        int32_t *match_row = kCounts ? match_out + row * (int64_t)n_hap : nullptr;
        const bool too_long = k1 - k0 > W * 32;  // block-uniform
        const int n_obs = too_long ? 0 : (int)(k1 - k0);

        if (!too_long) {
        // ---- 0. stage the row -------------------------------------------------------
        for (int k = tid; k < n_obs; k += kClassThreads) {
            const int p = pos_idx[k0 + k];
            int c = base_code[k0 + k];
            if (c >= tb.n_planes - 1) c = tb.n_planes - 1;
            const double2 hm = tb.hitmiss[p];
            const bool base_match = tb.plane_base[p * tb.n_planes + c] != 0;
            s_term[k] = base_match ? hm : make_double2(hm.y, hm.x);
            s_plane[k] = p * tb.n_planes + c;
            // the match flag rides in s_pcnt[k + 1] until the prefix pass
            s_pcnt[k + 1] = base_match ? 1 : 0;
        }
        for (int i = tid; i < n_groups * W; i += kClassThreads) s_gmap[i] = 0u;
        if (tid == 0) { s_overflow = 0; s_ndense = 0; }
        __syncthreads();

        if (warp == kWorkWarps) {
            // ---- 1'. baseline prefix sums (one dependent-add chain), off the others' path
            if (lane == 0) {
                double acc = 0.0;
                int cnt = 0;
                s_prefix[0] = acc;
                s_pcnt[0] = 0;
                int k = 0;
                for (; k + 8 <= n_obs; k += 8) {
                    double t[8];
                    int f[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) { t[u] = s_term[k + u].x; f[u] = s_pcnt[k + u + 1]; }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        acc += t[u];
                        cnt += f[u];
                        s_prefix[k + u + 1] = acc;
                        s_pcnt[k + u + 1] = (uint16_t)cnt;
                    }
                }
                for (; k < n_obs; ++k) {
                    acc += s_term[k].x;
                    cnt += s_pcnt[k + 1];
                    s_prefix[k + 1] = acc;
                    s_pcnt[k + 1] = (uint16_t)cnt;
                }
                s_val[0] = acc;   // class 0: the baseline pattern
                if (kCounts) s_icnt[0] = cnt;
                bar_arrive(&s_prefix_bar);
            }
        } else {
            // ---- 1. deviation entries of the row, grouped by 32-column group ------------------
            // 8 lanes walk the sparse list of one observation (5.7 entries on average)
            // (the loops are kept warp-uniform: the four lists advance together)
            const int sub = lane >> 3, sl = lane & 7;
#pragma unroll 1
            for (int kb = warp * 4; kb < n_obs; kb += kWorkWarps * 4) {
                const int k = kb + sub;
                int e = 0, e1 = 0;
                if (k < n_obs) {
                    const int plane = s_plane[k];
                    e = tb.dev_ptr[plane] + sl;
                    e1 = tb.dev_ptr[plane + 1];
                }
#pragma unroll 1
                while (__any_sync(0xffffffffu, e < e1)) {
                    if (e < e1) atomicOr(&s_gmap[tb.dev_ent[e].x * W + (k >> 5)], 1u << (k & 31));
                    e += 8;
                }
            }
            work_warps_sync<kWorkWarps * 32>();
            if (warp == 0) {  // entries per group, their exclusive scan, list of the groups with any
                int carry = 0, n_list = 0;
                for (int g0 = 0; g0 < n_groups; g0 += 32) {
                    const int g = g0 + lane;
                    int c = 0;
                    if (g < n_groups) {
#pragma unroll
                        for (int w = 0; w < W; ++w) c += __popc(s_gmap[g * W + w]);
                        s_gcnt[g] = c;
                        if (c == 0) s_gbase[g] = (uint16_t)kEmptyGroup;
                    }
                    const uint32_t some = __ballot_sync(0xffffffffu, c > 0);
                    if (c > 0) s_glist[n_list + __popc(some & ((1u << lane) - 1u))] = (uint16_t)g;
                    n_list += __popc(some);
                    int incl = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int v = __shfl_up_sync(0xffffffffu, incl, o);
                        if (lane >= o) incl += v;
                    }
                    if (g < n_groups) s_goff[g] = carry + incl - c;
                    carry += __shfl_sync(0xffffffffu, incl, 31);
                }
                if (lane == 0) {
                    s_nlist = n_list;
                    if (carry > Tier::kEntries) s_overflow = 1;
                }
            }
            work_warps_sync<kWorkWarps * 32>();
            // read once, before any warp can raise the flag again: the branch and the
            // loops below hold warp-synchronous intrinsics and must stay warp-uniform
            const bool too_many_entries = s_overflow != 0;
            if (!too_many_entries) {
#pragma unroll 1
                for (int kb = warp * 4; kb < n_obs; kb += kWorkWarps * 4) {
                    const int k = kb + sub;
                    int e = 0, e1 = 0;
                    if (k < n_obs) {
                        const int plane = s_plane[k];
                        e = tb.dev_ptr[plane] + sl;
                        e1 = tb.dev_ptr[plane + 1];
                    }
#pragma unroll 1
                    while (__any_sync(0xffffffffu, e < e1)) {
                        if (e < e1) {
                            // slot = rank of k among the group's deviating observations:
                            // the group's entries end up sorted by k without a sort
                            const uint2 ent = tb.dev_ent[e];
                            const uint32_t *map = s_gmap + ent.x * W;
                            int slot = s_goff[ent.x] + __popc(map[k >> 5] & ((1u << (k & 31)) - 1u));
                            for (int w = 0; w < (k >> 5); ++w) slot += __popc(map[w]);
                            s_ek[slot] = (uint16_t)k;
                            s_ew[slot] = ent.y;
                        }
                        e += 8;
                    }
                }
            }
            work_warps_sync<kWorkWarps * 32>();

            // ---- 2. classes of every 32-column group ------------------------------------------
            const int pool_base = 1 + warp * kPool;
            int my_items = 0;       // warp-uniform; items past kPool are counted but not stored
            const int n_list = too_many_entries ? 0 : s_nlist;
#pragma unroll 1
            for (int gi = warp; gi < n_list; gi += kWorkWarps) {
                const int g = s_glist[gi];
                const int a = s_gcnt[g];
                if (a > 32) {  // handled after the prefix pass
                    if (lane == 0) { s_gbase[g] = (uint16_t)kDenseGroup; atomicAdd(&s_ndense, 1); }
                    continue;
                }
                const uint32_t *w = s_ew + s_goff[g];
                const int base_idx = pool_base + my_items;
                if (a == 1) {  // a third of the groups: one deviating observation, one class
                    const uint32_t d = w[0];
                    if (lane == 0 && my_items < kPool) s_item[base_idx] = make_uint2(1u, (uint32_t)g);
                    my_items += 1;
                    s_cell[g * 32 + lane] = (uint8_t)((d >> lane) & 1u);
                    if (lane == 0) s_gbase[g] = (uint16_t)base_idx;
                    continue;
                }
                uint32_t pattern;   // bit e: this lane's column deviates at the group's e-th entry
                if (a <= 5) {       // nineteen groups in twenty: patterns are numbers below 32
                    const uint32_t w0 = w[0], w1 = w[1];
                    pattern = ((w0 >> lane) & 1u) | (((w1 >> lane) & 1u) << 1);
                    if (a > 2) pattern |= ((w[2] >> lane) & 1u) << 2;
                    if (a > 3) pattern |= ((w[3] >> lane) & 1u) << 3;
                    if (a > 4) pattern |= ((w[4] >> lane) & 1u) << 4;
                    // the set of patterns present in the group, as a bitmap: classes are numbered
                    // by pattern value, and lane p stores the item of pattern p
                    const uint32_t present = __reduce_or_sync(0xffffffffu, 1u << pattern) & ~1u;
                    const int n_lead = __popc(present);
                    if (((present >> lane) & 1u) && my_items + n_lead <= kPool)
                        s_item[base_idx + __popc(present & ((1u << lane) - 1u))] =
                            make_uint2((uint32_t)lane, (uint32_t)g);
                    my_items += n_lead;
                    s_cell[g * 32 + lane] =
                        (uint8_t)(pattern ? 1 + __popc(present & ((1u << pattern) - 1u)) : 0);
                    if (lane == 0) s_gbase[g] = (uint16_t)base_idx;
                    continue;
                }
                pattern = 0;
#pragma unroll 4
                for (int e = a - 1; e >= 0; --e) pattern = (pattern << 1) | ((w[e] >> lane) & 1u);
                const uint32_t peers = __match_any_sync(0xffffffffu, pattern);
                const int leader_lane = __ffs(peers) - 1;
                const bool leader = (lane == leader_lane) && pattern != 0u;
                const uint32_t lead_mask = __ballot_sync(0xffffffffu, leader);
                const int n_lead = __popc(lead_mask);
                int local = 1 + __popc(lead_mask & ((1u << lane) - 1u));  // 1-based within the group
                if (leader && my_items + n_lead <= kPool)
                    s_item[base_idx + local - 1] = make_uint2(pattern, (uint32_t)g);
                my_items += n_lead;
                local = __shfl_sync(0xffffffffu, local, leader_lane);
                s_cell[g * 32 + lane] = (uint8_t)(pattern ? local : 0);
                if (lane == 0) s_gbase[g] = (uint16_t)base_idx;
            }
            if (my_items > kPool) {   // the warp's pool is full: the row goes to the next tier
                if (lane == 0) s_overflow = 1;
                my_items = 0;
            }

            // ---- 3. one dependent-add chain per class, by the warp that found it (run_chains)
            __syncwarp();   // the warp's items are visible to all of its lanes
            bar_wait(&s_prefix_bar, prefix_parity);   // P[] is complete (every phase is waited on)
            // 64 items at a time (two independent chains per lane share every term load)
            // while the warp has more than 32 left, then one chain per lane
            int i0 = 0;
#pragma unroll 1
            for (; my_items - i0 > 32; i0 += 64)
                run_chains<kCounts, true>(pool_base + i0, my_items - i0, lane, n_obs, s_item, s_val,
                                          s_icnt, s_ek, s_goff, s_term, s_prefix, s_pcnt);
            if (i0 < my_items)
                run_chains<kCounts, false>(pool_base + i0, my_items - i0, lane, n_obs, s_item, s_val,
                                           s_icnt, s_ek, s_goff, s_term, s_prefix, s_pcnt);
        }
        __syncthreads();
        prefix_parity ^= 1u;
        }  // !too_long
        if (too_long || s_overflow) {  // block-uniform: the row does not fit this tier's pools
            if (overflow_list) {
                if (tid == 0) overflow_list[atomicAdd(overflow_count, 1)] = (int32_t)row;
            } else if constexpr (kLastTier) {
                build_dense_row<kClassThreads>(tb.bits, tb.hitmiss, tb.n_planes, tb.n_words, n_hap,
                                               k0, k1, pos_idx, base_code, out_row, match_row,
                                               s_term, s_off);
                if (route_out && tid == 0) route_out[row] = 2;
            }
            __syncthreads();  // the row's shared state is reused by the next row
            continue;
        }

        if (kLastTier && route_out && tid == 0) route_out[row] = 1 + 4 * s_ndense;
        // groups with more than 32 deviating positions: walk the dense table, one warp each
        if (s_ndense > 0) {   // block-uniform
            if (!kLastTier && route_out && tid == 0) route_out[row] = 4 * s_ndense;
#pragma unroll 1
            for (int g = warp; g < n_groups; g += kClassWarps) {
                if (s_gbase[g] != kDenseGroup) continue;
                const int j = g * 32 + lane;
                double acc = 0.0;
                int cnt = 0;
                for (int k = 0; k < n_obs; ++k) {
                    const uint32_t w = __ldg(tb.bits + (size_t)s_plane[k] * tb.n_words + g);
                    const uint32_t d = (w >> lane) & 1u;   // 1 = match
                    const double2 t = s_term[k];
                    const bool bm = s_pcnt[k + 1] != s_pcnt[k];
                    acc += (d != 0) == bm ? t.x : t.y;
                    cnt += d;
                }
                if (j < n_hap) {
                    out_row[j] = acc;
                    if (kCounts) match_row[j] = cnt;
                }
            }
        }

        // ---- 4. write the row -----------------------------------------------------------------
        if ((n_hap & 3) == 0) {   // four cells per thread: one group, one 32-bit load of the classes
            for (int j = tid * 4; j < n_hap; j += kClassThreads * 4) {
                const unsigned gb = s_gbase[j >> 5];
                if (gb == kDenseGroup) continue;
                const unsigned cc = gb == kEmptyGroup ? 0u : *reinterpret_cast<const uint32_t *>(s_cell + j);
                unsigned idx[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const unsigned c = (cc >> (8 * u)) & 0xFFu;
                    idx[u] = c ? gb + c - 1 : 0;
                }
                *reinterpret_cast<double2 *>(out_row + j) = make_double2(s_val[idx[0]], s_val[idx[1]]);
                *reinterpret_cast<double2 *>(out_row + j + 2) = make_double2(s_val[idx[2]], s_val[idx[3]]);
                if (kCounts)
                    *reinterpret_cast<int4 *>(match_row + j) =
                        make_int4(s_icnt[idx[0]], s_icnt[idx[1]], s_icnt[idx[2]], s_icnt[idx[3]]);
            }
        } else {
            for (int j = tid; j < n_hap; j += kClassThreads) {
                const unsigned gb = s_gbase[j >> 5];
                if (gb == kDenseGroup) continue;
                const unsigned c0 = gb == kEmptyGroup ? 0u : s_cell[j];
                const unsigned i0 = c0 ? gb + c0 - 1 : 0;
                out_row[j] = s_val[i0];
                if (kCounts) match_row[j] = s_icnt[i0];
            }
        }
        __syncthreads();  // the row's shared state is reused by the next row
    }
}

// One launch of the cascade: rows come from list_in (all rows when NULL), rows that do not
// fit the tier's pools go to list_out (dense path when NULL: last tier only).
template <bool kCounts, class Tier, int kMaxGroups>
static cudaError_t launch_tier(mxb_ctx *ctx, const BuildTables &tb, int64_t n_rows,
                               const int32_t *list_in, const int *n_in, int32_t *list_out,
                               int *n_out, int *work_counter, const int64_t *row_ptr,
                               const int32_t *pos_idx, const uint8_t *base_code, double *out,
                               int32_t *match_out, int32_t *route_out) {
    constexpr size_t smem_bytes = BuildSmem<Tier, kMaxGroups, kCounts>::total;
    auto fn = build_matrix_kernel<kCounts, Tier, kMaxGroups>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem_bytes);
    int per_sm = 0;
    if (e == cudaSuccess)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, Tier::kThreads, smem_bytes);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    const int grid = (int)std::min<int64_t>(n_rows, (int64_t)ctx->num_sms * per_sm);
    fn<<<grid, Tier::kThreads, smem_bytes, ctx->stream>>>(tb, n_rows, list_in, n_in, list_out,
                                                          n_out, work_counter, row_ptr, pos_idx,
                                                          base_code, out, match_out, route_out);
    ctx->launches++;
    return cudaGetLastError();
}

// kMaxGroups sizes the group arrays of the shared-memory layout: 176 groups hold
// Phylotree Build 17 (5408 haplotypes -> 169 groups), 256 groups everything up to 8192.
constexpr int kGroupsSmall = 176, kGroupsLarge = 256;

template <bool kCounts, class Tier>
static cudaError_t launch_tier_groups(mxb_ctx *ctx, const BuildTables &tb, int64_t n_rows,
                                      const int32_t *list_in, const int *n_in, int32_t *list_out,
                                      int *n_out, int *work_counter, const int64_t *row_ptr,
                                      const int32_t *pos_idx, const uint8_t *base_code, double *out,
                                      int32_t *match_out, int32_t *route_out) {
    if (tb.n_groups <= kGroupsSmall)
        return launch_tier<kCounts, Tier, kGroupsSmall>(ctx, tb, n_rows, list_in, n_in, list_out,
                                                        n_out, work_counter, row_ptr, pos_idx,
                                                        base_code, out, match_out, route_out);
    return launch_tier<kCounts, Tier, kGroupsLarge>(ctx, tb, n_rows, list_in, n_in, list_out, n_out,
                                                    work_counter, row_ptr, pos_idx, base_code, out,
                                                    match_out, route_out);
}

}  // namespace mxb

using namespace mxb;

extern "C" {

int mxb_phylo_pack(mxb_ctx *ctx, int32_t n_pos, int32_t n_hap, int32_t n_sym,
                   const double *hit, const double *miss, const uint8_t *ref_code,
                   const int64_t *marker_ptr, const int32_t *marker_pos_idx,
                   const uint8_t *marker_code, mxb_phylo **out) {
    MXB_REQUIRE(ctx != nullptr && out != nullptr, "NULL argument");
    MXB_REQUIRE(n_pos >= 0 && n_hap >= 0 && n_sym >= 1 && n_sym <= 254, "bad sizes");
    MXB_REQUIRE(n_pos == 0 || (hit && miss && ref_code), "NULL table");
    MXB_REQUIRE(n_hap == 0 || marker_ptr, "NULL marker_ptr");
    *out = nullptr;
    const int n_planes = n_sym + 1;
    const int n_words = (int)round_up(ceil_div(std::max(n_hap, 1), 32), 4);
    if ((int64_t)n_pos * n_planes * n_words >= ((int64_t)1 << 31)) {
        set_error("mxb_phylo_pack: bitset table too large (%d x %d x %d words)",
                  n_pos, n_planes, n_words);
        return MXB_ERR_ARG;
    }
    std::vector<uint32_t> bits;
    std::vector<double2> hm;
    try {
        bits.assign((size_t)n_pos * n_planes * n_words, 0u);
        hm.resize((size_t)n_pos);
    } catch (const std::bad_alloc &) {
        set_error("out of host memory");
        return MXB_ERR_NOMEM;
    }
    for (int p = 0; p < n_pos; ++p) {
        if (ref_code[p] >= n_sym) {
            set_error("mxb_phylo_pack: ref_code[%d]=%d outside the alphabet", p, ref_code[p]);
            return MXB_ERR_ARG;
        }
        uint32_t *plane = &bits[((size_t)p * n_planes + ref_code[p]) * n_words];
        for (int j = 0; j < n_hap; ++j) plane[j >> 5] |= 1u << (j & 31);
        hm[p] = make_double2(hit[p], miss[p]);
    }
    for (int j = 0; j < n_hap; ++j) {
        for (int64_t m = marker_ptr[j]; m < marker_ptr[j + 1]; ++m) {
            const int p = marker_pos_idx[m];
            const int c = marker_code[m];
            if (p < 0 || p >= n_pos || c >= n_sym) {
                set_error("mxb_phylo_pack: marker %lld of haplotype %d out of range",
                          (long long)m, j);
                return MXB_ERR_ARG;
            }
            for (int a = 0; a < n_sym; ++a)
                bits[((size_t)p * n_planes + a) * n_words + (j >> 5)] &= ~(1u << (j & 31));
            bits[((size_t)p * n_planes + c) * n_words + (j >> 5)] |= 1u << (j & 31);
        }
    }
    // sparse deviation lists: D = bits XOR (baseline outcome), non-zero words only.  The
    // baseline outcome of a plane is the one most haplotypes have: the marker-free outcome
    // (a == ref[p]) except where a derived allele is carried by more than half of them.
    std::vector<int32_t> dev_ptr;
    std::vector<uint2> dev_ent;
    std::vector<uint8_t> plane_base;
    try {
        dev_ptr.assign((size_t)n_pos * n_planes + 1, 0);
        plane_base.assign((size_t)n_pos * n_planes, 0);
        const int n_groups = (int)ceil_div(std::max(n_hap, 1), 32);
        const bool majority = getenv("MXB_BUILD_BASE_REF") == nullptr;
        for (int p = 0; p < n_pos; ++p) {
            for (int a = 0; a < n_planes; ++a) {
                const uint32_t *plane = &bits[((size_t)p * n_planes + a) * n_words];
                bool base_match = (a == (int)ref_code[p]);
                if (majority) {
                    int64_t n_match = 0;
                    for (int g = 0; g < n_groups; ++g) n_match += __builtin_popcount(plane[g]);
                    base_match = 2 * n_match > (int64_t)n_hap;
                }
                plane_base[(size_t)p * n_planes + a] = base_match ? 1 : 0;
                for (int g = 0; g < n_groups; ++g) {
                    const int valid = std::min(32, n_hap - g * 32);
                    const uint32_t vmask = valid >= 32 ? 0xFFFFFFFFu
                                           : (valid <= 0 ? 0u : ((1u << valid) - 1u));
                    const uint32_t d = (plane[g] ^ (base_match ? 0xFFFFFFFFu : 0u)) & vmask;
                    if (d) dev_ent.push_back(make_uint2((uint32_t)g, d));
                }
                dev_ptr[(size_t)p * n_planes + a + 1] = (int32_t)dev_ent.size();
            }
        }
    } catch (const std::bad_alloc &) {
        set_error("out of host memory");
        return MXB_ERR_NOMEM;
    }
    MXB_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<mxb_phylo> ph(new (std::nothrow) mxb_phylo());
    if (!ph) { set_error("out of host memory"); return MXB_ERR_NOMEM; }
    ph->ctx = ctx;
    ph->n_pos = n_pos;
    ph->n_hap = n_hap;
    ph->n_sym = n_sym;
    ph->n_words = n_words;
    ph->n_dev = (int64_t)dev_ent.size();
    if (!bits.empty()) {
        // [bits][hit, miss][plane baselines][deviation lists: offsets, entries]
        MXB_TRY(ph->mem.alloc_parts(ctx, "mxb_phylo_pack", [&](Carve &c) {
            ph->bits = c.part<uint32_t>(bits.size());
            ph->hitmiss = c.part<double2>(hm.size());
            ph->plane_base = c.part<uint8_t>(std::max<size_t>(1, plane_base.size()));
            ph->dev_ptr = c.part<int32_t>(dev_ptr.size());
            ph->dev_ent = c.part<uint2>(std::max<size_t>(1, dev_ent.size()));
        }));
        cudaStream_t s = ctx->stream;
        MXB_CUDA(cudaMemcpyAsync(ph->bits, bits.data(), bits.size() * sizeof(uint32_t),
                                 cudaMemcpyHostToDevice, s));
        MXB_CUDA(cudaMemcpyAsync(ph->hitmiss, hm.data(), hm.size() * sizeof(double2),
                                 cudaMemcpyHostToDevice, s));
        MXB_CUDA(cudaMemcpyAsync(ph->plane_base, plane_base.data(), plane_base.size(),
                                 cudaMemcpyHostToDevice, s));
        MXB_CUDA(cudaMemcpyAsync(ph->dev_ptr, dev_ptr.data(), dev_ptr.size() * sizeof(int32_t),
                                 cudaMemcpyHostToDevice, s));
        if (!dev_ent.empty())
            MXB_CUDA(cudaMemcpyAsync(ph->dev_ent, dev_ent.data(), dev_ent.size() * sizeof(uint2),
                                     cudaMemcpyHostToDevice, s));
        MXB_CUDA(cudaStreamSynchronize(s));
    }
    *out = ph.release();
    return MXB_OK;
}

int mxb_phylo_destroy(mxb_phylo *ph) {
    if (!ph) return MXB_OK;
    cudaSetDevice(ph->ctx->device);
    delete ph;   // (gives its tables back)
    return MXB_OK;
}

int mxb_build_matrix(mxb_ctx *ctx, const mxb_phylo *ph, int64_t n_rows,
                     const int64_t *row_ptr, const int32_t *pos_idx,
                     const uint8_t *base_code, double *out_host, int32_t *match_host,
                     int32_t *route_host, mxb_matrix **out_dev, float *elapsed_ms) {
    MXB_REQUIRE(ctx != nullptr && ph != nullptr, "NULL handle");
    MXB_REQUIRE(n_rows >= 0, "negative n_rows");
    MXB_REQUIRE(n_rows == 0 || row_ptr != nullptr, "row_ptr is NULL");
    if (out_dev) *out_dev = nullptr;
    if (elapsed_ms) *elapsed_ms = 0.f;
    MXB_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_obs = n_rows ? row_ptr[n_rows] : 0;
    MXB_REQUIRE(n_obs == 0 || (pos_idx && base_code), "NULL observation arrays");
    MXB_REQUIRE(n_obs == 0 || ph->n_pos > 0, "observations but no positions");

    mxb_matrix *mat = nullptr;
    MXB_TRY(mxb_matrix_alloc(ctx, n_rows, ph->n_hap, &mat));
    std::unique_ptr<mxb_matrix, decltype(&mxb_matrix_destroy)> m(mat, mxb_matrix_destroy);
    const size_t cells = (size_t)n_rows * (size_t)ph->n_hap;
    Prefault fault_out, fault_match;  // first-touch the result pages while the GPU works
    if (cells) {
        if (out_host) fault_out.start(out_host, cells * sizeof(double));
        if (match_host) fault_match.start(match_host, cells * sizeof(int32_t));
        // class kernel (two tiers) when its shared-memory layouts fit, else the dense kernel
        const bool counts = match_host != nullptr;
        const int n_groups = (int)ceil_div(ph->n_hap, 32);
        const bool use_class = getenv("MXB_BUILD_DENSE") == nullptr &&
                               n_groups <= kGroupsLarge && n_rows < ((int64_t)1 << 31);
        // MXB_BUILD_TIERS=2 skips tier 1 (cross-check of the large-pool launch)
        const char *tiers_env = getenv("MXB_BUILD_TIERS");
        const bool two_tiers = !(tiers_env && strcmp(tiers_env, "2") == 0);
        // [row offsets][observations: positions, codes][match counts][class kernel: overflow,
        // routes]; d_overflow[0] = number of rows deferred to tier 2, [1], [2] = the work counters
        // of the two launches, [3..] = the deferred rows
        DevBlock buf;
        int64_t *d_row_ptr = nullptr;
        int32_t *d_pos = nullptr, *d_match = nullptr, *d_overflow = nullptr, *d_route = nullptr;
        uint8_t *d_code = nullptr;
        MXB_TRY(buf.alloc_parts(ctx, "mxb_build_matrix", [&](Carve &c) {
            d_row_ptr = c.part<int64_t>(n_rows + 1);
            if (n_obs) {
                d_pos = c.part<int32_t>(n_obs);
                d_code = c.part<uint8_t>(n_obs);
            }
            if (counts) d_match = c.part<int32_t>(cells);
            if (use_class) d_overflow = c.part<int32_t>(n_rows + 3);
            if (use_class && route_host) d_route = c.part<int32_t>(n_rows);
        }));
        Events ev;   // around the kernels
        MXB_TRY(ev.create(2, cudaEventDefault, "mxb_build_matrix"));
        cudaStream_t s = ctx->stream;
        MXB_CUDA(cudaMemcpyAsync(d_row_ptr, row_ptr, (n_rows + 1) * sizeof(int64_t),
                                 cudaMemcpyHostToDevice, s));
        if (n_obs) {
            MXB_CUDA(cudaMemcpyAsync(d_pos, pos_idx, n_obs * sizeof(int32_t), cudaMemcpyHostToDevice, s));
            MXB_CUDA(cudaMemcpyAsync(d_code, base_code, n_obs * sizeof(uint8_t), cudaMemcpyHostToDevice, s));
        }
        if (use_class) {
            MXB_CUDA(cudaMemsetAsync(d_overflow, 0, 3 * sizeof(int32_t), s));
            // rows tier 1 finishes without dense groups stay 0
            if (d_route) MXB_CUDA(cudaMemsetAsync(d_route, 0, n_rows * sizeof(int32_t), s));
        } else if (route_host) {
            std::fill(route_host, route_host + n_rows, 3);
        }
        MXB_CUDA(cudaEventRecord(ev[0], s));
        if (use_class) {
            BuildTables tb;
            tb.bits = ph->bits;
            tb.hitmiss = ph->hitmiss;
            tb.plane_base = ph->plane_base;
            tb.dev_ptr = ph->dev_ptr;
            tb.dev_ent = ph->dev_ent;
            tb.n_planes = ph->n_sym + 1;
            tb.n_words = ph->n_words;
            tb.n_hap = ph->n_hap;
            tb.n_groups = n_groups;
            int *ov_count = reinterpret_cast<int *>(d_overflow);
            int32_t *ov_list = d_overflow + 3;
            cudaError_t e = cudaSuccess;
            if (two_tiers) {
                e = counts ? launch_tier_groups<true, Tier1>(ctx, tb, n_rows, nullptr, nullptr,
                                                             ov_list, ov_count, ov_count + 1,
                                                             d_row_ptr, d_pos, d_code, m->data,
                                                             d_match, d_route)
                           : launch_tier_groups<false, Tier1>(ctx, tb, n_rows, nullptr, nullptr,
                                                              ov_list, ov_count, ov_count + 1,
                                                              d_row_ptr, d_pos, d_code, m->data,
                                                              d_match, d_route);
            }
            const int32_t *in2 = two_tiers ? ov_list : nullptr;
            const int *n_in2 = two_tiers ? ov_count : nullptr;
            if (e == cudaSuccess)
                e = counts ? launch_tier_groups<true, Tier2>(ctx, tb, n_rows, in2, n_in2, nullptr,
                                                             nullptr, ov_count + 2, d_row_ptr,
                                                             d_pos, d_code, m->data, d_match,
                                                             d_route)
                           : launch_tier_groups<false, Tier2>(ctx, tb, n_rows, in2, n_in2, nullptr,
                                                              nullptr, ov_count + 2, d_row_ptr,
                                                              d_pos, d_code, m->data, d_match,
                                                              d_route);
            if (e != cudaSuccess) {
                cudaGetLastError();
                set_error("mxb_build_matrix: %s", cudaGetErrorString(e));
                return MXB_ERR_CUDA;
            }
            ctx->launches--;  // counted once more below
        } else {
            const int grid = (int)std::min<int64_t>(n_rows, (int64_t)ctx->num_sms * 4);
            build_matrix_dense_kernel<<<grid, kBuildThreads, 0, s>>>(
                ph->bits, ph->hitmiss, ph->n_sym + 1, ph->n_words, ph->n_hap, n_rows,
                d_row_ptr, d_pos, d_code, m->data, d_match);
        }
        ctx->launches++;
        MXB_CUDA(cudaGetLastError());
        MXB_CUDA(cudaEventRecord(ev[1], s));
        if (d_route)
            MXB_CUDA(cudaMemcpyAsync(route_host, d_route, n_rows * sizeof(int32_t),
                                     cudaMemcpyDeviceToHost, s));
        // pageable results leave through the staged copy engine (api.cu)
        if (out_host) {
            fault_out.join();
            MXB_TRY(copy_d2h(ctx, out_host, m->data, cells * sizeof(double)));
        }
        if (match_host) {
            fault_match.join();
            MXB_TRY(copy_d2h(ctx, match_host, d_match, cells * sizeof(int32_t)));
        }
        MXB_CUDA(cudaStreamSynchronize(s));
        if (elapsed_ms) MXB_CUDA(cudaEventElapsedTime(elapsed_ms, ev[0], ev[1]));
    }
    if (out_dev) *out_dev = m.release();
    return MXB_OK;
}

}  // extern "C"
