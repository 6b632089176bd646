/*
 * mixemt_b200.h -- C-ABI of the B200-native numeric core for svohr/mixemt.
 *
 * The reference has no FFI of its own (it is pure Python); the drop-in
 * boundary is two module attributes (SURVEY.md section 8b):
 *
 *   mixemt.preprocess.build_em_matrix(refseq, phylo, reads, haplogroups, args)
 *       reference: mixemt/preprocess.py:177-198
 *   mixemt.em.run_em(read_hap_mat, weights, args)
 *       reference: mixemt/em.py:94-165
 *   (and, for test parity) mixemt.em.em_step(...)   mixemt/em.py:57-91
 *
 * The Python host layer (mixemt_b200/preprocess.py, mixemt_b200/em.py) keeps
 * those signatures and binds the entry points below with ctypes.  Every entry
 * point is extern "C", takes plain pointers and sizes, returns an int status
 * (MXB_OK == 0) and never throws; mxb_last_error() returns the message of the
 * last failing call on the calling thread.  Host buffers are caller-owned;
 * opaque handles are library-owned and released by the matching *_destroy.
 *
 * There is no CPU fallback: every compute entry point needs a CUDA device and
 * fails with MXB_ERR_CUDA when there is none.
 */
#ifndef MIXEMT_B200_H
#define MIXEMT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MXB_ABI_VERSION 2

enum {
    MXB_OK = 0,
    MXB_ERR_CUDA = 1,      /* CUDA runtime / NCCL failure (message has detail)   */
    MXB_ERR_ARG = 2,       /* bad argument (NULL, negative size, bad handle)     */
    MXB_ERR_VALUE = 3,     /* malformed signature -> Python ValueError           */
    MXB_ERR_KEY = 4,       /* unknown variant position -> Python KeyError        */
    MXB_ERR_NOMEM = 5,     /* host or device allocation failed                   */
    MXB_ERR_RANGE = 6      /* EM left the representable range (non-finite sums)  */
};

typedef struct mxb_ctx mxb_ctx;       /* one device + stream + scratch + (optional) NCCL comm */
typedef struct mxb_phylo mxb_phylo;   /* packed haplotype bitsets + per-position log tables   */
typedef struct mxb_matrix mxb_matrix; /* device-resident row-major fp64 N x H matrix          */
typedef struct mxb_em mxb_em;         /* EM session over one matrix (row shard)               */

/* ---- library -------------------------------------------------------------- */
int mxb_abi_version(void);
const char *mxb_last_error(void);
/* Number of visible CUDA devices (0 when there is no GPU / no driver). */
int mxb_device_count(void);

/* ---- context -------------------------------------------------------------- */
int mxb_ctx_create(int device, mxb_ctx **out);
int mxb_ctx_destroy(mxb_ctx *ctx);
/* Launch on an externally owned cudaStream_t (e.g. torch's current stream). */
int mxb_ctx_set_stream(mxb_ctx *ctx, void *cuda_stream);
int mxb_ctx_synchronize(mxb_ctx *ctx);
/* Device blocks of >= 1 MiB freed through this context are kept for reuse,
 * up to MXB_CACHE_MB (default: a quarter of the device memory; 0 disables) -- cudaMalloc
 * and cudaFree of multi-GB blocks are slow and jittery.  mxb_ctx_trim hands them back. */
int mxb_ctx_trim(mxb_ctx *ctx);
/* Bytes of device memory this context has handed out and not yet freed (live), and bytes it
 * keeps cached for reuse.  MXB_DEBUG_FAIL_ALLOC=k, read by mxb_ctx_create, makes the k-th
 * device allocation of the new context fail as out of memory (error-path tests). */
int mxb_ctx_mem_stats(const mxb_ctx *ctx, int64_t *live_bytes, int64_t *cached_bytes);
/* Pinned host memory for matrix-sized results (no counterpart in the reference, which returns
 * numpy arrays: em.py:111, preprocess.py:183).  An N x H result that lives in one of these
 * blocks is downloaded by one DMA without staging copy or page faults.  Blocks are pooled
 * process-wide: mxb_host_free keeps them for the next mxb_host_alloc of about the same size
 * (up to MXB_PINNED_CACHE_MB, default a quarter of the host memory), mxb_host_trim releases
 * them.  mxb_host_alloc leaves *out NULL (and returns MXB_OK) when pinning fails or when
 * only_if_cached is set and no pooled block fits: the caller then uses pageable memory.
 * mxb_host_reserve pins `count` blocks ahead of time (pinning costs about a second per 6 GB). */
int mxb_host_alloc(size_t bytes, int only_if_cached, void **out);
int mxb_host_free(void *ptr);
int mxb_host_reserve(size_t bytes, int count);
int mxb_host_trim(void);
/* Stage times of the one-call entry points since the last mxb_stage_timing(1), milliseconds:
 * [0] host->device copies of matrices, [1] session set-up (class tiles or fp64 rows, result
 * allocation), [2] EM iterations, [3] read-matrix kernels, [4] device->host copy of the
 * result, [5] release.  Bench instrumentation; off by default (adds stream synchronisations). */
int mxb_stage_timing(int on);
int mxb_stage_times(double *ms_out, int n);
/* Kernel launches issued through this context since creation (bench evidence). */
int64_t mxb_ctx_launch_count(const mxb_ctx *ctx);
/* Multi-GPU: one process per GPU.  Rank 0 calls mxb_comm_unique_id, the host
 * layer broadcasts the 128 bytes (torch.distributed), every rank calls
 * mxb_comm_init.  After that mxb_em_* sessions created with sharded != 0
 * all-reduce the H column sums once per EM iteration (ncclAllReduce, fp64). */
int mxb_comm_unique_id(void *id128);
int mxb_comm_init(mxb_ctx *ctx, const void *id128, int rank, int world);
int mxb_comm_destroy(mxb_ctx *ctx);
/* 1 when the ranks of the comm mapped each other's mailboxes (CUDA IPC over
 * NVLink) and the per-iteration exchange of the column sums is fused into the
 * EM tail kernel as peer stores; 0 when ncclAllReduce is used instead. */
int mxb_comm_p2p_enabled(const mxb_ctx *ctx);
/* In-place sum / max all-reduce of a host fp64 vector across the comm
 * (restart fan-out: sum of log-proportions, reference em.py:155). */
int mxb_comm_allreduce_host(mxb_ctx *ctx, double *buf, int64_t n, int op_is_max);

/* ---- signatures -> CSR (host only; replaces preprocess.pos_obs_from_sig,
 *      mixemt/preprocess.py:151-160, 26 us/row in Python) -------------------- */
/* Count observations (comma-separated fields) of every signature.
 * buf: concatenated UTF-8 signatures; offsets[n_rows+1] delimit them.
 * row_ptr[n_rows+1] receives the exclusive prefix sum. */
int mxb_sig_count(const char *buf, const int64_t *offsets, int64_t n_rows,
                  int64_t *row_ptr);
/* Parse "pos:base,pos:base,...".  pos2idx[pos] maps a 0-based reference
 * position to its index in the packed position table (-1: not a variant
 * position).  sym2code[256] maps a single-byte base to its symbol code
 * (255: never matches).  On MXB_ERR_VALUE / MXB_ERR_KEY *bad_row is the first
 * offending row, in the order the reference would have hit it. */
int mxb_sig_parse(const char *buf, const int64_t *offsets, int64_t n_rows,
                  const int32_t *pos2idx, int64_t pos2idx_len,
                  const uint8_t *sym2code, const int64_t *row_ptr,
                  int32_t *pos_idx, uint8_t *base_code,
                  int64_t *bad_row, int64_t *bad_pos);

/* ---- fragments -> unique signatures (host only; replaces the string round trip of
 *      preprocess.read_signature / reduce_reads and the sorted()/weights of
 *      build_em_input, mixemt/preprocess.py:142-148, :163-174, :218-220) ---------- */
typedef struct mxb_sigset mxb_sigset;
/* frag_ptr[n_frag+1] delimits each fragment's observations: pos[] 0-based reference
 * positions ascending inside a fragment (like sorted(obs_by_pos)), base[] ASCII.
 * Equal observation lists collapse into one signature; rows are ordered like the
 * reference orders them (string sort of "pos:base,pos:base,..."). */
int mxb_reduce_reads(const int64_t *frag_ptr, const int32_t *pos, const uint8_t *base,
                     int64_t n_frag, mxb_sigset **out);
int mxb_sigset_sizes(const mxb_sigset *ss, int64_t *n_sig, int64_t *n_obs, int64_t *n_chars);
/* Every output is nullable.  row_ptr[n_sig+1], pos/base[n_obs]: CSR of the rows;
 * weights[n_sig]: fragments per row; first_frag[n_sig]: lowest fragment index of the
 * row; sig_of_frag[n_frag]: row of every fragment; frag_order[n_frag]: fragment
 * indexes grouped by row (ascending inside a row, weights[] delimit the groups);
 * strings[n_chars] + str_offsets[n_sig+1]: the signature strings, concatenated. */
int mxb_sigset_export(const mxb_sigset *ss, int64_t *row_ptr, int32_t *pos, uint8_t *base,
                      int64_t *weights, int64_t *first_frag, int64_t *sig_of_frag,
                      int64_t *frag_order, char *strings, int64_t *str_offsets);
int mxb_sigset_destroy(mxb_sigset *ss);

/* ---- haplotype tables (replaces HapVarBaseMatrix, preprocess.py:23-96) ----- */
/* n_sym symbols (codes 0..n_sym-1).  hit[p] = log(1-mut_prob), miss[p] =
 * log(mut_prob/3), computed by the host with math.log so they are
 * bit-identical to the reference's (preprocess.py:75-95).  ref_code[p] is the
 * code of refseq[pos]; markers are CSR per haplotype column
 * (marker_ptr[n_hap+1], marker_pos_idx, marker_code). */
int mxb_phylo_pack(mxb_ctx *ctx, int32_t n_pos, int32_t n_hap, int32_t n_sym,
                   const double *hit, const double *miss,
                   const uint8_t *ref_code, const int64_t *marker_ptr,
                   const int32_t *marker_pos_idx, const uint8_t *marker_code,
                   mxb_phylo **out);
int mxb_phylo_destroy(mxb_phylo *phylo);

/* ---- kernel 1: matrix build (replaces build_em_matrix, preprocess.py:177) --- */
/* CSR rows -> fp64 N x H log-likelihood matrix.  out_host (nullable) receives
 * the matrix, match_host (nullable) the int32 per-cell match counts
 * (mismatches = K_i - matches), route_host (nullable) the path that finished
 * each row: route_host[i] = path + 4 * (number of 32-column groups the class
 * kernel walked with its per-group dense loop), path 0 = class kernel tier 1,
 * 1 = tier 2, 2 = tier 2's dense row walk, 3 = dense kernel (H > 8192 or
 * MXB_BUILD_DENSE=1).  Nothing is written to it when H == 0.  out_dev
 * (nullable) keeps the matrix resident.  elapsed_ms (nullable) = device time
 * of the build kernel alone. */
int mxb_build_matrix(mxb_ctx *ctx, const mxb_phylo *phylo, int64_t n_rows,
                     const int64_t *row_ptr, const int32_t *pos_idx,
                     const uint8_t *base_code, double *out_host,
                     int32_t *match_host, int32_t *route_host,
                     mxb_matrix **out_dev, float *elapsed_ms);

/* ---- device matrices ------------------------------------------------------- */
int mxb_matrix_alloc(mxb_ctx *ctx, int64_t n_rows, int64_t n_cols, mxb_matrix **out);
int mxb_matrix_upload(mxb_ctx *ctx, const double *host, int64_t n_rows,
                      int64_t n_cols, mxb_matrix **out);
int mxb_matrix_download(mxb_ctx *ctx, const mxb_matrix *m, double *host);
int mxb_matrix_shape(const mxb_matrix *m, int64_t *n_rows, int64_t *n_cols);
/* Raw device pointer (for torch interop / tests); row stride == n_cols. */
void *mxb_matrix_data(const mxb_matrix *m);
/* Row-wise argmax (first maximum, like numpy.argmax axis=1;
 * consumers assemble.py:115, stats.py:39). */
int mxb_matrix_argmax_rows(mxb_ctx *ctx, const mxb_matrix *m, int64_t *out_host);
int mxb_matrix_destroy(mxb_matrix *m);

/* ---- consumers of the EM result, kept on the device (SURVEY.md 8f N2-N4) ---- */
/* preprocess.reduce_em_matrix (preprocess.py:230-251): out[i][k] = src[i][cols[k]]. */
int mxb_matrix_gather_cols(mxb_ctx *ctx, const mxb_matrix *src, const int64_t *cols,
                           int64_t n_out, mxb_matrix **out);
/* assemble._find_contribs_from_reads (assemble.py:102-124) / stats.report_read_votes
 * (stats.py:34-46): votes_out[j] = sum of weights[i] over rows whose first row maximum
 * is column j; argmax_out (nullable) receives the row maxima positions. */
int mxb_matrix_vote_count(mxb_ctx *ctx, const mxb_matrix *m, const int64_t *weights,
                          int64_t *votes_out, int64_t *argmax_out);
/* assemble._find_contribs_from_reads (assemble.py:102-124) over a row shard whose first row
 * is global row row0: votes_out[j] as mxb_matrix_vote_count; first_out[j] = smallest
 * row0 + r whose first row maximum is column j, -1 when no row's maximum is j.  Two launches
 * (row argmax, then integer-atomic votes and minima); only the 2 x n_cols results are copied
 * back, so rows-mode ranks merge them with an O(H) all-reduce (consumers.py). */
int mxb_matrix_vote_first(mxb_ctx *ctx, const mxb_matrix *m, const int64_t *weights,
                          int64_t row0, int64_t *votes_out, int64_t *first_out);
/* assemble.assign_read_indexes (assemble.py:267-334): per row the two contributor
 * columns with the highest read_mix[i][c] - con_lnprops[k]; assign_out[i] = k of the
 * best one when it leads the runner-up by at least ln_min_fold, else -1 (unassigned);
 * with a single contributor every row is assigned to it. */
int mxb_assign_reads(mxb_ctx *ctx, const mxb_matrix *read_mix, const int64_t *con_cols,
                     const double *con_lnprops, int32_t n_con, double ln_min_fold,
                     int32_t *assign_out);
/* Row-range transfers (streaming .npy save/load, bin/mixemt:168-245). */
int mxb_matrix_download_rows(mxb_ctx *ctx, const mxb_matrix *m, int64_t row0, int64_t n_rows,
                             double *host);
int mxb_matrix_upload_rows(mxb_ctx *ctx, mxb_matrix *m, int64_t row0, int64_t n_rows,
                           const double *host);

/* ---- kernel 2: EM (replaces em_step / run_em, em.py:57-165) ---------------- */
/* Session over one matrix shard.  weights[n_rows] (fp64).  sharded != 0 and a
 * comm on ctx: rows are a shard, column sums are all-reduced every iteration.
 * The session keeps L = exp(M - rowmax) either as class tiles (per 128-row batch the
 * bit-identical columns collapse into classes: exact, several times fewer bytes and FMAs;
 * needs rows in the reference's order, preprocess.py:219, to pay off) or, when the matrix does
 * not compress, as fp64 rows (see mxb_em_pass_bytes).  What an iteration runs (the pass over
 * tiles, fp64 rows or the general path, its restart slots and its tail) is decided once here
 * (em.cu: decide_form).  In a sharded session the call is collective: every rank zeroes its
 * peer mailboxes behind a barrier. */
int mxb_em_create(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                  int sharded, mxb_em **out);
int mxb_em_destroy(mxb_em *em);
/* Set the current log-proportions (em.py:123-124, host draws the Dirichlet). */
int mxb_em_set_lnprops(mxb_em *em, const double *lnprops);
/* Iterate em_step + converged (em.py:126-143) from the proportions mxb_em_set_lnprops set,
 * until sum|dprops| < tol or max_iter (max_iter <= 0 runs no iteration).  iters_out =
 * iterations run; converged_out = 1/0.  Driven by the same host loop as mxb_run_em's restarts.
 * An iteration in which a row's mixture likelihood underflows in linear space is redone in log
 * space (em.py:80-89); in a sharded session all ranks redo it together, so the call stays
 * collective. */
int mxb_em_iterate(mxb_em *em, int64_t max_iter, double tol,
                   int64_t *iters_out, int32_t *converged_out);
/* Bytes the kernels of one EM iteration read from HBM, and how the rows are stored:
 * *layout = -1 when the session keeps L as fp64 rows (N x ld x 8 bytes per pass), 0 when it
 * runs over class tiles (csrc/em_tiles.cuh: tiles + class maps + class vectors).
 * Measurement aid of bench.py; no counterpart in the reference (em.py:57-91 re-reads the
 * whole matrix several times). */
int mxb_em_pass_bytes(const mxb_em *em, int64_t *bytes_per_pass, int64_t *layout);

/* Host only (no device needed): the plan of the class-tile pass that mxb_em_create makes for
 * n_batches batches of 128 rows (the last one shorter, n_rows in all) whose columns fall into
 * n_cls[b] classes, on a GPU with num_sms SMs (csrc/tile_plan.h).  seg_out (nullable,
 * seg_cap x 8 int32) receives per segment, in CTA order, {CTA, batch, first row inside the
 * batch, rows, rows per copy, copies, log2 of the threads per row, row stride in doubles};
 * errors = violated invariants (0).  For the CPU tests of the host logic; no counterpart in the
 * reference, whose em_step (em.py:57-91) is three numpy expressions over the whole matrix. */
int mxb_tile_plan(const int32_t *n_cls, int64_t n_batches, int64_t n_rows, int32_t num_sms,
                  int32_t *seg_out, int64_t seg_cap, int32_t *n_cta, int32_t *n_seg,
                  int32_t *n_slots, int32_t *slot_bytes, int32_t *errors);

/* Exactly n_iter iterations without convergence test or host sync (bench); MXB_ERR_RANGE
 * when fewer ran (a row's mixture likelihood underflowed and the run stopped for the
 * log-space step, which only mxb_em_iterate and the one-call forms below take);
 * elapsed_ms (nullable) = device time between first and last launch,
 * pass_ms (nullable) = summed device time from the first pass kernel of an iteration to
 * its tail kernel (class sums + pass + gather for tiles; adds an event pair per iteration). */
int mxb_em_iterate_fixed(mxb_em *em, int64_t n_iter, float *elapsed_ms,
                         float *pass_ms);
/* Per-kernel attribution of an iteration (bench instrumentation): n_iter iterations with an
 * event between the kernels; ms_out[4] = average milliseconds of {class sums (tile_pi_kernel),
 * pass (tile_pass_kernel or em_pass_fast_kernel), gather (tile_gather_kernel), tail
 * (em_finish_kernel)}; the first and third are 0 for a session over fp64 rows. */
int mxb_em_profile(mxb_em *em, int64_t n_iter, float *ms_out);
/* which: 0 = latest log-proportions (new_props), 1 = the ones before them. */
int mxb_em_get_lnprops(mxb_em *em, int which, double *out);
/* Read matrix from the *previous* log-proportions (em.py:130 / F5), written or
 * folded into dst: mode 0 = store, 1 = dst = logaddexp(dst, Z) (em.py:156).
 * sub_log != 0.0 subtracts it afterwards (em.py:161, log(n_multi)). */
int mxb_em_read_mix(mxb_em *em, mxb_matrix *dst, int mode, double sub_log);

/* One-call forms with host buffers (what a reference-side FFI would bind). */
/* em.run_em (em.py:94-165): init_lnprops[n_multi*n_cols] drawn by the host;
 * props_out[n_cols] linear scale; read_mix_out (nullable) N x H log scale;
 * iters_out[n_multi], converged_out[n_multi] (nullable).  One scheduler runs the restarts,
 * one per pass or, over fp64 rows, two per pass (MXB_EM_NO_BATCH=1: one), and combines them in
 * restart order as em.py:145-163 does; with max_iter <= 0 every restart hands back its init.
 * Iterations whose row likelihoods underflow in linear space are redone in log space in every
 * kind of session (one GPU or row-sharded), as the reference computes them. */
/* flags: MXB_EM_SHARDED = the rows are this rank's shard of a larger matrix
 * (column sums all-reduced over the ctx comm every iteration);
 * MXB_EM_RAW = skip the final averaging (em.py:158-163): props_out then holds
 * the plain sum of the restarts' log-proportions and read_mix the plain
 * logaddexp fold, for combining restart subsets run on different GPUs. */
#define MXB_EM_SHARDED 1
#define MXB_EM_RAW 2
int mxb_run_em(mxb_ctx *ctx, const double *read_hap_mat, const double *weights,
               int64_t n_rows, int64_t n_cols, const double *init_lnprops,
               int32_t n_multi, int64_t max_iter, double tol, int32_t flags,
               double *props_out, double *read_mix_out,
               int64_t *iters_out, int32_t *converged_out);
/* Same, matrix already on the device (kept there by mxb_build_matrix);
 * read_mix_dev (nullable) keeps the result matrix resident as well. */
int mxb_run_em_dev(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                   const double *init_lnprops, int32_t n_multi,
                   int64_t max_iter, double tol, int32_t flags,
                   double *props_out, double *read_mix_out,
                   mxb_matrix **read_mix_dev,
                   int64_t *iters_out, int32_t *converged_out);
/* Cross-rank fold of per-rank read matrices (restart fan-out, em.py:156 and :161 across
 * ranks): m = logaddexp over ranks (in rank order) of m - sub_log, in place on every rank.
 * All-to-all of row shards (ncclSend/ncclRecv), local fold, shards broadcast back. */
int mxb_matrix_fold_ranks(mxb_ctx *ctx, mxb_matrix *m, double sub_log);
/* em.em_step (em.py:57-91): one E+M step, read_mix_out written in full.  The same as
 * mxb_run_em with MXB_EM_RAW, one restart, max_iter 1 and tol -1: new_props_out receives the
 * new log-proportions, read_mix_out the read matrix of ln_props. */
int mxb_em_step(mxb_ctx *ctx, const double *read_hap_mat, const double *weights,
                const double *ln_props, int64_t n_rows, int64_t n_cols,
                double *read_mix_out, double *new_props_out);

/* ---- nonparametric bootstrap of the proportions (no counterpart in the reference) ----
 * Replicate b draws W = sum(weights) fragments with replacement from the rows (row i carries
 * weights[i] fragments; the weights must be finite non-negative integers with 1 <= W < 2^32,
 * else MXB_ERR_VALUE): fragment f takes r = x0 | x1 << 32 of Philox4x32-10 with counter
 * {f_lo, f_hi, b, 0} and key {seed_lo, seed_hi}, t = mulhi64(r, W), and the first row i whose
 * inclusive prefix sum of the weights exceeds t.
 * counts_out[k][i] = draws of row i by replicate boot0 + k (k < n_boot). */
int mxb_boot_counts(mxb_ctx *ctx, const double *weights, int64_t n_rows, uint64_t seed,
                    int64_t boot0, int64_t n_boot, uint32_t *counts_out);
/* Replicates boot0 .. boot0 + n_boot - 1 of the fit start_lnprops (log-proportions, -inf for a
 * zero): replicate b's row of lnprops_out is the final log-proportions of one run_em restart
 * (em.py:117-143, with max_iter, tol, the swap back of em.py:141-143 and max_iter <= 0 handing
 * back the start) on the matrix with replicate b's counts as weights, started from
 * start_lnprops; iters_out / converged_out per replicate.  A replicate's result depends only on
 * (m, weights, start_lnprops, seed, b, max_iter, tol).  Over class tiles several replicates
 * iterate per launch; slots_out (nullable) = how many (chosen from the matrix by
 * mxb_boot_slots' rule), 1 over fp64 rows. */
int mxb_em_bootstrap(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                     const double *start_lnprops, int64_t boot0, int64_t n_boot, uint64_t seed,
                     int64_t max_iter, double tol, double *lnprops_out, int64_t *iters_out,
                     int32_t *converged_out, int32_t *slots_out);
/* Replicate slots of a bootstrap session over class tiles with these batch class counts (as
 * mxb_tile_plan takes them): the largest power of two R <= 16 whose tile plan for num_sms / R
 * CTAs models at most R times the time of the plan for num_sms, with R * bytes_per_slot at
 * most an eighth of free_bytes (a session passes the bytes of one slot's buffers, em.cu:
 * slot_block, plus its class vectors).  Host only, for the CPU tests. */
int mxb_boot_slots(const int32_t *n_cls, int64_t n_batches, int64_t n_rows, int32_t num_sms,
                   double bytes_per_slot, double free_bytes, int32_t *slots_out);

/* ---- log-likelihood of a fit and constrained refits (no counterpart in the reference) ----
 * out[k] = sum_i weights[i] * logsumexp_j(M_ij + lnprops[k][j]) for the n_vec log-proportion
 * vectors lnprops (n_vec x H, host; not renormalised here).  -inf cells and -inf log-proportions
 * add nothing, a row without a finite term gives -inf, a row of weight 0 adds exactly 0.  Up to
 * 16 vectors share one read of m; a vector's result is the same bits whichever vectors share the
 * call.  A row that would underflow in linear space (the EM's 2^-960 rule) is redone in log
 * space.  MXB_ERR_VALUE for a NaN log-proportion.  On a row shard the result covers the shard's
 * rows (the caller adds the ranks' values). */
int mxb_matrix_loglik(mxb_ctx *ctx, const mxb_matrix *m, const double *weights,
                      const double *lnprops, int64_t n_vec, double *out);
/* n_starts refits of the same matrix and weights: row k of lnprops_out (n_starts x H) is the
 * final log-proportions of one run_em restart from starts[k] (log-proportions, -inf for a zero,
 * which stays zero), as mxb_run_em_dev with MXB_EM_RAW and n_multi 1 returns them, with
 * iters_out[k] and converged_out[k]; max_iter <= 0 hands back the starts.  Over class tiles
 * several refits iterate per launch (slots_out, nullable: how many; mxb_boot_slots' rule), over
 * fp64 rows one at a time.  MXB_ERR_VALUE before any launch for a NaN in a start or a start
 * whose proportions sum to 0. */
int mxb_em_refit(mxb_ctx *ctx, const mxb_matrix *m, const double *weights, const double *starts,
                 int64_t n_starts, int64_t max_iter, double tol, double *lnprops_out,
                 int64_t *iters_out, int32_t *converged_out, int32_t *slots_out);

#ifdef __cplusplus
}
#endif
#endif /* MIXEMT_B200_H */
