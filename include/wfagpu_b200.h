/*
 * wfagpu_b200.h -- C-ABI between the C host code and the hand-written sm_100a
 * CUDA layer (wfa-gpu_b200/csrc), plus the B200-specific extensions of the
 * public API.  Plain pointers and sizes only; no CUDA or torch types.
 *
 * This is the boundary a reference maintainer would bind instead of
 * lib/sequence_packing.cuh:27-40 (pack_sequences_gpu_async) and
 * lib/sequence_alignment.cuh:29-114 (the allocate_xxx / reset_xxx helpers,
 * launch_alignments_async, launch_alignments_distance_async, copyInResults),
 * see INTEGRATION.md.
 */
#ifndef WFAGPU_B200_H
#define WFAGPU_B200_H

#include <stddef.h>
#include <stdint.h>
#include "wfa_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Longest sequence wfagpu_add_sequences accepts (the reference: MAX_SEQ_LEN - 1 = 32767). */
/* The large tier stages both packed sequences of a pair in one CTA's shared memory (227 KB): 2 x len / 2 bytes. */
#define WFAGPU_MAX_SEQ_LEN ((size_t)220000)

/* ---------------------------------------------------------- step table --- */
/* Per-score control record.  It depends on the penalties and the step budget
 * only (the existence logic of lib/kernels/sequence_alignment_kernel.cu:584-631
 * never looks at the sequences), so the host builds it once per launch. */
#define WFAGPU_STEP_NULL 0u
#define WFAGPU_STEP_M    1u
#define WFAGPU_STEP_MDI  2u
typedef struct {
    uint32_t row_off; /* offset of this score's decision row, in 16-byte units */
    uint16_t n;       /* half width of the diagonal range [-n, n] after this step */
    uint16_t kind;    /* WFAGPU_STEP_*                                          */
} wfagpu_step_t;

/* Builds the table for scores 0 .. d_end-1 (returns d_end; tab may be NULL to
 * size it).  `arena_units` receives the number of 16-byte decision units one
 * alignment can write.  Budget rule = reference: MDI steps stop once
 * steps >= max_steps-1 (sequence_alignment_kernel.cu:584, steps starts at 1).
 * banded_win == 0: exact kernels (n = computed half width, row_off = decision-byte row of the
 * warp-per-pair and large-tier kernels; the CTA kernels keep ring snapshots instead, laid out by the device layer);
 * banded_win  > 0: banded kernels (n = number of M/I/D steps so far, rows of
 * ceil(win/16) units).  A decision row holds one byte per diagonal. */
int wfagpu_build_step_table(int x, int o, int e, int max_steps, int max_dist, int banded_win,
                            wfagpu_step_t *tab, uint64_t *arena_units);

/* Ends-free alignments (exact kernels only): every score's range is widened by `start_half_width` diagonals on both
 * sides, the half width of the start row [-pattern_begin_free, text_begin_free].  -1 if it does not fit the table. */
int wfagpu_build_step_table_span(int x, int o, int e, int max_steps, int max_dist, int start_half_width,
                                 wfagpu_step_t *tab, uint64_t *arena_units);

/* Gap-affine 2-piece penalties (exact kernels, global alignment only): a second gap component (o2, e2).  A score is
 * an M/I/D step when a gap of either piece exists (gap_i[d] = M[d - o_i - e_i] || gap_i[d - e_i]), and its half width
 * is min(#M/I/D steps, max((d - o1) / e1, (d - o2) / e2)).  With o2 = o1, e2 = e1 the table equals
 * wfagpu_build_step_table(x, o1, e1, ...).  -1 for x < 1, e1 < 1, e2 < 1 or a negative opening. */
int wfagpu_build_step_table_affine2p(int x, int o1, int e1, int o2, int e2, int max_steps, int max_dist,
                                     wfagpu_step_t *tab, uint64_t *arena_units);

/* --------------------------------------------------- gap-affine 2-piece --- */
/* WFA2-lib's `affine2p` model: a gap of L bases costs min(o1 + e1 L, o2 + e2 L), a mismatch x.  Valid: x >= 1,
 * e1, e2 >= 1, o1, o2 >= 0, the pieces in either order.  Scores do not depend on the order; on equal offsets the
 * traceback prefers piece 1 (M: D1 > D2 > X > I1 > I2; I / D: extend beats open).  Identical pieces give the
 * single-piece scores and CIGAR text byte for byte.  Global alignment only: no band, no ends-free span. */
typedef struct {
    int x, o1, e1, o2, e2;
} wfagpu_affine2p_t;

/* ---------------------------------------------------------- ends-free --- */
/* Ends-free (semi-global) span of a call, WFA2-lib's `ends-free` order.  All zero = global alignment.  Per pair each
 * value is clamped to the sequence it applies to.  The score is the gap-affine cost of the aligned part: leading and
 * trailing pattern / text bases up to these counts are free.  The CIGAR still covers both full sequences: the free
 * parts print as leading / trailing I (text) or D (pattern) runs, joined with a gap run of the same letter next to
 * them. */
typedef struct {
    int pattern_begin_free, pattern_end_free, text_begin_free, text_end_free;
} wfagpu_span_t;

/* ------------------------------------------------------- device batches --- */
/* One pair as the device sees it (built by the host from sequence_pair_t). */
typedef struct {
    uint32_t p_ascii; /* byte offset of the pattern in the batch ASCII buffer */
    uint32_t t_ascii;
    uint32_t p_word;  /* u32 offset of the packed pattern in the packed buffer (multiple of 4) */
    uint32_t t_word;
    uint32_t plen;
    uint32_t tlen;
    uint32_t flags;   /* WFAGPU_PAIR_* (has_N written by the pack kernel)      */
    uint32_t reserved;
} wfagpu_pair_t;
#define WFAGPU_PAIR_HAS_N 1u

/* Per-pair result record written by the alignment kernels. */
typedef struct {
    int32_t distance;  /* score if finished                                     */
    uint32_t status;   /* WFAGPU_ST_*                                           */
    uint32_t ops_off;  /* u32 offset of the packed op stream in the ops pool    */
    uint32_t n_ops;    /* number of 2-bit backtrace ops, stored newest first    */
} wfagpu_pair_out_t;
#define WFAGPU_ST_FINISHED   1u
#define WFAGPU_ST_OVERBUDGET 2u /* needs a larger wavefront budget (re-dispatch) */
#define WFAGPU_ST_NEEDS_ASCII 4u /* flagged by the packer: byte-compare kernel    */
#define WFAGPU_ST_FAILED 8u      /* the GPU cannot finish this pair (> 60000 wavefront steps or wavefronts wider than
                                  * one CTA holds); set by wfagpu_device_download, the other pairs keep their results */

/* Where a pair's CIGAR text sits in the text pool returned by wfagpu_device_download_text. */
typedef struct {
    uint32_t off; /* byte offset in the text pool */
    uint32_t len; /* characters (no terminator); 0 = none */
} wfagpu_cigar_ref_t;

typedef struct wfagpu_device wfagpu_device_t; /* opaque: streams, buffers, arenas of one GPU */

typedef struct {
    int x, o, e;
    int max_steps;   /* budget of the first pass (reference `max_error`)        */
    int band;        /* <=0 exact                                               */
    int band_width;  /* banded window width (reference threads_per_block)       */
    int with_cigar;
    int threads_hint;
    int workers_hint;
    int o2, e2;      /* gap-affine 2-piece: second gap piece; e2 == 0 = one piece (o, e) */
    int with_ends;   /* ends-free, with_cigar == 0: also find where every alignment begins (k_begin of
                      * wfagpu_device_download_ends); 0 = score only, as before */
} wfagpu_plan_t;

/* Statistics of the last batch (kernel times from CUDA events on the launch
 * stream; counts of kernels launched). */
typedef struct {
    float ms_h2d, ms_pack, ms_align, ms_d2h, ms_total;
    uint32_t launches;        /* kernels launched for this batch                */
    uint32_t redispatched;    /* pairs that needed a larger budget              */
    uint32_t ascii_pairs;     /* pairs routed to the byte-compare kernel        */
    uint64_t cells;           /* wavefront cells computed (0 unless profiling)  */
    uint64_t h2d_bytes, d2h_bytes;
    float ms_wavefront;       /* the first pass's wavefront kernel alone (0 if it ran in several sub-launches) */
    uint32_t failed_pairs;    /* pairs reported as WFAGPU_ST_FAILED                                            */
    uint32_t pending_pairs;   /* after wfagpu_device_wait: pairs the first pass left to the re-dispatch tier   */
    uint32_t n_cap, cta_threads, ctas, d_end; /* launch shape of the first pass: ring half width, CTA size, grid, score limit */
    uint32_t reserved1;
} wfagpu_batch_stats_t;

/* Leases a context of CUDA device `dev`: an idle one from the pool (with its grown buffers) or a new one; the
 * caller owns it until wfagpu_device_release.  Two leases never share streams, slots or staging buffers, so
 * threads (or two workers on one GPU) do not interfere.  NULL on failure (message on stderr); never falls
 * back to the CPU.  wfagpu_device_close_all frees every context (none may be in use). */
wfagpu_device_t *wfagpu_device_open(int dev);
void wfagpu_device_release(wfagpu_device_t *d);
void wfagpu_device_close_all(void);

/*
 * One batch on one device, in three phases on the slot's own stream (two slots
 * per device let the host overlap batch c+1's copies with batch c's kernels):
 *   upload    H2D of the batch's ASCII (pairs[i].*_ascii are offsets into
 *             `ascii`), pair descriptors and the longest-first schedule;
 *   align     pack kernel, score-bound kernel, alignment kernel (+ traceback, CIGAR text); may be
 *             repeated on a resident batch.  Returns with the alignment kernels queued; for long
 *             reads it first waits for the bound kernel (the rings of the pass are sized from the
 *             batch's own bounds: 4 bytes per pair come back to the host), the rest is asynchronous;
 *   download  waits, finishes over-budget / non-ACGT pairs on the GPU
 *             (re-dispatch with a doubled budget, byte-compare kernel) and copies
 *             out[i] and the packed op streams back (`*ops` points into pinned
 *             memory owned by the slot, valid until the slot's next download).
 * All return 0 on success; failures print to stderr -- there is no CPU path.
 */
int wfagpu_device_upload(wfagpu_device_t *d, int slot, const char *ascii, size_t ascii_bytes,
                         const wfagpu_pair_t *pairs, size_t n);
int wfagpu_device_align(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan,
                        int resident);
int wfagpu_device_download(wfagpu_device_t *d, int slot, size_t n, wfagpu_pair_out_t *out,
                           uint32_t **ops, size_t *ops_used, uint32_t *pair_flags);
/* wfagpu_device_align with an ends-free span (NULL or all zero: exactly wfagpu_device_align).  A non-zero span runs
 * the one-diagonal-per-thread kernels with decision-byte traceback on every tier and neither reads nor updates the
 * provisioning hint of global batches.  -3 for negative values or band > 0 with a non-zero span. */
int wfagpu_device_align_span(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int resident,
                             const wfagpu_span_t *span);
/* The same with one span per pair of the batch (spans[i] for pair i; NULL: global).  The batch is ends-free when any
 * pair's span is non-zero; every pair is aligned under its own span, and a pair with an all-zero span gets its global
 * alignment.  -3 as above when any pair's span is rejected. */
int wfagpu_device_align_spans(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int resident,
                              const wfagpu_span_t *spans);
/* After wfagpu_device_download of an ends-free batch: per pair {k_begin, k_end} (2 n ints), the diagonals of the
 * alignment's first and last cell: it starts at (max(0, -k_begin), max(0, k_begin)) and ends at offset
 * min(tlen, plen + k_end).  k_end is always valid; k_begin only when the batch was aligned with with_cigar or
 * with_ends (a score-only batch without with_ends holds k_begin = k_end).  Pairs that did not finish hold no record.
 * -1 for a global batch. */
int wfagpu_device_download_ends(wfagpu_device_t *d, int slot, size_t n, int32_t *ends);
/* A plan with e2 > 0 (gap-affine 2-piece, through wfagpu_device_align / _align_span / _rescore) runs the
 * one-diagonal-per-thread kernels with decision-byte traceback, no score-bound kernel (pruning uses the launch bound)
 * and neither reads nor updates the provisioning hint.  Those calls return -3 for a 2-piece plan with band > 0, a
 * non-zero span, or a negative value. */
/* Waits for the slot's stream; event-timed durations (milliseconds) of the pack kernel and of the
 * first pass of the alignment: score bounds + wavefronts + traceback + CIGAR text. */
int wfagpu_device_wait(wfagpu_device_t *d, int slot, float *ms_pack, float *ms_align);
/* After wfagpu_device_download: CIGAR text emitted on the device (one warp per pair, the
 * reference's exact format) and compacted; `*text` / `*refs` point into pinned memory owned by
 * the slot.  Replaces the host loop over recover_cigar_affine (utils/wfa_cpu.c:88-107). */
int wfagpu_device_download_text(wfagpu_device_t *d, int slot, size_t n, const char **text, size_t *text_bytes,
                                const wfagpu_cigar_ref_t **refs);
void wfagpu_device_last_stats(wfagpu_device_t *d, int slot, wfagpu_batch_stats_t *st);
/* Page-locks a caller buffer (e.g. the aligner's sequence buffer) so that the
 * H2D copies run as asynchronous DMA. */
int wfagpu_host_register(void *ptr, size_t bytes);
int wfagpu_host_unregister(void *ptr);
/* 1 if `ptr` is page-locked memory. */
int wfagpu_host_is_pinned(const void *ptr);
/* Page-locked staging area of a slot for callers with a pageable sequence buffer (see driver.c). */
char *wfagpu_device_staging(wfagpu_device_t *d, int slot, size_t bytes);
/* Page-locked zeroed host memory (NULL without a usable CUDA device: callers fall back to calloc). */
void *wfagpu_host_alloc(size_t bytes);
void wfagpu_host_free(void *p);
int wfagpu_device_sm_count(wfagpu_device_t *d);

/* Builds the device-side descriptors of pairs [from, from+n) of a host buffer
 * (also rewrites their *_offset_packed like lib/align.cu:103-115). `base_out` /
 * `bytes_out`: the slice of the buffer to hand to wfagpu_device_upload. */
int wfagpu_pairs_from_metadata(sequence_pair_t *meta, size_t from, size_t n, size_t buf_size,
                               wfagpu_pair_t *pairs, size_t *base_out, size_t *bytes_out);

/* Pack kernel alone (tests, replaces prepare_pack_sequences_gpu +
 * pack_sequences_gpu_async, lib/sequence_packing.cu:27-116): uploads, packs and
 * returns the packed words (layout: word j = bases [8j, 8j+16), first base in
 * bits 31:30, code (c&6)>>1) and the has_N flags. */
int wfagpu_device_pack_only(wfagpu_device_t *d, const char *ascii, size_t ascii_bytes,
                            wfagpu_pair_t *pairs, size_t n, uint32_t *packed_out,
                            size_t packed_words);

/* ------------------------------------------------------------ host side --- */
/* CIGAR text from a packed op stream (newest op first, 16 ops per u32, op j
 * of a word in bits 2j+1:2j).  Same text as utils/cigar.c:96-272 produces
 * from the reference's backtrace chain.  Appends to `cigar`. */
bool wfagpu_ops_to_cigar(const char *pattern, size_t plen, const char *text, size_t tlen,
                         int distance, const uint32_t *ops, uint32_t n_ops, wfa_cigar_t *cigar);

/* The same for an ends-free alignment that starts on diagonal `k_begin` (wfagpu_device_download_ends): a leading
 * I (k_begin > 0) or D run of |k_begin|, the path from (max(0, -k_begin), max(0, k_begin)), and a trailing I / D run
 * to the end of both sequences; a free run joins the gap run of the same letter next to it. */
bool wfagpu_ops_to_cigar_span(const char *pattern, size_t plen, const char *text, size_t tlen, int k_begin,
                              const uint32_t *ops, uint32_t n_ops, wfa_cigar_t *cigar);

/* Appends formatted CIGAR text to a result buffer (growing it like insert_ops does). */
bool wfagpu_cigar_append(wfa_cigar_t *cigar, const char *text, size_t len);

/* Device selection for launch_alignments*: "0", "0,1,2", "all", or a count
 * ("n:4").  Default (NULL/unset): environment WFAGPU_DEVICES, else device 0. */
void wfagpu_set_devices(const char *spec);

/* Chunking of a job over `n_devices` GPUs (pure function, used by launch_alignments*). */
void wfagpu_plan_chunks(size_t n, size_t batch_size, int n_devices, size_t ascii_span,
                        size_t *chunk_out, size_t *n_chunks_out);

/* How the chunks of a job are dealt to `nworkers` host threads (one per device-list entry): every worker owns a contiguous
 * share [share_next[i], share_end[i]) and takes `want` pairs from its front; a worker whose share is used up takes `steal`
 * pairs from the back of the fullest share.  Pure functions on the share table (the caller serialises); false = nothing left. */
void wfagpu_plan_shares(size_t n, int nworkers, size_t *share_next, size_t *share_end);
bool wfagpu_share_take(size_t *share_next, size_t *share_end, int nworkers, int index, size_t want, size_t steal,
                       size_t *from, size_t *n);

/* Host threads this library may use per call (result loop, staging copies, generators); 0 = OpenMP default.
 * torchrun pins OMP_NUM_THREADS=1 per rank: a rank that works alone can lift that. */
void wfagpu_set_host_threads(int n);

/* Stats of the last launch_alignments* call (summed over batches/devices). */
typedef struct {
    double wall_s;
    double gpu_align_ms;  /* sum of alignment-kernel time over batches (max over devices per batch not tracked) */
    double gpu_pack_ms;
    uint64_t launches;
    uint64_t redispatched;
    uint64_t ascii_pairs;
    uint64_t h2d_bytes, d2h_bytes;
    int devices;          /* workers (one leased context each) */
    int staged;           /* 1: the caller's buffer was pageable, chunks went through page-locked staging */
    uint64_t failed_pairs; /* pairs the GPU could not finish (results[i].error == UINT_MAX)               */
    uint64_t checked, incorrect; /* check_correctness: pairs validated / found wrong                      */
} wfagpu_run_stats_t;
/* Statistics / outcome of the calling thread's last launch_alignments* call (thread-local). */
void wfagpu_last_run_stats(wfagpu_run_stats_t *st);
/* false when that call failed on the GPU or left pairs unaligned (nothing is computed on the CPU) */
bool wfagpu_last_launch_ok(void);
/* Device list syntax of wfagpu_set_devices / WFAGPU_DEVICES (pure function; -1 on a bad list). */
int wfagpu_parse_devices(const char *spec, int visible, int *devs, int max_devs);
/* Independent re-computation of the scores of the batch resident in `slot` (check_correctness): score only,
 * one-diagonal-per-thread kernels, launch bound only -- no per-pair bounds, packed-SIMD kernel, snapshots or
 * provisioning hints.  scores[i] = -1 for a pair it could not finish. */
int wfagpu_device_rescore(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int32_t *scores);
/* The same for an ends-free span (NULL = global).  with_cigar and with_ends of the plan are ignored. */
int wfagpu_device_rescore_span(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan,
                               const wfagpu_span_t *span, int32_t *scores);
/* The same with one span per pair (spans[i] for pair i; NULL = global). */
int wfagpu_device_rescore_spans(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan,
                                const wfagpu_span_t *spans, int32_t *scores);

/* Makes room for `bytes` more sequence bytes and `pairs` more pairs in one step (readers, generators). */
bool wfagpu_reserve(wfagpu_aligner_t *aligner, size_t bytes, size_t pairs);

/* Clears errors and CIGAR text of a previous wfagpu_align (the reference, like
 * this library, appends to results[i].cigar) so an aligner can be re-aligned. */
void wfagpu_reset_results(wfagpu_aligner_t *aligner);

/* CLI input formats (replace utils/sequence_reader.c:137-392): append the pairs of a .seq file
 * (">pattern" / "<text" lines) or of two FASTA files (n-th query record with n-th target record)
 * to the aligner. max_pairs == 0 reads everything. Return the number of pairs, -1 on error. */
long wfagpu_read_seq_file(wfagpu_aligner_t *aligner, const char *path, size_t max_pairs);
long wfagpu_read_fasta_files(wfagpu_aligner_t *aligner, const char *query_path, const char *target_path,
                             size_t max_pairs);

/* Incremental readers (streaming): every call appends the next `max_pairs` pairs (0 = all that are left) to the
 * aligner's page-locked buffer; returns how many (0 at the end of the input, -1 on a format error). */
typedef struct wfagpu_reader wfagpu_reader_t;
wfagpu_reader_t *wfagpu_reader_open_seq(const char *path);
wfagpu_reader_t *wfagpu_reader_open_fasta(const char *query_path, const char *target_path);
long wfagpu_reader_next(wfagpu_reader_t *r, wfagpu_aligner_t *aligner, size_t max_pairs);
long wfagpu_reader_total_bytes(const wfagpu_reader_t *r);
void wfagpu_reader_close(wfagpu_reader_t *r);
/* Forgets the pairs of an aligner but keeps its (page-locked) buffers, so that the next window of a stream reuses them. */
void wfagpu_clear_sequences(wfagpu_aligner_t *aligner);

/* `-c`: true iff `cigar` is a valid global alignment of (pattern, text) whose gap-affine cost is
 * `error` (replaces check_cigar_edit + check_affine_distance, utils/verification.c:27-146). */
bool wfagpu_check_result(const char *pattern, size_t plen, const char *text, size_t tlen,
                         affine_penalties_t pen, unsigned int error, const char *cigar);
/* The same under an ends-free span: a leading I run of length L costs 0 if L <= text_begin_free, else
 * o + e (L - text_begin_free); likewise a leading D run (pattern_begin_free), a trailing I run (text_end_free) and a
 * trailing D run (pattern_end_free).  A run that is both leading and trailing may use both allowances. */
bool wfagpu_check_result_span(const char *pattern, size_t plen, const char *text, size_t tlen,
                              affine_penalties_t pen, const wfagpu_span_t *span, unsigned int error, const char *cigar);

/* The same under gap-affine 2-piece penalties: every gap run of length L costs min(o1 + e1 L, o2 + e2 L). */
bool wfagpu_check_result_affine2p(const char *pattern, size_t plen, const char *text, size_t tlen,
                                  const wfagpu_affine2p_t *pen, unsigned int error, const char *cigar);

/* wfagpu_align under gap-affine 2-piece penalties: the five values replace the aligner's penalties for this call
 * (honours compute_cigar).  False, with a message and the results untouched, for an invalid set (see
 * wfagpu_affine2p_t), band > 0.  NULL: exactly wfagpu_align. */
bool wfagpu_align_affine2p(wfagpu_aligner_t *aligner, const wfagpu_affine2p_t *pen);
/* launch_alignments / launch_alignments_distance (cigar = false) under 2-piece penalties (options.penalties is not
 * used); check_correctness validates every CIGAR under them and re-computes every score.  NULL: the single-piece
 * function. */
void wfagpu_launch_alignments_affine2p(char *sequences_buffer, size_t sequences_buffer_size,
                                       sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                       wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                       const wfagpu_affine2p_t *pen);

/* wfagpu_align with an ends-free span (honours compute_cigar).  False, with a message, for negative values, or for
 * band > 0 together with a non-zero span.  NULL or all zero: exactly wfagpu_align. */
bool wfagpu_align_span(wfagpu_aligner_t *aligner, const wfagpu_span_t *span);
/* launch_alignments / launch_alignments_distance (cigar = false) with an ends-free span; check_correctness validates
 * every CIGAR under the span and re-computes every score with the same span. */
void wfagpu_launch_alignments_span(char *sequences_buffer, size_t sequences_buffer_size,
                                   sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                   wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                   const wfagpu_span_t *span);

/* The aligned part: pattern[pattern_begin, pattern_end) against text[text_begin, text_end).  From {k_begin, k_end}:
 * pattern_begin = max(0, -k_begin), text_begin = max(0, k_begin), text_end = min(tlen, plen + k_end),
 * pattern_end = text_end - k_end.  Global call (NULL / zero span): (0, plen, 0, tlen).  Pair not aligned: all -1. */
typedef struct {
    int pattern_begin, pattern_end, text_begin, text_end;
} wfagpu_coords_t;
/* wfagpu_align_span that also fills `coords` (one entry per pair, owned by the caller) in CIGAR and score-only mode.
 * NULL coords: exactly wfagpu_align_span. */
bool wfagpu_align_span_coords(wfagpu_aligner_t *aligner, const wfagpu_span_t *span, wfagpu_coords_t *coords);
/* wfagpu_launch_alignments_span that also fills `coords`; NULL coords: exactly wfagpu_launch_alignments_span. */
void wfagpu_launch_alignments_span_coords(char *sequences_buffer, size_t sequences_buffer_size,
                                          sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                          wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                          const wfagpu_span_t *span, wfagpu_coords_t *coords);

/* Per-pair spans: wfagpu_align_span_coords with spans[i] for pair i (num_sequence_pairs entries; honours compute_cigar;
 * coords may be NULL).  Pairs with an all-zero span get their global alignment; all-zero spans or NULL: exactly
 * wfagpu_align.  False, with a message, for a negative value, or for band > 0 with a non-zero span. */
bool wfagpu_align_spans(wfagpu_aligner_t *aligner, const wfagpu_span_t *spans, wfagpu_coords_t *coords);
/* wfagpu_launch_alignments_span_coords with spans[i] for pair i, indexed like sequences_metadata; check_correctness
 * validates every CIGAR under its pair's span and re-computes every score with the same spans. */
void wfagpu_launch_alignments_spans(char *sequences_buffer, size_t sequences_buffer_size,
                                    sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                    wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                    const wfagpu_span_t *spans, wfagpu_coords_t *coords);

/* The reference library's generic validators, same names, argument order (text first) and input format
 * (utils/verification.h:37-58): the op string may be UNROLLED ("MMXMMI", what the reference's recover_cigar
 * returns and lib/align.cu:284-293 passes) or the run-length text of results[i].cigar.buffer ("2M1X2M1I").
 * check_cigar_edit: the ops are a global alignment of (pattern, text); check_affine_distance: their gap-affine
 * cost equals `distance`. */
bool check_cigar_edit(const char *text, const char *pattern, const int tlen, const int plen, const char *curr_cigar);
bool check_affine_distance(const char *text, const char *pattern, const int tlen, const int plen, const int distance,
                           const affine_penalties_t penalties, const char *cigar);
/* recover_cigar (utils/verification.h:52-58): unrolled op string from a reference-format backtrace chain
 * (calloc'ed, caller frees). */
char *recover_cigar(const char *text, const char *pattern, const size_t tlen, const size_t plen,
                    wfa_backtrace_t final_backtrace, wfa_backtrace_t *offloaded_backtraces_array,
                    alignment_result_t result);
/* Unrolled op string of run-length CIGAR text (malloc'ed, caller frees; NULL on malformed text). */
char *wfagpu_unroll_cigar(const char *rle);

/* Deterministic synthetic pairs (SURVEY §8d: text uniform over ACGT, pattern =
 * text with ceil(L*err) edits, each uniformly mismatch / 1-base deletion /
 * 1-base insertion; splitmix64 seeded).  Appends n pairs to the aligner. */
bool wfagpu_synth_add_pairs(wfagpu_aligner_t *aligner, uint64_t seed, size_t n, int length,
                            double err_lo, double err_hi);

#ifdef __cplusplus
}
#endif
#endif
