/*
 * aligner.c -- the wfagpu_* public API (replaces lib/aligner.c:24-263).
 *
 * Same observable behaviour as the reference: sequences are copied into one
 * growing host buffer, each at a 4-byte aligned offset and followed by NULs;
 * metadata slots grow in blocks; defaults come from
 * wfagpu_set_default_options.  The reference's grow_* helpers store byte sizes
 * in element-count fields (lib/aligner.c:62-70,103-111) and leave the new
 * metadata tail uninitialised; here lengths are kept in their own units and new
 * memory is zeroed.
 */
#include <stdio.h>
#include <string.h>
#include "wfagpu_b200.h"

#define SEQ_BUF_CHUNK ((size_t)1 << 20)
#define META_CHUNK ((size_t)10000)
#define FIRST_CIGAR_LEN 50

#define WARN(...) do { fprintf(stderr, "WARNING: "); fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); } while (0)
#define ERR(...) do { fprintf(stderr, "[!] ERROR: "); fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); } while (0)

extern bool wfagpu_last_launch_ok(void); /* driver.c */

/* The aligner owns its result array.  The reference frees it with the *current*
 * pair count (lib/aligner.c:231-235), which overruns when pairs were added after
 * wfagpu_initialize_parameters; here the allocated count lives in a hidden
 * 16-byte prefix in front of the array. */
#define RES_PREFIX 16
static wfa_alignment_result_t *owned_results_new(size_t n, size_t cigar_len)
{
    char *blk = (char *)calloc(1, RES_PREFIX + (n ? n : 1) * sizeof(wfa_alignment_result_t));
    if (!blk) return NULL;
    *(size_t *)blk = n;
    wfa_alignment_result_t *r = (wfa_alignment_result_t *)(blk + RES_PREFIX);
    for (size_t i = 0; i < n; ++i) {
        r[i].cigar.buffer = (char *)calloc(cigar_len, 1);
        if (!r[i].cigar.buffer) return NULL;
        r[i].cigar.buffer_size = cigar_len;
    }
    return r;
}
static void owned_results_free(wfa_alignment_result_t *r)
{
    if (!r) return;
    char *blk = (char *)r - RES_PREFIX;
    const size_t n = *(size_t *)blk;
    for (size_t i = 0; i < n; ++i) free(r[i].cigar.buffer);
    free(blk);
}

/* The sequence buffer is what every batch is uploaded from.  The reference callocs it and leaves "CudaMallocHost
 * instead of calloc" as a TODO (utils/sequence_reader.c:73); here it is page-locked from the start, so an
 * unmodified caller of wfagpu_add_sequences / wfagpu_align gets asynchronous DMA uploads without calling any
 * extension.  A hidden 64-byte prefix remembers how the block was obtained (without a usable CUDA device it is
 * plain calloc memory).  Buffers that do not come from here -- a caller of launch_alignments with its own
 * malloc'ed buffer -- are staged chunk by chunk (driver.c). */
#define SEQ_PREFIX 64
#define SEQ_MAGIC 0x5746414750554231ull
typedef struct { unsigned long long magic; int pinned; } seq_prefix_t;

static char *seqbuf_new(size_t bytes)
{
    int pinned = 1;
    char *blk = (char *)wfagpu_host_alloc(bytes + SEQ_PREFIX);
    if (!blk) { pinned = 0; blk = (char *)calloc(bytes + SEQ_PREFIX, 1); }
    if (!blk) return NULL;
    seq_prefix_t *pf = (seq_prefix_t *)blk;
    pf->magic = SEQ_MAGIC;
    pf->pinned = pinned;
    return blk + SEQ_PREFIX;
}
static void seqbuf_free(char *buf)
{
    if (!buf) return;
    seq_prefix_t *pf = (seq_prefix_t *)(buf - SEQ_PREFIX);
    if (pf->magic != SEQ_MAGIC) { free(buf); return; }      /* not ours (a caller swapped the pointer) */
    pf->magic = 0;
    if (pf->pinned) wfagpu_host_free(pf); else free(pf);
}

bool wfagpu_initialize_aligner(wfagpu_aligner_t *aligner)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    memset(aligner, 0, sizeof(*aligner));
    aligner->last_sequence_pair_idx = -1;
    aligner->sequences_buffer = (wfagpu_seqbuf_t *)seqbuf_new(SEQ_BUF_CHUNK);
    aligner->sequences_metadata = (sequence_pair_t *)calloc(META_CHUNK, sizeof(sequence_pair_t));
    if (!aligner->sequences_buffer || !aligner->sequences_metadata) {
        ERR("Can not initialize the aligner buffers.");
        return false;
    }
    aligner->sequences_buffer_len = SEQ_BUF_CHUNK;
    aligner->sequences_metadata_len = META_CHUNK;
    return true;
}

static bool reserve_pairs(wfagpu_aligner_t *a, size_t need);
static bool reserve_bytes(wfagpu_aligner_t *a, size_t need)
{
    if (need < a->sequences_buffer_len) return true;
    size_t nlen = a->sequences_buffer_len;
    /* geometric growth: the reference adds 1 MiB at a time, which is quadratic for GB inputs */
    while (nlen <= need) nlen += (nlen / 2 > SEQ_BUF_CHUNK ? nlen / 2 : SEQ_BUF_CHUNK);
    char *nb = seqbuf_new(nlen);                             /* zeroed */
    if (!nb) return false;
    size_t used = 0;
    if (a->last_sequence_pair_idx >= 0) {
        const sequence_pair_t *last = &a->sequences_metadata[a->last_sequence_pair_idx];
        used = last->text_offset + last->text_len + 1;
        if (used > a->sequences_buffer_len) used = a->sequences_buffer_len;
    }
    memcpy(nb, a->sequences_buffer, used);
    seqbuf_free(a->sequences_buffer);
    a->sequences_buffer = nb;
    a->sequences_buffer_len = nlen;
    return true;
}

/* Extension for the readers and generators: make room for `bytes` more sequence bytes and `pairs` more pairs
 * in one step (a page-locked buffer is expensive to grow geometrically). */
bool wfagpu_reserve(wfagpu_aligner_t *aligner, size_t bytes, size_t pairs)
{
    if (!aligner || !aligner->sequences_buffer || !aligner->sequences_metadata) return false;
    size_t used = 0;
    if (aligner->last_sequence_pair_idx >= 0) {
        const sequence_pair_t *last = &aligner->sequences_metadata[aligner->last_sequence_pair_idx];
        used = WFA_ALIGN_32_BITS(last->text_offset + last->text_len + 1);
    }
    return reserve_bytes(aligner, used + bytes + 16) && reserve_pairs(aligner, (size_t)(aligner->last_sequence_pair_idx + 1) + pairs);
}

static bool reserve_pairs(wfagpu_aligner_t *a, size_t need)
{
    if (need <= a->sequences_metadata_len) return true;
    size_t nlen = a->sequences_metadata_len;
    while (nlen < need) nlen += (nlen / 2 > META_CHUNK ? nlen / 2 : META_CHUNK);
    sequence_pair_t *nm = (sequence_pair_t *)realloc(a->sequences_metadata, nlen * sizeof(sequence_pair_t));
    if (!nm) return false;
    memset(nm + a->sequences_metadata_len, 0, (nlen - a->sequences_metadata_len) * sizeof(sequence_pair_t));
    a->sequences_metadata = nm;
    a->sequences_metadata_len = nlen;
    return true;
}

bool wfagpu_add_sequences(wfagpu_aligner_t *aligner, const char *query, const char *target)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (!query || !target) { ERR("Invalid sequence pointers."); return false; }
    if (!aligner->sequences_buffer || !aligner->sequences_metadata) { ERR("Aligner is not initialized."); return false; }

    size_t p_off = 0;
    if (aligner->last_sequence_pair_idx >= 0) {
        const sequence_pair_t *last = &aligner->sequences_metadata[aligner->last_sequence_pair_idx];
        p_off = WFA_ALIGN_32_BITS(last->text_offset + last->text_len + 1);
    }
    /* The reference stops at MAX_SEQ_LEN - 1 = 32767 bases (int16 offsets, lib/aligner.c:139-142).
     * Longer sequences are accepted here and run on the int32 large tier. */
    const size_t plen = strnlen(query, WFAGPU_MAX_SEQ_LEN);
    const size_t tlen = strnlen(target, WFAGPU_MAX_SEQ_LEN);
    if (plen >= WFAGPU_MAX_SEQ_LEN || tlen >= WFAGPU_MAX_SEQ_LEN) {
        WARN("Sequences must be shorter than %lu.", (unsigned long)WFAGPU_MAX_SEQ_LEN - 1);
        return false;
    }
    const size_t t_off = WFA_ALIGN_32_BITS(p_off + plen + 1);
    if (!reserve_bytes(aligner, WFA_ALIGN_32_BITS(t_off + tlen + 1) + 8)) {
        ERR("Sequences do not fit in memory. Aborting.");
        return false;
    }
    const size_t slot = (size_t)(aligner->last_sequence_pair_idx + 1);
    if (!reserve_pairs(aligner, slot + 1)) {
        ERR("Can not resize sequence metadata buffer. Aborting.");
        return false;
    }
    memcpy(aligner->sequences_buffer + p_off, query, plen);
    memcpy(aligner->sequences_buffer + t_off, target, tlen);
    /* NUL padding up to the next sequence: a buffer reused after wfagpu_clear_sequences still holds the old bytes */
    memset(aligner->sequences_buffer + p_off + plen, 0, t_off - (p_off + plen));
    memset(aligner->sequences_buffer + t_off + tlen, 0, WFA_ALIGN_32_BITS(t_off + tlen + 1) - (t_off + tlen));
    sequence_pair_t *m = &aligner->sequences_metadata[slot];
    memset(m, 0, sizeof(*m));
    m->pattern_offset = p_off;
    m->pattern_len = (unsigned)plen;
    m->text_offset = t_off;
    m->text_len = (unsigned)tlen;
    aligner->last_sequence_pair_idx++;
    aligner->num_sequence_pairs++;
    return true;
}

bool wfagpu_initialize_parameters(wfagpu_aligner_t *aligner, affine_penalties_t penalties)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (penalties.x < 0 || penalties.o < 0 || penalties.e < 0) { ERR("Penalties must be >= 0."); return false; }
    if (penalties.x == 0 && penalties.o == 0 && penalties.e == 0) { ERR("All penalties can not be 0."); return false; }
    if (aligner->num_sequence_pairs == 0 || !aligner->sequences_metadata) {
        ERR("Add the sequences before initializing the parameters.");
        return false;
    }
    wfagpu_set_default_options(&aligner->alignment_options, aligner->sequences_metadata, penalties,
                               aligner->num_sequence_pairs);
    owned_results_free(aligner->results);
    aligner->results = owned_results_new(aligner->num_sequence_pairs, FIRST_CIGAR_LEN);
    return aligner->results != NULL;
}

bool wfagpu_set_batch_size(wfagpu_aligner_t *aligner, size_t batch_size)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (batch_size > aligner->num_sequence_pairs) {
        WARN("Batch size must be less or equal than the number of sequences. Setting batch size to %zu.",
             aligner->num_sequence_pairs);
        batch_size = aligner->num_sequence_pairs;
    }
    if (batch_size == 0) {
        WARN("Batch size can not be zero. Setting batch size to %zu.", aligner->num_sequence_pairs);
        batch_size = aligner->num_sequence_pairs;
    }
    aligner->alignment_options.batch_size = batch_size;
    return true;
}

void wfagpu_destroy_aligner(wfagpu_aligner_t *aligner)
{
    if (!aligner) return;
    seqbuf_free(aligner->sequences_buffer);
    free(aligner->sequences_metadata);
    owned_results_free(aligner->results);
    aligner->sequences_buffer = NULL;
    aligner->sequences_metadata = NULL;
    aligner->results = NULL;
}

bool wfagpu_align(wfagpu_aligner_t *aligner)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (!aligner->results || !aligner->sequences_metadata) { ERR("Aligner parameters are not initialized."); return false; }
    if (aligner->alignment_options.compute_cigar) {
        launch_alignments(aligner->sequences_buffer, aligner->sequences_buffer_len, aligner->sequences_metadata,
                          aligner->results, aligner->alignment_options, false);
    } else {
        launch_alignments_distance(aligner->sequences_buffer, aligner->sequences_buffer_len,
                                   aligner->sequences_metadata, aligner->results, aligner->alignment_options, false);
    }
    /* the reference always returns true here; a failed GPU launch is reported instead */
    return wfagpu_last_launch_ok();
}

bool wfagpu_align_span(wfagpu_aligner_t *aligner, const wfagpu_span_t *span)
{
    return wfagpu_align_span_coords(aligner, span, NULL);
}

bool wfagpu_align_span_coords(wfagpu_aligner_t *aligner, const wfagpu_span_t *span, wfagpu_coords_t *coords)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (!aligner->results || !aligner->sequences_metadata) { ERR("Aligner parameters are not initialized."); return false; }
    if (span && (span->pattern_begin_free < 0 || span->pattern_end_free < 0 || span->text_begin_free < 0 ||
                 span->text_end_free < 0)) {
        ERR("Ends-free span values must be >= 0.");
        return false;
    }
    const bool ef = span && (span->pattern_begin_free || span->pattern_end_free || span->text_begin_free ||
                             span->text_end_free);
    if (ef && aligner->alignment_options.band > 0) {
        ERR("Ends-free alignment cannot be combined with the adaptive band.");
        return false;
    }
    wfagpu_launch_alignments_span_coords(aligner->sequences_buffer, aligner->sequences_buffer_len,
                                         aligner->sequences_metadata, aligner->results, aligner->alignment_options,
                                         aligner->alignment_options.compute_cigar, false, ef ? span : NULL, coords);
    return wfagpu_last_launch_ok();
}

bool wfagpu_align_spans(wfagpu_aligner_t *aligner, const wfagpu_span_t *spans, wfagpu_coords_t *coords)
{
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (!aligner->results || !aligner->sequences_metadata) { ERR("Aligner parameters are not initialized."); return false; }
    /* the spans are validated by the driver, before anything is aligned */
    wfagpu_launch_alignments_spans(aligner->sequences_buffer, aligner->sequences_buffer_len, aligner->sequences_metadata,
                                   aligner->results, aligner->alignment_options, aligner->alignment_options.compute_cigar,
                                   false, spans, coords);
    return wfagpu_last_launch_ok();
}

bool wfagpu_align_affine2p(wfagpu_aligner_t *aligner, const wfagpu_affine2p_t *pen)
{
    if (!pen) return wfagpu_align(aligner);
    if (!aligner) { ERR("Invalid aligner."); return false; }
    if (!aligner->results || !aligner->sequences_metadata) { ERR("Aligner parameters are not initialized."); return false; }
    if (pen->x < 1 || pen->o1 < 0 || pen->e1 < 1 || pen->o2 < 0 || pen->e2 < 1) {
        ERR("Gap-affine 2-piece penalties must satisfy x >= 1, o1, o2 >= 0, e1, e2 >= 1.");
        return false;
    }
    if (aligner->alignment_options.band > 0) {
        ERR("Gap-affine 2-piece alignment cannot be combined with the adaptive band.");
        return false;
    }
    wfagpu_launch_alignments_affine2p(aligner->sequences_buffer, aligner->sequences_buffer_len,
                                      aligner->sequences_metadata, aligner->results, aligner->alignment_options,
                                      aligner->alignment_options.compute_cigar, false, pen);
    return wfagpu_last_launch_ok();
}

/* Extension: forget the pairs, keep the buffers (streaming: the next window is read into the same pinned memory). */
void wfagpu_clear_sequences(wfagpu_aligner_t *aligner)
{
    if (!aligner) return;
    aligner->last_sequence_pair_idx = -1;
    aligner->num_sequence_pairs = 0;
}

/* Extension: forget the CIGAR text of a previous wfagpu_align so that the same
 * aligner can be aligned again (the reference appends to the old text). */
void wfagpu_reset_results(wfagpu_aligner_t *aligner)
{
    if (!aligner || !aligner->results) return;
    const size_t n = *(size_t *)((char *)aligner->results - RES_PREFIX);
    for (size_t i = 0; i < n; ++i) {
        aligner->results[i].error = 0;
        aligner->results[i].cigar.last_free_position = 0;
        if (aligner->results[i].cigar.buffer && aligner->results[i].cigar.buffer_size)
            aligner->results[i].cigar.buffer[0] = 0;
    }
}
