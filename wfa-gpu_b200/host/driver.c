/*
 * driver.c -- batch driver behind launch_alignments / launch_alignments_distance
 * (replaces the host half of lib/align.cu:42-881 and utils/wfa_cpu.c:30-164).
 *
 * The pair range is cut into chunks of at most `batch_size` pairs.  Each
 * selected GPU is driven by one host thread that leases its own device context
 * (two slots): while the GPU aligns chunk c, the thread hands chunk c-1's
 * results to the caller.  Pairs are independent, so GPUs never exchange data
 * (no NCCL): results are written straight into alignment_results[i], disjoint
 * per chunk.  There is no CPU alignment path: over-budget and non-ACGT pairs
 * are finished on the GPU inside wfagpu_device_download().
 *
 * Re-entrant like the reference (lib/align.cu:63-162 allocates per call): a call
 * owns its job, its workers and their leased contexts; the only process-wide
 * state is the default device list (wfagpu_set_devices, mutex) and, per thread,
 * the statistics of that thread's last call.
 */
#include <pthread.h>
#include <stdio.h>
#include <string.h>
#include <time.h>
#include <limits.h>
#include <omp.h>
#include "wfagpu_b200.h"

#define MAX_DEVICES 64

static pthread_mutex_t g_spec_mu = PTHREAD_MUTEX_INITIALIZER;
static char g_device_spec[256] = "";
static __thread wfagpu_run_stats_t t_last_stats;
static __thread bool t_last_ok = true;

void wfagpu_set_devices(const char *spec)
{
    pthread_mutex_lock(&g_spec_mu);
    if (!spec) g_device_spec[0] = 0;
    else {
        strncpy(g_device_spec, spec, sizeof(g_device_spec) - 1);
        g_device_spec[sizeof(g_device_spec) - 1] = 0;
    }
    pthread_mutex_unlock(&g_spec_mu);
}

void wfagpu_set_host_threads(int n) { if (n > 0) omp_set_num_threads(n); }

void wfagpu_last_run_stats(wfagpu_run_stats_t *st) { if (st) *st = t_last_stats; }
bool wfagpu_last_launch_ok(void) { return t_last_ok; }

/* Device list of a call: "all", "n:4", or ids ("0,2,5"; an id may repeat: every entry is one worker with its
 * own context, "0,0" drives GPU 0 from two host threads).  Returns the number of workers, -1 on a bad id. */
int wfagpu_parse_devices(const char *spec, int visible, int *devs, int max_devs)
{
    int n = 0;
    if (!spec || !*spec) { devs[0] = 0; return 1; }
    if (!strcmp(spec, "all")) {
        for (int i = 0; i < visible && i < max_devs; ++i) devs[n++] = i;
        if (!n) { devs[0] = 0; n = 1; }
        return n;
    }
    if (!strncmp(spec, "n:", 2)) {
        const int want = atoi(spec + 2);
        for (int i = 0; i < want && i < visible && i < max_devs; ++i) devs[n++] = i;
        if (!n) { devs[0] = 0; n = 1; }
        return n;
    }
    const char *p = spec;
    while (*p && n < max_devs) {
        char *end;
        const long v = strtol(p, &end, 10);
        if (end == p) return -1;
        if (v < 0 || (visible > 0 && v >= visible)) return -1;
        devs[n++] = (int)v;
        if (*end == ',') p = end + 1;
        else if (*end == 0) break;
        else return -1;
    }
    if (!n) { devs[0] = 0; n = 1; }
    return n;
}

static int select_devices(int *devs)
{
    char spec[256];
    pthread_mutex_lock(&g_spec_mu);
    memcpy(spec, g_device_spec, sizeof(spec));
    pthread_mutex_unlock(&g_spec_mu);
    const char *sp = spec[0] ? spec : getenv("WFAGPU_DEVICES");
    int visible = 0;
    get_num_cuda_devices(&visible);
    const int n = wfagpu_parse_devices(sp, visible, devs, MAX_DEVICES);
    if (n < 0) fprintf(stderr, "[!] ERROR: bad device list \"%s\" (%d CUDA device(s) visible).\n", sp ? sp : "", visible);
    return n;
}

typedef struct {
    /* job */
    char *buf;
    size_t buf_size;
    sequence_pair_t *meta;
    wfa_alignment_result_t *res;
    wfa_alignment_options_t opt;
    bool cigar;
    bool check;             /* check_correctness: validate every result (see check_chunk) */
    bool pageable;          /* the caller's sequence buffer is not page-locked: stage every chunk */
    size_t n, chunk;
    size_t n_chunks;
    size_t share_next[MAX_DEVICES], share_end[MAX_DEVICES];   /* guarded by mu: what is left of every worker's share */
    size_t first_chunk;     /* size of the first chunk of every worker (ramp-up: its upload is not hidden) */
    int nworkers;           /* host threads (one per device-list entry) that share the stream of chunks */
    pthread_mutex_t mu;
    bool failed;
    bool verbose;
    bool host_cigar;        /* WFAGPU_HOST_CIGAR=1: print the CIGAR text on the host instead of the GPU */
    bool ef;                /* ends-free call: some pair's span is not all zero */
    const wfagpu_span_t *spans;   /* the caller's: pair i has spans[i * span_stride] (stride 0: one span for the call) */
    size_t span_stride;
    bool p2;                /* gap-affine 2-piece call: `pen2` replaces opt.penalties */
    wfagpu_affine2p_t pen2;
    wfagpu_coords_t *coords;  /* the caller's, one per pair, or NULL */
    int decode_threads;
    /* accumulated */
    wfagpu_run_stats_t stats;
    uint64_t failed_pairs, checked, incorrect;
    size_t first_failed[8];
    int n_first_failed;
} job_t;

typedef struct {
    job_t *job;
    int dev;
    int index;              /* which share of the stream is this worker's */
    bool first_taken;
} worker_t;

typedef struct {
    size_t from, n;
    bool active;
    wfagpu_pair_t *pairs;
    size_t pairs_cap;
    wfagpu_pair_out_t *out;
    size_t out_cap;
    int32_t *ends;          /* ends-free, CIGAR text on the host or coordinates: {k_begin, k_end} per pair */
    bool ef;                /* the chunk was aligned as an ends-free batch: some pair of it has a non-zero span */
} inflight_t;

static double now_s(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* Every worker owns a contiguous share of the stream and walks it front to back (first chunk, chunks, remainder): equal
 * GPUs finish together whatever the chunk sizes are.  A worker that runs dry takes `steal` pairs from the back of the
 * fullest share (a slower GPU, a device shared with another job).  Pure functions on the share table, so that the
 * policy is testable without a GPU; the caller serialises. */
void wfagpu_plan_shares(size_t n, int nworkers, size_t *share_next, size_t *share_end)
{
    if (nworkers < 1) return;
    const size_t per = (n + (size_t)nworkers - 1) / (size_t)nworkers;
    size_t at = 0;
    for (int i = 0; i < nworkers; ++i) {
        share_next[i] = at;
        at = (at + per < n && i + 1 < nworkers) ? at + per : n;
        share_end[i] = at;
    }
}

bool wfagpu_share_take(size_t *share_next, size_t *share_end, int nworkers, int index, size_t want, size_t steal,
                       size_t *from, size_t *n)
{
    if (index < 0 || index >= nworkers) return false;
    if (share_next[index] < share_end[index]) {
        const size_t left = share_end[index] - share_next[index];
        *from = share_next[index];
        *n = left < want ? left : (want > 0 ? want : 1);
        share_next[index] += *n;
        return true;
    }
    int best = -1;
    size_t most = 0;
    for (int k = 0; k < nworkers; ++k)
        if (share_end[k] - share_next[k] > most) { most = share_end[k] - share_next[k]; best = k; }
    if (best < 0) return false;
    size_t take = steal > 0 ? steal : 1;
    if (take > most) take = most;
    share_end[best] -= take;
    *from = share_end[best];
    *n = take;
    return true;
}

static bool take_chunk(worker_t *w, size_t *from, size_t *n)
{
    job_t *j = w->job;
    bool ok = false;
    pthread_mutex_lock(&j->mu);
    if (!j->failed) {
        const size_t want = w->first_taken ? j->chunk : j->first_chunk;
        ok = wfagpu_share_take(j->share_next, j->share_end, j->nworkers, w->index, want, j->chunk / 2, from, n);
        w->first_taken = true;
    }
    pthread_mutex_unlock(&j->mu);
    return ok;
}

static void fail_job(job_t *j)
{
    pthread_mutex_lock(&j->mu);
    j->failed = true;
    pthread_mutex_unlock(&j->mu);
}

/* Device-side view of pairs [from, from+n) of a host buffer laid out like
 * wfagpu_add_sequences / the readers do (increasing 4-byte aligned offsets). */
int wfagpu_pairs_from_metadata(sequence_pair_t *meta, size_t from, size_t n, size_t buf_size,
                               wfagpu_pair_t *pairs, size_t *base_out, size_t *bytes_out)
{
    if (!meta || !pairs || n == 0) return -1;
    sequence_pair_t *m = meta + from;
    const size_t base = m[0].pattern_offset;
    const size_t last = m[n - 1].text_offset + m[n - 1].text_len + 1;
    if (last < base || last > buf_size) {
        fprintf(stderr, "[!] ERROR: Reading out of sequences buffer. Aborting.\n");
        return -1;
    }
    const size_t bytes = last - base;
    if (bytes >= ((size_t)1 << 32)) {
        fprintf(stderr, "[!] ERROR: a batch of %zu pairs spans %zu bytes; lower the batch size (32-bit offsets).\n", n, bytes);
        return -1;
    }
    size_t words = 0;
    for (size_t i = 0; i < n; ++i) {
        wfagpu_pair_t *p = &pairs[i];
        if (m[i].pattern_offset < base || m[i].text_offset < base ||
            m[i].pattern_offset + m[i].pattern_len > last || m[i].text_offset + m[i].text_len > last) {
            fprintf(stderr, "[!] ERROR: sequence metadata is not laid out in increasing offsets.\n");
            return -1;
        }
        if (((m[i].pattern_offset - base) | (m[i].text_offset - base)) & 3) {
            /* the pack kernel reads 16-byte vectors and selects words: sequences start on 4-byte boundaries
             * (the layout of lib/aligner.c:127-166 and of the readers) */
            fprintf(stderr, "[!] ERROR: sequence %zu does not start on a 4-byte boundary of the batch.\n", from + i);
            return -1;
        }
        if (m[i].pattern_len >= WFAGPU_MAX_SEQ_LEN || m[i].text_len >= WFAGPU_MAX_SEQ_LEN) {
            fprintf(stderr, "[!] ERROR: pair %zu has a sequence of %u bases; the limit is %zu.\n", from + i,
                    m[i].pattern_len > m[i].text_len ? m[i].pattern_len : m[i].text_len, (size_t)WFAGPU_MAX_SEQ_LEN - 1);
            return -1;
        }
        p->p_ascii = (uint32_t)(m[i].pattern_offset - base);
        p->t_ascii = (uint32_t)(m[i].text_offset - base);
        p->plen = m[i].pattern_len;
        p->tlen = m[i].text_len;
        p->p_word = p->t_word = 0;
        p->flags = 0;
        p->reserved = 0;
        /* the reference rewrites the packed offsets of every batch (lib/align.cu:103-115, 363-377) */
        m[i].pattern_offset_packed = words * 4;
        words += ((((size_t)p->plen + 7) >> 3) + 1 + 3) & ~(size_t)3;
        m[i].text_offset_packed = words * 4;
        words += ((((size_t)p->tlen + 7) >> 3) + 1 + 3) & ~(size_t)3;
    }
    if (base_out) *base_out = base;
    if (bytes_out) *bytes_out = bytes;
    return 0;
}

static void fill_plan(const job_t *j, bool cigar, wfagpu_plan_t *plan)
{
    memset(plan, 0, sizeof(*plan));
    plan->x = j->opt.penalties.x;
    plan->o = j->opt.penalties.o;
    plan->e = j->opt.penalties.e;
    plan->max_steps = j->opt.max_error;
    plan->band = j->opt.band;
    plan->band_width = j->opt.threads_per_block;
    plan->with_cigar = cigar;
    plan->threads_hint = j->opt.threads_per_block;
    plan->workers_hint = j->opt.num_workers;
    if (j->p2) { plan->o2 = j->pen2.o2; plan->e2 = j->pen2.e2; }
    plan->with_ends = j->ef && j->coords;
}

/* wfagpu_coords_t of a finished pair from its {k_begin, k_end} (NULL: a global alignment covers both sequences) */
static wfagpu_coords_t coords_of(const sequence_pair_t *m, const int32_t *ends)
{
    const int plen = (int)m->pattern_len, tlen = (int)m->text_len;
    if (!ends) return (wfagpu_coords_t){0, plen, 0, tlen};
    const int kb = ends[0], ke = ends[1];
    const int te = tlen < plen + ke ? tlen : plen + ke;
    return (wfagpu_coords_t){kb < 0 ? -kb : 0, te - ke, kb > 0 ? kb : 0, te};
}

static bool span_is_free(const wfagpu_span_t *sp)
{
    return sp->pattern_begin_free || sp->pattern_end_free || sp->text_begin_free || sp->text_end_free;
}

/* the span of pair i of the job (NULL: a global call) */
static const wfagpu_span_t *span_of(const job_t *j, size_t i)
{
    return j->ef ? j->spans + i * j->span_stride : NULL;
}

static int submit(job_t *j, wfagpu_device_t *d, int slot, inflight_t *f)
{
    if (f->pairs_cap < f->n) {
        free(f->pairs);
        f->pairs = (wfagpu_pair_t *)malloc(f->n * sizeof(wfagpu_pair_t));
        f->pairs_cap = f->n;
    }
    if (f->out_cap < f->n) {
        free(f->out);
        f->out = (wfagpu_pair_out_t *)malloc(f->n * sizeof(wfagpu_pair_out_t));
        f->out_cap = f->n;
    }
    if (!f->pairs || !f->out) return -1;
    size_t base = 0, bytes = 0;
    if (wfagpu_pairs_from_metadata(j->meta, f->from, f->n, j->buf_size, f->pairs, &base, &bytes)) return -1;
    wfagpu_plan_t plan;
    fill_plan(j, j->cigar, &plan);
    const char *src = j->buf + base;
    if (j->pageable) {
        /* A caller that did not get its buffer from this library (calloc'ed like the reference's readers,
         * utils/sequence_reader.c:73-78): copy the chunk into the slot's page-locked staging area with this
         * worker's host threads, so that the upload is asynchronous DMA and overlaps the other slot's kernels. */
        char *stage = wfagpu_device_staging(d, slot, bytes);
        if (!stage) return -1;
        const size_t blk = (size_t)1 << 20;
        const long nblk = (long)((bytes + blk - 1) / blk);
        #pragma omp parallel for schedule(static) num_threads(j->decode_threads) if (nblk > 8)
        for (long b = 0; b < nblk; ++b) {
            const size_t off = (size_t)b * blk;
            memcpy(stage + off, src + off, off + blk <= bytes ? blk : bytes - off);
        }
        src = stage;
    }
    if (wfagpu_device_upload(d, slot, src, bytes, f->pairs, f->n)) return -1;
    f->ef = false;
    for (size_t i = 0; j->ef && !f->ef && i < (j->span_stride ? f->n : 1); ++i) f->ef = span_is_free(span_of(j, f->from + i));
    if (j->span_stride ? wfagpu_device_align_spans(d, slot, f->n, &plan, 0, span_of(j, f->from))
                       : wfagpu_device_align_span(d, slot, f->n, &plan, 0, span_of(j, f->from)))
        return -1;
    f->active = true;
    return 0;
}

/* check_correctness (the reference: lib/align.cu:258-326 validates the CIGAR with check_cigar_edit /
 * check_affine_distance and compares the score with its CPU WFA).  There is no CPU aligner here: the CIGAR is
 * validated on the host (it must be an alignment of the two sequences whose gap-affine cost is the reported
 * score), and the score is compared with an INDEPENDENT GPU computation of the same chunk -- score only, through
 * the one-diagonal-per-thread kernels without per-pair bounds, snapshots or provisioning hints
 * (wfagpu_device_rescore).  A wrong optimum or a wrong path is counted as incorrect. */
static void check_chunk(job_t *j, wfagpu_device_t *d, int slot, inflight_t *f)
{
    const sequence_pair_t *m = j->meta + f->from;
    const wfa_alignment_result_t *res = j->res + f->from;
    int32_t *ref = (int32_t *)malloc(f->n * sizeof(int32_t));
    wfagpu_plan_t plan;
    fill_plan(j, false, &plan);
    plan.band = 0;                                            /* the exact optimum, also for banded runs */
    const bool have_ref = ref && (j->span_stride ? wfagpu_device_rescore_spans(d, slot, f->n, &plan, span_of(j, f->from), ref)
                                                 : wfagpu_device_rescore_span(d, slot, f->n, &plan, span_of(j, f->from), ref)) == 0;
    long bad = 0, sum = 0;
    #pragma omp parallel for schedule(dynamic, 64) num_threads(j->decode_threads) reduction(+:bad,sum) if (f->n > 256)
    for (long i = 0; i < (long)f->n; ++i) {
        if (!(f->out[i].status & WFAGPU_ST_FINISHED)) continue;
        bool ok = true;
        if (j->cigar && j->p2)
            ok = wfagpu_check_result_affine2p(j->buf + m[i].pattern_offset, m[i].pattern_len, j->buf + m[i].text_offset,
                                              m[i].text_len, &j->pen2, res[i].error, res[i].cigar.buffer);
        else if (j->cigar)
            ok = wfagpu_check_result_span(j->buf + m[i].pattern_offset, m[i].pattern_len, j->buf + m[i].text_offset,
                                          m[i].text_len, j->opt.penalties, span_of(j, f->from + (size_t)i), res[i].error,
                                          res[i].cigar.buffer);
        /* a banded score may legitimately exceed the optimum; an exact one must equal it */
        if (have_ref && ref[i] >= 0 && (j->opt.band > 0 ? (long)res[i].error < ref[i] : (long)res[i].error != ref[i])) {
            fprintf(stderr, "[!] ERROR: Incorrect distance (%zu). GPU=%u, independent GPU check=%d\n", f->from + (size_t)i,
                    res[i].error, ref[i]);
            ok = false;
        }
        if (!ok) bad++;
        sum += res[i].error;
    }
    free(ref);
    pthread_mutex_lock(&j->mu);
    j->checked += f->n;
    j->incorrect += (uint64_t)bad;
    pthread_mutex_unlock(&j->mu);
    fprintf(stderr, "(Batch from %zu) correct=%ld Incorrect=%ld Average score=%f%s\n", f->from, (long)f->n - bad, bad,
            f->n ? (double)sum / (double)f->n : 0.0, have_ref ? "" : " (scores not re-computed)");
}

static int collect(job_t *j, wfagpu_device_t *d, int slot, inflight_t *f, wfagpu_run_stats_t *acc)
{
    uint32_t *ops = NULL;
    size_t ops_used = 0;
    const double t_a = now_s();
    if (wfagpu_device_download(d, slot, f->n, f->out, &ops, &ops_used, NULL)) return -1;
    const double t_b = now_s();
    f->active = false;
    wfagpu_batch_stats_t bs;
    wfagpu_device_last_stats(d, slot, &bs);
    acc->gpu_align_ms += bs.ms_align;
    acc->gpu_pack_ms += bs.ms_pack;
    acc->redispatched += bs.redispatched;
    acc->ascii_pairs += bs.ascii_pairs;
    acc->h2d_bytes += bs.h2d_bytes;

    const char *text = NULL;
    size_t text_bytes = 0;
    const wfagpu_cigar_ref_t *refs = NULL;
    if (j->cigar && !j->host_cigar) {
        if (wfagpu_device_download_text(d, slot, f->n, &text, &text_bytes, &refs)) return -1;
        wfagpu_device_last_stats(d, slot, &bs);
    }
    if (f->ef && (j->coords || (j->cigar && j->host_cigar))) {
        /* the coordinates and the host decoder need the diagonals every alignment starts and ends on */
        free(f->ends);
        f->ends = (int32_t *)malloc(2 * f->n * sizeof(int32_t));
        if (!f->ends || wfagpu_device_download_ends(d, slot, f->n, f->ends)) return -1;
    }
    acc->launches += bs.launches;
    acc->d2h_bytes += bs.d2h_bytes;
    const double t_c = now_s();

    const sequence_pair_t *m = j->meta + f->from;
    wfa_alignment_result_t *res = j->res + f->from;
    int bad = 0, failed = 0;
    const int nthreads = j->decode_threads;
    #pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads) reduction(+:bad,failed) if (f->n > 256)
    for (long i = 0; i < (long)f->n; ++i) {
        const wfagpu_pair_out_t *o = &f->out[i];
        if (o->status & WFAGPU_ST_FAILED) {
            /* the GPU cannot finish this pair and nothing is computed on the CPU: never report a score for it */
            res[i].error = UINT_MAX;
            failed++;
            continue;
        }
        if (!(o->status & WFAGPU_ST_FINISHED)) { bad++; continue; }
        res[i].error = (unsigned int)o->distance;
        if (j->coords) j->coords[f->from + (size_t)i] = coords_of(&m[i], f->ef ? f->ends + 2 * i : NULL);
        if (j->cigar && refs) {
            /* text was printed on the GPU: append it to the caller's buffer */
            if (!wfagpu_cigar_append(&res[i].cigar, text + refs[i].off, refs[i].len)) bad++;
        } else if (j->cigar && f->ef) {
            if (!wfagpu_ops_to_cigar_span(j->buf + m[i].pattern_offset, m[i].pattern_len, j->buf + m[i].text_offset,
                                          m[i].text_len, f->ends[2 * i], ops + o->ops_off, o->n_ops, &res[i].cigar))
                bad++;
        } else if (j->cigar) {
            if (!wfagpu_ops_to_cigar(j->buf + m[i].pattern_offset, m[i].pattern_len, j->buf + m[i].text_offset,
                                     m[i].text_len, o->distance, ops + o->ops_off, o->n_ops, &res[i].cigar))
                bad++;
        }
    }
    if (failed) {
        pthread_mutex_lock(&j->mu);
        for (size_t i = 0; i < f->n && j->n_first_failed < 8; ++i)
            if (f->out[i].status & WFAGPU_ST_FAILED) j->first_failed[j->n_first_failed++] = f->from + i;
        j->failed_pairs += (uint64_t)failed;
        pthread_mutex_unlock(&j->mu);
    }
    if (bad) {
        fprintf(stderr, "[!] ERROR: %d alignments of the batch starting at %zu were not completed on the GPU.\n", bad, f->from);
        return -1;
    }
    if (j->check) check_chunk(j, d, slot, f);
    if (j->verbose)
        fprintf(stderr, "[wfagpu] chunk from=%zu n=%zu: wait+download %.2f ms, text %.2f ms, host results %.2f ms (kernel %.2f ms)\n",
                f->from, f->n, (t_b - t_a) * 1e3, (t_c - t_b) * 1e3, (now_s() - t_c) * 1e3, bs.ms_align);
    return 0;
}

static void *worker_main(void *arg)
{
    worker_t *w = (worker_t *)arg;
    job_t *j = w->job;
    wfagpu_device_t *d = wfagpu_device_open(w->dev);
    if (!d) { fail_job(j); return NULL; }
    inflight_t fl[2];
    memset(fl, 0, sizeof(fl));
    wfagpu_run_stats_t acc;
    memset(&acc, 0, sizeof(acc));
    int slot = 0;
    bool ok = true;
    while (ok) {
        size_t from, n;
        const bool got = take_chunk(w, &from, &n);
        if (got) {
            fl[slot].from = from;
            fl[slot].n = n;
            if (submit(j, d, slot, &fl[slot])) { ok = false; break; }
        }
        const int other = slot ^ 1;
        if (fl[other].active && collect(j, d, other, &fl[other], &acc)) { ok = false; break; }
        if (!got) {
            if (fl[slot].active && collect(j, d, slot, &fl[slot], &acc)) ok = false;
            break;
        }
        slot = other;
    }
    if (!ok) fail_job(j);
    for (int s = 0; s < 2; ++s) { free(fl[s].pairs); free(fl[s].out); free(fl[s].ends); }
    wfagpu_device_release(d);
    pthread_mutex_lock(&j->mu);
    j->stats.gpu_align_ms += acc.gpu_align_ms;
    j->stats.gpu_pack_ms += acc.gpu_pack_ms;
    j->stats.launches += acc.launches;
    j->stats.redispatched += acc.redispatched;
    j->stats.ascii_pairs += acc.ascii_pairs;
    j->stats.h2d_bytes += acc.h2d_bytes;
    j->stats.d2h_bytes += acc.d2h_bytes;
    pthread_mutex_unlock(&j->mu);
    return NULL;
}

/* How the pair range is cut: chunks of at most `batch_size` pairs; at least two chunks per worker so that
 * uploads hide behind kernels and the tail balances -- eight per worker once a worker's share reaches 32768
 * pairs, as long as a chunk keeps >= 1024 pairs (measured on B200, one 8192 x 10 kbp call: 2 x 4096 32.5 ms,
 * 4 x 2048 33.5 ms, 8 x 1024 37.6 ms: every launch has a ragged tail of one pair's run time); a chunk's ASCII
 * stays below the 32-bit offset limit of the device descriptors. */
void wfagpu_plan_chunks(size_t n, size_t batch_size, int n_devices, size_t ascii_span,
                        size_t *chunk_out, size_t *n_chunks_out)
{
    size_t chunk = batch_size;
    if (n == 0) { *chunk_out = 0; *n_chunks_out = 0; return; }
    if (chunk == 0 || chunk > n) chunk = n;
    if (n_devices < 1) n_devices = 1;
    const size_t share = (n + (size_t)n_devices - 1) / (size_t)n_devices;
    const size_t parts = share >= 32768 ? 8 : 2;
    const size_t per = (share + parts - 1) / parts;
    if (per < chunk && (per >= 1024 || n_devices > 1)) chunk = per;
    const size_t avg = ascii_span / n + 1;
    const size_t max_pairs = ((size_t)3 << 30) / avg;
    if (max_pairs > 0 && chunk > max_pairs) chunk = max_pairs;
    if (chunk == 0) chunk = 1;
    *chunk_out = chunk;
    *n_chunks_out = (n + chunk - 1) / chunk;
}

static void run_job(char *buf, size_t buf_size, sequence_pair_t *meta, wfa_alignment_result_t *res,
                    wfa_alignment_options_t opt, bool cigar, bool check, const wfagpu_span_t *ends_free,
                    size_t span_stride, const wfagpu_affine2p_t *affine2p, wfagpu_coords_t *coords)
{
    const double t0 = now_s();
    memset(&t_last_stats, 0, sizeof(t_last_stats));
    t_last_ok = false;
    if (!buf || !meta || !res) { fprintf(stderr, "[!] ERROR: invalid buffers.\n"); return; }
    if (affine2p) {
        const wfagpu_affine2p_t *q = affine2p;
        if (q->x < 1 || q->o1 < 0 || q->e1 < 1 || q->o2 < 0 || q->e2 < 1) {
            fprintf(stderr, "[!] ERROR: gap-affine 2-piece penalties must satisfy x >= 1, o1, o2 >= 0, e1, e2 >= 1.\n");
            return;
        }
        if (opt.band > 0) {
            fprintf(stderr, "[!] ERROR: gap-affine 2-piece alignment cannot be combined with the adaptive band (-B).\n");
            return;
        }
        opt.penalties.x = q->x; opt.penalties.o = q->o1; opt.penalties.e = q->e1;
    }
    if (opt.num_alignments == 0) { t_last_ok = true; return; }
    if (opt.penalties.x < 1 || opt.penalties.e < 1 || opt.penalties.o < 0) {
        /* x = 0 or e = 0 make a wavefront depend on itself; the reference reads
         * half-written memory in that case (lib/kernels/sequence_alignment_kernel.cu:149-152) */
        fprintf(stderr, "[!] ERROR: penalties must satisfy x >= 1, e >= 1, o >= 0.\n");
        return;
    }
    /* every span is checked before anything is aligned */
    bool ef = false;
    for (size_t i = 0; ends_free && i < (span_stride ? opt.num_alignments : 1); ++i) {
        const wfagpu_span_t *sp = ends_free + i * span_stride;
        if (sp->pattern_begin_free < 0 || sp->pattern_end_free < 0 || sp->text_begin_free < 0 || sp->text_end_free < 0) {
            fprintf(stderr, "[!] ERROR: ends-free span values must be >= 0 (pair %zu: %d,%d,%d,%d).\n", i,
                    sp->pattern_begin_free, sp->pattern_end_free, sp->text_begin_free, sp->text_end_free);
            return;
        }
        ef = ef || span_is_free(sp);
    }
    if (ef && opt.band > 0) {
        fprintf(stderr, "[!] ERROR: ends-free alignment cannot be combined with the adaptive band (-B).\n");
        return;
    }
    if (ef && affine2p) {
        fprintf(stderr, "[!] ERROR: gap-affine 2-piece alignment cannot be combined with an ends-free span.\n");
        return;
    }
    int devs[MAX_DEVICES];
    const int ndev = select_devices(devs);
    if (ndev < 1) return;

    job_t job;
    memset(&job, 0, sizeof(job));
    job.buf = buf; job.buf_size = buf_size; job.meta = meta; job.res = res; job.opt = opt; job.cigar = cigar;
    job.check = check;
    job.ef = ef;
    job.spans = ends_free;
    job.span_stride = span_stride;
    job.p2 = affine2p != NULL;
    if (affine2p) job.pen2 = *affine2p;
    job.coords = coords;
    if (coords)
        for (size_t i = 0; i < opt.num_alignments; ++i) coords[i] = (wfagpu_coords_t){-1, -1, -1, -1};   /* until aligned */
    job.n = opt.num_alignments;
    job.pageable = !wfagpu_host_is_pinned(buf);
    const size_t span = meta[job.n - 1].text_offset + meta[job.n - 1].text_len + 1 - meta[0].pattern_offset;
    size_t chunk = 0, n_chunks_unused = 0;
    /* `batch_size` is an upper bound a caller sets to limit what one device batch holds.  The value
     * wfagpu_set_default_options puts there (a tenth of the pairs, lib/alignment_parameters.h:100-104) is not such a
     * request: 819-pair batches of an 8192-pair call leave every launch with a ragged tail (43 ms per call against
     * 32.5 ms with two chunks, B200) -- the default means "the library plans the chunks". */
    size_t batch = opt.batch_size;
    if (batch == (job.n > 10 ? job.n / 10 : job.n)) batch = job.n;
    wfagpu_plan_chunks(job.n, batch, ndev, span, &chunk, &n_chunks_unused);
    job.chunk = chunk;
    job.n_chunks = (job.n + chunk - 1) / chunk;
    /* Ramp-up: the upload of a worker's first chunk cannot hide behind kernels, so that chunk is smaller than the
     * others -- but never so small that its kernels leave the GPU half empty: at least 10 pairs per SM
     * (measured on B200, 8192 x 10 kbp: first chunk 512 of 2048 -> 37.7 ms per call, no ramp -> 33.5 ms).
     * WFAGPU_RAMP=0 disables, WFAGPU_FIRST_CHUNK=n sets the size. */
    job.first_chunk = chunk;
    {
        const char *rp = getenv("WFAGPU_RAMP");
        const char *fc = getenv("WFAGPU_FIRST_CHUNK");
        const int ramp = rp ? atoi(rp) : 4;
        size_t first = chunk;
        if (fc && atol(fc) > 0) first = (size_t)atol(fc);
        else if (ramp > 1 && job.n_chunks >= (size_t)4 * (size_t)ndev) {
            const int sms = get_cuda_SM_count(devs[0]);
            const size_t floor_pairs = (size_t)10 * (size_t)(sms > 0 ? sms : 148);
            first = chunk / (size_t)ramp;
            if (first < floor_pairs) first = floor_pairs;
        } else if (ramp > 1 && opt.band <= 0 && job.n_chunks >= (size_t)2 * (size_t)ndev && (span / job.n) * chunk >= ((size_t)16 << 20)) {
            /* two big chunks per worker (long reads): half a chunk first -- its upload (and the bound pass the launch
             * waits for) is the exposed part of the call (measured on B200, 8192 x 10 kbp: 4096 + 4096 -> 31.6 ms,
             * 2048 + 4096 + 2048 -> 30.7 ms; the banded launch does not wait for anything: 28.8 against 29.8 ms) */
            const int sms = get_cuda_SM_count(devs[0]);
            const size_t floor_pairs = (size_t)10 * (size_t)(sms > 0 ? sms : 148);
            if (chunk / 2 >= floor_pairs) first = chunk / 2;
        }
        if (first < chunk && first >= 1) {
            job.first_chunk = first;
            job.n_chunks += (size_t)ndev;         /* upper bound: used to size the worker pool only */
        }
    }
    pthread_mutex_init(&job.mu, NULL);
    /* host threads per GPU worker for the result loop: respect OMP_NUM_THREADS (torchrun sets it to 1
     * per rank) and never oversubscribe when several workers share the box */
    int cores = omp_get_num_procs();
    if (omp_get_max_threads() < cores) cores = omp_get_max_threads();
    const char *ht = getenv("WFAGPU_HOST_THREADS");
    if (ht && atoi(ht) > 0) cores = atoi(ht);
    job.decode_threads = cores / ndev > 0 ? cores / ndev : 1;
    const char *vb = getenv("WFAGPU_VERBOSE");
    job.verbose = vb && atoi(vb) != 0;
    const char *hc = getenv("WFAGPU_HOST_CIGAR");
    job.host_cigar = hc && atoi(hc) != 0;
    if (!job.host_cigar && !job.check && job.decode_threads > 4) job.decode_threads = 4;   /* only memcpy of finished text is left */

    const int nworkers = (size_t)ndev < job.n_chunks ? ndev : (int)job.n_chunks;
    job.nworkers = nworkers;
    worker_t workers[MAX_DEVICES];
    pthread_t th[MAX_DEVICES];
    wfagpu_plan_shares(job.n, nworkers, job.share_next, job.share_end);
    for (int i = 0; i < nworkers; ++i) { workers[i].job = &job; workers[i].dev = devs[i]; workers[i].index = i; workers[i].first_taken = false; }
    if (nworkers == 1) {
        worker_main(&workers[0]);
    } else {
        for (int i = 0; i < nworkers; ++i) pthread_create(&th[i], NULL, worker_main, &workers[i]);
        for (int i = 0; i < nworkers; ++i) pthread_join(th[i], NULL);
    }
    pthread_mutex_destroy(&job.mu);
    t_last_stats = job.stats;
    t_last_stats.devices = nworkers;
    t_last_stats.failed_pairs = job.failed_pairs;
    t_last_stats.checked = job.checked;
    t_last_stats.incorrect = job.incorrect;
    t_last_stats.staged = job.pageable ? 1 : 0;
    t_last_stats.wall_s = now_s() - t0;
    t_last_ok = !job.failed && job.failed_pairs == 0;
    if (job.failed_pairs) {
        fprintf(stderr, "[!] ERROR: %llu pair(s) could not be aligned on the GPU (error = UINT_MAX, no CIGAR); first indices:",
                (unsigned long long)job.failed_pairs);
        for (int i = 0; i < job.n_first_failed; ++i) fprintf(stderr, " %zu", job.first_failed[i]);
        fprintf(stderr, "\n");
    }
    if (job.failed) fprintf(stderr, "[!] ERROR: alignment failed on the GPU (no CPU fallback exists in this library).\n");
}

void launch_alignments(char *sequences_buffer, const size_t sequences_buffer_size,
                       sequence_pair_t *const sequences_metadata,
                       wfa_alignment_result_t *const alignment_results,
                       wfa_alignment_options_t options, bool check_correctness)
{
    run_job(sequences_buffer, sequences_buffer_size, sequences_metadata, alignment_results, options, true,
            check_correctness, NULL, 0, NULL, NULL);
}

void launch_alignments_distance(char *sequences_buffer, const size_t sequences_buffer_size,
                                sequence_pair_t *const sequences_metadata,
                                wfa_alignment_result_t *const alignment_results,
                                wfa_alignment_options_t options, bool check_correctness)
{
    run_job(sequences_buffer, sequences_buffer_size, sequences_metadata, alignment_results, options, false,
            check_correctness, NULL, 0, NULL, NULL);
}

void wfagpu_launch_alignments_span(char *sequences_buffer, size_t sequences_buffer_size,
                                   sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                   wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                   const wfagpu_span_t *span)
{
    run_job(sequences_buffer, sequences_buffer_size, sequences_metadata, alignment_results, options, cigar,
            check_correctness, span, 0, NULL, NULL);
}

void wfagpu_launch_alignments_span_coords(char *sequences_buffer, size_t sequences_buffer_size,
                                          sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                          wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                          const wfagpu_span_t *span, wfagpu_coords_t *coords)
{
    run_job(sequences_buffer, sequences_buffer_size, sequences_metadata, alignment_results, options, cigar,
            check_correctness, span, 0, NULL, coords);
}

void wfagpu_launch_alignments_spans(char *sequences_buffer, size_t sequences_buffer_size,
                                    sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                    wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                    const wfagpu_span_t *spans, wfagpu_coords_t *coords)
{
    run_job(sequences_buffer, sequences_buffer_size, sequences_metadata, alignment_results, options, cigar,
            check_correctness, spans, 1, NULL, coords);
}

void wfagpu_launch_alignments_affine2p(char *sequences_buffer, size_t sequences_buffer_size,
                                       sequence_pair_t *sequences_metadata, wfa_alignment_result_t *alignment_results,
                                       wfa_alignment_options_t options, bool cigar, bool check_correctness,
                                       const wfagpu_affine2p_t *pen)
{
    run_job(sequences_buffer, sequences_buffer_size, sequences_metadata, alignment_results, options, cigar,
            check_correctness, NULL, 0, pen, NULL);
}
