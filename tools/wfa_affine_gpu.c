/*
 * wfa_affine_gpu.c -- the command line aligner `bin/wfa.affine.gpu`
 * (replaces tools/aligner.c:58-517 + utils/arg_handler.c of the reference).
 *
 * Same flags, defaults and output format:
 *   -i/--input-seq FILE              .seq input (">pattern" / "<text")
 *   -Q/--input-fasta-query FILE      paired FASTA input ...
 *   -T/--input-fasta-target FILE     ... n-th query record vs n-th target record
 *   -n/--num-alignments N            read only the first N pairs
 *   -g/--affine-penalties x,o,e      default 2,3,1 (signs are stripped)
 *   -x/--compute-cigar               CIGAR (otherwise score only)
 *   -e/--max-distance E              wavefront budget of the first GPU pass
 *                                    (default 0.1 * maxlen(pair 0) * max(x,o,e), at least 20; with -G the maximum
 *                                    of the five values)
 *   -t/--threads-per-block T         hint; the band width when -B is given
 *   -b/--batch-size B, -w/--workers W
 *   -B/--band L                      adaptive band, re-centred every L scores; "auto"/0 = 25
 *   -c/--check                       validate every result: CIGAR on the host, score against an independent GPU pass
 *   -F/--ends-free P0,Pf,T0,Tf       ends-free alignment (WFA2-lib's order): that many leading / trailing pattern and
 *                                    text bases are free; not with -B
 *   -E/--ends-free-file FILE         ends-free with a span per pair: one "P0,Pf,T0,Tf" line per pair, in input order
 *                                    (as many lines as pairs read); not with -F, -B or -G
 *   -G/--affine2p-penalties x,o1,e1,o2,e2
 *                                    gap-affine 2-piece penalties (WFA2-lib's affine2p): a gap of L bases costs
 *                                    min(o1 + e1 L, o2 + e2 L); signs are stripped, e1, e2 >= 1; not with -g, -B or -F
 *   -P/--print-coords                append where each alignment lies: pattern_begin, pattern_end, text_begin, text_end
 *                                    (pattern[pb, pe) against text[tb, te); the full sequences without -F); not with -G
 *   -o/--output-file FILE, -p/--print-output, -O/--output-verbose
 * Output lines: "-score\tCIGAR" (then "\tpb\tpe\ttb\tte" with -P, then "\tpattern\ttext" with -O).
 * Pairs whose score exceeds -e are NOT sent to a CPU: they are re-dispatched on the GPU.
 * Extra: -D/--devices SPEC ("all", "n:4", "0,1") shards the batches over several GPUs;
 *        -S/--stream N streams the input in windows of N pairs (the next window is read into page-locked memory
 *        while the GPU aligns the current one; automatic for inputs above 2 GiB).
 */
#include <limits.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "wfagpu_b200.h"

typedef struct {
    const char *seq, *fq, *ft, *out, *pen, *devices, *ends_free, *pen2, *span_file;
    long n, e, t, b, w, band, stream;
    int have_e, have_t, have_b, have_w, have_band, have_stream, cigar, check, print, verbose, coords;
} args_t;

static void usage(void)
{
    fprintf(stderr,
            "Options:\n[Input/Output]\n"
            "\t-i, --input-seq FILE            sequences in .seq format\n"
            "\t-Q, --input-fasta-query FILE    query sequences (FASTA)\n"
            "\t-T, --input-fasta-target FILE   target sequences (FASTA)\n"
            "\t-n, --num-alignments N          number of alignments to read (default all)\n"
            "\t-o, --output-file FILE          where the alignment output is saved\n"
            "\t-p, --print-output              print the output to stderr\n"
            "\t-O, --output-verbose            add query/target to the output\n"
            "\t-P, --print-coords              add the aligned intervals: pattern begin, end, text begin, end\n"
            "[Alignment Options]\n"
            "\t-g, --affine-penalties x,o,e    gap-affine penalties (default 2,3,1)\n"
            "\t-x, --compute-cigar             compute the CIGAR, not only the score\n"
            "\t-e, --max-distance E            error budget of the first GPU pass\n"
            "\t-b, --batch-size B              alignments per batch\n"
            "\t-B, --band L                    banded heuristic, re-centre every L scores (auto = 25)\n"
            "\t-c, --check                     check the alignments\n"
            "\t-F, --ends-free P0,Pf,T0,Tf     ends-free: free leading/trailing pattern (P) and text (T) bases\n"
            "\t-E, --ends-free-file FILE       ends-free with one P0,Pf,T0,Tf line per pair, in input order\n"
            "\t-G, --affine2p-penalties x,o1,e1,o2,e2  gap-affine 2-piece: a gap of L costs min(o1+e1*L, o2+e2*L)\n"
            "[System]\n"
            "\t-t, --threads-per-block T       threads per alignment (band width with -B)\n"
            "\t-w, --workers W                 GPU workers (hint)\n"
            "\t-D, --devices SPEC              GPUs to use: all, n:<count> or a list 0,1,..\n"
            "\t-S, --stream N                  read / align / write N pairs at a time (0 = 65536); reading overlaps the GPU\n"
            "[Examples]\n"
            "\t./bin/wfa.affine.gpu -i sequences.seq -b <batch_size> -o scores.out\n"
            "\t./bin/wfa.affine.gpu -i sequences.seq -b <batch_size> -B auto -o scores-banded.out\n"
            "\t./bin/wfa.affine.gpu -Q queries.fasta -T targets.fasta -b <batch_size> -x -o cigars.out\n");
}

static const struct { char s; const char *l; int has_val; } OPTS[] = {
    {'i', "input-seq", 1}, {'Q', "input-fasta-query", 1}, {'T', "input-fasta-target", 1}, {'n', "num-alignments", 1},
    {'g', "affine-penalties", 1}, {'x', "compute-cigar", 0}, {'c', "check", 0}, {'e', "max-distance", 1},
    {'t', "threads-per-block", 1}, {'b', "batch-size", 1}, {'w', "workers", 1}, {'B', "band", 1},
    {'o', "output-file", 1}, {'p', "print-output", 0}, {'O', "output-verbose", 0}, {'D', "devices", 1},
    {'S', "stream", 1}, {'F', "ends-free", 1}, {'G', "affine2p-penalties", 1}, {'P', "print-coords", 0},
    {'E', "ends-free-file", 1},
};

static int parse(int argc, char **argv, args_t *a)
{
    int seen = 0;
    for (int i = 1; i < argc; ++i) {
        const char *arg = argv[i];
        if (arg[0] != '-') continue;                       /* stray values are ignored like the reference does */
        int idx = -1;
        for (size_t k = 0; k < sizeof(OPTS) / sizeof(OPTS[0]); ++k) {
            if (arg[1] == '-' ? !strcmp(arg + 2, OPTS[k].l) : (arg[1] == OPTS[k].s && arg[2] == 0)) idx = (int)k;
        }
        if (idx < 0) continue;
        const char *val = NULL;
        if (OPTS[idx].has_val) {
            if (i + 1 >= argc) { fprintf(stderr, "Error parsing argument: %s.\n", OPTS[idx].l); return 0; }
            val = argv[++i];
        }
        ++seen;
        switch (OPTS[idx].s) {
        case 'i': a->seq = val; break;
        case 'Q': a->fq = val; break;
        case 'T': a->ft = val; break;
        case 'o': a->out = val; break;
        case 'g': a->pen = val; break;
        case 'D': a->devices = val; break;
        case 'F': a->ends_free = val; break;
        case 'E': a->span_file = val; break;
        case 'G': a->pen2 = val; break;
        case 'S': a->stream = atol(val); a->have_stream = 1; break;
        case 'n': a->n = atoll(val); break;
        case 'e': a->e = atoll(val); a->have_e = 1; break;
        case 't': a->t = atoll(val); a->have_t = 1; break;
        case 'b': a->b = atoll(val); a->have_b = 1; break;
        case 'w': a->w = atoll(val); a->have_w = 1; break;
        case 'B': a->band = atoll(val); a->have_band = 1; break;   /* atoll("auto") == 0 -> 25 */
        case 'x': a->cigar = 1; break;
        case 'c': a->check = 1; break;
        case 'p': a->print = 1; break;
        case 'O': a->verbose = 1; break;
        case 'P': a->coords = 1; break;
        }
    }
    return seen;
}

static double now_s(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* -E: the spans of the next `n` pairs, one "P0,Pf,T0,Tf" line each (surrounding blanks allowed).  0, or -1 with a
 * message for a missing, malformed or negative line. */
static int read_spans(FILE *fp, const char *path, long first_pair, long n, wfagpu_span_t *spans)
{
    char line[256];
    for (long i = 0; i < n; ++i) {
        wfagpu_span_t *sp = &spans[i];
        char tail = 0;
        if (!fgets(line, sizeof(line), fp)) {
            fprintf(stderr, "[!] ERROR: --ends-free-file %s has %ld line(s) but there are more pairs.\n", path, first_pair + i);
            return -1;
        }
        if (sscanf(line, " %d , %d , %d , %d %c", &sp->pattern_begin_free, &sp->pattern_end_free, &sp->text_begin_free,
                   &sp->text_end_free, &tail) != 4 ||
            sp->pattern_begin_free < 0 || sp->pattern_end_free < 0 || sp->text_begin_free < 0 || sp->text_end_free < 0) {
            line[strcspn(line, "\r\n")] = 0;
            fprintf(stderr, "[!] ERROR: --ends-free-file %s line %ld: expected four values >= 0, P0,Pf,T0,Tf (got \"%s\").\n",
                    path, first_pair + i + 1, line);
            return -1;
        }
    }
    return 0;
}

/* -E after the last pair: anything but blank lines left means the file does not match the input */
static int spans_left_over(FILE *fp, const char *path, long pairs)
{
    char line[256];
    while (fgets(line, sizeof(line), fp))
        if (line[strspn(line, " \t\r\n")]) {
            fprintf(stderr, "[!] ERROR: --ends-free-file %s has more lines than the %ld pairs read.\n", path, pairs);
            return -1;
        }
    return 0;
}

/* ---- streaming: window w + 1 is read (into page-locked memory) by a helper thread while the GPU aligns window w ---- */
typedef struct {
    wfagpu_reader_t *reader;
    wfagpu_aligner_t *al;
    size_t want;
    long got;
} fill_t;

static void *fill_main(void *arg)
{
    fill_t *f = (fill_t *)arg;
    wfagpu_clear_sequences(f->al);
    f->got = wfagpu_reader_next(f->reader, f->al, f->want);
    return NULL;
}

int main(int argc, char **argv)
{
    args_t a;
    memset(&a, 0, sizeof(a));
    int ndev = 0;
    get_num_cuda_devices(&ndev);
    if (ndev == 0) { fprintf(stderr, "[!] ERROR: No CUDA devices detected.\n"); return -1; }
    int major = 0, minor = 0;
    get_cuda_capability(0, &major, &minor);
    char *name = get_cuda_dev_name(0);
    fprintf(stderr, "INFO: Using CUDA device \"%s\" with capability %d.%d\n", name ? name : "?", major, minor);
    free(name);

    if (!parse(argc, argv, &a)) { usage(); return 1; }
    if (!a.seq && !(a.fq && a.ft)) { fprintf(stderr, "[!] ERROR: No input file provided.\n"); return 1; }
    FILE *span_fp = NULL;
    if (a.span_file) {
        if (a.ends_free) { fprintf(stderr, "[!] ERROR: --ends-free-file cannot be combined with --ends-free (-F).\n"); return 1; }
        if (a.have_band) { fprintf(stderr, "[!] ERROR: --ends-free-file cannot be combined with the band (-B).\n"); return 1; }
        if (!a.pen2 && !(span_fp = fopen(a.span_file, "r"))) {
            fprintf(stderr, "[!] ERROR: Could not open --ends-free-file %s\n", a.span_file);
            return 1;
        }
    }

    /* -G: gap-affine 2-piece penalties instead of -g */
    wfagpu_affine2p_t pen2 = {0, 0, 0, 0, 0};
    if (a.pen2) {
        if (a.pen) { fprintf(stderr, "[!] ERROR: --affine2p-penalties cannot be combined with --affine-penalties (-g).\n"); return 1; }
        if (a.have_band) { fprintf(stderr, "[!] ERROR: --affine2p-penalties cannot be combined with the band (-B).\n"); return 1; }
        if (a.ends_free) { fprintf(stderr, "[!] ERROR: --affine2p-penalties cannot be combined with --ends-free (-F).\n"); return 1; }
        if (a.span_file) { fprintf(stderr, "[!] ERROR: --affine2p-penalties cannot be combined with --ends-free-file (-E).\n"); return 1; }
        if (a.coords) { fprintf(stderr, "[!] ERROR: --affine2p-penalties cannot be combined with --print-coords (-P).\n"); return 1; }
        if (sscanf(a.pen2, "%d,%d,%d,%d,%d", &pen2.x, &pen2.o1, &pen2.e1, &pen2.o2, &pen2.e2) != 5) {
            fprintf(stderr, "[!] ERROR: --affine2p-penalties takes five values: x,o1,e1,o2,e2 (got %s).\n", a.pen2);
            return 1;
        }
        if (pen2.x < 0) pen2.x = -pen2.x;
        if (pen2.o1 < 0) pen2.o1 = -pen2.o1;
        if (pen2.e1 < 0) pen2.e1 = -pen2.e1;
        if (pen2.o2 < 0) pen2.o2 = -pen2.o2;
        if (pen2.e2 < 0) pen2.e2 = -pen2.e2;
        if (pen2.x < 1 || pen2.e1 < 1 || pen2.e2 < 1) {
            fprintf(stderr, "[!] ERROR: --affine2p-penalties needs x, e1, e2 >= 1 (got %s).\n", a.pen2);
            return 1;
        }
    }
    int x = 2, o = 3, e = 1;
    if (a.pen && sscanf(a.pen, "%d,%d,%d", &x, &o, &e) != 3) {
        fprintf(stderr, "WARNING: Invalid penalties format provided. Using default penalties (0,2,3,1).\n");
        x = 2; o = 3; e = 1;
    }
    if (x < 0) x = -x;
    if (o < 0) o = -o;
    if (e < 0) e = -e;
    if (a.pen2) {
        x = pen2.x; o = pen2.o1; e = pen2.e1;
        fprintf(stderr, "INFO: Gap-affine 2-piece penalties: M=0, X=%d, O1=%d, E1=%d, O2=%d, E2=%d.\n", pen2.x, pen2.o1, pen2.e1,
                pen2.o2, pen2.e2);
    } else {
        fprintf(stderr, "INFO: Penalties: M=0, X=%d, O=%d, E=%d.\n", x, o, e);
    }
    if (a.devices) wfagpu_set_devices(a.devices);

    wfagpu_reader_t *reader = a.seq ? wfagpu_reader_open_seq(a.seq) : wfagpu_reader_open_fasta(a.fq, a.ft);
    if (!reader) return 1;
    /* One window = everything (the reference's behaviour) unless -S asks for windows of N pairs or the input is
     * larger than 2 GiB, in which case it is streamed in windows of 65536 pairs. */
    const long limit = a.n > 0 ? a.n : 0;
    size_t window = 0;
    if (a.have_stream) window = (size_t)(a.stream > 0 ? a.stream : 65536);
    else if (wfagpu_reader_total_bytes(reader) > ((long)2 << 30)) window = 65536;
    if (window && limit && (size_t)limit < window) window = 0;

    wfagpu_aligner_t al[2];
    if (!wfagpu_initialize_aligner(&al[0])) return 1;
    if (window && !wfagpu_initialize_aligner(&al[1])) return 1;
    fprintf(stderr, "INFO: Reading sequences file...\n");
    double t0 = now_s();
    if (!window && !limit && wfagpu_reader_total_bytes(reader) > 0) {
        const size_t tb = (size_t)wfagpu_reader_total_bytes(reader);
        wfagpu_reserve(&al[0], tb + tb / 16 + 4096, 0);              /* one page-locked allocation */
    }
    long first = wfagpu_reader_next(reader, &al[0], window ? window : (size_t)limit);
    if (first <= 0) { fprintf(stderr, "[!] ERROR: Error reading input.\n"); return 1; }
    if (!window) fprintf(stderr, "INFO: File read: %.3fs (%ld pairs)\n", now_s() - t0, first);
    else fprintf(stderr, "INFO: Streaming in windows of %zu pairs (first window read in %.3fs)\n", window, now_s() - t0);

    int max_distance;
    if (a.have_e) {
        max_distance = (int)a.e;
        if (max_distance <= 0) { fprintf(stderr, "[!] ERROR: Maximum error supported by the kernel must be > 0. Aborting.\n"); return -1; }
    } else {
        const sequence_pair_t *m0 = &al[0].sequences_metadata[0];
        max_distance = (int)((m0->text_len > m0->pattern_len ? m0->text_len : m0->pattern_len) * 0.1);
        int pm = x > o ? x : o;
        if (e > pm) pm = e;
        if (a.pen2 && pen2.o2 > pm) pm = pen2.o2;
        if (a.pen2 && pen2.e2 > pm) pm = pen2.e2;
        max_distance *= pm;
        if (max_distance <= 20) max_distance = 20;
        fprintf(stderr, "INFO: No maximum error provided by the user, using %d\n", max_distance);
    }
    int tpb = a.have_t ? (int)a.t : wfa_get_threads_per_alignment((size_t)max_distance);
    if (a.have_b && a.b <= 0) { fprintf(stderr, "[!] ERROR: Incorrect batch size (%ld).\n", a.b); return -1; }
    int workers = a.have_w ? (int)a.w : get_num_workers(tpb);
    wfagpu_span_t span = {0, 0, 0, 0};
    if (a.ends_free) {
        if (sscanf(a.ends_free, "%d,%d,%d,%d", &span.pattern_begin_free, &span.pattern_end_free, &span.text_begin_free,
                   &span.text_end_free) != 4 || span.pattern_begin_free < 0 || span.pattern_end_free < 0 ||
            span.text_begin_free < 0 || span.text_end_free < 0) {
            fprintf(stderr, "[!] ERROR: --ends-free takes four values >= 0: P0,Pf,T0,Tf (got %s).\n", a.ends_free);
            return -1;
        }
        if (a.have_band) { fprintf(stderr, "[!] ERROR: --ends-free cannot be combined with the band (-B).\n"); return -1; }
        fprintf(stderr, "INFO: Ends-free alignment: pattern %d,%d text %d,%d free bases at begin,end.\n",
                span.pattern_begin_free, span.pattern_end_free, span.text_begin_free, span.text_end_free);
    }
    int band = -1;
    if (a.have_band) {
        if (a.band < 0) { fprintf(stderr, "[!] ERROR: Band must positive (band=%ld).\n", a.band); return -1; }
        band = a.band == 0 ? 25 : (int)a.band;
        fprintf(stderr, "INFO: Banded execution. Band width: %d. Band re-centering every %d steps\n", tpb, band);
    }

    FILE *fp = NULL;
    if (a.out || a.print) {
        fp = a.print ? stderr : fopen(a.out, "w");
        if (!fp) { fprintf(stderr, "[!] ERROR: Could not open file %s\n", a.out); return -1; }
    }

    double t_align = 0;
    long total = 0;
    bool ok_run = true;
    wfagpu_run_stats_t sum;
    memset(&sum, 0, sizeof(sum));
    int cur = 0;
    long pairs = first;
    while (pairs > 0) {
        /* start reading the next window while this one is aligned */
        pthread_t th;
        fill_t fill = {reader, &al[cur ^ 1], window, 0};
        bool filling = false;
        const bool more = window && (!limit || total + pairs < limit);
        if (more) {
            if (limit && (size_t)(limit - total - pairs) < fill.want) fill.want = (size_t)(limit - total - pairs);
            filling = pthread_create(&th, NULL, fill_main, &fill) == 0;
            if (!filling) fill_main(&fill);
        }
        wfagpu_aligner_t *A = &al[cur];
        wfa_alignment_result_t *results = NULL;
        if (!initialize_wfa_results(&results, (size_t)pairs, (size_t)max_distance * 5)) {
            fprintf(stderr, "[!] ERROR: Can not initialise CIGAR buffer.\n");
            return -1;
        }
        wfagpu_coords_t *coords = a.coords ? (wfagpu_coords_t *)malloc((size_t)pairs * sizeof(wfagpu_coords_t)) : NULL;
        if (a.coords && !coords) { fprintf(stderr, "[!] ERROR: Can not allocate the coordinates.\n"); return -1; }
        wfagpu_span_t *spans = span_fp ? (wfagpu_span_t *)malloc((size_t)pairs * sizeof(wfagpu_span_t)) : NULL;
        if (span_fp && (!spans || read_spans(span_fp, a.span_file, total, pairs, spans))) return -1;
        if (span_fp && !more && spans_left_over(span_fp, a.span_file, total + pairs)) return -1;   /* the last window */
        wfa_alignment_options_t opt;
        memset(&opt, 0, sizeof(opt));
        opt.max_error = max_distance;
        opt.threads_per_block = tpb;
        opt.num_workers = workers;
        opt.band = band;
        opt.batch_size = a.have_b ? ((size_t)a.b < (size_t)pairs ? (size_t)a.b : (size_t)pairs)
                                  : ((size_t)pairs > 10 ? (size_t)pairs / 10 : (size_t)pairs);   /* library default: it plans the chunks */
        opt.num_alignments = (size_t)pairs;
        opt.penalties.x = x; opt.penalties.o = o; opt.penalties.e = e;
        opt.compute_cigar = a.cigar;

        t0 = now_s();
        if (a.pen2)
            wfagpu_launch_alignments_affine2p(A->sequences_buffer, A->sequences_buffer_len, A->sequences_metadata, results,
                                              opt, a.cigar, a.check, &pen2);
        else if (spans)
            wfagpu_launch_alignments_spans(A->sequences_buffer, A->sequences_buffer_len, A->sequences_metadata, results,
                                           opt, a.cigar, a.check, spans, coords);
        else if (a.ends_free || a.coords)
            wfagpu_launch_alignments_span_coords(A->sequences_buffer, A->sequences_buffer_len, A->sequences_metadata,
                                                 results, opt, a.cigar, a.check, a.ends_free ? &span : NULL, coords);
        else if (a.cigar) launch_alignments(A->sequences_buffer, A->sequences_buffer_len, A->sequences_metadata, results, opt, a.check);
        else launch_alignments_distance(A->sequences_buffer, A->sequences_buffer_len, A->sequences_metadata, results, opt, a.check);
        t_align += now_s() - t0;
        ok_run = ok_run && wfagpu_last_launch_ok();
        wfagpu_run_stats_t st;
        wfagpu_last_run_stats(&st);
        sum.launches += st.launches; sum.redispatched += st.redispatched; sum.ascii_pairs += st.ascii_pairs;
        sum.checked += st.checked; sum.incorrect += st.incorrect; sum.failed_pairs += st.failed_pairs;
        if (st.devices > sum.devices) sum.devices = st.devices;

        if (fp) {
            for (long i = 0; i < pairs; ++i) {
                const sequence_pair_t *m = &A->sequences_metadata[i];
                const char *cigar = a.cigar ? results[i].cigar.buffer : "";
                if (results[i].error == UINT_MAX) {              /* the GPU could not finish this pair: no score is invented */
                    fprintf(fp, "NA\t\n");
                    continue;
                }
                fprintf(fp, "%d\t%s", -(int)results[i].error, cigar);
                if (coords)
                    fprintf(fp, "\t%d\t%d\t%d\t%d", coords[i].pattern_begin, coords[i].pattern_end, coords[i].text_begin,
                            coords[i].text_end);
                if (a.verbose)
                    fprintf(fp, "\t%s\t%s", A->sequences_buffer + m->pattern_offset, A->sequences_buffer + m->text_offset);
                fputc('\n', fp);
            }
        }
        free(coords);
        free(spans);
        destroy_wfa_results(results, (size_t)pairs);
        total += pairs;
        pairs = 0;
        if (more) {
            if (filling) pthread_join(th, NULL);
            if (fill.got < 0) { fprintf(stderr, "[!] ERROR: Error reading input.\n"); ok_run = false; break; }
            pairs = fill.got;
            cur ^= 1;
        }
    }
    if (span_fp && ok_run && spans_left_over(span_fp, a.span_file, total)) return -1;
    if (span_fp) fclose(span_fp);
    printf("Alignment computed. Wall time: %.3fs (%.3f alignments per second)\n", t_align, (double)total / t_align);
    fprintf(stderr, "INFO: %d GPU(s), %llu kernel launches, %llu pairs re-dispatched on the GPU, %llu byte-compare pairs\n",
            sum.devices, (unsigned long long)sum.launches, (unsigned long long)sum.redispatched,
            (unsigned long long)sum.ascii_pairs);
    if (a.check)
        /* validated inside the library, batch by batch (CIGAR on the host, score against an independent GPU pass) */
        fprintf(stderr, "DEBUG: (all batches) correct=%llu Incorrect=%llu\n",
                (unsigned long long)(sum.checked - sum.incorrect), (unsigned long long)sum.incorrect);
    if (fp && !a.print) fclose(fp);
    wfagpu_reader_close(reader);
    wfagpu_destroy_aligner(&al[0]);
    if (window) wfagpu_destroy_aligner(&al[1]);
    wfagpu_device_close_all();
    return ok_run ? 0 : 2;
}
