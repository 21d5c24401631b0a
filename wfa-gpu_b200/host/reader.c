/*
 * reader.c -- input formats of the CLI (replaces utils/sequence_reader.c:137-392).
 *
 *   .seq   : one pair per two lines, ">PATTERN" then "<TEXT"; blank lines are skipped.
 *   FASTA  : two files, the n-th record of the query file pairs with the n-th record of
 *            the target file; sequences may span several lines; header lines start with
 *            '>' (leading blanks allowed).
 *
 * Both fill a wfagpu_aligner_t through wfagpu_add_sequences, i.e. the same host layout
 * (4-byte aligned, NUL padded) the reference readers produce.  Unlike the reference, a
 * final line without a newline keeps its last base and '\r' is dropped.
 */
#define _GNU_SOURCE
#include <stdio.h>
#include <string.h>
#include "wfagpu_b200.h"

static long file_size(FILE *fp)
{
    long sz = -1;
    if (fseek(fp, 0, SEEK_END) == 0) sz = ftell(fp);
    rewind(fp);
    return sz;
}

static size_t chomp(char *line, ssize_t n)
{
    while (n > 0 && (line[n - 1] == '\n' || line[n - 1] == '\r')) line[--n] = 0;
    return (size_t)n;
}

/* ---- incremental readers: the next `max_pairs` pairs of a .seq file or of a FASTA pair go straight into the
 * aligner's page-locked buffer.  The CLI streams with them (window w + 1 is read while the GPU aligns window w)
 * instead of "load everything, then align" (README.md:120-121 of the reference). ---- */
typedef struct { FILE *fp; char *line; size_t cap; bool eof; bool pending_header; } fasta_t;

struct wfagpu_reader {
    bool fasta;
    FILE *fp;              /* .seq */
    char *line;
    size_t cap, lineno;
    fasta_t q, t;          /* FASTA */
    char *qs, *ts;
    size_t qc, tc;
    long total_bytes;      /* size of the input (both files), for one up-front reservation */
};

static bool is_header(const char *s) { while (*s == ' ') ++s; return *s == '>'; }

/* Reads the next record's sequence into *seq (realloc'ed). Returns false when no record is left. */
static bool fasta_next(fasta_t *f, char **seq, size_t *seq_cap)
{
    if (f->eof) return false;
    size_t len = 0;
    bool any = false;
    ssize_t n;
    if (*seq_cap == 0) { *seq_cap = 1 << 16; *seq = (char *)malloc(*seq_cap); }
    (*seq)[0] = 0;
    while ((n = getline(&f->line, &f->cap, f->fp)) != -1) {
        const size_t l = chomp(f->line, n);
        if (l == 0) continue;
        if (is_header(f->line)) {
            if (!f->pending_header) { f->pending_header = true; continue; }  /* very first header */
            return true;                                                       /* next record starts */
        }
        f->pending_header = true;
        if (len + l + 1 > *seq_cap) { while (len + l + 1 > *seq_cap) *seq_cap *= 2; *seq = (char *)realloc(*seq, *seq_cap); }
        memcpy(*seq + len, f->line, l + 1);
        len += l;
        any = true;
    }
    f->eof = true;
    return any;
}

wfagpu_reader_t *wfagpu_reader_open_seq(const char *path)
{
    FILE *fp = fopen(path, "r");
    if (!fp) { fprintf(stderr, "[!] ERROR: Could not open %s\n", path); return NULL; }
    wfagpu_reader_t *r = (wfagpu_reader_t *)calloc(1, sizeof(*r));
    if (!r) { fclose(fp); return NULL; }
    r->fp = fp;
    r->total_bytes = file_size(fp);
    return r;
}

wfagpu_reader_t *wfagpu_reader_open_fasta(const char *query_path, const char *target_path)
{
    FILE *q = fopen(query_path, "r"), *t = fopen(target_path, "r");
    if (!q || !t) {
        fprintf(stderr, "[!] ERROR: Could not open %s\n", !q ? query_path : target_path);
        if (q) fclose(q);
        if (t) fclose(t);
        return NULL;
    }
    wfagpu_reader_t *r = (wfagpu_reader_t *)calloc(1, sizeof(*r));
    if (!r) { fclose(q); fclose(t); return NULL; }
    r->fasta = true;
    r->q.fp = q;
    r->t.fp = t;
    const long a = file_size(q), b = file_size(t);
    r->total_bytes = (a > 0 && b > 0) ? a + b : -1;
    return r;
}

long wfagpu_reader_total_bytes(const wfagpu_reader_t *r) { return r ? r->total_bytes : -1; }

long wfagpu_reader_next(wfagpu_reader_t *r, wfagpu_aligner_t *aligner, size_t max_pairs)
{
    if (!r || !aligner) return -1;
    long pairs = 0;
    bool ok = true;
    if (r->fasta) {
        while (ok && (max_pairs == 0 || (size_t)pairs < max_pairs)) {
            const bool hq = fasta_next(&r->q, &r->qs, &r->qc);
            const bool ht = fasta_next(&r->t, &r->ts, &r->tc);
            if (!hq || !ht) break;
            ok = wfagpu_add_sequences(aligner, r->qs, r->ts);
            ++pairs;
        }
        return ok ? pairs : -1;
    }
    char *pattern = NULL;
    ssize_t n;
    while (ok && (max_pairs == 0 || (size_t)pairs < max_pairs) && (n = getline(&r->line, &r->cap, r->fp)) != -1) {
        ++r->lineno;
        const size_t len = chomp(r->line, n);
        if (len == 0) continue;
        if (!pattern) {
            if (r->line[0] != '>') { fprintf(stderr, "[!] ERROR: Invalid file format. Could not read pattern in line %zu\n", r->lineno); ok = false; break; }
            pattern = strdup(r->line + 1);
        } else {
            if (r->line[0] != '<') { fprintf(stderr, "[!] ERROR: Invalid file format. Could not read text in line %zu\n", r->lineno); ok = false; break; }
            ok = wfagpu_add_sequences(aligner, pattern, r->line + 1);
            free(pattern);
            pattern = NULL;
            ++pairs;
        }
    }
    free(pattern);
    return ok ? pairs : -1;
}

void wfagpu_reader_close(wfagpu_reader_t *r)
{
    if (!r) return;
    if (r->fp) fclose(r->fp);
    if (r->q.fp) fclose(r->q.fp);
    if (r->t.fp) fclose(r->t.fp);
    free(r->line); free(r->q.line); free(r->t.line); free(r->qs); free(r->ts);
    free(r);
}

static long read_all(wfagpu_reader_t *r, wfagpu_aligner_t *aligner, size_t max_pairs)
{
    if (!r) return -1;
    if (max_pairs == 0 && r->total_bytes > 0)
        /* one page-locked allocation for the whole input instead of geometric growth */
        wfagpu_reserve(aligner, (size_t)r->total_bytes + (size_t)r->total_bytes / 16 + 4096, 0);
    const long pairs = wfagpu_reader_next(r, aligner, max_pairs);
    wfagpu_reader_close(r);
    return pairs;
}

long wfagpu_read_seq_file(wfagpu_aligner_t *aligner, const char *path, size_t max_pairs)
{
    return read_all(wfagpu_reader_open_seq(path), aligner, max_pairs);
}

long wfagpu_read_fasta_files(wfagpu_aligner_t *aligner, const char *query_path, const char *target_path, size_t max_pairs)
{
    const long pairs = read_all(wfagpu_reader_open_fasta(query_path, target_path), aligner, max_pairs);
    if (pairs == 0) { fprintf(stderr, "[!] ERROR: Empty FASTA file.\n"); return -1; }
    return pairs;
}

/* -c: validates a result without any CPU aligner (replaces check_cigar_edit +
 * check_affine_distance, utils/verification.c:27-146): the CIGAR must transform the pattern
 * into the text (I consumes text, D consumes pattern) and its gap-affine cost must be `error`. */
bool wfagpu_check_result(const char *pattern, size_t plen, const char *text, size_t tlen,
                         affine_penalties_t pen, unsigned int error, const char *cigar)
{
    size_t v = 0, h = 0;
    unsigned long score = 0;
    const char *c = cigar;
    if (!c) return false;
    while (*c) {
        unsigned long rep = 0;
        if (*c < '0' || *c > '9') return false;
        while (*c >= '0' && *c <= '9') rep = rep * 10 + (unsigned long)(*c++ - '0');
        const char op = *c++;
        if (op == 'M' || op == 'X') {
            if (v + rep > plen || h + rep > tlen) return false;
            for (unsigned long i = 0; i < rep; ++i)
                if ((pattern[v + i] == text[h + i]) != (op == 'M')) return false;
            v += rep; h += rep;
            if (op == 'X') score += rep * (unsigned long)pen.x;
        } else if (op == 'I') { h += rep; score += (unsigned long)pen.o + rep * (unsigned long)pen.e; }
        else if (op == 'D') { v += rep; score += (unsigned long)pen.o + rep * (unsigned long)pen.e; }
        else return false;
        if (v > plen || h > tlen) return false;
    }
    return v == plen && h == tlen && score == error;
}

/* The same under an ends-free span: the first and the last run of the CIGAR, when they are I or D runs, are free up
 * to the span's allowance for that end (wfagpu_b200.h). */
bool wfagpu_check_result_span(const char *pattern, size_t plen, const char *text, size_t tlen,
                              affine_penalties_t pen, const wfagpu_span_t *span, unsigned int error, const char *cigar)
{
    if (!span) return wfagpu_check_result(pattern, plen, text, tlen, pen, error, cigar);
    if (span->pattern_begin_free < 0 || span->pattern_end_free < 0 || span->text_begin_free < 0 || span->text_end_free < 0)
        return false;
    size_t v = 0, h = 0;
    unsigned long score = 0;
    const char *c = cigar;
    bool first = true;
    if (!c) return false;
    while (*c) {
        unsigned long rep = 0;
        if (*c < '0' || *c > '9') return false;
        while (*c >= '0' && *c <= '9') rep = rep * 10 + (unsigned long)(*c++ - '0');
        const char op = *c++;
        const bool last = (*c == 0);
        if (op == 'M' || op == 'X') {
            if (v + rep > plen || h + rep > tlen) return false;
            for (unsigned long i = 0; i < rep; ++i)
                if ((pattern[v + i] == text[h + i]) != (op == 'M')) return false;
            v += rep; h += rep;
            if (op == 'X') score += rep * (unsigned long)pen.x;
        } else if (op == 'I' || op == 'D') {
            unsigned long free_bases = 0;
            if (first) free_bases += (unsigned long)(op == 'I' ? span->text_begin_free : span->pattern_begin_free);
            if (last) free_bases += (unsigned long)(op == 'I' ? span->text_end_free : span->pattern_end_free);
            if (rep > free_bases) score += (unsigned long)pen.o + (rep - free_bases) * (unsigned long)pen.e;
            if (op == 'I') h += rep; else v += rep;
        } else {
            return false;
        }
        if (v > plen || h > tlen) return false;
        first = false;
    }
    return v == plen && h == tlen && score == error;
}

/* The same under gap-affine 2-piece penalties: a gap run of length L costs min(o1 + e1 L, o2 + e2 L). */
bool wfagpu_check_result_affine2p(const char *pattern, size_t plen, const char *text, size_t tlen,
                                  const wfagpu_affine2p_t *pen, unsigned int error, const char *cigar)
{
    if (!pen || pen->x < 1 || pen->o1 < 0 || pen->e1 < 1 || pen->o2 < 0 || pen->e2 < 1) return false;
    size_t v = 0, h = 0;
    unsigned long score = 0;
    const char *c = cigar;
    if (!c) return false;
    while (*c) {
        unsigned long rep = 0;
        if (*c < '0' || *c > '9') return false;
        while (*c >= '0' && *c <= '9') rep = rep * 10 + (unsigned long)(*c++ - '0');
        const char op = *c++;
        if (op == 'M' || op == 'X') {
            if (v + rep > plen || h + rep > tlen) return false;
            for (unsigned long i = 0; i < rep; ++i)
                if ((pattern[v + i] == text[h + i]) != (op == 'M')) return false;
            v += rep; h += rep;
            if (op == 'X') score += rep * (unsigned long)pen->x;
        } else if (op == 'I' || op == 'D') {
            const unsigned long c1 = (unsigned long)pen->o1 + rep * (unsigned long)pen->e1;
            const unsigned long c2 = (unsigned long)pen->o2 + rep * (unsigned long)pen->e2;
            score += c1 < c2 ? c1 : c2;
            if (op == 'I') h += rep; else v += rep;
        } else {
            return false;
        }
        if (v > plen || h > tlen) return false;
    }
    return v == plen && h == tlen && score == error;
}

/* ---------------------------------------------------------------------------------------------
 * The reference library's validators under their own names, argument order (text first) and input format
 * (utils/verification.h:37-58).  The reference hands them the UNROLLED op string that its recover_cigar
 * produces ("MMMXMMIIM", one letter per column; lib/align.cu:284-293); results[i].cigar.buffer holds the
 * run-length text ("3M1X2M2I1M").  Both spellings are accepted: a CIGAR that starts with a digit is read as
 * run-length text, anything else letter by letter.
 * --------------------------------------------------------------------------------------------- */
typedef struct { const char *c; unsigned long left; char op; bool rle; bool bad; } cigar_it_t;

static void cig_begin(cigar_it_t *it, const char *cigar)
{
    it->c = cigar; it->left = 0; it->op = 0; it->bad = false;
    it->rle = cigar && cigar[0] >= '0' && cigar[0] <= '9';
}
/* next column of the alignment: 'M', 'X', 'I', 'D'; 0 at the end (or on malformed run-length text: it->bad) */
static char cig_next(cigar_it_t *it)
{
    if (it->left) { it->left--; return it->op; }
    if (!it->c || !*it->c) return 0;
    if (!it->rle) return *it->c++;
    unsigned long rep = 0;
    if (*it->c < '0' || *it->c > '9') { it->bad = true; return 0; }
    while (*it->c >= '0' && *it->c <= '9') rep = rep * 10 + (unsigned long)(*it->c++ - '0');
    it->op = *it->c ? *it->c++ : 0;
    if (!it->op || rep == 0) { it->bad = true; return 0; }
    it->left = rep - 1;
    return it->op;
}

bool check_cigar_edit(const char *text, const char *pattern, const int tlen, const int plen, const char *curr_cigar)
{
    if (!curr_cigar || !text || !pattern || tlen < 0 || plen < 0) return false;
    long h = 0, v = 0;
    cigar_it_t it;
    cig_begin(&it, curr_cigar);
    for (char op; (op = cig_next(&it)) != 0;) {
        switch (op) {
        case 'M':
            if (v >= plen || h >= tlen || pattern[v] != text[h]) return false;
            ++v; ++h;
            break;
        case 'X':
            if (v >= plen || h >= tlen || pattern[v] == text[h]) return false;
            ++v; ++h;
            break;
        case 'I': ++h; break;
        case 'D': ++v; break;
        default:                      /* the reference skips letters it does not know (verification.c:71-73) */
            if (it.rle) return false;
            break;
        }
        if (v > plen || h > tlen) return false;
    }
    return !it.bad && v == plen && h == tlen;
}

bool check_affine_distance(const char *text, const char *pattern, const int tlen, const int plen, const int distance,
                           const affine_penalties_t penalties, const char *cigar)
{
    (void)text; (void)pattern; (void)tlen; (void)plen;      /* like the reference, only the op string is scored */
    if (!cigar || distance < 0) return false;
    long score = 0;
    char gap = 0;                                           /* 'I' / 'D' while inside a gap of that kind */
    cigar_it_t it;
    cig_begin(&it, cigar);
    for (char op; (op = cig_next(&it)) != 0;) {
        if (op == 'I' || op == 'D') {
            score += (gap == op) ? penalties.e : penalties.o + penalties.e;
            gap = op;
            /* run-length text prints two same-type gaps that only a gap-close separates as two runs ("1I1I") */
            if (it.rle && it.left == 0) gap = 0;
        } else {
            gap = 0;
            if (op == 'X') score += penalties.x;
            else if (op != 'M' && it.rle) return false;
        }
    }
    return !it.bad && score == (long)distance;
}

/* Unrolled op string ("MMXMMI...", malloc'ed, caller frees) of run-length CIGAR text: what the reference's
 * recover_cigar returns for the same alignment. */
char *wfagpu_unroll_cigar(const char *rle)
{
    if (!rle) return NULL;
    size_t n = 0;
    cigar_it_t it;
    cig_begin(&it, rle);
    if (!it.rle && rle[0]) return strdup(rle);
    while (cig_next(&it)) ++n;
    if (it.bad) return NULL;
    char *out = (char *)malloc(n + 1);
    if (!out) return NULL;
    cig_begin(&it, rle);
    size_t i = 0;
    for (char op; (op = cig_next(&it)) != 0;) out[i++] = op;
    out[i] = 0;
    return out;
}

/* recover_cigar (utils/verification.h:52-58): unrolled op string from a backtrace chain in the REFERENCE's own
 * format -- `offloaded_backtraces_array[num_bt_blocks - 1]` is the oldest full word, `final_backtrace` the last,
 * 16 two-bit ops per word filled from the least significant end, the op of a word's first step in its highest
 * used bits.  This library's kernels do not produce such chains (they emit a flat 2-bit op stream, see
 * wfagpu_ops_to_cigar); the function is kept for callers that hold reference-format results. */
static long common_prefix(const char *pattern, long plen, const char *text, long tlen, long v, long h)
{
    long n = 0;
    while (v + n < plen && h + n < tlen && pattern[v + n] == text[h + n]) ++n;
    return n;
}

char *recover_cigar(const char *text, const char *pattern, const size_t tlen, const size_t plen,
                    wfa_backtrace_t final_backtrace, wfa_backtrace_t *offloaded_backtraces_array,
                    alignment_result_t result)
{
    char *out = (char *)calloc(tlen + plen + 1, 1);
    if (!out) return NULL;
    size_t w = 0;
    long k = 0, off = 0;
    bool in_gap = false;
    for (int blk = result.num_bt_blocks; blk >= 0; --blk) {
        const uint32_t word = blk > 0 ? offloaded_backtraces_array[blk - 1].backtrace : final_backtrace.backtrace;
        const int used = word ? 16 - (__builtin_clz(word) >> 1) : 0;
        for (int i = used - 1; i >= 0; --i) {
            if (!in_gap) {
                const long m = common_prefix(pattern, (long)plen, text, (long)tlen, off - k, off);
                for (long j = 0; j < m && w < tlen + plen; ++j) out[w++] = 'M';
                off += m;
            }
            const unsigned op = (word >> (2 * i)) & 3u;
            if (op == OP_DEL) { in_gap = true; --k; if (w < tlen + plen) out[w++] = 'D'; }
            else if (op == OP_INS) { in_gap = true; ++k; ++off; if (w < tlen + plen) out[w++] = 'I'; }
            else if (op == OP_SUB) {
                if (in_gap) in_gap = false;                 /* gap-close delimiter */
                else { ++off; if (w < tlen + plen) out[w++] = 'X'; }
            }
        }
    }
    if (!in_gap) {
        const long m = common_prefix(pattern, (long)plen, text, (long)tlen, off - k, off);
        for (long j = 0; j < m && w < tlen + plen; ++j) out[w++] = 'M';
    }
    return out;
}
