/*
 * cigar.c -- CIGAR text from the kernel's 2-bit op stream.
 *
 * Produces byte-for-byte what the reference's host decoder
 * (recover_cigar_affine, utils/cigar.c:96-272) prints for the same alignment
 * path: match runs are re-derived on the ASCII sequences between ops, `X`
 * inside a gap is the gap-close delimiter and prints nothing, equal ops are
 * run-length merged unless a delimiter or a match run separates them, a zero
 * score prints "<tlen>M".  The ops arrive newest first (traceback order),
 * 16 per 32-bit word, so they are walked backwards.
 */
#include <string.h>
#include "wfagpu_b200.h"

static inline size_t match_run(const char *p, size_t plen, const char *t, size_t tlen, long v, long h)
{
    if (v < 0 || h < 0) return 0;
    size_t n = 0;
    const size_t room_p = (size_t)v <= plen ? plen - (size_t)v : 0;
    const size_t room_t = (size_t)h <= tlen ? tlen - (size_t)h : 0;
    const size_t room = room_p < room_t ? room_p : room_t;
    const char *a = p + v, *b = t + h;
    while (n + 8 <= room) {
        uint64_t wa, wb;
        memcpy(&wa, a + n, 8);
        memcpy(&wb, b + n, 8);
        const uint64_t diff = wa ^ wb;
        if (diff) return n + (size_t)(__builtin_ctzll(diff) >> 3);
        n += 8;
    }
    while (n < room && a[n] == b[n]) ++n;
    return n;
}

bool wfagpu_ops_to_cigar(const char *pattern, size_t plen, const char *text, size_t tlen,
                         int distance, const uint32_t *ops, uint32_t n_ops, wfa_cigar_t *cigar)
{
    if (distance == 0) return insert_ops(cigar, 'M', (unsigned)tlen);
    static const char letter[4] = {'?', 'I', 'X', 'D'};
    long k = 0, off = 0;
    bool in_gap = false;
    int run_op = OP_NOOP;      /* op of the pending run */
    unsigned run_len = 0;
    bool ok = true;
    for (uint32_t i = n_ops; i-- > 0;) {
        int op = (int)((ops[i >> 4] >> (2 * (i & 15u))) & 3u);
        if (op != run_op && run_len) { ok &= insert_ops(cigar, letter[run_op], run_len); run_len = 0; }
        if (!in_gap) {
            const size_t m = match_run(pattern, plen, text, tlen, off - k, off);
            if (m) {
                if (run_len) { ok &= insert_ops(cigar, letter[run_op], run_len); run_len = 0; }
                ok &= insert_ops(cigar, 'M', (unsigned)m);
                off += (long)m;
            }
        }
        if (op == OP_DEL) { in_gap = true; --k; ++run_len; }
        else if (op == OP_INS) { in_gap = true; ++k; ++off; ++run_len; }
        else if (op == OP_SUB) {
            if (in_gap) { in_gap = false; op = OP_NOOP; /* delimiter: the gap run was flushed above */ }
            else { ++off; ++run_len; }
        }
        run_op = op;
    }
    if (run_len) ok &= insert_ops(cigar, letter[run_op], run_len);
    if (!in_gap) {
        const size_t m = match_run(pattern, plen, text, tlen, off - k, off);
        ok &= insert_ops(cigar, 'M', (unsigned)m);
    }
    return ok;
}

/* Ends-free twin of cigar_text_kernel<true>: the same walk from (max(0, -k_begin), max(0, k_begin)) behind the leading
 * run, and the trailing run to the end of both sequences.  A free run joins the gap run of the same letter next to it:
 * the leading run through the run tracking, the trailing run through the gap run held back at the last delimiter. */
bool wfagpu_ops_to_cigar_span(const char *pattern, size_t plen, const char *text, size_t tlen, int k_begin,
                              const uint32_t *ops, uint32_t n_ops, wfa_cigar_t *cigar)
{
    static const char letter[4] = {'?', 'I', 'X', 'D'};
    long k = k_begin, off = k_begin > 0 ? k_begin : 0;
    bool in_gap = false;
    int run_op = k_begin > 0 ? OP_INS : (k_begin < 0 ? OP_DEL : OP_NOOP);
    unsigned run_len = (unsigned)(k_begin < 0 ? -(long)k_begin : k_begin);
    bool ok = true;
    for (uint32_t i = n_ops; i-- > 0;) {
        int op = (int)((ops[i >> 4] >> (2 * (i & 15u))) & 3u);
        const bool hold = i == 0 && in_gap && op == OP_SUB;   /* the last gap's delimiter: the trailing run may join it */
        if (op != run_op && run_len && !hold) { ok &= insert_ops(cigar, letter[run_op], run_len); run_len = 0; }
        if (!in_gap) {
            const size_t m = match_run(pattern, plen, text, tlen, off - k, off);
            if (m) {
                if (run_len) { ok &= insert_ops(cigar, letter[run_op], run_len); run_len = 0; }
                ok &= insert_ops(cigar, 'M', (unsigned)m);
                off += (long)m;
            }
        }
        if (op == OP_DEL) { in_gap = true; --k; ++run_len; }
        else if (op == OP_INS) { in_gap = true; ++k; ++off; ++run_len; }
        else if (op == OP_SUB) {
            if (in_gap) { in_gap = false; op = hold ? run_op : OP_NOOP; }
            else { ++off; ++run_len; }
        }
        run_op = op;
    }
    const size_t m = in_gap ? 0 : match_run(pattern, plen, text, tlen, off - k, off);
    if (m) {
        if (run_len) ok &= insert_ops(cigar, letter[run_op], run_len);
        run_len = 0;
        ok &= insert_ops(cigar, 'M', (unsigned)m);
        off += (long)m;
    }
    if (off > (long)tlen || off - k > (long)plen) return false;
    const unsigned tail_i = (unsigned)((long)tlen - off), tail_d = (unsigned)((long)plen - (off - k));
    const unsigned tail = tail_i ? tail_i : tail_d;
    const int tail_op = tail_i ? OP_INS : OP_DEL;
    if (tail) {
        if (run_len && run_op == tail_op) {
            run_len += tail;
        } else {
            if (run_len) ok &= insert_ops(cigar, letter[run_op], run_len);
            run_op = tail_op;
            run_len = tail;
        }
    }
    if (run_len) ok &= insert_ops(cigar, letter[run_op], run_len);
    return ok;
}
