/*
 * step_table.c -- per-score control table shared by the forward kernel and the
 * traceback (include/wfagpu_b200.h).
 *
 * Which scores are null steps, mismatch-only steps (next_M) or full M/I/D steps
 * (next_MDI) is decided in the reference by the `exist` flags of the ring
 * (lib/kernels/sequence_alignment_kernel.cu:584-631); those flags depend on the
 * penalties alone, so the whole schedule -- including the wavefront half-width
 * and where each score's decision row lives -- is computed once on the host.
 */
#include <stdlib.h>
#include "wfagpu_b200.h"

/* `extra`: diagonals added on both sides of every score's range (the start row of an ends-free alignment).
 * e2 > 0: gap-affine 2-piece, a second gap component (o2, e2) next to (o, e); e2 == 0: one piece. */
static int build_step_table(int x, int o, int e, int o2, int e2, int max_steps, int max_dist, int banded_win, int extra,
                            wfagpu_step_t *tab, uint64_t *arena_units)
{
    if (max_dist < 1) max_dist = 1;
    unsigned char *has_m = (unsigned char *)calloc((size_t)max_dist + 1, 1);
    unsigned char *has_gap = (unsigned char *)calloc((size_t)max_dist + 1, 1);
    unsigned char *has_gap2 = e2 > 0 ? (unsigned char *)calloc((size_t)max_dist + 1, 1) : NULL;
    if (!has_m || !has_gap || (e2 > 0 && !has_gap2)) { free(has_m); free(has_gap); free(has_gap2); return -1; }
    uint64_t units = 0;
    int steps = 1; /* the reference counts the score-0 wavefront as step 1 (kernel.cu:580-581) */
    int n = 0;     /* half width of the computed diagonal range                                  */
    int mdi = 0;   /* number of M/I/D steps so far (the reference's wavefront growth)            */
    /* one decision byte per cell, rows padded to 16-byte units; a banded row starts at the window's first diagonal rounded
     * down to a multiple of four (wfa_bandq_kernel) and holds whole quads: up to win + 6 bytes */
    const uint64_t band_units = banded_win > 0 ? (uint64_t)((banded_win + 8 + 15) / 16) : 0;
    int d;
    has_m[0] = 1;
    if (tab) { tab[0].row_off = 0; tab[0].n = (uint16_t)extra; tab[0].kind = WFAGPU_STEP_M; }
    for (d = 1; d < max_dist; ++d) {
        if (steps >= max_steps - 1) break;          /* while (steps < max_steps - 1) */
        if (n + extra >= 65535 || mdi >= 65535) break;
        int gap = 0, m = 0;
        if (d - o - e >= 0) gap = has_m[d - o - e] || has_gap[d - e];
        int gap2 = 0;
        if (e2 > 0 && d - o2 - e2 >= 0) gap2 = has_m[d - o2 - e2] || has_gap2[d - e2];
        if (gap2) has_gap2[d] = 1;
        if (gap) has_gap[d] = 1;
        gap = gap || gap2;
        if (gap) m = 1;
        else if (d - x >= 0) m = has_m[d - x];
        unsigned kind = WFAGPU_STEP_NULL;
        if (gap) {
            kind = WFAGPU_STEP_MDI; has_m[d] = 1; ++mdi; ++steps;
            if (banded_win > 0) {
                n = mdi;                             /* banded: n counts the M/I/D steps (row index + 1) */
            } else {
                /* The reference widens the range by one diagonal per M/I/D step.  A diagonal k
                 * needs a gap of |k| bases, i.e. a score of at least o + |k| e, so everything
                 * beyond (d - o) / e is NULL and need not be computed (e >= 2 halves the work).  2-piece: a gap
                 * of |k| bases costs at least min(o + |k| e, o2 + |k| e2), so the reach is the larger of the two. */
                int reach = (d - o) / e;
                if (e2 > 0 && (d - o2) / e2 > reach) reach = (d - o2) / e2;
                n = mdi < reach ? mdi : reach;
                if (n < 0) n = 0;
            }
        } else if (m) { kind = WFAGPU_STEP_M; has_m[d] = 1; }
        if (units > 0xffffffffull) break;           /* row offsets are 32-bit */
        if (tab) { tab[d].row_off = (uint32_t)units; tab[d].n = (uint16_t)(n + extra); tab[d].kind = (uint16_t)kind; }
        if (kind == WFAGPU_STEP_MDI) units += banded_win > 0 ? band_units : (uint64_t)((2 * (n + extra) + 1 + 15) / 16);
    }
    free(has_m);
    free(has_gap);
    free(has_gap2);
    if (arena_units) *arena_units = units;
    return d;
}

int wfagpu_build_step_table(int x, int o, int e, int max_steps, int max_dist, int banded_win,
                            wfagpu_step_t *tab, uint64_t *arena_units)
{
    return build_step_table(x, o, e, 0, 0, max_steps, max_dist, banded_win, 0, tab, arena_units);
}

int wfagpu_build_step_table_span(int x, int o, int e, int max_steps, int max_dist, int start_half_width,
                                 wfagpu_step_t *tab, uint64_t *arena_units)
{
    if (start_half_width < 0 || start_half_width >= 65535) return -1;
    return build_step_table(x, o, e, 0, 0, max_steps, max_dist, 0, start_half_width, tab, arena_units);
}

int wfagpu_build_step_table_affine2p(int x, int o1, int e1, int o2, int e2, int max_steps, int max_dist,
                                     wfagpu_step_t *tab, uint64_t *arena_units)
{
    if (x < 1 || o1 < 0 || e1 < 1 || o2 < 0 || e2 < 1) return -1;
    return build_step_table(x, o1, e1, o2, e2, max_steps, max_dist, 0, 0, tab, arena_units);
}
