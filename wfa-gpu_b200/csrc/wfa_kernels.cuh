/*
 * wfa_kernels.cuh -- device code of the B200-native gap-affine WFA hot path.
 *
 * Kernels (all integer SIMT work; no tensor cores -- there is no contraction):
 *   pack_kernel          ASCII -> 2-bit, one warp per sequence, 128-bit aligned loads
 *                        (replaces lib/kernels/sequence_packing_kernel.cu:28-116)
 *   wfa_bound_kernel     per-pair score upper bound: the recurrence on a re-centred window of 32
 *                        diagonals, one warp per pair (feeds the exact kernel's pruning)
 *   wfa_exact_kernel     M/I/D offset recurrence + extend on the score-bound-pruned window, one CTA
 *                        (or one warp) per pair, persistent, next pair prefetched with
 *                        cp.async.bulk (TMA 1-D); backtrace state = ring snapshots every P scores
 *                        (CTA kernels) or one decision byte per cell (warp kernel, large tier)
 *                        (replaces lib/kernels/sequence_alignment_kernel.cu:355-688,
 *                         lib/kernels/sequence_distance_kernel.cu:175-423)
 *   wfa_traceback_kernel ring snapshots -> 2-bit op stream by recomputing the dependency cone under
 *                        the path, one warp per pair (replaces the bt-word/offload chain of
 *                        sequence_alignment_kernel.cu and the gather in lib/align.cu)
 *   wfa_banded_kernel    adaptive band (-B), the reference's heuristic bit for bit
 *   wfa_bandq_kernel     the same, four diagonals per thread on packed int16 (packed pairs)
 *   cigar_text_kernel    op stream + sequences -> CIGAR text on the device (utils/cigar.c)
 *
 * Semantics reproduced from the reference (see SURVEY.md S1-S10):
 *   k = h - v, offset = h; NULL = -32000 (int16, drifts upward, stays < 0);
 *   I = max(M[d-o-e][k-1], I[d-e][k-1]) + 1   ties: extend beats open
 *   D = max(M[d-o-e][k+1], D[d-e][k+1])       ties: extend beats open
 *   M = extend(max(M[d-x][k]+1, I, D))        ties: D beats X beats I
 *   an M cell whose winning candidate is outside the sequences becomes NULL,
 *   I/D offsets are not bounds-checked (common_alignment_kernels.cuh:38).
 */
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "wfagpu_b200.h"

namespace wfagpu {

constexpr int kOffNull = -32000;
constexpr uint32_t kInvalidIdx = 0xffffffffu;

struct KernelParams {
    /* inputs */
    const uint32_t *packed;       /* packed sequences, overlapped 8-base stride words        */
    const char *ascii;            /* batch ASCII (byte-compare kernel only)                  */
    wfagpu_pair_t *pairs;
    const uint32_t *order;        /* pair indices, longest first                             */
    uint32_t n_items;             /* entries of `order`                                      */
    uint32_t *queue;              /* atomic work-queue head                                  */
    uint32_t *tb_queue;           /* same for the traceback kernel                           */
    uint32_t *bound_queue;        /* same for the bound kernel                               */
    int32_t *bound;               /* per pair: upper bound of its score (wfa_bound_kernel), or null:
                                   * the pruning then uses the launch bound d_end - 1         */
    const wfagpu_step_t *steps;
    int d_end;                    /* scores 1 .. d_end-1 may be computed                     */
    int n_cap;                    /* largest half width the rings of this launch can hold    */
    int x, o, e;
    int A, E1, G;                 /* ring depths (M: A, I/D: E1) and guard width             */
    int row_stride;               /* int16 elements per ring row                             */
    int center;                   /* index of k = 0 inside a row                             */
    int seq_words;                /* u32 capacity of one packed sequence buffer in smem      */
    int with_bt;
    int band;                     /* banded kernel: re-centre every `band` scores           */
    int win;                      /* banded kernel: window width in diagonals               */
    int32_t *band_lo;             /* banded kernel: per group, lo of every score (traceback) */
    uint32_t band_lo_words;
    int band_tb;                  /* wfa_bandq_kernel: arena and band_lo are per queue position and the backtrace is walked
                                   * by wfa_band_traceback_kernel (a thread per pair) after the launch */
    int stages;                   /* 1 or 2 sequence buffers per group (2 = prefetch next pair) */
    int quad_pairs;               /* quad kernel: two scores per barrier (needs ring_m = A + 1, ring_g = E1 + 1) */
    int ring_m, ring_g;           /* quad kernel: rows of the M ring and of the I / D rings */
    /* decision arena: one region per worker group */
    int32_t *gring;               /* large tier: per-group rings in global memory, else null */
    uint64_t gring_elems;         /* int32 elements per group                                */
    uint4 *arena;
    uint64_t arena_units;         /* uint4 units per group                                   */
    const uint32_t *ck_off;       /* checkpointed traceback: arena offset (units) of the snapshot of
                                   * score j * ck_period; null = one decision byte per cell  */
    int ck_period;                /* 7, 15 or 31                                              */
    uint32_t *ops_scratch;        /* per-group scratch for the traceback's op words          */
    uint32_t ops_scratch_words;
    /* outputs */
    uint32_t *ops_pool;
    uint32_t *ops_pool_head;      /* bump allocator                                          */
    uint32_t ops_pool_words;
    wfagpu_pair_out_t *out;
    uint32_t *retry_list;         /* pairs that ran out of budget                            */
    uint32_t *retry_count;
    uint32_t *ascii_list;         /* pairs the packer flagged (byte-compare launch)          */
    uint32_t *ascii_count;
    unsigned long long *cells;    /* optional work counter (may be null)                     */
    /* ends-free alignment (wfa_exact_kernel<..., EF = true>): free leading / trailing bases of the pattern and the
     * text, clamped per pair; the step table's half widths include the start row's max(pb, tb) */
    int ef_pb, ef_pe, ef_tb, ef_te;
    int2 *ends;                   /* ends-free: per pair {k_begin, k_end}; null in global mode */
    /* gap-affine 2-piece (wfa_exact_kernel<..., P2 = true>): second gap piece and the depth of its I2 / D2 rings (e2 + 1);
     * e2 == 0: one piece.  With P2, A = max(x, o + e, o2 + e2) + 1 */
    int o2, e2, E2;
};

struct PackParams {
    const char *ascii;
    uint32_t *packed;
    wfagpu_pair_t *pairs;
    uint32_t n_pairs;
};

struct CigarParams {
    const char *ascii;
    const wfagpu_pair_t *pairs;
    const wfagpu_pair_out_t *out;
    const uint32_t *ops_pool;
    uint32_t n_pairs;
    char *slots;                      /* slack slots, bump-allocated in 8-byte units            */
    unsigned long long slot_bytes;
    unsigned long long *slot_head;
    char *text;                       /* dense text pool                                        */
    unsigned long long *text_head;
    wfagpu_cigar_ref_t *refs;         /* per pair: offset (bytes) + length of its text          */
    uint32_t *overflow;
    const int2 *ends;                 /* ends-free: per pair {k_begin, k_end} (leading / trailing runs); null = global */
};

void launch_pack(const PackParams &p, cudaStream_t s);
void launch_cigar_text(const CigarParams &p, cudaStream_t s);
/* group_threads == 32 -> warp-per-pair variant; otherwise CTA-per-pair.  p.ends != null runs the ends-free
 * variant, p.e2 > 0 the gap-affine 2-piece variant (both: decision-byte traceback only, p.ck_off must be null) */
cudaError_t launch_exact(const KernelParams &p, int group_threads, int groups_per_cta, int ctas,
                         size_t smem_bytes, bool ascii_extend, cudaStream_t s);
/* CTA per pair, four diagonals per thread (packed sequences, shared-memory rings whose diagonal 0 is 16-byte
 * aligned; with backtrace it writes ring snapshots: p.ck_off must be set) */
cudaError_t launch_quad(const KernelParams &p, int threads, int ctas, size_t smem_bytes, cudaStream_t s);
int quad_max_ctas_per_sm(int threads, size_t smem_bytes, bool bt);
/* large tier: int32 rings in global memory (p.gring, rows of p.row_stride elements, multiple of 4, diagonal 0 at p.center,
 * multiple of 4), four diagonals per thread; shared memory = exact_smem_bytes(A, E1, 0, seq_words, 1, 1, true) */
cudaError_t launch_quadg(const KernelParams &p, int threads, int ctas, size_t smem_bytes, cudaStream_t s);
int quadg_max_ctas_per_sm(int threads, size_t smem_bytes, bool bt);
/* per-pair score upper bounds for the pruning (warp per pair) */
cudaError_t launch_bound(const KernelParams &p, int ctas, int warps, cudaStream_t s);
size_t bound_smem_bytes(int A, int E1, int warps);
int bound_max_ctas_per_sm(int A, int E1, int warps);
/* traceback of the checkpointed path: `warps` pairs per CTA */
cudaError_t launch_traceback(const KernelParams &p, int ctas, int warps, bool ascii_extend, cudaStream_t s);
size_t traceback_smem_bytes(int A, int period, int warps);
int traceback_max_ctas_per_sm(int A, int period, int warps, bool ascii_extend);
/* sched: CTA-per-pair kernels with shared-memory rings keep per-score schedule records (3 KB; not the 2-piece kernels).
 * E2 > 0: the two extra I2 / D2 rings of a 2-piece launch */
size_t exact_smem_bytes(int A, int E1, int row_stride, int seq_words, int groups_per_cta, int stages, bool sched = false,
                        int E2 = 0);
cudaError_t launch_banded(const KernelParams &p, int threads, int ctas, size_t smem_bytes, bool ascii_extend,
                          cudaStream_t s);
size_t banded_smem_bytes(int A, int win, int seq_words, int stages);
int banded_max_ctas_per_sm(int threads, size_t smem_bytes, bool ascii_extend, bool with_bt);
/* the same heuristic, four diagonals per thread on packed int16 (packed pairs only) */
cudaError_t launch_bandq(const KernelParams &p, int threads, int ctas, size_t smem_bytes, cudaStream_t s);
size_t bandq_smem_bytes(int A, int win, int seq_words, int stages);
int bandq_max_ctas_per_sm(int threads, size_t smem_bytes, bool with_bt);
/* decision bytes of wfa_bandq_kernel -> 2-bit ops, one thread per pair of the launch */
cudaError_t launch_band_traceback(const KernelParams &p, cudaStream_t s);
int large_max_ctas_per_sm(int threads, size_t smem_bytes, bool ascii_extend, bool with_bt, bool ef = false,
                          bool p2 = false);
int exact_max_ctas_per_sm(int group_threads, int groups_per_cta, size_t smem_bytes, bool ascii_extend, bool with_bt,
                          bool ckpt = false, bool ef = false, bool p2 = false);

} // namespace wfagpu
