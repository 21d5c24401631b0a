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
    /* ends-free alignment (wfa_exact_kernel<..., EF = true>): per pair its free leading / trailing bases of the pattern
     * and the text {pb, pe, tb, te}, already clamped to that pair; the step table's half widths include the widest start
     * row of the batch, max(pb, tb) over its pairs */
    const int4 *spans;
    int spans_pad[2];             /* keeps the offsets of the fields below, and with them the code of the kernels that read them */
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

/* Which wavefront kernel a launch runs.  It is decided once per launch shape: the occupancy questions that size the
 * launch and the launch itself ask with the same value. */
enum class Family : uint8_t {
    Exact,    /* wfa_exact_kernel: one diagonal per thread, warp or CTA per pair */
    Quad,     /* wfa_quad_kernel: CTA per pair, four diagonals per thread on packed int16, shared-memory rings whose
               * diagonal 0 is 16-byte aligned; with backtrace it writes ring snapshots (ckpt) */
    QuadG,    /* wfa_quadg_kernel: the large tier's quad kernel, int32 rings in global memory (gring): rows a multiple of 4,
               * diagonal 0 at a multiple of 4; shared memory = exact_smem_bytes(A, E1, 0, seq_words, 1, 1, true) */
    Banded,   /* wfa_banded_kernel: adaptive band (-B) */
    BandQ,    /* wfa_bandq_kernel: the same, four diagonals per thread on packed int16 (packed pairs only) */
};
struct KernelChoice {
    Family family = Family::Exact;
    bool warp = false;    /* exact: warp per pair (threads = 32 x pairs per CTA) */
    bool ascii = false;   /* byte-compare extend on the ASCII copy */
    bool bt = false;      /* backtrace (CIGAR) */
    bool gring = false;   /* rings in global memory, int32 offsets (RingG32); else shared memory (RingS16) */
    bool ckpt = false;    /* ring snapshots for wfa_traceback_kernel instead of decision bytes */
    bool ef = false;      /* exact: ends-free (decision-byte traceback on every tier) */
    bool p2 = false;      /* exact: gap-affine 2-piece (likewise) */
    bool org = false;     /* exact, ends-free, score only: origin rows carry each alignment's start diagonal to p.ends */
    int threads = 0;      /* threads per CTA; QuadG picks its register budget (MAXT) from it */
    bool quad() const { return family == Family::Quad || family == Family::QuadG || family == Family::BandQ; }
};
using kernel_fn = void (*)(const KernelParams);
/* the __global__ function of `k`, null for a combination that has no kernel.  count_cells: the instrumented
 * wfa_quad_kernel (COUNT = true) that fills p.cells; occupancy is always asked without it, so that counting cells does
 * not change the launch shape */
kernel_fn wavefront_kernel(const KernelChoice &k, bool count_cells = false);
/* allow the opt-in shared memory, launch, and report the launch error (null kfn: cudaErrorInvalidValue) */
cudaError_t launch(kernel_fn kfn, const KernelParams &p, int ctas, int threads, size_t smem, cudaStream_t s);
/* resident CTAs per SM at that shape, 0 if none (or null kfn) */
int max_ctas_per_sm(kernel_fn kfn, int threads, size_t smem);

/* per-pair score upper bounds for the pruning (warp per pair) */
cudaError_t launch_bound(const KernelParams &p, int ctas, int warps, cudaStream_t s);
size_t bound_smem_bytes(int A, int E1, int warps);
int bound_max_ctas_per_sm(int A, int E1, int warps);
/* traceback of the checkpointed path: `warps` pairs per CTA */
cudaError_t launch_traceback(const KernelParams &p, int ctas, int warps, bool ascii_extend, cudaStream_t s);
size_t traceback_smem_bytes(int A, int period, int warps);
int traceback_max_ctas_per_sm(int A, int period, int warps, bool ascii_extend);
/* sched: CTA-per-pair kernels with shared-memory rings keep per-score schedule records (3 KB; not the 2-piece kernels).
 * E2 > 0: the two extra I2 / D2 rings of a 2-piece launch.  org: every ring row has an origin row (KernelChoice::org) */
size_t exact_smem_bytes(int A, int E1, int row_stride, int seq_words, int groups_per_cta, int stages, bool sched = false,
                        int E2 = 0, bool org = false);
size_t banded_smem_bytes(int A, int win, int seq_words, int stages);
size_t bandq_smem_bytes(int A, int win, int seq_words, int stages);
/* decision bytes of wfa_bandq_kernel -> 2-bit ops, one thread per pair of the launch */
cudaError_t launch_band_traceback(const KernelParams &p, cudaStream_t s);

} // namespace wfagpu
