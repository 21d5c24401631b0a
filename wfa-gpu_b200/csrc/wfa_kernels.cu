/*
 * wfa_kernels.cu -- hand-written sm_100a kernels of the gap-affine WFA hot path.
 * See wfa_kernels.cuh for the kernel list and the reference lines each replaces.
 */
#include "wfa_kernels.cuh"

#include <climits>
#include <mutex>
#include <type_traits>
#include <unordered_map>
#include <unordered_set>

namespace wfagpu {

/* Every kernel may use up to the opt-in maximum of dynamic shared memory (227 KB on B200).  The limit is a per-function,
 * per-device attribute: it is always set to the same value, never to the size of one launch, because two host threads that
 * drive the same GPU (two workers of one call, or two calls) would otherwise lower it under each other's launches. */
struct LaunchMemo {                /* what the host already asked the runtime, per device and kernel */
    std::mutex mu;
    std::unordered_set<uint64_t> smem_allowed;
    std::unordered_map<uint64_t, int> occupancy;
};
static LaunchMemo &launch_memo() { static LaunchMemo m; return m; }

static inline uint64_t memo_key(int dev, const void *kfn, uint64_t a, uint64_t b)
{
    uint64_t h = 0x9E3779B97F4A7C15ull * (uint64_t)(uintptr_t)kfn + (uint64_t)dev;
    h = (h ^ (h >> 29)) * 0xBF58476D1CE4E5B9ull + a;
    h = (h ^ (h >> 32)) * 0x94D049BB133111EBull + b;
    return h ^ (h >> 31);
}

template <typename K>
static cudaError_t allow_max_smem(K kfn)
{
    int dev = 0, optin = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return err;
    LaunchMemo &m = launch_memo();
    const uint64_t key = memo_key(dev, (const void *)kfn, 0, 0);
    {
        std::lock_guard<std::mutex> g(m.mu);
        if (m.smem_allowed.count(key)) return cudaSuccess;
    }
    err = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (err != cudaSuccess) return err;
    std::lock_guard<std::mutex> g(m.mu);
    m.smem_allowed.insert(key);
    return cudaSuccess;
}

/* cudaOccupancyMaxActiveBlocksPerMultiprocessor, remembered: the chunk planner asks the same few questions for every chunk
 * of a stream (10-20 us each, several dozen per pass). */
template <typename K>
static cudaError_t occupancy_of(int *n, K kfn, int threads, size_t smem)
{
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return err;
    LaunchMemo &m = launch_memo();
    const uint64_t key = memo_key(dev, (const void *)kfn, (uint64_t)threads, (uint64_t)smem + 1);
    {
        std::lock_guard<std::mutex> g(m.mu);
        auto it = m.occupancy.find(key);
        if (it != m.occupancy.end()) { *n = it->second; return cudaSuccess; }
    }
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, kfn, threads, smem);
    if (err != cudaSuccess) return err;
    std::lock_guard<std::mutex> g(m.mu);
    if (m.occupancy.size() > 65536) m.occupancy.clear();
    m.occupancy[key] = *n;
    return cudaSuccess;
}

/* ======================================================================== */
/*                               PTX helpers                                */
/* ======================================================================== */

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

/* 1-D bulk copy global -> shared through the TMA unit (SASS: UBLKCP). */
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

/* ======================================================================== */
/*                               pack kernel                                */
/* ======================================================================== */
/*
 * One warp per sequence.  Per iteration a warp consumes 512 ASCII bytes: lane i
 * reads two 16-byte aligned uint4 (its own and the next one), picks the 24
 * bytes that start at sequence byte 16*i (the sequence start is only 4-byte
 * aligned, lib/aligner.c:127-166), and emits two packed words:
 *   word j = bases [8j, 8j+16), base 8j in bits 31:30, code (c & 6) >> 1
 * (A=0 C=1 T=2 G=3, lib/kernels/sequence_packing_kernel.cu:79).  The 8-base
 * stride makes every extend start with >= 9 bases in a single word.
 * The has_N flag follows sequence_packing_kernel.cu:54-76 literally.
 */
__device__ __forceinline__ uint32_t pack4(uint32_t w)
{
    /* 4 ASCII bytes (first base in the low byte) -> 8 bits, first base in bits 7:6 */
    return (((w >> 1) & 0x03030303u) * 0x40100401u) >> 24;
}

__device__ __forceinline__ uint32_t keep_bytes(uint32_t w, int nbytes)
{
    /* keep the first nbytes (low) bytes of a little-endian word, zero the rest */
    if (nbytes >= 4) return w;
    if (nbytes <= 0) return 0u;
    return w & (0xffffffffu >> (32 - 8 * nbytes));
}

__global__ void __launch_bounds__(256) pack_kernel(PackParams p)
{
    const int lane = threadIdx.x & 31;
    const uint32_t seq = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (seq >= 2u * p.n_pairs) return;
    wfagpu_pair_t *pr = p.pairs + (seq >> 1);
    const bool is_text = seq & 1u;
    const uint32_t len = is_text ? pr->tlen : pr->plen;
    const uint32_t a_off = is_text ? pr->t_ascii : pr->p_ascii;
    uint32_t *dst = p.packed + (is_text ? pr->t_word : pr->p_word);
    const uint32_t nwords = ((len + 7u) >> 3) + 1u;          /* words that carry data or the terminator */
    const uint32_t nwords_pad = (nwords + 3u) & ~3u;           /* TMA copies whole 16-byte units */
    const char *src = p.ascii + a_off;
    const uintptr_t addr = (uintptr_t)src;
    const uint4 *base16 = (const uint4 *)(addr & ~(uintptr_t)15);
    const int q = (int)((addr & 15) >> 2);                      /* misalignment in words: 0..3 */
    /* groups of 4 bytes the reference's flag loop visits */
    const uint32_t ngroups = (len + (4u - (len & 3u))) >> 2;
    /* number of aligned uint4 that may be touched without leaving the batch buffer */
    const uint32_t n16 = (uint32_t)(((addr & 15) + len + 1 + 15) >> 4);
    bool flag = false;   /* (the reference also flags len >= 32768 because of its int16 offsets; the large tier takes those) */

    for (uint32_t it = 0; it * 64u < nwords_pad; ++it) {
        const uint32_t u = it * 32u + lane;                     /* index of this lane's first uint4 */
        uint4 a = make_uint4(0, 0, 0, 0), b = make_uint4(0, 0, 0, 0), c = make_uint4(0, 0, 0, 0);
        if (u < n16) a = __ldg(base16 + u);
        if (u + 1 < n16) b = __ldg(base16 + u + 1);
        if (q == 3 && u + 2 < n16) c = __ldg(base16 + u + 2);
        uint32_t w[9] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x};
        uint32_t s[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            uint32_t v = w[j];
            v = (q == 1) ? w[j + 1] : v;
            v = (q == 2) ? w[j + 2] : v;
            v = (q == 3) ? w[j + 3] : v;
            s[j] = v;
        }
        /* s[j] = sequence bytes [16u*... ] i.e. bytes 16*u + 4j .. +3 */
        const uint32_t byte0 = 16u * u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t g = (byte0 >> 2) + j;                /* 4-byte group index */
            if (g < ngroups && s[j] != 0u) {
                const uint32_t t = s[j] ^ 0x4e4e4e4eu;
                const uint32_t f = (t & 0xff) & ((t >> 8) & 0xff) & ((t >> 16) & 0xff) & (t >> 24);
                flag |= (f == 0u);
            }
        }
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const int nb = (int)len - (int)(byte0 + 4u * j);
            s[j] = keep_bytes(s[j], nb);
        }
        const uint32_t w0 = (pack4(s[0]) << 24) | (pack4(s[1]) << 16) | (pack4(s[2]) << 8) | pack4(s[3]);
        const uint32_t w1 = (pack4(s[2]) << 24) | (pack4(s[3]) << 16) | (pack4(s[4]) << 8) | pack4(s[5]);
        const uint32_t j0 = 2u * u;
        if (j0 + 1 < nwords_pad) {
            *reinterpret_cast<uint2 *>(dst + j0) = make_uint2(w0, w1);
        } else if (j0 < nwords_pad) {
            dst[j0] = w0;
        }
    }
    flag = __any_sync(0xffffffffu, flag);
    if (flag && lane == 0) atomicOr(&pr->flags, WFAGPU_PAIR_HAS_N);
}

void launch_pack(const PackParams &p, cudaStream_t s)
{
    if (p.n_pairs == 0) return;
    const uint32_t warps = 2u * p.n_pairs;
    const uint32_t blocks = (warps + 7u) / 8u;
    pack_kernel<<<blocks, 256, 0, s>>>(p);
}

/* ======================================================================== */
/*                            alignment kernel                              */
/* ======================================================================== */
/*
 * All wavefront state lives in shared memory and is addressed through 32-bit
 * shared-window addresses with explicit ld.shared / st.shared (one LDS.S16 per
 * source offset, no generic-pointer arithmetic, no sign-extension fix-ups).
 */
__device__ __forceinline__ int lds_s16(uint32_t a)
{
    int v;
    asm volatile("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_16(uint32_t a, int v)
{
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "h"((short)v) : "memory");
}
__device__ __forceinline__ void sts_v4(uint32_t a, uint4 v)
{
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}

/* Where the wavefront rings live.  RingS16: shared memory, int16 offsets (sequences
 * < 32768 bases, the reference's wfa_offset_t).  RingG32: global memory (L2), int32
 * offsets -- the large tier for wavefronts wider than an SM's shared memory and for
 * sequences the reference cannot take at all (>= 32768 bases, lib/wfa_types.h:28-32). */
struct RingS16 {
    using addr_t = uint32_t;                       /* shared-window address of diagonal 0 of a row */
    static constexpr int kNull = kOffNull;
    static constexpr uint32_t kElem = 2;
    __device__ static __forceinline__ int ld(addr_t row, int k) { return lds_s16(row + (uint32_t)(2 * k)); }
    __device__ static __forceinline__ void st(addr_t row, int k, int v) { sts_16(row + (uint32_t)(2 * k), v); }
    __device__ static __forceinline__ addr_t add(addr_t a, uint32_t bytes) { return a + bytes; }
};
struct RingG32 {
    using addr_t = int32_t *;
    static constexpr int kNull = -(1 << 28);
    static constexpr uint32_t kElem = 4;
    __device__ static __forceinline__ int ld(addr_t row, int k) { return row[k]; }
    __device__ static __forceinline__ void st(addr_t row, int k, int v) { row[k] = v; }
    __device__ static __forceinline__ addr_t add(addr_t a, uint32_t bytes)
    {
        return reinterpret_cast<addr_t>(reinterpret_cast<char *>(a) + bytes);
    }
};

template <bool WARP>
struct Group {
    __device__ static __forceinline__ int tid() { return WARP ? (threadIdx.x & 31) : threadIdx.x; }
    __device__ static __forceinline__ int size() { return WARP ? 32 : blockDim.x; }
    __device__ static __forceinline__ int id_in_cta() { return WARP ? (threadIdx.x >> 5) : 0; }
    __device__ static __forceinline__ void sync()
    {
        if (WARP) __syncwarp(); else __syncthreads();
    }
};

/* Bounded common prefix on packed words (replaces WF_extend_kernel,
 * lib/kernels/common_alignment_kernels.cuh:29-111): XOR + count-leading-zeros
 * on 32-bit windows.  With the 8-base stride layout a window of >= 9 bases
 * starts inside one word, so the common case (a mismatch within 9 bases) costs
 * two shared loads and no loop. */
__device__ __forceinline__ int extend_packed(uint32_t Pa, uint32_t Ta, int plen, int tlen, int k, int off,
                                             const int null_v = kOffNull)
{
    const int v = off - k, h = off;
    const int rem = min(plen - v, tlen - h);
    if (rem < 0) return null_v;
    const uint32_t uv = (uint32_t)v, uh = (uint32_t)h;
    const uint32_t wp = lds_u32(Pa + ((uv >> 3) << 2)) << ((uv & 7u) * 2u);
    const uint32_t wt = lds_u32(Ta + ((uh >> 3) << 2)) << ((uh & 7u) * 2u);
    const int run = __clz((int)(wp ^ wt)) >> 1;
    /* at least 9 bases of each window are real: a run of up to 8 needs no further look */
    if (run <= 8) return off + min(run, rem);
    const int nvalid = 16 - (int)max(uv & 7u, uh & 7u);
    int e1 = min(run, rem);
    if (e1 >= nvalid) {
        /* long match (rare off the optimal path): keep going window by window */
        int acc = nvalid;
        while (acc < rem) {
            const uint32_t v2 = uv + (uint32_t)acc, h2 = uh + (uint32_t)acc;
            const uint32_t a = lds_u32(Pa + ((v2 >> 3) << 2)) << ((v2 & 7u) * 2u);
            const uint32_t b = lds_u32(Ta + ((h2 >> 3) << 2)) << ((h2 & 7u) * 2u);
            const int nv = 16 - (int)max(v2 & 7u, h2 & 7u);
            const int eq = min(__clz((int)(a ^ b)) >> 1, nv);
            acc += eq;
            if (eq < nv) break;
        }
        e1 = min(acc, rem);
    }
    return off + e1;
}

/* Byte-compare variant for pairs the packer flagged (non-ACGT bytes): plain
 * byte equality like the CPU WFA the reference falls back to
 * (utils/wfa_cpu.c:57-85), straight from the ASCII copy in global memory. */
__device__ __forceinline__ int extend_ascii(const char *__restrict__ P, const char *__restrict__ T, int plen,
                                            int tlen, int k, int off, const int null_v = kOffNull)
{
    const int v = off - k, h = off;
    const int rem = min(plen - v, tlen - h);
    if (rem < 0) return null_v;
    int acc = 0;
    while (acc < rem && P[v + acc] == T[h + acc]) ++acc;
    return off + acc;
}

/* extend_packed on the packed words in global memory (the warp-per-pair kernels) */
__device__ __forceinline__ int extend_packed_g(const uint32_t *__restrict__ Pw, const uint32_t *__restrict__ Tw,
                                               int plen, int tlen, int k, int off)
{
    const int v = off - k, h = off;
    const int rem = min(plen - v, tlen - h);
    if (rem < 0) return kOffNull;
    {
        /* common case: the run ends within the 9 bases every window is good for */
        const uint32_t a = __ldg(Pw + ((uint32_t)v >> 3)) << (((uint32_t)v & 7u) * 2u);
        const uint32_t b = __ldg(Tw + ((uint32_t)h >> 3)) << (((uint32_t)h & 7u) * 2u);
        const int run = __clz((int)(a ^ b)) >> 1;
        if (run <= 8) return off + min(run, rem);
    }
    int acc = 0;
    while (acc < rem) {
        const uint32_t v2 = (uint32_t)(v + acc), h2 = (uint32_t)(h + acc);
        const uint32_t a = __ldg(Pw + (v2 >> 3)) << ((v2 & 7u) * 2u);
        const uint32_t b = __ldg(Tw + (h2 >> 3)) << ((h2 & 7u) * 2u);
        const int nv = 16 - (int)max(v2 & 7u, h2 & 7u);
        const int eq = min(__clz((int)(a ^ b)) >> 1, nv);
        acc += eq;
        if (eq < nv) break;
    }
    return off + min(acc, rem);
}

/* extend for the warp-per-pair kernels, called by all 32 lanes together: a lane that `want`s it gets
 * off + (common prefix of P[off-k ..] and T[off ..]), or null_v outside the sequences; the others get
 * `off` back.  A run of up to 8 bases is settled by the lane itself.  The one or two lanes on the
 * alignment path have long runs, and instead of dragging the warp through their serial loops the whole
 * warp compares 256 bases of such a run per round (8 per lane: every window has >= 9 real bases). */
__device__ __forceinline__ int warp_extend_packed(const uint32_t *__restrict__ Pw, const uint32_t *__restrict__ Tw,
                                                  int plen, int tlen, bool want, int k, int off, int null_v, int lane)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int ev = off - k, eh = off;
    int rem = -1, res = off;
    bool lng = false;
    if (want) {
        rem = min(plen - ev, tlen - eh);
        if (rem >= 0) {
            const uint32_t a = __ldg(Pw + ((uint32_t)ev >> 3)) << (((uint32_t)ev & 7u) * 2u);
            const uint32_t b = __ldg(Tw + ((uint32_t)eh >> 3)) << (((uint32_t)eh & 7u) * 2u);
            const int run = __clz((int)(a ^ b)) >> 1;
            if (run <= 8) res = eh + min(run, rem); else lng = true;
        } else {
            res = null_v;
        }
    }
    unsigned need = __ballot_sync(FULL, lng);
    while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        const int v0 = __shfl_sync(FULL, ev, src), h0 = __shfl_sync(FULL, eh, src);
        const int rem0 = __shfl_sync(FULL, rem, src);
        int total = rem0;
        for (int base = 0; base < rem0; base += 256) {
            const int start = base + 8 * lane;
            int eq = 0;
            if (start < rem0) {
                const uint32_t pv = (uint32_t)(v0 + start), ph = (uint32_t)(h0 + start);
                const uint32_t a = __ldg(Pw + (pv >> 3)) << ((pv & 7u) * 2u);
                const uint32_t b = __ldg(Tw + (ph >> 3)) << ((ph & 7u) * 2u);
                eq = min(min(__clz((int)(a ^ b)) >> 1, 8), rem0 - start);
            }
            const unsigned stop = __ballot_sync(FULL, eq < 8);
            if (stop) {
                const int f = __ffs(stop) - 1;
                total = base + 8 * f + __shfl_sync(FULL, eq, f);
                break;
            }
        }
        if (lane == src) res = eh + min(total, rem);
    }
    return res;
}

/* Score-bound pruning window of one score: the diagonals of [-n, n] within q = (Dmax - d) / e of
 * the target diagonal.  When none is (an all-NULL step) the window is the clamped full range, so
 * that the rows still read as NULL wherever a later score may look.  Returns whether any cell is
 * computed.  Used identically by the forward pass and by the checkpointed traceback. */
__device__ __forceinline__ bool prune_window(int n, int kt, int q, int n_cap, int &lo, int &hi)
{
    lo = max(-n, kt - q);
    hi = min(n, kt + q);
    const bool live = lo <= hi;
    if (!live) { hi = min(n, n_cap); lo = -hi; }
    return live;
}

/* The same for an ends-free alignment: the diagonals within q of the target range [tlo, thi] that the pair's own start
 * row reaches, [dp - n, n - dt].  The step table's n = W + r(d) is sized for the widest start row W of the batch, so
 * dp = W - pb and dt = W - tb narrow it to [-pb - r(d), tb + r(d)]: a cell further from the pair's start row needs a gap
 * longer than r(d) and is NULL (DESIGN.md §9).  An all-NULL step NULLs that reach, clamped to the rings. */
__device__ __forceinline__ bool prune_window_range(int n, int tlo, int thi, int q, int n_cap, int dp, int dt, int &lo, int &hi)
{
    lo = max(dp - n, tlo - q);
    hi = min(n - dt, thi + q);
    const bool live = lo <= hi;
    if (!live) { lo = max(dp - n, -n_cap); hi = min(n - dt, n_cap); }
    return live;
}

struct GroupCtl {
    uint64_t bar[2];     /* TMA completion barriers, one per sequence stage */
    uint32_t idx[2];     /* pair index staged in each buffer                */
    uint32_t n_ops;
    uint32_t ops_off;
    uint32_t pos[2];     /* queue position of that pair (its snapshot arena) */
    int32_t k_end;       /* ends-free CTA kernels: lowest finishing diagonal of the current score */
    uint32_t pad;
};

/* Per-score schedule record (CTA-per-pair kernels with shared-memory rings).  Everything a thread
 * needs to start a score -- the pruning window, the step kind, the ring rows of the score and of
 * its sources -- is the same for the whole CTA and costs ~60 instructions to derive, a third of
 * what a warp spends on a score at 10 kbp / 5 %.  Warp 0 derives the records of kSchedBlock scores at a
 * time (one per lane, double-buffered in shared memory) and every thread fetches its score's
 * record with three 128-bit broadcast loads. */
struct __align__(16) StepRec {
    int lo, hi;             /* window of diagonals computed at this score                       */
    uint32_t flags;         /* bits 1:0 kind, 2 live, 3 stop, 4 target diagonal inside, 5 snapshot */
    int n;                  /* half width of the unpruned wavefront (snapshot pitch)            */
    uint32_t aMc, aMx, aMo, aIc;
    uint32_t aIe, aDc, aDe, ck_j;   /* ck_j: snapshot index (CKPT) or decision-byte row offset */
};
constexpr uint32_t kRecLive = 4u, kRecStop = 8u, kRecTarget = 16u, kRecSnap = 32u;
constexpr int kSchedBlock = 16;                 /* scores per block of records (power of two, <= 32) */
constexpr uint32_t kSchedBytes = 2u * kSchedBlock * (uint32_t)sizeof(StepRec);

/* Gap-affine 2-piece state of wfa_exact_kernel<..., P2 = true>: the second piece and its I2 / D2 rings (after D, depth
 * e2 + 1), and the rows of the current score.  One piece uses the empty NoPiece2, so those kernels carry nothing extra. */
template <typename RA>
struct Piece2 {
    int e2, oe2, ep;            /* e2, o2 + e2, min(e1, e2) (pruning)                                    */
    RA I0, D0, Iend, Dend;      /* the I2 / D2 rings                                                      */
    RA Ic, Dc, Mo, Ie, De;      /* rows of score d: I2 / D2 at d and d - e2, M at d - o2 - e2             */
};
struct NoPiece2 {};

/* CKPT (CTA per pair, shared-memory rings, with backtrace): instead of a decision byte per
 * cell the forward pass snapshots the ring rows every p.ck_period scores, and the traceback
 * recomputes the offsets it needs on the dependency cone below the cell it stands on
 * (model + proof of equivalence: oracle/kernel_model.c, km_align_pair_ckpt).
 *
 * EF (ends-free, DESIGN.md §9): score 0 holds the extend of (max(0, -k), max(0, k)) on every diagonal of
 * [-pb, tb]; the pruning measures the distance to the target range [kt - te, kt + pe] instead of kt; an M cell on
 * a target diagonal finishes when its offset reaches min(tlen, plen + k), the lowest such k of the first finishing
 * score wins; the traceback starts there and stops at score 0.  k_begin / k_end go to p.ends[idx].
 *
 * ORG (score-only ends-free with coordinates, DESIGN.md §9): every M, I and D cell also stores the origin of its value,
 * the score-0 diagonal its path started on, in an origin row at a fixed byte offset (the value rows' size) from its
 * value row.  The origin follows the winner the decision byte of the CIGAR kernel records (I / D: extend beats open;
 * M: D > X > I), so the origin of the finishing cell is the traceback's k_begin, ties included.  Only a winner's
 * origin is read and a winner with a valid offset always has a written origin: origin rows need no prologue and no
 * NULL stores (tests/endsfree_origin_model.py checks this with poisoned origin cells). */
template <bool WARP, bool ASCII, bool BT, typename R, bool CKPT, bool EF = false, bool P2 = false, bool ORG = false>
__global__ void __launch_bounds__(WARP ? 256 : 1024, WARP ? 4 : 1) wfa_exact_kernel(const __grid_constant__ KernelParams p)
{
    static_assert(!CKPT || (BT && !WARP && R::kElem == 2), "checkpointed traceback: CTA groups with shared-memory rings");
    static_assert(!(EF && CKPT), "ends-free: decision-byte traceback only");
    static_assert(!(P2 && (CKPT || EF)), "gap-affine 2-piece: global alignment, decision-byte traceback only");
    static_assert(!ORG || (EF && !BT && !CKPT && !P2), "origins: score-only ends-free only");
    using G = Group<WARP>;
    using RA = typename R::addr_t;
    constexpr bool GR = (R::kElem == 4);          /* rings in global memory */
    constexpr bool SCHED = !WARP && !GR && !P2;   /* per-score schedule records (see StepRec); 2-piece: rows in registers */
    constexpr int NULLV = R::kNull;
    extern __shared__ __align__(16) unsigned char smem_raw[];

    const int tid = G::tid();
    const int gsz = G::size();
    const int groups_per_cta = WARP ? (blockDim.x >> 5) : 1;
    const uint32_t group = blockIdx.x * groups_per_cta + G::id_in_cta();

    /* ---- carve shared memory: [rings][sequence stages][ctl] per group ---- */
    const int rows = p.A + 2 * p.E1 + (P2 ? 2 * p.E2 : 0);
    const uint32_t row_bytes = (uint32_t)p.row_stride * R::kElem;
    const uint32_t org_off = (uint32_t)rows * row_bytes;          /* ORG: origin row = value row + org_off */
    const uint32_t ring_bytes = GR ? 0u : (((ORG ? 2u : 1u) * org_off + 15u) & ~15u);
    const uint32_t seq_bytes = (uint32_t)p.seq_words * 4u;          /* one sequence, one stage */
    const uint32_t seq_total = ASCII ? 0u : 2u * (uint32_t)p.stages * seq_bytes;
    const uint32_t group_bytes = (ring_bytes + seq_total + (uint32_t)sizeof(GroupCtl) + (SCHED ? kSchedBytes : 0u) + 15u) & ~15u;
    unsigned char *gbase = smem_raw + (size_t)G::id_in_cta() * group_bytes;
    const uint32_t ring_sa = smem_u32(gbase);
    const uint32_t seq_sa = ring_sa + ring_bytes;
    GroupCtl *ctl = reinterpret_cast<GroupCtl *>(gbase + ring_bytes + seq_total);
    const uint32_t sched_sa = ring_sa + ring_bytes + seq_total + (uint32_t)sizeof(GroupCtl);   /* GroupCtl is 48 bytes */

    const int x = p.x, e = p.e, A = p.A, E1 = p.E1, GW = p.G;
    const int oe = p.o + p.e;
    RA M0;                                                          /* row 0 of M, diagonal 0 */
    if constexpr (GR) {
        M0 = reinterpret_cast<RA>(p.gring + (size_t)group * p.gring_elems + p.center);
    } else {
        M0 = (RA)(ring_sa + 2u * (uint32_t)p.center);
    }
    const RA I0 = R::add(M0, (uint32_t)A * row_bytes);
    const RA D0 = R::add(I0, (uint32_t)E1 * row_bytes);
    /* 2-piece: state of the second gap piece (an empty struct for one piece) */
    std::conditional_t<P2, Piece2<RA>, NoPiece2> q2;
    if constexpr (P2) {
        q2.e2 = p.e2; q2.oe2 = p.o2 + p.e2; q2.ep = min(e, p.e2);
        q2.I0 = R::add(D0, (uint32_t)E1 * row_bytes);
        q2.D0 = R::add(q2.I0, (uint32_t)p.E2 * row_bytes);
        q2.Iend = R::add(q2.I0, (uint32_t)p.E2 * row_bytes);
        q2.Dend = R::add(q2.D0, (uint32_t)p.E2 * row_bytes);
    }

    uint4 *arena = p.arena + (size_t)group * p.arena_units;    /* CKPT: one arena per pair, set below */
    uint32_t *const scratch = p.ops_scratch + (size_t)group * p.ops_scratch_words;

    auto issue_load = [&](int stage, uint32_t idx) {
        /* leader only: both packed sequences of pair idx -> stage buffers, via TMA */
        if (ASCII) return;
        const wfagpu_pair_t pr = p.pairs[idx];
        const uint32_t pw = ((((pr.plen + 7u) >> 3) + 1u) + 3u) & ~3u;
        const uint32_t tw = ((((pr.tlen + 7u) >> 3) + 1u) + 3u) & ~3u;
        unsigned char *dp = gbase + ring_bytes + (size_t)(2 * stage) * seq_bytes;
        unsigned char *dt = dp + seq_bytes;
        fence_proxy_async();
        mbar_expect_tx(&ctl->bar[stage], (pw + tw) * 4u);
        tma_load_1d(dp, p.packed + pr.p_word, pw * 4u, &ctl->bar[stage]);
        tma_load_1d(dt, p.packed + pr.t_word, tw * 4u, &ctl->bar[stage]);
    };
    auto pop = [&](int slot) -> uint32_t {
        const uint32_t pos = atomicAdd(p.queue, 1u);
        ctl->pos[slot] = pos;
        return pos < p.n_items ? p.order[pos] : kInvalidIdx;
    };

    if (tid == 0) {
        if (!ASCII) {
            mbar_init(&ctl->bar[0], 1);
            mbar_init(&ctl->bar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        const uint32_t first = pop(0);
        ctl->idx[0] = first;
        if (first != kInvalidIdx) issue_load(0, first);
    }
    G::sync();

    int stage = 0;
    uint32_t phase_bits = 0; /* bit s = parity to wait for on stage s */

    while (true) {
        const uint32_t idx = ctl->idx[stage];
        if (idx == kInvalidIdx) break;
        if (CKPT) arena = p.arena + (size_t)ctl->pos[stage] * p.arena_units;
        if (tid == 0 && p.stages == 2) {
            /* prefetch the next pair into the other stage while this one computes */
            const uint32_t nxt = pop(stage ^ 1);
            ctl->idx[stage ^ 1] = nxt;
            if (nxt != kInvalidIdx) issue_load(stage ^ 1, nxt);
        }
        const wfagpu_pair_t pr = p.pairs[idx];
        const int plen = (int)pr.plen, tlen = (int)pr.tlen;
        const int kt = tlen - plen;
        /* ends-free: this pair's span (clamped by the host), its target diagonals, and how much narrower than the batch's
         * widest start row W = steps[0].n its own start row [-pb, tb] is on either side (prune_window_range) */
        const int4 sp = EF ? p.spans[idx] : make_int4(0, 0, 0, 0);
        const int ef_w = EF ? (int)p.steps[0].n : 0;
        const int ef_dp = ef_w - sp.x, ef_dt = ef_w - sp.z;
        const int klo_t = EF ? kt - sp.w : kt, khi_t = EF ? kt + sp.y : kt;

        const uint32_t Pa = seq_sa + (uint32_t)(2 * stage) * seq_bytes;
        const uint32_t Ta = Pa + seq_bytes;
        const char *const Pg = p.ascii + pr.p_ascii;
        const char *const Tg = p.ascii + pr.t_ascii;
        auto extend = [&](int k, int off) -> int {
            if (ASCII) return extend_ascii(Pg, Tg, plen, tlen, k, off, NULLV);
            return extend_packed(Pa, Ta, plen, tlen, k, off, NULLV);
        };

        /* pairs flagged by the packer are left to the byte-compare launch */
        const bool skip = !ASCII && (pr.flags & WFAGPU_PAIR_HAS_N);

        /* ---- ring prologue: NULL over [-2G, 2G] on every row (no full re-init) ---- */
        if constexpr (EF) {
            /* ... widened by this pair's start row half width max(pb, tb): its windows of the first A scores reach that
             * + A - 1 (own reach, prune_window_range) */
            const int wz = min(max(sp.x, sp.z), p.n_cap);
            const int span = 4 * GW + 2 * wz + 1;
            const int total = rows * span;
            for (int i = tid; i < total; i += gsz) {
                const int r = i / span;
                const int k = i - r * span - 2 * GW - wz;
                R::st(R::add(M0, (uint32_t)r * row_bytes), k, NULLV);
            }
            if (tid == 0) ctl->k_end = INT_MAX;
        } else {
            const int span = 4 * GW + 1;
            const int total = rows * span;
            for (int i = tid; i < total; i += gsz) {
                const int r = i / span;
                const int k = i - r * span - 2 * GW;
                R::st(R::add(M0, (uint32_t)r * row_bytes), k, NULLV);
            }
        }
        if (!ASCII) mbar_wait(&ctl->bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        G::sync();

        int dist = 0;
        bool finished = false;
        int k_end = kt;                              /* ends-free: diagonal of the finishing cell */
        int k_org = 0;                               /* ORG: origin of the finishing cell (score > 0) */
        /* ends-free end test: the lowest finishing diagonal of the group (kb = INT_MAX: none on this thread); also the
         * barrier after the score's cells */
        auto ef_lowest = [&](int kb) -> int {
            if constexpr (WARP) {
                __syncwarp();
                return __reduce_min_sync(0xffffffffu, kb);
            } else {
                if (kb != INT_MAX) atomicMin(&ctl->k_end, kb);
                return __syncthreads_or(kb != INT_MAX) ? ctl->k_end : INT_MAX;
            }
        };

        if (!skip) {
            /* Score-bound pruning: this launch only reports pairs that finish with a score <= Dmax
             * (d_end - 1, or the pair's own bound from wfa_bound_kernel), and every diagonal between k
             * and the target diagonal kt costs at least one gap extension, so a cell (d, k) with
             * d + e * |k - kt| > Dmax cannot be on such an alignment.  Those cells are not computed and
             * read as NULL; the cells of the optimal path keep their offsets and win the same
             * tie-breaks (proof and poisoned-cell model: oracle/kernel_model.c, km_prune_range).
             * Ends-free: the same with the distance to the target range. */
            const int Dmax = p.bound ? min(p.d_end - 1, p.bound[idx]) : p.d_end - 1;
            /* schedule records of scores dbase .. dbase + kSchedBlock - 1 (warp 0, one score per lane) */
            auto fill_sched = [&](int dbase, int buf) {
                if constexpr (SCHED) {
                    const int d = dbase + tid;
                    StepRec r;
                    r.lo = 0; r.hi = -1; r.flags = kRecStop; r.n = 0; r.ck_j = 0;
                    r.aMc = r.aMx = r.aMo = r.aIc = r.aIe = r.aDc = r.aDe = 0;
                    if (d <= Dmax) {
                        const wfagpu_step_t st = p.steps[d];
                        int lo, hi;
                        const bool live = EF ? prune_window_range((int)st.n, klo_t, khi_t, (Dmax - d) / e, p.n_cap, ef_dp, ef_dt, lo, hi)
                                             : prune_window((int)st.n, kt, (Dmax - d) / e, p.n_cap, lo, hi);
                        const bool stop = live && (lo < -p.n_cap || hi > p.n_cap);     /* wider than the rings */
                        const bool work = live && st.kind != WFAGPU_STEP_NULL;
                        r.lo = lo; r.hi = hi; r.n = (int)st.n;
                        r.flags = (uint32_t)st.kind | (live ? kRecLive : 0u) | (stop ? kRecStop : 0u) |
                                  ((work && (EF ? (khi_t >= lo && klo_t <= hi) : (kt >= lo && kt <= hi))) ? kRecTarget : 0u) |
                                  ((CKPT && d % p.ck_period == 0) ? kRecSnap : 0u);
                        r.ck_j = CKPT ? (uint32_t)(d / p.ck_period) : st.row_off;    /* snapshot index, or decision row */
                        const int dm = d % A, de1 = d % E1;
                        int sx = dm - x % A; if (sx < 0) sx += A;
                        int so = dm - oe % A; if (so < 0) so += A;
                        int se = de1 - e % E1; if (se < 0) se += E1;
                        r.aMc = (uint32_t)M0 + (uint32_t)dm * row_bytes;
                        r.aMx = (uint32_t)M0 + (uint32_t)sx * row_bytes;
                        r.aMo = (uint32_t)M0 + (uint32_t)so * row_bytes;
                        r.aIc = (uint32_t)I0 + (uint32_t)de1 * row_bytes;
                        r.aIe = (uint32_t)I0 + (uint32_t)se * row_bytes;
                        r.aDc = (uint32_t)D0 + (uint32_t)de1 * row_bytes;
                        r.aDe = (uint32_t)D0 + (uint32_t)se * row_bytes;
                    }
                    const uint32_t a = sched_sa + (uint32_t)(buf * kSchedBlock + tid) * (uint32_t)sizeof(StepRec);
                    sts_v4(a, make_uint4((uint32_t)r.lo, (uint32_t)r.hi, r.flags, (uint32_t)r.n));
                    sts_v4(a + 16u, make_uint4(r.aMc, r.aMx, r.aMo, r.aIc));
                    sts_v4(a + 32u, make_uint4(r.aIe, r.aDc, r.aDe, r.ck_j));
                }
            };
            bool stop0 = false;                      /* ends-free: finished (or too wide for the rings) at score 0 */
            if constexpr (EF) {
                /* score 0: the start row [-pb, tb] (the own reach of score 0), within the pruning window of score 0 */
                int lo0, hi0;
                const bool live0 = prune_window_range(ef_w, klo_t, khi_t, Dmax / e, p.n_cap, ef_dp, ef_dt, lo0, hi0);
                const int slo = live0 ? lo0 : 1, shi = live0 ? hi0 : 0;
                int kb = INT_MAX;
                if (slo >= -p.n_cap && shi <= p.n_cap) {
                    for (int k = slo + tid; k <= shi; k += gsz) {
                        const int m = extend(k, max(0, k));
                        R::st(M0, k, m);
                        if constexpr (ORG) R::st(R::add(M0, org_off), k, k);
                        if (k >= klo_t && k <= khi_t && m == min(tlen, plen + k)) kb = min(kb, k);
                    }
                } else {
                    stop0 = true;                    /* re-dispatched with wider rings */
                }
                if (SCHED && tid < kSchedBlock) fill_sched(1, 0);
                kb = ef_lowest(kb);
                if (kb != INT_MAX) { finished = true; k_end = kb; stop0 = true; }
            } else {
                if (tid == 0) R::st(M0, 0, extend(0, 0));
                if (SCHED && tid < kSchedBlock) fill_sched(1, 0);
                G::sync();
            }
            if (EF ? stop0 : (kt == 0 && R::ld(M0, 0) == tlen)) {
                finished = EF ? finished : true;
            } else {
                wfagpu_step_t st_next = p.steps[1 < p.d_end ? 1 : 0];
                /* Row addresses of the current score and of its sources are carried from
                 * score to score (one add + wrap each) so that the diagonal loop sees them
                 * as plain live values instead of re-deriving them. */
                const RA Mend = R::add(M0, (uint32_t)A * row_bytes);
                const RA Iend = R::add(I0, (uint32_t)E1 * row_bytes);
                const RA Dend = R::add(D0, (uint32_t)E1 * row_bytes);
                RA aMc = M0, aIc = I0, aDc = D0;                                    /* rows of score d (d = 0 now) */
                RA aMx = R::add(M0, (uint32_t)((A - x % A) % A) * row_bytes);       /* row of score d - x     */
                RA aMo = R::add(M0, (uint32_t)((A - oe % A) % A) * row_bytes);      /* row of score d - o - e */
                RA aIe = R::add(I0, (uint32_t)((E1 - e % E1) % E1) * row_bytes);    /* row of score d - e     */
                RA aDe = R::add(D0, (uint32_t)((E1 - e % E1) % E1) * row_bytes);
                /* 2-piece: rows of I2 / D2 at d and d - e2, and of M at d - o2 - e2.  In an M/I/D step driven by
                 * piece 1 with d < o2 + e2 (or the other way round) the M row of d - o2 - e2 is a row no score has
                 * written yet: it reads as NULL only because the prologue covers [-2G, 2G] and the windows of the
                 * first A scores (half width <= d < A = G) stay inside it. */
                if constexpr (P2) {
                    const int E2 = p.E2;
                    q2.Ic = q2.I0; q2.Dc = q2.D0;
                    q2.Mo = R::add(M0, (uint32_t)((A - q2.oe2 % A) % A) * row_bytes);
                    q2.Ie = R::add(q2.I0, (uint32_t)((E2 - q2.e2 % E2) % E2) * row_bytes);
                    q2.De = R::add(q2.D0, (uint32_t)((E2 - q2.e2 % E2) % E2) * row_bytes);
                }
                int ck_left = p.ck_period, ck_j = 0;
                /* snapshot of the ring rows the scores above d can still read: M of scores d .. d-A+2,
                 * I and D of d .. d-e+1.  A snapshot row covers [-n, n] rounded out to 16-byte units;
                 * only the units of [lo - 1, hi + 1] (all that later scores can read) are copied. */
                auto checkpoint = [&](int n, int lo, int hi) {
                    if constexpr (CKPT) {
                        const int pitch = (((n + 7) & ~7) + ((n + 8) & ~7)) >> 3;       /* units per snapshot row */
                        const int k0 = max((lo - 1) & ~7, -((n + 7) & ~7));               /* floor to 8 diagonals   */
                        const int units = ((min((hi + 1) | 7, ((n + 8) & ~7) - 1) - k0) + 1) >> 3;
                        uint4 *dst = arena + p.ck_off[ck_j] + ((k0 + ((n + 7) & ~7)) >> 3);
                        uint32_t row = (uint32_t)aMc;
                        for (int a = 0; a < A - 1; ++a) {
                            for (int q = tid; q < units; q += gsz) __stcs(dst + q, lds_v4(row + (uint32_t)(2 * k0) + 16u * (uint32_t)q));
                            dst += pitch;
                            row = (row == (uint32_t)M0) ? (uint32_t)Mend - row_bytes : row - row_bytes;
                        }
                        row = (uint32_t)aIc;
                        for (int a = 0; a < e; ++a) {
                            for (int q = tid; q < units; q += gsz) __stcs(dst + q, lds_v4(row + (uint32_t)(2 * k0) + 16u * (uint32_t)q));
                            dst += pitch;
                            row = (row == (uint32_t)I0) ? (uint32_t)Iend - row_bytes : row - row_bytes;
                        }
                        row = (uint32_t)aDc;
                        for (int a = 0; a < e; ++a) {
                            for (int q = tid; q < units; q += gsz) __stcs(dst + q, lds_v4(row + (uint32_t)(2 * k0) + 16u * (uint32_t)q));
                            dst += pitch;
                            row = (row == (uint32_t)D0) ? (uint32_t)Dend - row_bytes : row - row_bytes;
                        }
                    }
                };
                int pr_q = Dmax / e, pr_r = Dmax % e;        /* (Dmax - d) = q * e + r */
                if constexpr (P2) { pr_q = Dmax / q2.ep; pr_r = Dmax % q2.ep; }     /* 2-piece: q * min(e1, e2) + r */
                unsigned long long n_cells = 0;              /* cells computed for this pair (optional counter) */
                for (int d = 1; d <= Dmax; ++d) {
                    int n, lo, hi, kind;
                    uint32_t row_off = 0;                        /* decision-byte row of this score (!CKPT) */
                    bool live, target_in, snap_now;
                    if constexpr (SCHED) {
                        const int ri = (d - 1) & (kSchedBlock - 1), buf = ((d - 1) / kSchedBlock) & 1;
                        if (ri == 0 && tid < kSchedBlock) fill_sched(d + kSchedBlock, buf ^ 1);       /* the block after this one */
                        const uint32_t a = sched_sa + (uint32_t)(buf * kSchedBlock + ri) * (uint32_t)sizeof(StepRec);
                        const uint4 r0 = lds_v4(a), r1 = lds_v4(a + 16u), r2 = lds_v4(a + 32u);
                        if (r0.z & kRecStop) break;
                        lo = (int)r0.x; hi = (int)r0.y; n = (int)r0.w;
                        kind = (int)(r0.z & 3u);
                        live = (r0.z & kRecLive) != 0;
                        target_in = (r0.z & kRecTarget) != 0;
                        snap_now = (r0.z & kRecSnap) != 0;
                        aMc = r1.x; aMx = r1.y; aMo = r1.z; aIc = r1.w;
                        aIe = r2.x; aDc = r2.y; aDe = r2.z;
                        if (CKPT) ck_j = (int)r2.w; else row_off = r2.w;
                        if (p.cells && live && kind != WFAGPU_STEP_NULL) n_cells += (unsigned)(hi - lo + 1);
                    } else {
                        const wfagpu_step_t st = st_next;
                        if (d + 1 < p.d_end) st_next = p.steps[d + 1];
                        n = st.n;
                        kind = st.kind;
                        row_off = st.row_off;
                        if constexpr (P2) {
                            if (pr_r == 0) { pr_r = q2.ep - 1; --pr_q; } else --pr_r;
                        } else {
                            if (pr_r == 0) { pr_r = e - 1; --pr_q; } else --pr_r;
                        }
                        live = EF ? prune_window_range(n, klo_t, khi_t, pr_q, p.n_cap, ef_dp, ef_dt, lo, hi)
                                  : prune_window(n, kt, pr_q, p.n_cap, lo, hi);
                        if (live && (lo < -p.n_cap || hi > p.n_cap)) break;     /* wider than the rings of this launch */
                        if (live && kind != WFAGPU_STEP_NULL) n_cells += (unsigned)(hi - lo + 1);
                        target_in = live && kind != WFAGPU_STEP_NULL && kt >= lo && kt <= hi;
                        aMc = R::add(aMc, row_bytes); if (aMc == Mend) aMc = M0;
                        aMx = R::add(aMx, row_bytes); if (aMx == Mend) aMx = M0;
                        aMo = R::add(aMo, row_bytes); if (aMo == Mend) aMo = M0;
                        aIc = R::add(aIc, row_bytes); if (aIc == Iend) aIc = I0;
                        aIe = R::add(aIe, row_bytes); if (aIe == Iend) aIe = I0;
                        aDc = R::add(aDc, row_bytes); if (aDc == Dend) aDc = D0;
                        aDe = R::add(aDe, row_bytes); if (aDe == Dend) aDe = D0;
                        if constexpr (P2) {
                            q2.Mo = R::add(q2.Mo, row_bytes); if (q2.Mo == Mend) q2.Mo = M0;
                            q2.Ic = R::add(q2.Ic, row_bytes); if (q2.Ic == q2.Iend) q2.Ic = q2.I0;
                            q2.Ie = R::add(q2.Ie, row_bytes); if (q2.Ie == q2.Iend) q2.Ie = q2.I0;
                            q2.Dc = R::add(q2.Dc, row_bytes); if (q2.Dc == q2.Dend) q2.Dc = q2.D0;
                            q2.De = R::add(q2.De, row_bytes); if (q2.De == q2.Dend) q2.De = q2.D0;
                        }
                        snap_now = false;
                        if (CKPT && --ck_left == 0) { ck_left = p.ck_period; ++ck_j; snap_now = true; }
                    }

                    if (kind == WFAGPU_STEP_NULL || !live) {
                        for (int k = lo - GW + tid; k <= hi + GW; k += gsz) {
                            R::st(aMc, k, NULLV);
                            R::st(aIc, k, NULLV);
                            R::st(aDc, k, NULLV);
                            if constexpr (P2) { R::st(q2.Ic, k, NULLV); R::st(q2.Dc, k, NULLV); }
                        }
                        G::sync();
                        if (CKPT && snap_now) checkpoint(n, lo, hi);
                        continue;
                    }
                    int kb = INT_MAX;                            /* ends-free: lowest finishing diagonal of this thread */
                    if (kind == WFAGPU_STEP_M) {
                        for (int k = lo - GW + tid; k <= hi + GW; k += gsz) {
                            R::st(aIc, k, NULLV);
                            R::st(aDc, k, NULLV);
                            if constexpr (P2) { R::st(q2.Ic, k, NULLV); R::st(q2.Dc, k, NULLV); }
                            int m = NULLV;
                            if (k >= lo && k <= hi) {
                                m = R::ld(aMx, k) + 1;
                                if (m >= 0) m = extend(k, m);
                                if (EF && k >= klo_t && k <= khi_t && m == min(tlen, plen + k)) kb = min(kb, k);
                                if constexpr (ORG) R::st(R::add(aMc, org_off), k, R::ld(R::add(aMx, org_off), k));
                            }
                            R::st(aMc, k, m);
                        }
                    } else {
                        /* guard cells: NULL on both sides of [lo, hi] */
                        for (int g = tid; g < 2 * GW; g += gsz) {
                            const int k = (g < GW) ? (lo - 1 - g) : (hi + 1 + (g - GW));
                            R::st(aMc, k, NULLV);
                            R::st(aIc, k, NULLV);
                            R::st(aDc, k, NULLV);
                            if constexpr (P2) { R::st(q2.Ic, k, NULLV); R::st(q2.Dc, k, NULLV); }
                        }
                        /* one decision byte per cell: bit0 I extends, bit1 D extends, bits 3:2 the winner of M
                         * (1 = I, 2 = X, 3 = D); a warp writes 32 consecutive bytes of the pair's row */
                        uint8_t *const rowb = reinterpret_cast<uint8_t *>(arena + row_off) + n;
                        if constexpr (P2) {
                            /* 2-piece decision byte: bit0 I1 extends, bit1 D1, bit2 I2, bit3 D2; bits 5:4 the op of M's
                             * source (1 = I, 2 = X, 3 = D); bit6 that source is piece 2.  M: D1 > D2 > X > I1 > I2. */
                            for (int k = lo + tid; k <= hi; k += gsz) {
                                const int io1 = R::ld(aMo, k - 1) + 1, ie1 = R::ld(aIe, k - 1) + 1;
                                const int io2 = R::ld(q2.Mo, k - 1) + 1, ie2 = R::ld(q2.Ie, k - 1) + 1;
                                const int do1 = R::ld(aMo, k + 1), de1 = R::ld(aDe, k + 1);
                                const int do2 = R::ld(q2.Mo, k + 1), de2 = R::ld(q2.De, k + 1);
                                const int X = R::ld(aMx, k) + 1;
                                const int I1 = max(io1, ie1), D1 = max(do1, de1);
                                const int I2 = max(io2, ie2), D2 = max(do2, de2);
                                const int I = max(I1, I2), D = max(D1, D2);
                                int M = max(max(X, D), I);
                                uint32_t src;
                                if (D >= X && D >= I) src = D1 >= D2 ? 0x30u : 0x70u;
                                else if (X >= I) src = 0x20u;
                                else src = I1 >= I2 ? 0x10u : 0x50u;
                                if (M >= 0) M = extend(k, M);
                                R::st(aIc, k, I1);
                                R::st(aDc, k, D1);
                                R::st(q2.Ic, k, I2);
                                R::st(q2.Dc, k, D2);
                                R::st(aMc, k, M);
                                if (BT) rowb[k] = (uint8_t)((ie1 >= io1 ? 1u : 0u) | (de1 >= do1 ? 2u : 0u) |
                                                            (ie2 >= io2 ? 4u : 0u) | (de2 >= do2 ? 8u : 0u) | src);
                            }
                        } else
                        for (int k = lo + tid; k <= hi; k += gsz) {
                            const int io = R::ld(aMo, k - 1) + 1;
                            const int ie = R::ld(aIe, k - 1) + 1;
                            const int dopen = R::ld(aMo, k + 1);
                            const int dext = R::ld(aDe, k + 1);
                            const int X = R::ld(aMx, k) + 1;
                            /* Offsets by plain max; the tie-breaks only decide the backtrace bits:
                             * I/D: extend beats open on equal offsets; M: D beats X beats I. */
                            const int I = max(io, ie);
                            const int D = max(dopen, dext);
                            int M = max(max(X, D), I);
                            const bool bI = ie >= io;
                            const bool bD = dext >= dopen;
                            const bool bM0 = (D >= X) || (I > X);      /* winner is I(1) or D(3): not X */
                            const bool bM1 = (D >= I) || (X >= I);      /* winner is X(2) or D(3): not I */
                            if (M >= 0) M = extend(k, M);
                            R::st(aIc, k, I);
                            R::st(aDc, k, D);
                            R::st(aMc, k, M);
                            if (BT && !CKPT) rowb[k] = (uint8_t)((bI ? 1u : 0u) | (bD ? 2u : 0u) | (bM0 ? 4u : 0u) | (bM1 ? 8u : 0u));
                            if constexpr (ORG) {
                                /* the origin of the winner the decision byte would record */
                                const int oI = R::ld(R::add(bI ? aIe : aMo, org_off), k - 1);
                                const int oD = R::ld(R::add(bD ? aDe : aMo, org_off), k + 1);
                                const int oM = bM1 ? (bM0 ? oD : R::ld(R::add(aMx, org_off), k)) : oI;
                                R::st(R::add(aIc, org_off), k, oI);
                                R::st(R::add(aDc, org_off), k, oD);
                                R::st(R::add(aMc, org_off), k, oM);
                            }
                            if (EF && k >= klo_t && k <= khi_t && M == min(tlen, plen + k)) kb = min(kb, k);
                        }
                    }
                    if constexpr (EF) {
                        kb = ef_lowest(kb);
                        if (kb != INT_MAX) {
                            finished = true;
                            dist = d;
                            k_end = kb;
                            if constexpr (ORG) k_org = R::ld(R::add(aMc, org_off), kb);
                            break;
                        }
                    } else {
                        G::sync();
                        if (target_in && R::ld(aMc, kt) == tlen) {
                            finished = true;
                            dist = d;
                            break;
                        }
                    }
                    if (CKPT && snap_now) checkpoint(n, lo, hi);
                }
                if (p.cells && tid == 0) atomicAdd(p.cells, n_cells);
            }
        }

        /* ---- traceback -> 2-bit ops, newest first ---- */
        uint32_t n_ops = 0;
        if (tid == 0) {
            uint32_t ops_off = 0;
            int k_begin = (ORG && dist > 0) ? k_org : k_end;    /* ends-free: diagonal of the path's score-0 cell */
            if (BT && finished && dist > 0) {
              if constexpr (!CKPT) {
                int cd = dist, ck = EF ? k_end : kt, comp = 0;
                uint32_t word = 0;
                while (!(comp == 0 && cd == 0)) {
                    const wfagpu_step_t st = p.steps[cd];
                    uint32_t op;
                    if (comp == 0) {
                        op = OP_SUB;
                        if (st.kind == WFAGPU_STEP_M) {
                            cd -= x;
                        } else {
                            const int ii = ck + (int)st.n;
                            if (ii < 0 || ii > 2 * (int)st.n) { n_ops = 0; finished = false; break; }
                            const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                            const int mop = (int)(dec >> (P2 ? 4 : 2)) & 3;
                            if (mop == OP_SUB) cd -= x;
                            else if (mop == OP_INS) comp = (P2 && (dec & 64u)) ? 3 : 1;
                            else comp = (P2 && (dec & 64u)) ? 4 : 2;
                        }
                    } else if constexpr (P2) {
                        /* comp 1 I1, 2 D1, 3 I2, 4 D2: the extend bit of comp c is bit c - 1; closing a gap of piece i
                         * steps o_i + e_i down */
                        const int ii = ck + (int)st.n;
                        if (ii < 0 || ii > 2 * (int)st.n || st.kind != WFAGPU_STEP_MDI) { n_ops = 0; finished = false; break; }
                        const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                        const bool ins = (comp & 1) != 0, second = comp >= 3;
                        op = ins ? OP_INS : OP_DEL;
                        ck += ins ? -1 : 1;
                        if (dec & (1u << (comp - 1))) cd -= second ? q2.e2 : e;
                        else { cd -= second ? q2.oe2 : oe; comp = 0; }
                    } else {
                        const int ii = ck + (int)st.n;
                        if (ii < 0 || ii > 2 * (int)st.n || st.kind != WFAGPU_STEP_MDI) { n_ops = 0; finished = false; break; }
                        const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                        if (comp == 1) {
                            op = OP_INS;
                            ck -= 1;
                            if (dec & 1u) cd -= e; else { cd -= oe; comp = 0; }
                        } else {
                            op = OP_DEL;
                            ck += 1;
                            if (dec & 2u) cd -= e; else { cd -= oe; comp = 0; }
                        }
                    }
                    word |= op << (2 * (n_ops & 15u));
                    ++n_ops;
                    if ((n_ops & 15u) == 0) {
                        scratch[(n_ops >> 4) - 1] = word;
                        word = 0;
                    }
                    if (cd < 0 || (n_ops >> 4) >= p.ops_scratch_words) { n_ops = 0; finished = false; break; }
                }
                if (n_ops & 15u) scratch[n_ops >> 4] = word;
                const uint32_t nw = (n_ops + 15u) >> 4;
                ops_off = atomicAdd(p.ops_pool_head, nw);
                if (ops_off + nw > p.ops_pool_words) { n_ops = 0; finished = false; }
                if (EF) k_begin = ck;
              }
            }
            if (EF && finished) p.ends[idx] = make_int2(k_begin, k_end);
            ctl->n_ops = n_ops;
            ctl->ops_off = ops_off;
            wfagpu_pair_out_t r;
            r.distance = finished ? dist : 0;
            r.ops_off = ops_off;
            r.n_ops = n_ops;
            if (skip) {
                r.status = WFAGPU_ST_NEEDS_ASCII;
                p.ascii_list[atomicAdd(p.ascii_count, 1u)] = idx;
            } else if (finished) {
                r.status = WFAGPU_ST_FINISHED;
            } else {
                r.status = WFAGPU_ST_OVERBUDGET;
                p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
            }
            p.out[idx] = r;
        }
        G::sync();
        if (BT && !CKPT) {
            /* copy the op words from the group's scratch into the pool (coalesced) */
            const uint32_t nw = (ctl->n_ops + 15u) >> 4;
            const uint32_t off = ctl->ops_off;
            for (uint32_t i = tid; i < nw; i += gsz) p.ops_pool[off + i] = scratch[i];
        }
        G::sync();
        if (p.stages == 2) {
            stage ^= 1;
        } else {
            if (tid == 0) {
                /* single buffer (shared memory is tight): fetch the next pair now */
                const uint32_t nxt = pop(0);
                ctl->idx[0] = nxt;
                if (nxt != kInvalidIdx) issue_load(0, nxt);
            }
            G::sync();
        }
    }
}

/* ======================================================================== */
/*    CTA-per-pair wavefront kernel, four diagonals per thread (s16x2)      */
/* ======================================================================== */
/*
 * Same recurrence, windows, ring layout, schedule records and snapshots as
 * wfa_exact_kernel<false, false, BT, RingS16, CKPT> (so the traceback kernel and the
 * parity argument are unchanged), but
 *  (1) a thread owns FOUR adjacent diagonals k .. k+3 (k a multiple of 4) per trip:
 *      the source rows arrive as LDS.64 + LDS.32/U16 (the k-1 / k+4 neighbours) instead of
 *      20 x LDS.S16, the results leave as 3 x STS.64; I, D and the max of M run on packed
 *      int16 pairs (VIMNMX.S16x2, VIADD.16x2, VIMNMX3.S16x2 -- the DPX integer SIMD of
 *      sm_90+), the k-1 / k+1 shifts are PRMTs;
 *  (2) the extend keeps one cell per lane-slot but its common case (the run ends within the
 *      9 bases every packed window is good for, and the cell is more than 8 bases away from
 *      both sequence ends) is branch-free: predicated LDS x 2, XOR, FLO, predicated add --
 *      no clamping; everything else calls the out-of-line general extend;
 *  (3) TWO scores per barrier when the penalties allow it (x >= 2, o + e >= 2, e == 1):
 *      score d + 1 reads M of d - 1 and d - 3 and the I / D cells of score d, never the extended
 *      M of score d, so a thread computes its quad for d and d + 1 back to back; the two I / D cells
 *      of score d it needs from its neighbours (k - 1 for I, k + 4 for D) it recomputes from the old
 *      rows (two packed ops).  Halves the barriers and the per-score control work.
 * Cells of a quad outside a score's window [lo, hi] are written as NULL, so the rings hold exactly
 * what the one-diagonal-per-thread kernel leaves in them wherever a later score or a snapshot reads.
 */
__device__ __forceinline__ uint2 lds_v2(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_v2(uint32_t a, uint32_t x, uint32_t y)
{
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

__device__ __noinline__ int extend_packed_general(uint32_t Pa, uint32_t Ta, int plen, int tlen, int k, int off, int null_v)
{
    return extend_packed(Pa, Ta, plen, tlen, k, off, null_v);
}

/* The common case of an extend, branch-free so that the four cells of a quad overlap: returns the
 * XOR of the two 16-base windows at (m - k, m), or 0 when the cell is NULL or within 8 bases of the end of a
 * sequence (limp = max(min(plen + k, tlen) - 8, 0)).  A result >= 0x4000 means the run ends within the 9
 * bases every window is good for and nothing has to be clamped: m += clz >> 1. */
__device__ __forceinline__ uint32_t extend_probe(uint32_t Pa, uint32_t Ta, int k, int m, int limp)
{
    const uint32_t uv = (uint32_t)(m - k), uh = (uint32_t)m;
    uint32_t ap, at, wp = 0, wt = 0;
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(ap) : "r"(uv >> 3), "r"(Pa));
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(at) : "r"(uh >> 3), "r"(Ta));
    /* predicated loads (no branch): a NULL or near-the-end cell loads nothing and yields 0 */
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "setp.lt.u32 p, %4, %5;\n"
                 "@p ld.shared.u32 %0, [%2];\n"
                 "@p ld.shared.u32 %1, [%3];\n"
                 "}\n" : "+r"(wp), "+r"(wt) : "r"(ap), "r"(at), "r"((uint32_t)m), "r"((uint32_t)limp));
    return (wp << ((uv & 7u) * 2u)) ^ (wt << ((uh & 7u) * 2u));
}

/* m += clz(f) >> 1 when f >= 0x4000 (a run of at most 8 bases), predicated */
__device__ __forceinline__ int add_run(int m, uint32_t f)
{
    asm("{\n"
        ".reg .pred p;\n"
        ".reg .u32 t;\n"
        "setp.ge.u32 p, %1, 0x4000;\n"
        "bfind.u32 t, %1;\n"
        "shr.u32 t, t, 1;\n"
        "sub.s32 t, 15, t;\n"
        "@p add.s32 %0, %0, t;\n"
        "}\n" : "+r"(m) : "r"(f));
    return m;
}

constexpr uint32_t kNull2 = 0x83008300u;          /* two int16 NULLs (-32000) */
constexpr uint32_t kOnes2 = 0x00010001u;

/* mask of the cells (k, k+1) inside [lo, hi]; packed value with the cells outside replaced by NULL */
__device__ __forceinline__ uint32_t in2(int k, int lo, int hi)
{
    return ((k >= lo && k <= hi) ? 0xffffu : 0u) | ((k + 1 >= lo && k + 1 <= hi) ? 0xffff0000u : 0u);
}
__device__ __forceinline__ uint32_t sel2(uint32_t v, uint32_t mask) { return (v & mask) | (kNull2 & ~mask); }

/* extend the four M cells m0 .. m3 of the quad that starts at diagonal kq (null_v: what a cell outside the
 * sequences becomes; the probes treat every negative offset as NULL) */
__device__ __forceinline__ void extend_cells(uint32_t Pa, uint32_t Ta, int plen, int tlen, int kq, int tl8,
                                             int &m0, int &m1, int &m2, int &m3, const int null_v)
{
    const int c8 = kq + plen - 8;
    const uint32_t f0 = extend_probe(Pa, Ta, kq, m0, __viaddmin_s32_relu(c8, 0, tl8));
    const uint32_t f1 = extend_probe(Pa, Ta, kq + 1, m1, __viaddmin_s32_relu(c8, 1, tl8));
    const uint32_t f2 = extend_probe(Pa, Ta, kq + 2, m2, __viaddmin_s32_relu(c8, 2, tl8));
    const uint32_t f3 = extend_probe(Pa, Ta, kq + 3, m3, __viaddmin_s32_relu(c8, 3, tl8));
    /* z < 0x4000: a valid cell whose probe did not settle it -- a long run (the cells on the alignment
     * path) or a cell next to the end of a sequence: rare, out of line */
    const uint32_t z0 = f0 | ((uint32_t)m0 & 0x80000000u), z1 = f1 | ((uint32_t)m1 & 0x80000000u);
    const uint32_t z2 = f2 | ((uint32_t)m2 & 0x80000000u), z3 = f3 | ((uint32_t)m3 & 0x80000000u);
    m0 = add_run(m0, f0);
    m1 = add_run(m1, f1);
    m2 = add_run(m2, f2);
    m3 = add_run(m3, f3);
    if (min(min(z0, z1), min(z2, z3)) < 0x4000u) {
        if (z0 < 0x4000u) m0 = extend_packed_general(Pa, Ta, plen, tlen, kq, m0, null_v);
        if (z1 < 0x4000u) m1 = extend_packed_general(Pa, Ta, plen, tlen, kq + 1, m1, null_v);
        if (z2 < 0x4000u) m2 = extend_packed_general(Pa, Ta, plen, tlen, kq + 2, m2, null_v);
        if (z3 < 0x4000u) m3 = extend_packed_general(Pa, Ta, plen, tlen, kq + 3, m3, null_v);
    }
}

/* the same on two packed int16 pairs (M01 | M23) */
__device__ __forceinline__ void extend_quad(uint32_t Pa, uint32_t Ta, int plen, int tlen, int kq, int tl8,
                                            uint32_t &M01, uint32_t &M23)
{
    int m0 = (int)(short)(M01 & 0xffffu), m1 = (int)M01 >> 16;
    int m2 = (int)(short)(M23 & 0xffffu), m3 = (int)M23 >> 16;
    extend_cells(Pa, Ta, plen, tlen, kq, tl8, m0, m1, m2, m3, kOffNull);
    M01 = __byte_perm((uint32_t)m0, (uint32_t)m1, 0x5410);
    M23 = __byte_perm((uint32_t)m2, (uint32_t)m3, 0x5410);
}

template <bool BT, bool COUNT>
__global__ void __launch_bounds__(512, 1) wfa_quad_kernel(const __grid_constant__ KernelParams p)
{
    constexpr bool CKPT = BT;                     /* with backtrace: ring snapshots (wfa_traceback_kernel follows) */
    constexpr int NULLV = kOffNull;
    extern __shared__ __align__(16) unsigned char smem_raw[];

    const int tid = threadIdx.x, gsz = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, last_warp = (gsz >> 5) - 1;

    /* ---- shared memory: [rings][sequence stages][ctl][schedule records] (layout of wfa_exact_kernel) ---- */
    /* ring depths: one row more than the recurrence needs when two scores share a barrier interval (the
     * second score would otherwise overwrite rows d - A and d - e - 1 = sources of the first) */
    const int RM = p.ring_m, RG = p.ring_g;
    const int rows = RM + 2 * RG;
    const uint32_t row_bytes = (uint32_t)p.row_stride * 2u;
    const uint32_t ring_bytes = ((uint32_t)rows * row_bytes + 15u) & ~15u;
    const uint32_t seq_bytes = (uint32_t)p.seq_words * 4u;
    const uint32_t seq_total = 2u * (uint32_t)p.stages * seq_bytes;
    unsigned char *gbase = smem_raw;
    const uint32_t ring_sa = smem_u32(gbase);
    const uint32_t seq_sa = ring_sa + ring_bytes;
    GroupCtl *ctl = reinterpret_cast<GroupCtl *>(gbase + ring_bytes + seq_total);
    const uint32_t sched_sa = ring_sa + ring_bytes + seq_total + (uint32_t)sizeof(GroupCtl);

    const int x = p.x, e = p.e, A = p.A, GW = p.G;
    const int oe = p.o + p.e;
    const bool pairable = p.quad_pairs != 0;      /* two scores per barrier (host: x >= 2, o + e >= 2, e == 1, deeper rings) */
    const uint32_t M0 = ring_sa + 2u * (uint32_t)p.center;            /* row 0 of M, diagonal 0 (16-byte aligned) */
    const uint32_t I0 = M0 + (uint32_t)RM * row_bytes;
    const uint32_t D0 = I0 + (uint32_t)RG * row_bytes;
    const uint32_t Mend = M0 + (uint32_t)RM * row_bytes, Iend = I0 + (uint32_t)RG * row_bytes, Dend = D0 + (uint32_t)RG * row_bytes;

    uint4 *arena = p.arena;

    auto issue_load = [&](int stage, uint32_t idx) {
        const wfagpu_pair_t pr = p.pairs[idx];
        const uint32_t pw = ((((pr.plen + 7u) >> 3) + 1u) + 3u) & ~3u;
        const uint32_t tw = ((((pr.tlen + 7u) >> 3) + 1u) + 3u) & ~3u;
        unsigned char *dp = gbase + ring_bytes + (size_t)(2 * stage) * seq_bytes;
        unsigned char *dt = dp + seq_bytes;
        fence_proxy_async();
        mbar_expect_tx(&ctl->bar[stage], (pw + tw) * 4u);
        tma_load_1d(dp, p.packed + pr.p_word, pw * 4u, &ctl->bar[stage]);
        tma_load_1d(dt, p.packed + pr.t_word, tw * 4u, &ctl->bar[stage]);
    };
    auto pop = [&](int slot) -> uint32_t {
        const uint32_t pos = atomicAdd(p.queue, 1u);
        ctl->pos[slot] = pos;
        return pos < p.n_items ? p.order[pos] : kInvalidIdx;
    };

    if (tid == 0) {
        mbar_init(&ctl->bar[0], 1);
        mbar_init(&ctl->bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t first = pop(0);
        ctl->idx[0] = first;
        if (first != kInvalidIdx) issue_load(0, first);
    }
    __syncthreads();

    int stage = 0;
    uint32_t phase_bits = 0;

    while (true) {
        const uint32_t idx = ctl->idx[stage];
        if (idx == kInvalidIdx) break;
        if (CKPT) arena = p.arena + (size_t)ctl->pos[stage] * p.arena_units;
        if (tid == 0 && p.stages == 2) {
            const uint32_t nxt = pop(stage ^ 1);
            ctl->idx[stage ^ 1] = nxt;
            if (nxt != kInvalidIdx) issue_load(stage ^ 1, nxt);
        }
        const wfagpu_pair_t pr = p.pairs[idx];
        const int plen = (int)pr.plen, tlen = (int)pr.tlen;
        const int kt = tlen - plen;
        const uint32_t Pa = seq_sa + (uint32_t)(2 * stage) * seq_bytes;
        const uint32_t Ta = Pa + seq_bytes;
        const bool skip = (pr.flags & WFAGPU_PAIR_HAS_N) != 0;       /* left to the byte-compare launch */

        /* ring prologue: NULL over [-2G - 4, 2G + 4] on every row */
        {
            const int span = 4 * GW + 9;
            const int total = rows * span;
            for (int i = tid; i < total; i += gsz) {
                const int r = i / span;
                const int k = i - r * span - 2 * GW - 4;
                sts_16(M0 + (uint32_t)r * row_bytes + (uint32_t)(2 * k), NULLV);
            }
        }
        mbar_wait(&ctl->bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        __syncthreads();

        int dist = 0;
        bool finished = false;

        if (!skip) {
            const int Dmax = p.bound ? min(p.d_end - 1, p.bound[idx]) : p.d_end - 1;
            /* schedule records of scores dbase .. dbase + kSchedBlock - 1 (warp 0, one score per lane) */
            auto fill_sched = [&](int dbase, int buf) {
                const int d = dbase + tid;
                StepRec r;
                r.lo = 0; r.hi = -1; r.flags = kRecStop; r.n = 0; r.ck_j = 0;
                r.aMc = r.aMx = r.aMo = r.aIc = r.aIe = r.aDc = r.aDe = 0;
                if (d <= Dmax) {
                    const wfagpu_step_t st = p.steps[d];
                    int lo, hi;
                    const bool live = prune_window((int)st.n, kt, (Dmax - d) / e, p.n_cap, lo, hi);
                    const bool stop = live && (lo < -p.n_cap || hi > p.n_cap);
                    const bool work = live && st.kind != WFAGPU_STEP_NULL;
                    r.lo = lo; r.hi = hi; r.n = (int)st.n;
                    r.flags = (uint32_t)st.kind | (live ? kRecLive : 0u) | (stop ? kRecStop : 0u) |
                              ((work && kt >= lo && kt <= hi) ? kRecTarget : 0u) |
                              ((CKPT && d % p.ck_period == 0) ? kRecSnap : 0u);
                    r.ck_j = CKPT ? (uint32_t)(d / p.ck_period) : 0u;
                    const int dm = d % RM, de1 = d % RG;
                    int sx = dm - x % RM; if (sx < 0) sx += RM;
                    int so = dm - oe % RM; if (so < 0) so += RM;
                    int se = de1 - e % RG; if (se < 0) se += RG;
                    r.aMc = M0 + (uint32_t)dm * row_bytes;
                    r.aMx = M0 + (uint32_t)sx * row_bytes;
                    r.aMo = M0 + (uint32_t)so * row_bytes;
                    r.aIc = I0 + (uint32_t)de1 * row_bytes;
                    r.aIe = I0 + (uint32_t)se * row_bytes;
                    r.aDc = D0 + (uint32_t)de1 * row_bytes;
                    r.aDe = D0 + (uint32_t)se * row_bytes;
                }
                const uint32_t a = sched_sa + (uint32_t)(buf * kSchedBlock + tid) * (uint32_t)sizeof(StepRec);
                sts_v4(a, make_uint4((uint32_t)r.lo, (uint32_t)r.hi, r.flags, (uint32_t)r.n));
                sts_v4(a + 16u, make_uint4(r.aMc, r.aMx, r.aMo, r.aIc));
                sts_v4(a + 32u, make_uint4(r.aIe, r.aDc, r.aDe, r.ck_j));
            };
            auto rec_addr = [&](int d) -> uint32_t {
                return sched_sa + (uint32_t)((((d - 1) / kSchedBlock) & 1) * kSchedBlock + ((d - 1) & (kSchedBlock - 1))) * (uint32_t)sizeof(StepRec);
            };
            if (tid == 0) sts_16(M0, extend_packed(Pa, Ta, plen, tlen, 0, 0, NULLV));
            if (tid < kSchedBlock) fill_sched(1, 0);
            __syncthreads();
            if (kt == 0 && lds_s16(M0) == tlen) {
                finished = true;
            } else {
                const int tl8 = tlen - 8;
                unsigned long long n_cells = 0;
                /* snapshot of the ring rows later scores can still read (layout: wfa_exact_kernel) */
                auto checkpoint = [&](uint32_t aMc, uint32_t aIc, uint32_t aDc, int ck_j, int n, int lo, int hi) {
                    if constexpr (CKPT) {
                        const int pitch = (((n + 7) & ~7) + ((n + 8) & ~7)) >> 3;
                        const int k0 = max((lo - 1) & ~7, -((n + 7) & ~7));
                        const int units = ((min((hi + 1) | 7, ((n + 8) & ~7) - 1) - k0) + 1) >> 3;
                        uint4 *dst = arena + p.ck_off[ck_j] + ((k0 + ((n + 7) & ~7)) >> 3);
                        uint32_t row = aMc;
                        for (int a = 0; a < A - 1; ++a) {
                            for (int q = tid; q < units; q += gsz) __stcs(dst + q, lds_v4(row + (uint32_t)(2 * k0) + 16u * (uint32_t)q));
                            dst += pitch;
                            row = (row == M0) ? Mend - row_bytes : row - row_bytes;
                        }
                        row = aIc;
                        for (int a = 0; a < e; ++a) {
                            for (int q = tid; q < units; q += gsz) __stcs(dst + q, lds_v4(row + (uint32_t)(2 * k0) + 16u * (uint32_t)q));
                            dst += pitch;
                            row = (row == I0) ? Iend - row_bytes : row - row_bytes;
                        }
                        row = aDc;
                        for (int a = 0; a < e; ++a) {
                            for (int q = tid; q < units; q += gsz) __stcs(dst + q, lds_v4(row + (uint32_t)(2 * k0) + 16u * (uint32_t)q));
                            dst += pitch;
                            row = (row == D0) ? Dend - row_bytes : row - row_bytes;
                        }
                    }
                };
                /* guard cells: NULL on both sides of the quads [kq0, kend] of a row triple (one warp writes them) */
                auto guards = [&](uint32_t aMc, uint32_t aIc, uint32_t aDc, int kq0, int kend) {
                    for (int g = lane; g < 2 * GW; g += 32) {
                        const int k = (g < GW) ? (kq0 - 1 - g) : (kend + 1 + (g - GW));
                        sts_16(aMc + (uint32_t)(2 * k), NULLV);
                        sts_16(aIc + (uint32_t)(2 * k), NULLV);
                        sts_16(aDc + (uint32_t)(2 * k), NULLV);
                    }
                };
                int last_blk = -1;
                int d = 1;
                while (d <= Dmax) {
                    const int blk = (d - 1) / kSchedBlock;
                    if (blk != last_blk) {
                        /* first trip in this block of records: warp 0 derives the next block (the other buffer
                         * held block blk - 1, which nobody reads any more: a barrier has passed since) */
                        last_blk = blk;
                        if (tid < kSchedBlock) fill_sched((blk + 1) * kSchedBlock + 1, (blk + 1) & 1);
                    }
                    const uint32_t ra = rec_addr(d);
                    const uint4 r0 = lds_v4(ra), r1 = lds_v4(ra + 16u), r2 = lds_v4(ra + 32u);
                    if (r0.z & kRecStop) break;
                    const int lo = (int)r0.x, hi = (int)r0.y;
                    const int kind = (int)(r0.z & 3u);
                    const bool live = (r0.z & kRecLive) != 0;
                    const uint32_t aMc = r1.x, aMx = r1.y, aMo = r1.z, aIc = r1.w, aIe = r2.x, aDc = r2.y, aDe = r2.z;
                    if (COUNT && live && kind != WFAGPU_STEP_NULL) n_cells += (unsigned)(hi - lo + 1);

                    if (kind == WFAGPU_STEP_MDI && live) {
                        /* ---- can the next score ride along? ---- */
                        uint4 s0 = make_uint4(0, 0, 0, 0), s1 = s0, s2 = s0;
                        bool two = false;
                        if (pairable && d < Dmax) {
                            const uint32_t rb = rec_addr(d + 1);
                            s0 = lds_v4(rb);
                            two = (s0.z & (3u | kRecLive | kRecStop)) == (WFAGPU_STEP_MDI | kRecLive);
                            if (two) { s1 = lds_v4(rb + 16u); s2 = lds_v4(rb + 32u); }
                        }
                        if (!two) {
                            const int kq0 = lo & ~3, kend = hi | 3;
                            if (warp == last_warp) guards(aMc, aIc, aDc, kq0, kend);
                            for (int kq = kq0 + 4 * tid; kq <= hi; kq += 4 * gsz) {
                                const uint32_t o2 = (uint32_t)(2 * kq);
                                const uint2 mo = lds_v2(aMo + o2);
                                const uint32_t ml = lds_u16(aMo + o2 - 2u), mr = lds_u16(aMo + o2 + 8u);
                                const uint2 ie = lds_v2(aIe + o2);
                                const uint32_t il = lds_u16(aIe + o2 - 2u);
                                const uint2 de = lds_v2(aDe + o2);
                                const uint32_t dr = lds_u16(aDe + o2 + 8u);
                                const uint2 mx = lds_v2(aMx + o2);
                                /* (k-1 | k), (k+1 | k+2) and (k+3 | k+4) views of the open-gap source row */
                                const uint32_t moL01 = __byte_perm(ml, mo.x, 0x5410);
                                const uint32_t moMid = __byte_perm(mo.x, mo.y, 0x5432);
                                const uint32_t moR23 = __byte_perm(mo.y, mr, 0x5432);
                                uint32_t I01 = __vadd2(__vmaxs2(moL01, __byte_perm(il, ie.x, 0x5410)), kOnes2);
                                uint32_t I23 = __vadd2(__vmaxs2(moMid, __byte_perm(ie.x, ie.y, 0x5432)), kOnes2);
                                uint32_t D01 = __vmaxs2(moMid, __byte_perm(de.x, de.y, 0x5432));
                                uint32_t D23 = __vmaxs2(moR23, __byte_perm(de.y, dr, 0x5432));
                                uint32_t M01 = __vimax3_s16x2(__vadd2(mx.x, kOnes2), D01, I01);
                                uint32_t M23 = __vimax3_s16x2(__vadd2(mx.y, kOnes2), D23, I23);
                                if (kq < lo || kq + 3 > hi) {
                                    /* quad straddles the window: cells outside [lo, hi] read as NULL */
                                    const uint32_t k01 = in2(kq, lo, hi), k23 = in2(kq + 2, lo, hi);
                                    I01 = sel2(I01, k01); D01 = sel2(D01, k01); M01 = sel2(M01, k01);
                                    I23 = sel2(I23, k23); D23 = sel2(D23, k23); M23 = sel2(M23, k23);
                                }
                                sts_v2(aIc + o2, I01, I23);
                                sts_v2(aDc + o2, D01, D23);
                                extend_quad(Pa, Ta, plen, tlen, kq, tl8, M01, M23);
                                sts_v2(aMc + o2, M01, M23);
                            }
                            __syncthreads();
                            if ((r0.z & kRecTarget) != 0 && lds_s16(aMc + (uint32_t)(2 * kt)) == tlen) { finished = true; dist = d; break; }
                            if ((r0.z & kRecSnap) != 0) checkpoint(aMc, aIc, aDc, (int)r2.w, (int)r0.w, lo, hi);
                            d += 1;
                            continue;
                        }
                        /* ---- scores d and d + 1 in one barrier interval (e == 1: the extend sources of d + 1
                         *      are the I / D cells of d, kept in registers; its M sources are older rows) ---- */
                        const int lo2 = (int)s0.x, hi2 = (int)s0.y;
                        const uint32_t bMc = s1.x, bMx = s1.y, bMo = s1.z, bIc = s1.w, bDc = s2.y;
                        if (COUNT) n_cells += (unsigned)(hi2 - lo2 + 1);
                        const int kq0 = min(lo, lo2) & ~3, kend = max(hi, hi2) | 3;
                        if (warp == last_warp) { guards(aMc, aIc, aDc, kq0, kend); guards(bMc, bIc, bDc, kq0, kend); }
                        for (int kq = kq0 + 4 * tid; kq <= kend; kq += 4 * gsz) {
                            const uint32_t o2 = (uint32_t)(2 * kq);
                            /* score d: rows d-4 (open), d-1 (extend), d-2 (mismatch); the words at k-2 and k+4 carry
                             * the neighbours' cells and what their I / D cells of score d are made of */
                            const uint2 mo = lds_v2(aMo + o2);
                            const uint32_t mlw = lds_u32(aMo + o2 - 4u), mrw = lds_u32(aMo + o2 + 8u);   /* (k-2|k-1), (k+4|k+5) */
                            const uint2 ie = lds_v2(aIe + o2);
                            const uint32_t ilw = lds_u32(aIe + o2 - 4u);
                            const uint2 de = lds_v2(aDe + o2);
                            const uint32_t drw = lds_u32(aDe + o2 + 8u);
                            const uint2 mx = lds_v2(aMx + o2);
                            const uint32_t moL01 = __byte_perm(mlw, mo.x, 0x5432);                        /* (k-1 | k)   */
                            const uint32_t moMid = __byte_perm(mo.x, mo.y, 0x5432);                       /* (k+1 | k+2) */
                            const uint32_t moR23 = __byte_perm(mo.y, mrw, 0x5432);                        /* (k+3 | k+4) */
                            uint32_t I01 = __vadd2(__vmaxs2(moL01, __byte_perm(ilw, ie.x, 0x5432)), kOnes2);
                            uint32_t I23 = __vadd2(__vmaxs2(moMid, __byte_perm(ie.x, ie.y, 0x5432)), kOnes2);
                            uint32_t D01 = __vmaxs2(moMid, __byte_perm(de.x, de.y, 0x5432));
                            uint32_t D23 = __vmaxs2(moR23, __byte_perm(de.y, drw, 0x5432));
                            /* neighbours' cells of score d: I of (k-1 | k) and D of (k+3 | k+4) */
                            uint32_t IL = __vadd2(__vmaxs2(mlw, ilw), kOnes2);
                            uint32_t DR = __vmaxs2(mrw, drw);
                            uint32_t M01 = __vimax3_s16x2(__vadd2(mx.x, kOnes2), D01, I01);
                            uint32_t M23 = __vimax3_s16x2(__vadd2(mx.y, kOnes2), D23, I23);
                            if (kq - 1 < lo || kq + 4 > hi) {
                                const uint32_t k01 = in2(kq, lo, hi), k23 = in2(kq + 2, lo, hi);
                                I01 = sel2(I01, k01); D01 = sel2(D01, k01); M01 = sel2(M01, k01);
                                I23 = sel2(I23, k23); D23 = sel2(D23, k23); M23 = sel2(M23, k23);
                                IL = sel2(IL, in2(kq - 1, lo, hi));
                                DR = sel2(DR, in2(kq + 3, lo, hi));
                            }
                            sts_v2(aIc + o2, I01, I23);
                            sts_v2(aDc + o2, D01, D23);
                            extend_quad(Pa, Ta, plen, tlen, kq, tl8, M01, M23);
                            sts_v2(aMc + o2, M01, M23);
                            /* score d + 1: rows d-3 (open), d-1 (mismatch); extend sources from the registers */
                            const uint2 no = lds_v2(bMo + o2);
                            const uint32_t nl = lds_u16(bMo + o2 - 2u), nr = lds_u16(bMo + o2 + 8u);
                            const uint2 nx = lds_v2(bMx + o2);
                            const uint32_t noMid = __byte_perm(no.x, no.y, 0x5432);
                            uint32_t J01 = __vadd2(__vmaxs2(__byte_perm(nl, no.x, 0x5410), IL), kOnes2);
                            uint32_t J23 = __vadd2(__vmaxs2(noMid, __byte_perm(I01, I23, 0x5432)), kOnes2);
                            uint32_t E01 = __vmaxs2(noMid, __byte_perm(D01, D23, 0x5432));
                            uint32_t E23 = __vmaxs2(__byte_perm(no.y, nr, 0x5432), DR);
                            uint32_t N01 = __vimax3_s16x2(__vadd2(nx.x, kOnes2), E01, J01);
                            uint32_t N23 = __vimax3_s16x2(__vadd2(nx.y, kOnes2), E23, J23);
                            if (kq < lo2 || kq + 3 > hi2) {
                                const uint32_t k01 = in2(kq, lo2, hi2), k23 = in2(kq + 2, lo2, hi2);
                                J01 = sel2(J01, k01); E01 = sel2(E01, k01); N01 = sel2(N01, k01);
                                J23 = sel2(J23, k23); E23 = sel2(E23, k23); N23 = sel2(N23, k23);
                            }
                            sts_v2(bIc + o2, J01, J23);
                            sts_v2(bDc + o2, E01, E23);
                            extend_quad(Pa, Ta, plen, tlen, kq, tl8, N01, N23);
                            sts_v2(bMc + o2, N01, N23);
                        }
                        __syncthreads();
                        /* same order as score by score: an alignment that ends at d + 1 is traced back from the snapshot of d */
                        if ((r0.z & kRecTarget) != 0 && lds_s16(aMc + (uint32_t)(2 * kt)) == tlen) { finished = true; dist = d; break; }
                        if ((r0.z & kRecSnap) != 0) checkpoint(aMc, aIc, aDc, (int)r2.w, (int)r0.w, lo, hi);
                        if ((s0.z & kRecTarget) != 0 && lds_s16(bMc + (uint32_t)(2 * kt)) == tlen) { finished = true; dist = d + 1; break; }
                        if ((s0.z & kRecSnap) != 0) checkpoint(bMc, bIc, bDc, (int)s2.w, (int)s0.w, lo2, hi2);
                        /* the next interval recycles the rows of scores d - 3 (M) and d (I, D), which the snapshot of
                         * score d is still copying in slower warps */
                        if ((r0.z & kRecSnap) != 0) __syncthreads();
                        d += 2;
                        continue;
                    }
                    if (kind == WFAGPU_STEP_NULL || !live) {
                        for (int k = lo - GW - 4 + tid; k <= hi + GW + 4; k += gsz) {
                            sts_16(aMc + (uint32_t)(2 * k), NULLV);
                            sts_16(aIc + (uint32_t)(2 * k), NULLV);
                            sts_16(aDc + (uint32_t)(2 * k), NULLV);
                        }
                        __syncthreads();
                        if ((r0.z & kRecSnap) != 0) checkpoint(aMc, aIc, aDc, (int)r2.w, (int)r0.w, lo, hi);
                        d += 1;
                        continue;
                    }
                    /* mismatch-only step (the first scores, before any gap wavefront exists) */
                    for (int k = lo - GW - 4 + tid; k <= hi + GW + 4; k += gsz) {
                        sts_16(aIc + (uint32_t)(2 * k), NULLV);
                        sts_16(aDc + (uint32_t)(2 * k), NULLV);
                        int m = NULLV;
                        if (k >= lo && k <= hi) {
                            m = lds_s16(aMx + (uint32_t)(2 * k)) + 1;
                            if (m >= 0) m = extend_packed(Pa, Ta, plen, tlen, k, m, NULLV);
                        }
                        sts_16(aMc + (uint32_t)(2 * k), m);
                    }
                    __syncthreads();
                    if ((r0.z & kRecTarget) != 0 && lds_s16(aMc + (uint32_t)(2 * kt)) == tlen) { finished = true; dist = d; break; }
                    if ((r0.z & kRecSnap) != 0) checkpoint(aMc, aIc, aDc, (int)r2.w, (int)r0.w, lo, hi);
                    d += 1;
                }
                if (COUNT && tid == 0) atomicAdd(p.cells, n_cells);
            }
        }

        if (tid == 0) {
            wfagpu_pair_out_t r;
            r.distance = finished ? dist : 0;
            r.ops_off = 0;
            r.n_ops = 0;
            if (skip) {
                r.status = WFAGPU_ST_NEEDS_ASCII;
                p.ascii_list[atomicAdd(p.ascii_count, 1u)] = idx;
            } else if (finished) {
                r.status = WFAGPU_ST_FINISHED;
            } else {
                r.status = WFAGPU_ST_OVERBUDGET;
                p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
            }
            p.out[idx] = r;
        }
        __syncthreads();
        if (p.stages == 2) {
            stage ^= 1;
        } else {
            if (tid == 0) {
                const uint32_t nxt = pop(0);
                ctl->idx[0] = nxt;
                if (nxt != kInvalidIdx) issue_load(0, nxt);
            }
            __syncthreads();
        }
    }
}


/* ======================================================================== */
/*   large tier: rings in global memory (L2), int32, four diagonals/thread  */
/* ======================================================================== */
/*
 * For wavefronts wider than one CTA's shared memory and for sequences of 32768 bases and more (BASELINE
 * config 5: 50 kbp / 15 % has windows of ~20 000 diagonals, 720 KB of rings per pair).  Same recurrence,
 * pruning windows, schedule records and extend as wfa_quad_kernel; the rings are int32 rows in global memory that
 * stay resident in L2 (one CTA per SM: 148 x 0.7 MB), read with 128-bit loads (4 x LDG.128 + 4 x LDG.32 per four
 * cells instead of 20 scalar loads with 64-bit address arithmetic), written with 3 x STG.128; the backtrace is one
 * decision byte per cell (bit0 I extends, bit1 D extends, bits 3:2 the winner of M), walked by the CTA's leader.
 * Only the packed sequences and the schedule records live in shared memory.
 */
__device__ __forceinline__ int selnull(int v, bool in, int null_v) { return in ? v : null_v; }

template <bool BT, int MAXT>
__global__ void __launch_bounds__(MAXT, 1) wfa_quadg_kernel(const __grid_constant__ KernelParams p)
{
    constexpr int NULLV = RingG32::kNull;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, gsz = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, last_warp = (gsz >> 5) - 1;

    /* shared memory: [sequences, one stage][ctl][schedule records] */
    const uint32_t seq_bytes = (uint32_t)p.seq_words * 4u;
    const uint32_t seq_sa = smem_u32(smem_raw);
    GroupCtl *ctl = reinterpret_cast<GroupCtl *>(smem_raw + 2u * seq_bytes);
    const uint32_t sched_sa = seq_sa + 2u * seq_bytes + (uint32_t)sizeof(GroupCtl);

    const int x = p.x, e = p.e, A = p.A, E1 = p.E1, GW = p.G;
    const int oe = p.o + p.e;
    const uint32_t RS = (uint32_t)p.row_stride;                          /* int32 elements per row, multiple of 4 */
    int32_t *const ring = p.gring + (size_t)blockIdx.x * p.gring_elems;     /* 16-byte aligned */
    const uint32_t M0 = (uint32_t)p.center, I0 = M0 + (uint32_t)A * RS, D0 = I0 + (uint32_t)E1 * RS;   /* diagonal 0 of row 0 */
    const int rows = A + 2 * E1;
    uint4 *const arena = p.arena + (size_t)blockIdx.x * p.arena_units;
    uint32_t *const scratch = p.ops_scratch + (size_t)blockIdx.x * p.ops_scratch_words;

    auto issue_load = [&](uint32_t idx) {
        const wfagpu_pair_t pr = p.pairs[idx];
        const uint32_t pw = ((((pr.plen + 7u) >> 3) + 1u) + 3u) & ~3u;
        const uint32_t tw = ((((pr.tlen + 7u) >> 3) + 1u) + 3u) & ~3u;
        fence_proxy_async();
        mbar_expect_tx(&ctl->bar[0], (pw + tw) * 4u);
        tma_load_1d(smem_raw, p.packed + pr.p_word, pw * 4u, &ctl->bar[0]);
        tma_load_1d(smem_raw + seq_bytes, p.packed + pr.t_word, tw * 4u, &ctl->bar[0]);
    };
    auto pop = [&]() -> uint32_t {
        const uint32_t pos = atomicAdd(p.queue, 1u);
        return pos < p.n_items ? p.order[pos] : kInvalidIdx;
    };
    if (tid == 0) {
        mbar_init(&ctl->bar[0], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t first = pop();
        ctl->idx[0] = first;
        if (first != kInvalidIdx) issue_load(first);
    }
    __syncthreads();
    uint32_t phase = 0;

    while (true) {
        const uint32_t idx = ctl->idx[0];
        if (idx == kInvalidIdx) break;
        const wfagpu_pair_t pr = p.pairs[idx];
        const int plen = (int)pr.plen, tlen = (int)pr.tlen;
        const int kt = tlen - plen;
        const uint32_t Pa = seq_sa, Ta = seq_sa + seq_bytes;
        const bool skip = (pr.flags & WFAGPU_PAIR_HAS_N) != 0;

        /* ring prologue: NULL over [-2G - 4, 2G + 4] on every row */
        {
            const int span = 4 * GW + 9;
            const int total = rows * span;
            for (int i = tid; i < total; i += gsz) {
                const int r = i / span;
                ring[M0 + (uint32_t)r * RS + (uint32_t)(i - r * span - 2 * GW - 4)] = NULLV;
            }
        }
        mbar_wait(&ctl->bar[0], phase);
        phase ^= 1u;
        __syncthreads();

        int dist = 0;
        bool finished = false;
        if (!skip) {
            const int Dmax = p.bound ? min(p.d_end - 1, p.bound[idx]) : p.d_end - 1;
            auto fill_sched = [&](int dbase, int buf) {
                const int d = dbase + tid;
                StepRec r;
                r.lo = 0; r.hi = -1; r.flags = kRecStop; r.n = 0; r.ck_j = 0;
                r.aMc = r.aMx = r.aMo = r.aIc = r.aIe = r.aDc = r.aDe = 0;
                if (d <= Dmax) {
                    const wfagpu_step_t st = p.steps[d];
                    int lo, hi;
                    const bool live = prune_window((int)st.n, kt, (Dmax - d) / e, p.n_cap, lo, hi);
                    const bool stop = live && (lo < -p.n_cap || hi > p.n_cap);
                    const bool work = live && st.kind != WFAGPU_STEP_NULL;
                    r.lo = lo; r.hi = hi; r.n = (int)st.n;
                    r.flags = (uint32_t)st.kind | (live ? kRecLive : 0u) | (stop ? kRecStop : 0u) |
                              ((work && kt >= lo && kt <= hi) ? kRecTarget : 0u);
                    r.ck_j = st.row_off;                                   /* decision row of this score */
                    const int dm = d % A, de1 = d % E1;
                    int sx = dm - x % A; if (sx < 0) sx += A;
                    int so = dm - oe % A; if (so < 0) so += A;
                    int se = de1 - e % E1; if (se < 0) se += E1;
                    r.aMc = M0 + (uint32_t)dm * RS; r.aMx = M0 + (uint32_t)sx * RS; r.aMo = M0 + (uint32_t)so * RS;
                    r.aIc = I0 + (uint32_t)de1 * RS; r.aIe = I0 + (uint32_t)se * RS;
                    r.aDc = D0 + (uint32_t)de1 * RS; r.aDe = D0 + (uint32_t)se * RS;
                }
                const uint32_t a = sched_sa + (uint32_t)(buf * kSchedBlock + tid) * (uint32_t)sizeof(StepRec);
                sts_v4(a, make_uint4((uint32_t)r.lo, (uint32_t)r.hi, r.flags, (uint32_t)r.n));
                sts_v4(a + 16u, make_uint4(r.aMc, r.aMx, r.aMo, r.aIc));
                sts_v4(a + 32u, make_uint4(r.aIe, r.aDc, r.aDe, r.ck_j));
            };
            if (tid == 0) ring[M0] = extend_packed(Pa, Ta, plen, tlen, 0, 0, NULLV);
            if (tid < kSchedBlock) fill_sched(1, 0);
            __syncthreads();
            if (kt == 0 && ring[M0] == tlen) {
                finished = true;
            } else {
                const int tl8 = tlen - 8;
                unsigned long long n_cells = 0;
                int last_blk = -1;
                for (int d = 1; d <= Dmax; ++d) {
                    const int blk = (d - 1) / kSchedBlock;
                    if (blk != last_blk) {
                        last_blk = blk;
                        if (tid < kSchedBlock) fill_sched((blk + 1) * kSchedBlock + 1, (blk + 1) & 1);
                    }
                    const uint32_t ra = sched_sa + (uint32_t)((blk & 1) * kSchedBlock + ((d - 1) & (kSchedBlock - 1))) * (uint32_t)sizeof(StepRec);
                    const uint4 r0 = lds_v4(ra), r1 = lds_v4(ra + 16u), r2 = lds_v4(ra + 32u);
                    if (r0.z & kRecStop) break;
                    const int lo = (int)r0.x, hi = (int)r0.y, n = (int)r0.w;
                    const int kind = (int)(r0.z & 3u);
                    const bool live = (r0.z & kRecLive) != 0;
                    int32_t *const rMc = ring + r1.x, *const rIc = ring + r1.w, *const rDc = ring + r2.y;
                    const int32_t *const rMx = ring + r1.y, *const rMo = ring + r1.z, *const rIe = ring + r2.x, *const rDe = ring + r2.z;
                    if (p.cells && live && kind != WFAGPU_STEP_NULL) n_cells += (unsigned)(hi - lo + 1);

                    if (kind == WFAGPU_STEP_MDI && live) {
                        const int kq0 = lo & ~3, kend = hi | 3;
                        if (warp == last_warp) {
                            for (int g = lane; g < 2 * GW; g += 32) {
                                const int k = (g < GW) ? (kq0 - 1 - g) : (kend + 1 + (g - GW));
                                rMc[k] = NULLV; rIc[k] = NULLV; rDc[k] = NULLV;
                            }
                        }
                        uint8_t *const rowb = reinterpret_cast<uint8_t *>(arena + r2.w) + n;      /* decision row, indexed by k */
                        for (int kq = kq0 + 4 * tid; kq <= hi; kq += 4 * gsz) {
                            const int4 mo = *reinterpret_cast<const int4 *>(rMo + kq);
                            const int ml = rMo[kq - 1], mr = rMo[kq + 4];
                            const int4 ie = *reinterpret_cast<const int4 *>(rIe + kq);
                            const int il = rIe[kq - 1];
                            const int4 de = *reinterpret_cast<const int4 *>(rDe + kq);
                            const int dr = rDe[kq + 4];
                            const int4 mx = *reinterpret_cast<const int4 *>(rMx + kq);
                            /* offsets by plain max; the tie-breaks only decide the backtrace bits: I / D: extend beats open
                             * on equal offsets; M: D beats X beats I */
                            int i0 = max(ml, il) + 1, i1 = max(mo.x, ie.x) + 1, i2 = max(mo.y, ie.y) + 1, i3 = max(mo.z, ie.z) + 1;
                            int d0 = max(mo.y, de.y), d1 = max(mo.z, de.z), d2 = max(mo.w, de.w), d3 = max(mr, dr);
                            const int x0 = mx.x + 1, x1 = mx.y + 1, x2 = mx.z + 1, x3 = mx.w + 1;
                            int m0 = max(max(x0, d0), i0), m1 = max(max(x1, d1), i1), m2 = max(max(x2, d2), i2), m3 = max(max(x3, d3), i3);
                            if (BT) {
                                const uint32_t c0 = (il >= ml ? 1u : 0u) | (de.y >= mo.y ? 2u : 0u) | ((d0 >= x0 || i0 > x0) ? 4u : 0u) | ((d0 >= i0 || x0 >= i0) ? 8u : 0u);
                                const uint32_t c1 = (ie.x >= mo.x ? 1u : 0u) | (de.z >= mo.z ? 2u : 0u) | ((d1 >= x1 || i1 > x1) ? 4u : 0u) | ((d1 >= i1 || x1 >= i1) ? 8u : 0u);
                                const uint32_t c2 = (ie.y >= mo.y ? 1u : 0u) | (de.w >= mo.w ? 2u : 0u) | ((d2 >= x2 || i2 > x2) ? 4u : 0u) | ((d2 >= i2 || x2 >= i2) ? 8u : 0u);
                                const uint32_t c3 = (ie.z >= mo.z ? 1u : 0u) | (dr >= mr ? 2u : 0u) | ((d3 >= x3 || i3 > x3) ? 4u : 0u) | ((d3 >= i3 || x3 >= i3) ? 8u : 0u);
                                /* cells outside the window keep their byte unwritten: the traceback never visits them */
                                if (kq >= lo) rowb[kq] = (uint8_t)c0;
                                if (kq + 1 >= lo && kq + 1 <= hi) rowb[kq + 1] = (uint8_t)c1;
                                if (kq + 2 >= lo && kq + 2 <= hi) rowb[kq + 2] = (uint8_t)c2;
                                if (kq + 3 <= hi) rowb[kq + 3] = (uint8_t)c3;
                            }
                            if (kq < lo || kq + 3 > hi) {
                                const bool in0 = kq >= lo, in1 = kq + 1 >= lo && kq + 1 <= hi, in2 = kq + 2 >= lo && kq + 2 <= hi, in3 = kq + 3 <= hi;
                                i0 = selnull(i0, in0, NULLV); d0 = selnull(d0, in0, NULLV); m0 = selnull(m0, in0, NULLV);
                                i1 = selnull(i1, in1, NULLV); d1 = selnull(d1, in1, NULLV); m1 = selnull(m1, in1, NULLV);
                                i2 = selnull(i2, in2, NULLV); d2 = selnull(d2, in2, NULLV); m2 = selnull(m2, in2, NULLV);
                                i3 = selnull(i3, in3, NULLV); d3 = selnull(d3, in3, NULLV); m3 = selnull(m3, in3, NULLV);
                            }
                            *reinterpret_cast<int4 *>(rIc + kq) = make_int4(i0, i1, i2, i3);
                            *reinterpret_cast<int4 *>(rDc + kq) = make_int4(d0, d1, d2, d3);
                            extend_cells(Pa, Ta, plen, tlen, kq, tl8, m0, m1, m2, m3, NULLV);
                            *reinterpret_cast<int4 *>(rMc + kq) = make_int4(m0, m1, m2, m3);
                        }
                    } else if (kind == WFAGPU_STEP_NULL || !live) {
                        for (int k = lo - GW - 4 + tid; k <= hi + GW + 4; k += gsz) { rMc[k] = NULLV; rIc[k] = NULLV; rDc[k] = NULLV; }
                        __syncthreads();
                        continue;
                    } else {
                        for (int k = lo - GW - 4 + tid; k <= hi + GW + 4; k += gsz) {
                            rIc[k] = NULLV; rDc[k] = NULLV;
                            int m = NULLV;
                            if (k >= lo && k <= hi) {
                                m = rMx[k] + 1;
                                if (m >= 0) m = extend_packed(Pa, Ta, plen, tlen, k, m, NULLV);
                            }
                            rMc[k] = m;
                        }
                    }
                    __syncthreads();
                    if ((r0.z & kRecTarget) != 0 && rMc[kt] == tlen) { finished = true; dist = d; break; }
                }
                if (p.cells && tid == 0) atomicAdd(p.cells, n_cells);
            }
        }

        /* ---- traceback over the decision bytes -> 2-bit ops, newest first (leader) ---- */
        uint32_t n_ops = 0;
        if (tid == 0) {
            uint32_t ops_off = 0;
            if (BT && finished && dist > 0) {
                int cd = dist, ck = kt, comp = 0;
                uint32_t word = 0;
                while (!(comp == 0 && cd == 0)) {
                    const wfagpu_step_t st = p.steps[cd];
                    uint32_t op;
                    if (comp == 0) {
                        op = OP_SUB;
                        if (st.kind == WFAGPU_STEP_M) {
                            cd -= x;
                        } else {
                            const int ii = ck + (int)st.n;
                            if (ii < 0 || ii > 2 * (int)st.n) { n_ops = 0; finished = false; break; }
                            const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                            const int mop = (int)(dec >> 2) & 3;
                            if (mop == OP_SUB) cd -= x;
                            else if (mop == OP_INS) comp = 1;
                            else comp = 2;
                        }
                    } else {
                        const int ii = ck + (int)st.n;
                        if (ii < 0 || ii > 2 * (int)st.n || st.kind != WFAGPU_STEP_MDI) { n_ops = 0; finished = false; break; }
                        const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                        if (comp == 1) {
                            op = OP_INS;
                            ck -= 1;
                            if (dec & 1u) cd -= e; else { cd -= oe; comp = 0; }
                        } else {
                            op = OP_DEL;
                            ck += 1;
                            if (dec & 2u) cd -= e; else { cd -= oe; comp = 0; }
                        }
                    }
                    word |= op << (2 * (n_ops & 15u));
                    ++n_ops;
                    if ((n_ops & 15u) == 0) { scratch[(n_ops >> 4) - 1] = word; word = 0; }
                    if (cd < 0 || (n_ops >> 4) >= p.ops_scratch_words) { n_ops = 0; finished = false; break; }
                }
                if (n_ops & 15u) scratch[n_ops >> 4] = word;
                const uint32_t nw = (n_ops + 15u) >> 4;
                ops_off = atomicAdd(p.ops_pool_head, nw);
                if (ops_off + nw > p.ops_pool_words) { n_ops = 0; finished = false; }
            }
            ctl->n_ops = n_ops;
            ctl->ops_off = ops_off;
            wfagpu_pair_out_t r;
            r.distance = finished ? dist : 0;
            r.ops_off = ops_off;
            r.n_ops = n_ops;
            if (skip) {
                r.status = WFAGPU_ST_NEEDS_ASCII;
                p.ascii_list[atomicAdd(p.ascii_count, 1u)] = idx;
            } else if (finished) {
                r.status = WFAGPU_ST_FINISHED;
            } else {
                r.status = WFAGPU_ST_OVERBUDGET;
                p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
            }
            p.out[idx] = r;
        }
        __syncthreads();
        if (BT) {
            const uint32_t nw = (ctl->n_ops + 15u) >> 4;
            const uint32_t off = ctl->ops_off;
            for (uint32_t i = tid; i < nw; i += gsz) p.ops_pool[off + i] = scratch[i];
        }
        __syncthreads();
        if (tid == 0) {
            const uint32_t nxt = pop();
            ctl->idx[0] = nxt;
            if (nxt != kInvalidIdx) issue_load(nxt);
        }
        __syncthreads();
    }
}

/* ======================================================================== */
/*              score upper bound (warp per pair, 32 diagonals)             */
/* ======================================================================== */
/*
 * Feeds the score-bound pruning of wfa_exact_kernel with a per-pair bound.  A warp runs the
 * same M/I/D recurrence on a window of 32 diagonals (one per lane) that is re-centred every
 * few scores on the diagonal closest to the end of both sequences -- the idea of the
 * reference's adaptive band (sequence_distance_kernel_aband.cu:99-147) at the width of a warp.
 * Every offset it holds is the end of a real partial alignment, so the score at which it
 * reaches (plen, tlen) is the score of a real alignment: an upper bound of the optimum, and
 * in practice the optimum itself (16 diagonals already find it on 10 kbp / 5 % reads).
 * Its result only narrows the exact kernel's work, never its result: any bound >= the optimum
 * gives identical scores and CIGARs, and a pair that misses here just keeps the launch bound.
 * Cost: 32 cells per score against ~score/2 in the exact kernel.
 */
constexpr int kBoundNull = -(1 << 28);

__device__ __forceinline__ int lds_s32(uint32_t a)
{
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_32(uint32_t a, int v)
{
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

__global__ void __launch_bounds__(256) wfa_bound_kernel(const __grid_constant__ KernelParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = p.x, e = p.e, A = p.A, E1 = p.E1, oe = p.o + p.e;
    const int rows = A + 2 * E1;
    /* per warp: rows x 32 int32 offsets (128 bytes per row), explicit shared addresses.  Every row
     * shares one window [wlo, wlo + 31]; diagonal k lives in slot k & 31, so moving the window only
     * has to clear the slots that change owner. */
    const uint32_t ring_sa = smem_u32(smem_raw) + (uint32_t)(warp * rows) * 128u;
    const uint32_t Mr = ring_sa, Ir = ring_sa + (uint32_t)A * 128u, Dr = Ir + (uint32_t)E1 * 128u;
    const uint32_t Mend = (uint32_t)A * 128u, Gend = (uint32_t)E1 * 128u;      /* ring sizes in bytes */
    const int Dlaunch = p.d_end - 1;
    const uint32_t me = (uint32_t)lane * 4u, left = (uint32_t)((lane + 31) & 31) * 4u, right = (uint32_t)((lane + 1) & 31) * 4u;

    while (true) {
        uint32_t pos = 0;
        if (lane == 0) pos = atomicAdd(p.bound_queue, 1u);
        pos = __shfl_sync(FULL, pos, 0);
        if (pos >= p.n_items) break;
        const uint32_t idx = p.order[pos];
        const wfagpu_pair_t pr = p.pairs[idx];
        if (pr.flags & WFAGPU_PAIR_HAS_N) { if (lane == 0) p.bound[idx] = 0x7fffffff; continue; }    /* byte-compare pair: no bound, and the host can tell */
        const int plen = (int)pr.plen, tlen = (int)pr.tlen, kt = tlen - plen;
        const uint32_t *const Pw = p.packed + pr.p_word;
        const uint32_t *const Tw = p.packed + pr.t_word;
        for (int r = 0; r < rows; ++r) sts_32(ring_sa + (uint32_t)r * 128u + me, kBoundNull);
        int wlo = -16;
        int result = Dlaunch;
        {
            const int m = extend_packed_g(Pw, Tw, plen, tlen, 0, 0);
            __syncwarp();
            if (lane == 0) sts_32(Mr, m);                    /* score 0: k = 0 sits in slot 0 */
            if (kt == 0 && m == tlen) result = 0;
        }
        __syncwarp();
        if (result != 0) {
            /* byte offsets of the ring rows of the current score and of its sources, stepped with the score */
            uint32_t mc = 0, mx = (uint32_t)((A - x) % A) * 128u, mo = (uint32_t)((A - oe) % A) * 128u;
            uint32_t ic = 0, ie = (uint32_t)((E1 - e) % E1) * 128u;
            int my_m = kBoundNull, my_k = 0;
            wfagpu_step_t st_next = p.steps[1 < p.d_end ? 1 : 0];
            for (int d = 1; d <= Dlaunch; ++d) {
                const wfagpu_step_t st = st_next;
                if (d + 1 < p.d_end) st_next = p.steps[d + 1];
                mc += 128u; if (mc == Mend) mc = 0;
                mx += 128u; if (mx == Mend) mx = 0;
                mo += 128u; if (mo == Mend) mo = 0;
                ic += 128u; if (ic == Gend) ic = 0;
                ie += 128u; if (ie == Gend) ie = 0;
                if ((d & 7) == 0) {
                    /* re-centre on the diagonal with the least sequence left */
                    unsigned key = 0xffffffffu;
                    if (my_m >= 0) key = ((unsigned)max((plen - (my_m - my_k)) + (tlen - my_m), 0) << 5) | (unsigned)lane;
                    const unsigned best = __reduce_min_sync(FULL, key);
                    if (best != 0xffffffffu) {
                        const int nlo = __shfl_sync(FULL, my_k, (int)(best & 31u)) - 16;
                        if (nlo != wlo) {
                            const int k_old = wlo + ((lane - wlo) & 31), k_new = nlo + ((lane - nlo) & 31);
                            if (k_old != k_new)
                                for (int r = 0; r < rows; ++r) sts_32(ring_sa + (uint32_t)r * 128u + me, kBoundNull);
                            wlo = nlo;
                            __syncwarp();
                        }
                    }
                }
                const int k = wlo + ((lane - wlo) & 31);
                int vM = kBoundNull, vI = kBoundNull, vD = kBoundNull;
                if (st.kind != WFAGPU_STEP_NULL) {                 /* uniform */
                    const int n = st.n;
                    const bool in = (k >= -n && k <= n);
                    if (in) {
                        vM = lds_s32(Mr + mx + me) + 1;
                        if (st.kind == WFAGPU_STEP_MDI) {
                            /* neighbours outside the window read as NULL (selects, no branches) */
                            const int moL = lds_s32(Mr + mo + left), ieL = lds_s32(Ir + ie + left);
                            const int moR = lds_s32(Mr + mo + right), deR = lds_s32(Dr + ie + right);
                            vI = (k != wlo) ? max(moL, ieL) + 1 : kBoundNull;
                            vD = (k != wlo + 31) ? max(moR, deR) : kBoundNull;
                            vM = max(max(vM, vD), vI);
                        }
                    }
                    vM = warp_extend_packed(Pw, Tw, plen, tlen, in && vM >= 0, k, vM, kBoundNull, lane);
                    if (vM < 0) vM = kBoundNull;
                    if (vI < 0) vI = kBoundNull;
                    if (vD < 0) vD = kBoundNull;
                    my_m = vM; my_k = k;
                }
                /* the rows being replaced (scores d - A, d - e - 1) are no source of this score */
                sts_32(Mr + mc + me, vM);
                sts_32(Ir + ic + me, vI);
                sts_32(Dr + ic + me, vD);
                __syncwarp();
                if (__any_sync(FULL, k == kt && vM == tlen)) { result = d; break; }
            }
        }
        if (lane == 0) p.bound[idx] = result;
        __syncwarp();
    }
}

/* ======================================================================== */
/*                 checkpointed traceback (warp per pair)                   */
/* ======================================================================== */
/*
 * Second half of the CKPT path.  The forward kernel left, for every pair, a snapshot of
 * the ring rows every P = p.ck_period scores (one arena per pair, indexed by queue position).
 * A warp walks its pair from (distance, k_target) down to (0, 0), segment by segment:
 * stage the window of snapshot c = P * floor((d-1)/P) under the cell, recompute scores
 * c+1 .. d on the dependency cone |k - k_apex| <= d_apex - d level by level (same
 * recurrence, same extend), then follow the path while it stays above c using the
 * forward tie-breaks on the recomputed offsets (I/D: extend beats open; M: D beats X
 * beats I).  Emits the same newest-first 2-bit op stream as the decision-byte walk.
 * Running it as its own kernel puts thousands of these latency-bound walks in flight
 * instead of one per resident CTA (model: oracle/kernel_model.c, km_align_pair_ckpt).
 */
template <bool ASCII, int P>
__global__ void __launch_bounds__(256) wfa_traceback_kernel(const __grid_constant__ KernelParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    /* Per warp and component: a rectangle of levels -(A-2) .. P (score c + level) by 2P+1
     * diagonals around the apex; levels <= 0 hold the staged snapshot window. */
    constexpr int WP = 2 * P + 1;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int NULLV = kOffNull;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = p.x, e = p.e, A = p.A, oe = p.o + p.e;
    const int L0 = A - 2;                                      /* row of level 0 */
    const uint32_t comp_bytes = (uint32_t)((P + A - 1) * WP * 2);
    const uint32_t warp_bytes = (3u * comp_bytes + 15u) & ~15u;
    const uint32_t sM = smem_u32(smem_raw) + (uint32_t)warp * warp_bytes;
    const uint32_t sI = sM + comp_bytes, sD = sI + comp_bytes;
    /* address of (level, k): base + 2 * ((level + L0) * WP + (k - kc + P)) */

    while (true) {
        uint32_t pos = 0;
        if (lane == 0) pos = atomicAdd(p.tb_queue, 1u);
        pos = __shfl_sync(FULL, pos, 0);
        if (pos >= p.n_items) break;
        const uint32_t idx = p.order[pos];
        const wfagpu_pair_out_t res = p.out[idx];
        if (!(res.status & WFAGPU_ST_FINISHED) || res.distance <= 0) continue;
        const wfagpu_pair_t pr = p.pairs[idx];
        const int plen = (int)pr.plen, tlen = (int)pr.tlen, dist = res.distance;
        const uint32_t *const Pw = p.packed + pr.p_word;
        const uint32_t *const Tw = p.packed + pr.t_word;
        const char *const Pg = p.ascii + pr.p_ascii;
        const char *const Tg = p.ascii + pr.t_ascii;
        auto extend = [&](int k, int off) -> int {
            if (ASCII) return extend_ascii(Pg, Tg, plen, tlen, k, off, NULLV);
            return extend_packed_g(Pw, Tw, plen, tlen, k, off);
        };
        const uint4 *const arena = p.arena + (size_t)pos * p.arena_units;
        /* op words go straight to the pool: at most 2 ops per score */
        const uint32_t nw_max = ((2u * (uint32_t)dist + 15u) >> 4) + 1u;
        uint32_t ops_off = 0;
        if (lane == 0) ops_off = atomicAdd(p.ops_pool_head, nw_max);
        ops_off = __shfl_sync(FULL, ops_off, 0);
        bool tb_ok = (ops_off + nw_max <= p.ops_pool_words);
        uint32_t *const ops = p.ops_pool + ops_off;

        const int m00 = extend(0, 0);
        const int kt = tlen - plen;                              /* same pruning window as the forward pass */
        const int Dmax = p.bound ? min(p.d_end - 1, p.bound[idx]) : p.d_end - 1;
        int cd = dist, ck = kt, comp = 0;
        uint32_t word = 0, n_ops = 0;
        while (!(comp == 0 && cd == 0) && tb_ok) {
            if (cd <= 0) { tb_ok = false; break; }
            const int c = ((cd - 1) / P) * P, Rr = cd - c, kc = ck;
            const int jlo = P - Rr, jhi = P + Rr;                  /* columns of the cone's base */
            /* ---- stage snapshot c as levels 0, -1, ...: M ages 0..A-2, I/D ages 0..e-1 ---- */
            if (c == 0) {
                for (int a = 0; a < A - 1; ++a)
                    for (int j = jlo + lane; j <= jhi; j += 32) {
                        sts_16(sM + 2u * (uint32_t)((L0 - a) * WP + j), (a == 0 && j == P - kc) ? m00 : NULLV);
                        if (a < e) {
                            sts_16(sI + 2u * (uint32_t)((L0 - a) * WP + j), NULLV);
                            sts_16(sD + 2u * (uint32_t)((L0 - a) * WP + j), NULLV);
                        }
                    }
            } else {
                const int nc = p.steps[c].n;
                int wlo, whi;
                prune_window(nc, kt, (Dmax - c) / e, p.n_cap, wlo, whi);
                wlo = max(-nc, wlo - 1);
                whi = min(nc, whi + 1);
                const int k0 = -((nc + 7) & ~7);
                const int units = (((nc + 7) & ~7) + ((nc + 8) & ~7)) >> 3;
                const int16_t *snap = reinterpret_cast<const int16_t *>(arena + p.ck_off[c / P]) - k0;
                const size_t pitch = (size_t)units * 8;
                for (int j = jlo + lane; j <= jhi; j += 32) {
                    const int k = kc - P + j;
                    const bool in = (k >= wlo && k <= whi);
                    for (int a = 0; a < A - 1; ++a)
                        sts_16(sM + 2u * (uint32_t)((L0 - a) * WP + j), in ? (int)__ldcs(snap + (size_t)a * pitch + k) : NULLV);
                    for (int a = 0; a < e; ++a) {
                        sts_16(sI + 2u * (uint32_t)((L0 - a) * WP + j), in ? (int)__ldcs(snap + (size_t)(A - 1 + a) * pitch + k) : NULLV);
                        sts_16(sD + 2u * (uint32_t)((L0 - a) * WP + j), in ? (int)__ldcs(snap + (size_t)(A - 1 + e + a) * pitch + k) : NULLV);
                    }
                }
            }
            uint32_t my_nk = 0;          /* lane l: half width | kind << 16 of score c + 1 + l */
            if (lane < Rr) { const wfagpu_step_t t = p.steps[c + 1 + lane]; my_nk = (uint32_t)t.n | ((uint32_t)t.kind << 16); }
            __syncwarp();
            /* ---- recompute levels 1 .. Rr on the cone ---- */
            /* (Dmax - (c + i)) = q * e + r and the row offsets are stepped with the level */
            int pq = (Dmax - c) / e, prr = (Dmax - c) % e;
            uint32_t rowC = 2u * (uint32_t)(L0 * WP);
            for (int i = 1; i <= Rr; ++i) {
                const uint32_t nk = __shfl_sync(FULL, my_nk, i - 1);
                const int n_i = (int)(nk & 0xffffu), kind_i = (int)(nk >> 16);
                const int half = Rr - i;
                if (prr == 0) { prr = e - 1; --pq; } else --prr;
                int lo_i, hi_i;
                if (!prune_window(n_i, kt, pq, p.n_cap, lo_i, hi_i)) { lo_i = 1; hi_i = 0; }
                rowC += 2u * (uint32_t)WP;
                const uint32_t rowX = rowC - 2u * (uint32_t)(x * WP);
                const uint32_t rowO = rowC - 2u * (uint32_t)(oe * WP);
                const uint32_t rowE = rowC - 2u * (uint32_t)(e * WP);
                for (int j0 = P - half; j0 <= P + half; j0 += 32) {          /* uniform trip count */
                    const int j = j0 + lane;
                    const bool act = j <= P + half;
                    const int k = kc - P + j;
                    const uint32_t cj = 2u * (uint32_t)j;
                    int vM = NULLV, vI = NULLV, vD = NULLV;
                    const bool live = act && kind_i != WFAGPU_STEP_NULL && k >= lo_i && k <= hi_i;
                    if (live) {
                        if (kind_i == WFAGPU_STEP_M) {
                            vM = lds_s16(sM + rowX + cj) + 1;
                        } else {
                            vI = max(lds_s16(sM + rowO + cj - 2u), lds_s16(sI + rowE + cj - 2u)) + 1;
                            vD = max(lds_s16(sM + rowO + cj + 2u), lds_s16(sD + rowE + cj + 2u));
                            vM = max(max(lds_s16(sM + rowX + cj) + 1, vD), vI);
                        }
                    }
                    if constexpr (ASCII) {
                        if (live && vM >= 0) vM = extend(k, vM);
                    } else {
                        vM = warp_extend_packed(Pw, Tw, plen, tlen, live && vM >= 0, k, vM, NULLV, lane);
                    }
                    if (act) {
                        sts_16(sM + rowC + cj, vM);
                        sts_16(sI + rowC + cj, vI);
                        sts_16(sD + rowC + cj, vD);
                    }
                }
                __syncwarp();
            }
            /* ---- walk while the path stays above c (uniform across the warp; lane 0 stores) ---- */
            auto at = [&](uint32_t base, int d2, int k) -> int {
                return lds_s16(base + 2u * (uint32_t)((d2 - c + L0) * WP + (k - kc + P)));
            };
            while (cd > c && !(comp == 0 && cd == 0)) {
                const uint32_t nk = __shfl_sync(FULL, my_nk, cd - c - 1);
                const int kind_c = (int)(nk >> 16);
                uint32_t op;
                if (comp == 0) {
                    op = OP_SUB;
                    if (kind_c == WFAGPU_STEP_M) {
                        cd -= x;
                    } else {
                        const int X = at(sM, cd - x, ck) + 1;
                        const int I = at(sI, cd, ck), D = at(sD, cd, ck);
                        if (D >= X && D >= I) comp = 2;          /* D beats X beats I */
                        else if (X >= I) cd -= x;
                        else comp = 1;
                    }
                } else if (comp == 1) {
                    op = OP_INS;
                    const int opn = at(sM, cd - oe, ck - 1), ext = at(sI, cd - e, ck - 1);
                    ck -= 1;
                    if (ext >= opn) cd -= e; else { cd -= oe; comp = 0; }   /* extend beats open */
                } else {
                    op = OP_DEL;
                    const int opn = at(sM, cd - oe, ck + 1), ext = at(sD, cd - e, ck + 1);
                    ck += 1;
                    if (ext >= opn) cd -= e; else { cd -= oe; comp = 0; }
                }
                word |= op << (2 * (n_ops & 15u));
                ++n_ops;
                if ((n_ops & 15u) == 0) {
                    if (lane == 0) ops[(n_ops >> 4) - 1] = word;
                    word = 0;
                }
                if (cd < 0 || (n_ops >> 4) >= nw_max) { tb_ok = false; break; }
            }
            __syncwarp();
        }
        if (lane == 0) {
            wfagpu_pair_out_t r = res;
            if (tb_ok) {
                if (n_ops & 15u) ops[n_ops >> 4] = word;
                r.ops_off = ops_off;
                r.n_ops = n_ops;
            } else {
                /* cannot happen with a consistent snapshot arena; leave the pair to the re-dispatch loop */
                r.distance = 0; r.ops_off = 0; r.n_ops = 0;
                r.status = WFAGPU_ST_OVERBUDGET;
                p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
            }
            p.out[idx] = r;
        }
        __syncwarp();
    }
}

/* ======================================================================== */
/*                         banded (adaptive band) kernel                    */
/* ======================================================================== */
/*
 * Replaces alignment_kernel_aband / distance_kernel_aband
 * (lib/kernels/sequence_alignment_kernel_aband.cu:145-391, 596-725;
 *  lib/kernels/sequence_distance_kernel_aband.cu:99-147).
 *
 * The heuristic is not exact, so the reference's memory semantics are kept
 * as they are: rings of depth A for M, I and D, every slot with its own [lo, hi]
 * window (offsets stored at k - lo), slots are not cleared on null steps and
 * reads outside a slot's window return NULL.  Window rule (aband.cu:167-205):
 * grow by one on both sides, clip alternately hi--, lo++ to the band width,
 * and every `band` scores -- once the mismatch source is full width --
 * re-centre on the first diagonal with the smallest distance to the target.
 * The serial O(W) scan every thread runs in the reference ("TODO: make
 * cooperative") is a lexicographic (distance, diagonal) block reduction here.
 */
struct BandCtl {
    uint64_t bar[2];
    uint32_t idx[2];
    uint32_t n_ops;
    uint32_t ops_off;
    int new_center;
    int pad;
    unsigned long long red[32];
};

__device__ __forceinline__ int band_get(uint32_t row, int lo, int hi, int k)
{
    return (k >= lo && k <= hi) ? lds_s16(row + (uint32_t)(2 * (k - lo))) : kOffNull;
}

template <bool ASCII, bool BT>
__global__ void __launch_bounds__(1024, 1) wfa_banded_kernel(const __grid_constant__ KernelParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, gsz = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = gsz >> 5;
    const int x = p.x, e = p.e, A = p.A, W = p.win;
    const int oe = p.o + p.e;
    const uint32_t row_bytes = (uint32_t)((W + 7) & ~7) * 2u;
    const uint32_t comp_bytes = (uint32_t)A * row_bytes;
    const uint32_t ring_bytes = (3u * comp_bytes + 15u) & ~15u;
    const uint32_t lohi_bytes = (uint32_t)(((3 * A * 2 * (int)sizeof(int)) + 15) & ~15);
    const uint32_t seq_bytes = (uint32_t)p.seq_words * 4u;
    const uint32_t seq_total = ASCII ? 0u : 2u * (uint32_t)p.stages * seq_bytes;
    const uint32_t M0 = smem_u32(smem_raw);
    const uint32_t I0 = M0 + comp_bytes, D0 = I0 + comp_bytes;
    int *const LO = reinterpret_cast<int *>(smem_raw + ring_bytes);   /* [comp][slot] */
    int *const HI = LO + 3 * A;
    const uint32_t seq_sa = M0 + ring_bytes + lohi_bytes;
    BandCtl *ctl = reinterpret_cast<BandCtl *>(smem_raw + ring_bytes + lohi_bytes + seq_total);

    const uint32_t group = blockIdx.x;
    uint4 *const arena = p.arena + (size_t)group * p.arena_units;
    int32_t *const lo_tab = p.band_lo + (size_t)group * p.band_lo_words;
    uint32_t *const scratch = p.ops_scratch + (size_t)group * p.ops_scratch_words;

    auto issue_load = [&](int stage, uint32_t idx) {
        if (ASCII) return;
        const wfagpu_pair_t pr = p.pairs[idx];
        const uint32_t pw = ((((pr.plen + 7u) >> 3) + 1u) + 3u) & ~3u;
        const uint32_t tw = ((((pr.tlen + 7u) >> 3) + 1u) + 3u) & ~3u;
        unsigned char *dp = smem_raw + ring_bytes + lohi_bytes + (size_t)(2 * stage) * seq_bytes;
        unsigned char *dt = dp + seq_bytes;
        fence_proxy_async();
        mbar_expect_tx(&ctl->bar[stage], (pw + tw) * 4u);
        tma_load_1d(dp, p.packed + pr.p_word, pw * 4u, &ctl->bar[stage]);
        tma_load_1d(dt, p.packed + pr.t_word, tw * 4u, &ctl->bar[stage]);
    };
    auto pop = [&](int slot) -> uint32_t {
        const uint32_t pos = atomicAdd(p.queue, 1u);
        return pos < p.n_items ? p.order[pos] : kInvalidIdx;
    };
    if (tid == 0) {
        if (!ASCII) {
            mbar_init(&ctl->bar[0], 1);
            mbar_init(&ctl->bar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        const uint32_t first = pop(0);
        ctl->idx[0] = first;
        if (first != kInvalidIdx) issue_load(0, first);
    }
    __syncthreads();

    int stage = 0;
    uint32_t phase_bits = 0;
    while (true) {
        const uint32_t idx = ctl->idx[stage];
        if (idx == kInvalidIdx) break;
        if (tid == 0 && p.stages == 2) {
            const uint32_t nxt = pop(stage ^ 1);
            ctl->idx[stage ^ 1] = nxt;
            if (nxt != kInvalidIdx) issue_load(stage ^ 1, nxt);
        }
        const wfagpu_pair_t pr = p.pairs[idx];
        const int plen = (int)pr.plen, tlen = (int)pr.tlen;
        const int kt = tlen - plen;
        const int kt_abs = kt < 0 ? -kt : kt;
        const uint32_t Pa = seq_sa + (uint32_t)(2 * stage) * seq_bytes;
        const uint32_t Ta = Pa + seq_bytes;
        const char *const Pg = p.ascii + pr.p_ascii;
        const char *const Tg = p.ascii + pr.t_ascii;
        auto extend = [&](int k, int off) -> int {
            if (ASCII) return extend_ascii(Pg, Tg, plen, tlen, k, off);
            return extend_packed(Pa, Ta, plen, tlen, k, off);
        };
        const bool skip = !ASCII && (pr.flags & WFAGPU_PAIR_HAS_N);

        /* every slot starts as the one-diagonal window [0, 0] holding NULL (aband.cu:543-578) */
        for (int i = tid; i < 3 * A; i += gsz) {
            LO[i] = 0;
            HI[i] = 0;
            sts_16(M0 + (uint32_t)i * row_bytes, kOffNull);
        }
        if (!ASCII) mbar_wait(&ctl->bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        __syncthreads();

        int dist = 0;
        bool finished = false;
        if (!skip) {
            if (tid == 0) sts_16(M0, extend(0, 0));
            __syncthreads();
            if (kt == 0 && lds_s16(M0) == tlen) {
                finished = true;
            } else {
                int sM = 0;                                  /* ring slot of the current score: d mod A */
                for (int d = 1; d < p.d_end; ++d) {
                    const wfagpu_step_t st = p.steps[d];
                    sM = (sM + 1 == A) ? 0 : sM + 1;
                    if (st.kind == WFAGPU_STEP_NULL) continue;
                    int sx = sM - x;  if (sx < 0) sx += A;
                    const uint32_t aMx = M0 + (uint32_t)sx * row_bytes;
                    const int xlo = LO[sx], xhi = HI[sx];
                    const uint32_t aMc = M0 + (uint32_t)sM * row_bytes;
                    int lo, hi;
                    if (st.kind == WFAGPU_STEP_M) {
                        lo = xlo; hi = xhi;
                        for (int k = lo + tid; k <= hi; k += gsz) {
                            int m = lds_s16(aMx + (uint32_t)(2 * (k - xlo))) + 1;
                            if (m >= 0) m = extend(k, m);
                            sts_16(aMc + (uint32_t)(2 * (k - lo)), m);
                        }
                        if (tid == 0) { LO[sM] = lo; HI[sM] = hi; }
                    } else {
                        int so = sM - oe; if (so < 0) so += A;
                        int sg = sM - e;  if (sg < 0) sg += A;
                        const uint32_t aMo = M0 + (uint32_t)so * row_bytes;
                        const uint32_t aIe = I0 + (uint32_t)sg * row_bytes;
                        const uint32_t aDe = D0 + (uint32_t)sg * row_bytes;
                        const uint32_t aIc = I0 + (uint32_t)sM * row_bytes;
                        const uint32_t aDc = D0 + (uint32_t)sM * row_bytes;
                        const int olo = LO[so], ohi = HI[so];
                        const int ilo = LO[A + sg], ihi = HI[A + sg];
                        const int dlo = LO[2 * A + sg], dhi = HI[2 * A + sg];
                        const int hi_ID = max(ohi, max(ihi, dhi)) + 1;
                        const int lo_ID = min(olo, min(ilo, dlo)) - 1;
                        hi = max(xhi, hi_ID);
                        lo = min(xlo, lo_ID);
                        const int excess = (hi - lo) - (W - 1);
                        if (excess > 0) { hi -= (excess + 1) >> 1; lo += excess >> 1; }
                        if ((xhi - xlo) >= W - 1 && (d % p.band) == 0) {
                            /* first diagonal of [xlo, xhi) with the smallest distance to the target */
                            unsigned long long best = ~0ull;
                            for (int i = xlo + tid; i < xhi; i += gsz) {
                                const int off = lds_s16(aMx + (uint32_t)(2 * (i - xlo)));
                                const int left_v = (int)(short)(plen - (off - i));
                                const int left_h = (int)(short)(tlen - off);
                                const int dt = off >= 0 ? max(left_v, left_h) : 0x7fffffff;
                                const unsigned long long key =
                                    ((unsigned long long)((unsigned)dt ^ 0x80000000u) << 32) | (unsigned)(i - xlo);
                                best = key < best ? key : best;
                            }
                            for (int s = 16; s > 0; s >>= 1) {
                                const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, s);
                                best = o < best ? o : best;
                            }
                            if (lane == 0) ctl->red[warp] = best;
                            __syncthreads();
                            if (warp == 0) {
                                unsigned long long b = lane < nwarps ? ctl->red[lane] : ~0ull;
                                for (int s = 16; s > 0; s >>= 1) {
                                    const unsigned long long o = __shfl_xor_sync(0xffffffffu, b, s);
                                    b = o < b ? o : b;
                                }
                                if (lane == 0) {
                                    int c = xlo;
                                    if (b != ~0ull) {
                                        const int dt = (int)((unsigned)(b >> 32) ^ 0x80000000u);
                                        if (dt < 2 * (tlen + plen)) c = xlo + (int)(unsigned)(b & 0xffffffffu);
                                    }
                                    ctl->new_center = c;
                                }
                            }
                            __syncthreads();
                            lo = ctl->new_center - (W / 2);
                            hi = lo + W - 1;
                        }
                        /* nobody reads the window of the slot being rewritten during this score (it is
                         * never one of its own sources: x, o+e, e < A), so it can be updated right away */
                        if (tid == 0) {
                            LO[sM] = lo; HI[sM] = hi;
                            LO[A + sM] = lo; HI[A + sM] = hi;
                            LO[2 * A + sM] = lo; HI[2 * A + sM] = hi;
                            if (BT) lo_tab[d] = lo;
                        }
                        uint8_t *const rowb = reinterpret_cast<uint8_t *>(arena + st.row_off);
                        const int width = hi - lo + 1;
                        for (int idc = tid; idc < width; idc += gsz) {
                            const int k = lo + idc;
                            const int io = band_get(aMo, olo, ohi, k - 1) + 1;
                            const int ie = band_get(aIe, ilo, ihi, k - 1) + 1;
                            const int dopen = band_get(aMo, olo, ohi, k + 1);
                            const int dext = band_get(aDe, dlo, dhi, k + 1);
                            const int X = band_get(aMx, xlo, xhi, k) + 1;
                            /* the reference keeps int16 values between the steps */
                            const int pI = max((int)(short)io * 2, (int)(short)ie * 2 + 1);
                            const int pD = max(dopen * 2, dext * 2 + 1);
                            const int I = pI >> 1;
                            const int D = pD >> 1;
                            const int pM = max(max((int)(short)X * 4 + 2, D * 4 + 3), I * 4 + 1);
                            int M = pM >> 2;
                            if (M >= 0) M = extend(k, M);
                            const uint32_t kk = (uint32_t)(2 * idc);
                            sts_16(aIc + kk, I);
                            sts_16(aDc + kk, D);
                            sts_16(aMc + kk, M);
                            if (BT) rowb[idc] = (uint8_t)((pI & 1) | ((pD & 1) << 1) | ((pM & 3) << 2));
                        }
                    }
                    __syncthreads();
                    if (kt_abs <= d) {
                        const int t = band_get(aMc, lo, hi, kt);
                        if (t == tlen) { finished = true; dist = d; break; }
                        if (t > tlen) break;                 /* aband.cu:678-681 */
                    }
                }
            }
        }

        /* ---- traceback: like the exact kernel, plus the per-score window origin and the
         * resolution of stale ring slots (a null score keeps the slot's previous owner) ---- */
        if (tid == 0) {
            uint32_t n_ops = 0, ops_off = 0;
            if (BT && finished && dist > 0) {
                int cd = dist, ck = kt, comp = 0;
                uint32_t word = 0;
                bool bad = false;
                auto resolveM = [&](int dd) { while (dd > 0 && p.steps[dd].kind == WFAGPU_STEP_NULL) dd -= A; return dd; };
                auto resolveG = [&](int dd) { while (dd > 0 && p.steps[dd].kind != WFAGPU_STEP_MDI) dd -= A; return dd; };
                while (!(comp == 0 && cd == 0)) {
                    if (cd < 0) { bad = true; break; }
                    const wfagpu_step_t st = p.steps[cd];
                    uint32_t op;
                    if (comp == 0 && st.kind == WFAGPU_STEP_M) {
                        op = OP_SUB;
                        cd = resolveM(cd - x);
                    } else {
                        if (st.kind != WFAGPU_STEP_MDI) { bad = true; break; }
                        const int ii = ck - lo_tab[cd];
                        if (ii < 0 || ii >= W) { bad = true; break; }
                        const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                        if (comp == 0) {
                            op = OP_SUB;
                            const int mop = (int)(dec >> 2) & 3;
                            if (mop == OP_SUB) cd = resolveM(cd - x);
                            else if (mop == OP_INS) comp = 1;
                            else comp = 2;
                        } else if (comp == 1) {
                            op = OP_INS;
                            ck -= 1;
                            if (dec & 1u) cd = resolveG(cd - e); else { cd = resolveM(cd - oe); comp = 0; }
                        } else {
                            op = OP_DEL;
                            ck += 1;
                            if (dec & 2u) cd = resolveG(cd - e); else { cd = resolveM(cd - oe); comp = 0; }
                        }
                    }
                    word |= op << (2 * (n_ops & 15u));
                    ++n_ops;
                    if ((n_ops & 15u) == 0) { scratch[(n_ops >> 4) - 1] = word; word = 0; }
                    if ((n_ops >> 4) >= p.ops_scratch_words) { bad = true; break; }
                }
                if (bad) { n_ops = 0; finished = false; }
                if (n_ops & 15u) scratch[n_ops >> 4] = word;
                const uint32_t nw = (n_ops + 15u) >> 4;
                ops_off = atomicAdd(p.ops_pool_head, nw);
                if (ops_off + nw > p.ops_pool_words) { n_ops = 0; finished = false; }
            }
            ctl->n_ops = n_ops;
            ctl->ops_off = ops_off;
            wfagpu_pair_out_t r;
            r.distance = finished ? dist : 0;
            r.ops_off = ops_off;
            r.n_ops = n_ops;
            if (skip) {
                r.status = WFAGPU_ST_NEEDS_ASCII;
                p.ascii_list[atomicAdd(p.ascii_count, 1u)] = idx;
            } else if (finished) {
                r.status = WFAGPU_ST_FINISHED;
            } else {
                r.status = WFAGPU_ST_OVERBUDGET;
                p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
            }
            p.out[idx] = r;
        }
        __syncthreads();
        if (BT) {
            const uint32_t nw = (ctl->n_ops + 15u) >> 4;
            const uint32_t off = ctl->ops_off;
            for (uint32_t i = tid; i < nw; i += gsz) p.ops_pool[off + i] = scratch[i];
        }
        __syncthreads();
        if (p.stages == 2) {
            stage ^= 1;
        } else {
            if (tid == 0) {
                const uint32_t nxt = pop(0);
                ctl->idx[0] = nxt;
                if (nxt != kInvalidIdx) issue_load(0, nxt);
            }
            __syncthreads();
        }
    }
}

size_t banded_smem_bytes(int A, int win, int seq_words, int stages)
{
    const size_t row_bytes = (size_t)((win + 7) & ~7) * 2;
    const size_t ring_bytes = (3 * (size_t)A * row_bytes + 15) & ~(size_t)15;
    const size_t lohi_bytes = ((3 * (size_t)A * 2 * sizeof(int)) + 15) & ~(size_t)15;
    return ring_bytes + lohi_bytes + 2 * (size_t)stages * seq_words * 4 + sizeof(BandCtl) + 16;
}

/* ======================================================================== */
/*        adaptive band, four diagonals per thread on packed int16          */
/* ======================================================================== */
/*
 * Same heuristic, same results as wfa_banded_kernel, for packed (ACGT) pairs.  A ring row stores the cells of its score's
 * window [lo, hi] at index k - base with base = lo rounded down to a multiple of four, whole quads, cells outside the window
 * as NULL: every quad a thread reads (its own four diagonals in the rows of d - x, d - o - e, d - e and the two neighbours
 * k - 1, k + 4) is one aligned LDS.64 / LDS.U16 whatever the windows of the source scores are -- a quad or neighbour outside
 * the stored part of a row is a predicated-off load that leaves NULL in the register.  The recurrence runs on packed int16
 * pairs; with backtrace the max instructions also return which operand won (VIMNMX.S16x2 with predicate outputs), which
 * gives the decision byte of wfa_banded_kernel (bit0 I extends, bit1 D extends, bits 3:2 the winner of M: ties
 * extend > open, D > X > I) -- four of them per 32-bit store, at byte k - base of the score's row (band_lo holds base).
 */
__device__ __forceinline__ uint2 lds_v2_or_null(uint32_t a, uint32_t idx, uint32_t n)
{
    uint2 v = make_uint2(kNull2, kNull2);
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "setp.lt.u32 p, %3, %4;\n"
                 "@p ld.shared.v2.u32 {%0, %1}, [%2];\n"
                 "}\n" : "+r"(v.x), "+r"(v.y) : "r"(a), "r"(idx), "r"(n));
    return v;
}
__device__ __forceinline__ uint32_t lds_u16_or_null(uint32_t a, uint32_t idx, uint32_t n)
{
    uint32_t v = kNull2 & 0xffffu;
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "setp.lt.u32 p, %2, %3;\n"
                 "@p ld.shared.u16 %0, [%1];\n"
                 "}\n" : "+r"(v) : "r"(a), "r"(idx), "r"(n));
    return v;
}

/* cells a row stores for the window [.., hi] with this base: whole quads */
__device__ __forceinline__ uint32_t bandq_cells(int hi, int base) { return (uint32_t)(((hi - base) | 3) + 1); }

struct BandQCtl {
    uint64_t bar[2];
    uint32_t idx[2];
    uint32_t pos[2];
    uint32_t n_ops;
    uint32_t ops_off;
    int new_center;
    int pad;
    unsigned long long red[32];
};

template <bool BT>
__global__ void __launch_bounds__(512, 1) wfa_bandq_kernel(const __grid_constant__ KernelParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, gsz = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = gsz >> 5;
    const int x = p.x, e = p.e, A = p.A, W = p.win;
    const int oe = p.o + p.e;
    const int RW = ((W + 3) & ~3) + 8;                         /* cells per row: a window plus alignment slack */
    const uint32_t row_bytes = ((uint32_t)RW * 2u + 15u) & ~15u;
    const uint32_t comp_bytes = (uint32_t)A * row_bytes;
    const uint32_t ring_bytes = 3u * comp_bytes;
    const uint32_t win_bytes = (uint32_t)(2 * A) * 16u;             /* window records: {lo, hi, base, cells} per slot */
    const uint32_t seq_bytes = (uint32_t)p.seq_words * 4u;
    const uint32_t seq_total = 2u * (uint32_t)p.stages * seq_bytes;
    const uint32_t M0 = smem_u32(smem_raw);
    const uint32_t I0 = M0 + comp_bytes, D0 = I0 + comp_bytes;
    const uint32_t WM = M0 + ring_bytes;                             /* M rows; the I and D rows of a slot share a window */
    const uint32_t WG = WM + (uint32_t)A * 16u;
    const uint32_t seq_sa = M0 + ring_bytes + win_bytes;
    BandQCtl *ctl = reinterpret_cast<BandQCtl *>(smem_raw + ring_bytes + win_bytes + seq_total);

    const uint32_t group = blockIdx.x;
    uint32_t *const scratch = p.ops_scratch + (size_t)group * p.ops_scratch_words;

    auto issue_load = [&](int stage, uint32_t idx) {
        const wfagpu_pair_t pr = p.pairs[idx];
        const uint32_t pw = ((((pr.plen + 7u) >> 3) + 1u) + 3u) & ~3u;
        const uint32_t tw = ((((pr.tlen + 7u) >> 3) + 1u) + 3u) & ~3u;
        unsigned char *dp = smem_raw + ring_bytes + win_bytes + (size_t)(2 * stage) * seq_bytes;
        unsigned char *dt = dp + seq_bytes;
        fence_proxy_async();
        mbar_expect_tx(&ctl->bar[stage], (pw + tw) * 4u);
        tma_load_1d(dp, p.packed + pr.p_word, pw * 4u, &ctl->bar[stage]);
        tma_load_1d(dt, p.packed + pr.t_word, tw * 4u, &ctl->bar[stage]);
    };
    auto pop = [&](int slot) -> uint32_t {
        const uint32_t pos = atomicAdd(p.queue, 1u);
        ctl->pos[slot] = pos;
        return pos < p.n_items ? p.order[pos] : kInvalidIdx;
    };
    if (tid == 0) {
        mbar_init(&ctl->bar[0], 1);
        mbar_init(&ctl->bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t first = pop(0);
        ctl->idx[0] = first;
        if (first != kInvalidIdx) issue_load(0, first);
    }
    __syncthreads();

    int stage = 0;
    uint32_t phase_bits = 0;
    while (true) {
        const uint32_t idx = ctl->idx[stage];
        if (idx == kInvalidIdx) break;
        if (tid == 0 && p.stages == 2) {
            const uint32_t nxt = pop(stage ^ 1);
            ctl->idx[stage ^ 1] = nxt;
            if (nxt != kInvalidIdx) issue_load(stage ^ 1, nxt);
        }
        /* decision rows and row bases: per queue position (walked by wfa_band_traceback_kernel), else per CTA */
        const size_t region = p.band_tb ? (size_t)ctl->pos[stage] : (size_t)group;
        uint4 *const arena = p.arena + region * p.arena_units;
        int32_t *const lo_tab = p.band_lo + region * p.band_lo_words;
        const wfagpu_pair_t pr = p.pairs[idx];
        const int plen = (int)pr.plen, tlen = (int)pr.tlen;
        const int kt = tlen - plen;
        const int kt_abs = kt < 0 ? -kt : kt;
        const int tl8 = tlen - 8;
        const uint32_t Pa = seq_sa + (uint32_t)(2 * stage) * seq_bytes;
        const uint32_t Ta = Pa + seq_bytes;
        const bool skip = (pr.flags & WFAGPU_PAIR_HAS_N) != 0;

        /* every slot starts as the one-diagonal window [0, 0] holding NULL (aband.cu:543-578): one quad of NULLs at base 0 */
        for (int i = tid; i < 3 * A; i += gsz) {
            if (i < 2 * A) sts_v4(WM + (uint32_t)i * 16u, make_uint4(0u, 0u, 0u, 4u));
            sts_v2(M0 + (uint32_t)i * row_bytes, kNull2, kNull2);
        }
        mbar_wait(&ctl->bar[stage], (phase_bits >> stage) & 1u);
        phase_bits ^= (1u << stage);
        __syncthreads();

        int dist = 0;
        bool finished = false;
        if (!skip) {
            if (tid == 0) sts_16(M0, extend_packed(Pa, Ta, plen, tlen, 0, 0));
            __syncthreads();
            if (kt == 0 && lds_s16(M0) == tlen) {
                finished = true;
            } else {
                int sM = 0;                                  /* ring slot of the current score: d mod A */
                int d_rc = p.band;                           /* next score that is a multiple of `band` */
                for (int d = 1; d < p.d_end; ++d) {
                    const wfagpu_step_t st = p.steps[d];
                    sM = (sM + 1 == A) ? 0 : sM + 1;
                    if (d > d_rc) d_rc += p.band;
                    if (st.kind == WFAGPU_STEP_NULL) continue;
                    int sx = sM - x;  if (sx < 0) sx += A;
                    const uint32_t aMx = M0 + (uint32_t)sx * row_bytes;
                    const uint4 wx = lds_v4(WM + (uint32_t)sx * 16u);
                    const int xlo = (int)wx.x, xhi = (int)wx.y, bx = (int)wx.z;
                    const uint32_t aMc = M0 + (uint32_t)sM * row_bytes;
                    int lo, hi, base;
                    if (st.kind == WFAGPU_STEP_M) {
                        lo = xlo; hi = xhi; base = bx;
                        const int nq = ((hi - base) >> 2) + 1;
                        for (int q = tid; q < nq; q += gsz) {
                            const int kq = base + 4 * q;
                            const uint32_t o2 = (uint32_t)(8 * q);
                            const uint2 mx = lds_v2(aMx + o2);
                            uint32_t M01 = __vadd2(mx.x, kOnes2), M23 = __vadd2(mx.y, kOnes2);
                            if (kq < lo || kq + 3 > hi) {
                                M01 = sel2(M01, in2(kq, lo, hi));
                                M23 = sel2(M23, in2(kq + 2, lo, hi));
                            }
                            extend_quad(Pa, Ta, plen, tlen, kq, tl8, M01, M23);
                            sts_v2(aMc + o2, M01, M23);
                        }
                        if (tid == 0) sts_v4(WM + (uint32_t)sM * 16u, wx);
                    } else {
                        int so = sM - oe; if (so < 0) so += A;
                        int sg = sM - e;  if (sg < 0) sg += A;
                        const uint32_t aMo = M0 + (uint32_t)so * row_bytes;
                        const uint32_t aIe = I0 + (uint32_t)sg * row_bytes;
                        const uint32_t aDe = D0 + (uint32_t)sg * row_bytes;
                        const uint32_t aIc = I0 + (uint32_t)sM * row_bytes;
                        const uint32_t aDc = D0 + (uint32_t)sM * row_bytes;
                        const uint4 wo = lds_v4(WM + (uint32_t)so * 16u), wg = lds_v4(WG + (uint32_t)sg * 16u);
                        const int olo = (int)wo.x, ohi = (int)wo.y, bo = (int)wo.z;
                        const int glo = (int)wg.x, ghi = (int)wg.y, bg = (int)wg.z;
                        const int hi_ID = max(ohi, ghi) + 1;
                        const int lo_ID = min(olo, glo) - 1;
                        hi = max(xhi, hi_ID);
                        lo = min(xlo, lo_ID);
                        const int excess = (hi - lo) - (W - 1);
                        if (excess > 0) { hi -= (excess + 1) >> 1; lo += excess >> 1; }
                        if ((xhi - xlo) >= W - 1 && d == d_rc) {
                            /* first diagonal of [xlo, xhi) with the smallest distance to the target */
                            unsigned long long best = ~0ull;
                            for (int i = xlo + tid; i < xhi; i += gsz) {
                                const int off = lds_s16(aMx + (uint32_t)(2 * (i - bx)));
                                const int left_v = (int)(short)(plen - (off - i));
                                const int left_h = (int)(short)(tlen - off);
                                const int dt = off >= 0 ? max(left_v, left_h) : 0x7fffffff;
                                const unsigned long long key =
                                    ((unsigned long long)((unsigned)dt ^ 0x80000000u) << 32) | (unsigned)(i - xlo);
                                best = key < best ? key : best;
                            }
                            for (int s = 16; s > 0; s >>= 1) {
                                const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, s);
                                best = o < best ? o : best;
                            }
                            if (lane == 0) ctl->red[warp] = best;
                            __syncthreads();
                            if (warp == 0) {
                                unsigned long long b = lane < nwarps ? ctl->red[lane] : ~0ull;
                                for (int s = 16; s > 0; s >>= 1) {
                                    const unsigned long long o = __shfl_xor_sync(0xffffffffu, b, s);
                                    b = o < b ? o : b;
                                }
                                if (lane == 0) {
                                    int c = xlo;
                                    if (b != ~0ull) {
                                        const int dt = (int)((unsigned)(b >> 32) ^ 0x80000000u);
                                        if (dt < 2 * (tlen + plen)) c = xlo + (int)(unsigned)(b & 0xffffffffu);
                                    }
                                    ctl->new_center = c;
                                }
                            }
                            __syncthreads();
                            lo = ctl->new_center - (W / 2);
                            hi = lo + W - 1;
                        }
                        base = lo & ~3;
                        /* nobody reads the window of the slot being rewritten during this score (it is
                         * never one of its own sources: x, o+e, e < A), so it can be updated right away */
                        if (tid == 0) {
                            const uint4 w = make_uint4((uint32_t)lo, (uint32_t)hi, (uint32_t)base, bandq_cells(hi, base));
                            sts_v4(WM + (uint32_t)sM * 16u, w);
                            sts_v4(WG + (uint32_t)sM * 16u, w);
                            if (BT) lo_tab[d] = base;
                        }
                        uint8_t *const rowb = reinterpret_cast<uint8_t *>(arena + st.row_off);
                        const uint32_t nx = wx.w, no = wo.w, ng = wg.w;
                        const int nq = ((hi - base) >> 2) + 1;
                        for (int q = tid; q < nq; q += gsz) {
                            const int kq = base + 4 * q;
                            const uint32_t o2 = (uint32_t)(8 * q);
                            const int jo = kq - bo, jg = kq - bg, jx = kq - bx;
                            const uint32_t ao = aMo + (uint32_t)(2 * jo), ai = aIe + (uint32_t)(2 * jg), ad = aDe + (uint32_t)(2 * jg);
                            const uint2 mo = lds_v2_or_null(ao, (uint32_t)jo, no);
                            const uint32_t ml = lds_u16_or_null(ao - 2u, (uint32_t)(jo - 1), no);
                            const uint32_t mr = lds_u16_or_null(ao + 8u, (uint32_t)(jo + 4), no);
                            const uint2 ie = lds_v2_or_null(ai, (uint32_t)jg, ng);
                            const uint32_t il = lds_u16_or_null(ai - 2u, (uint32_t)(jg - 1), ng);
                            const uint2 de = lds_v2_or_null(ad, (uint32_t)jg, ng);
                            const uint32_t dr = lds_u16_or_null(ad + 8u, (uint32_t)(jg + 4), ng);
                            const uint2 mx = lds_v2_or_null(aMx + (uint32_t)(2 * jx), (uint32_t)jx, nx);
                            const uint32_t oL01 = __byte_perm(ml, mo.x, 0x5410);          /* Mo (k-1 | k)   */
                            const uint32_t oMid = __byte_perm(mo.x, mo.y, 0x5432);        /* Mo (k+1 | k+2) */
                            const uint32_t oR23 = __byte_perm(mo.y, mr, 0x5432);          /* Mo (k+3 | k+4) */
                            const uint32_t eI01 = __byte_perm(il, ie.x, 0x5410), eI23 = __byte_perm(ie.x, ie.y, 0x5432);
                            const uint32_t eD01 = __byte_perm(de.x, de.y, 0x5432), eD23 = __byte_perm(de.y, dr, 0x5432);
                            const uint32_t X01 = __vadd2(mx.x, kOnes2), X23 = __vadd2(mx.y, kOnes2);
                            uint32_t I01, I23, D01, D23, M01, M23, dec = 0;
                            if (BT) {
                                bool i0, i1, i2, i3, d0, d1, d2, d3, a0, a1, a2, a3, b0, b1, b2, b3;
                                I01 = __vadd2(__vibmax_s16x2(eI01, oL01, &i1, &i0), kOnes2);      /* pred: extend >= open */
                                I23 = __vadd2(__vibmax_s16x2(eI23, oMid, &i3, &i2), kOnes2);
                                D01 = __vibmax_s16x2(eD01, oMid, &d1, &d0);
                                D23 = __vibmax_s16x2(eD23, oR23, &d3, &d2);
                                const uint32_t T01 = __vibmax_s16x2(D01, X01, &a1, &a0);          /* pred: D >= X */
                                const uint32_t T23 = __vibmax_s16x2(D23, X23, &a3, &a2);
                                M01 = __vibmax_s16x2(T01, I01, &b1, &b0);                          /* pred: max(D, X) >= I */
                                M23 = __vibmax_s16x2(T23, I23, &b3, &b2);
                                dec = ((i0 ? 1u : 0u) + (d0 ? 2u : 0u) + (b0 ? (a0 ? 12u : 8u) : 4u)) +
                                      ((i1 ? 1u : 0u) + (d1 ? 2u : 0u) + (b1 ? (a1 ? 12u : 8u) : 4u)) * 0x100u +
                                      ((i2 ? 1u : 0u) + (d2 ? 2u : 0u) + (b2 ? (a2 ? 12u : 8u) : 4u)) * 0x10000u +
                                      ((i3 ? 1u : 0u) + (d3 ? 2u : 0u) + (b3 ? (a3 ? 12u : 8u) : 4u)) * 0x1000000u;
                            } else {
                                I01 = __vadd2(__vmaxs2(eI01, oL01), kOnes2);
                                I23 = __vadd2(__vmaxs2(eI23, oMid), kOnes2);
                                D01 = __vmaxs2(eD01, oMid);
                                D23 = __vmaxs2(eD23, oR23);
                                M01 = __vimax3_s16x2(X01, D01, I01);
                                M23 = __vimax3_s16x2(X23, D23, I23);
                            }
                            if (kq < lo || kq + 3 > hi) {
                                /* quad straddles the window: stores outside [lo, hi] are dropped, i.e. read back as NULL */
                                const uint32_t k01 = in2(kq, lo, hi), k23 = in2(kq + 2, lo, hi);
                                I01 = sel2(I01, k01); D01 = sel2(D01, k01); M01 = sel2(M01, k01);
                                I23 = sel2(I23, k23); D23 = sel2(D23, k23); M23 = sel2(M23, k23);
                            }
                            sts_v2(aIc + o2, I01, I23);
                            sts_v2(aDc + o2, D01, D23);
                            if (BT) *reinterpret_cast<uint32_t *>(rowb + 4 * q) = dec;
                            extend_quad(Pa, Ta, plen, tlen, kq, tl8, M01, M23);
                            sts_v2(aMc + o2, M01, M23);
                        }
                    }
                    __syncthreads();
                    if (kt_abs <= d) {
                        const int t = (kt >= lo && kt <= hi) ? lds_s16(aMc + (uint32_t)(2 * (kt - base))) : kOffNull;
                        if (t == tlen) { finished = true; dist = d; break; }
                        if (t > tlen) break;                 /* aband.cu:678-681 */
                    }
                }
            }
        }

        /* ---- traceback: as in wfa_banded_kernel; lo_tab holds the base of every score's row ---- */
        if (tid == 0) {
            uint32_t n_ops = 0, ops_off = 0;
            if (BT && finished && dist > 0 && !p.band_tb) {
                int cd = dist, ck = kt, comp = 0;
                uint32_t word = 0;
                bool bad = false;
                auto resolveM = [&](int dd) { while (dd > 0 && p.steps[dd].kind == WFAGPU_STEP_NULL) dd -= A; return dd; };
                auto resolveG = [&](int dd) { while (dd > 0 && p.steps[dd].kind != WFAGPU_STEP_MDI) dd -= A; return dd; };
                while (!(comp == 0 && cd == 0)) {
                    if (cd < 0) { bad = true; break; }
                    const wfagpu_step_t st = p.steps[cd];
                    uint32_t op;
                    if (comp == 0 && st.kind == WFAGPU_STEP_M) {
                        op = OP_SUB;
                        cd = resolveM(cd - x);
                    } else {
                        if (st.kind != WFAGPU_STEP_MDI) { bad = true; break; }
                        const int ii = ck - lo_tab[cd];
                        if (ii < 0 || ii >= RW) { bad = true; break; }
                        const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
                        if (comp == 0) {
                            op = OP_SUB;
                            const int mop = (int)(dec >> 2) & 3;
                            if (mop == OP_SUB) cd = resolveM(cd - x);
                            else if (mop == OP_INS) comp = 1;
                            else comp = 2;
                        } else if (comp == 1) {
                            op = OP_INS;
                            ck -= 1;
                            if (dec & 1u) cd = resolveG(cd - e); else { cd = resolveM(cd - oe); comp = 0; }
                        } else {
                            op = OP_DEL;
                            ck += 1;
                            if (dec & 2u) cd = resolveG(cd - e); else { cd = resolveM(cd - oe); comp = 0; }
                        }
                    }
                    word |= op << (2 * (n_ops & 15u));
                    ++n_ops;
                    if ((n_ops & 15u) == 0) { scratch[(n_ops >> 4) - 1] = word; word = 0; }
                    if ((n_ops >> 4) >= p.ops_scratch_words) { bad = true; break; }
                }
                if (bad) { n_ops = 0; finished = false; }
                if (n_ops & 15u) scratch[n_ops >> 4] = word;
                const uint32_t nw = (n_ops + 15u) >> 4;
                ops_off = atomicAdd(p.ops_pool_head, nw);
                if (ops_off + nw > p.ops_pool_words) { n_ops = 0; finished = false; }
            }
            ctl->n_ops = n_ops;
            ctl->ops_off = ops_off;
            wfagpu_pair_out_t r;
            r.distance = finished ? dist : 0;
            r.ops_off = ops_off;
            r.n_ops = n_ops;
            if (skip) {
                r.status = WFAGPU_ST_NEEDS_ASCII;
                p.ascii_list[atomicAdd(p.ascii_count, 1u)] = idx;
            } else if (finished) {
                r.status = WFAGPU_ST_FINISHED;
            } else {
                r.status = WFAGPU_ST_OVERBUDGET;
                p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
            }
            p.out[idx] = r;
        }
        __syncthreads();
        if (BT) {
            const uint32_t nw = (ctl->n_ops + 15u) >> 4;
            const uint32_t off = ctl->ops_off;
            for (uint32_t i = tid; i < nw; i += gsz) p.ops_pool[off + i] = scratch[i];
        }
        __syncthreads();
        if (p.stages == 2) {
            stage ^= 1;
        } else {
            if (tid == 0) {
                const uint32_t nxt = pop(0);
                ctl->idx[0] = nxt;
                if (nxt != kInvalidIdx) issue_load(0, nxt);
            }
            __syncthreads();
        }
    }
}

/* The backtrace of wfa_bandq_kernel's decision bytes, one thread per pair of the launch: a walk of dependent loads (the
 * score's row base, then the byte), so thousands of them in flight beat one walk per CTA while its other threads wait
 * (17 % of the warp time of the fused version).  Ops oldest-last, 16 per word, straight into the pool. */
__global__ void __launch_bounds__(128) wfa_band_traceback_kernel(const __grid_constant__ KernelParams p)
{
    const uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= p.n_items) return;
    const uint32_t idx = p.order[pos];
    wfagpu_pair_out_t res = p.out[idx];
    if (!(res.status & WFAGPU_ST_FINISHED) || res.distance <= 0) return;
    const int x = p.x, e = p.e, A = p.A, oe = p.o + p.e;
    const int RW = ((p.win + 3) & ~3) + 8;
    const wfagpu_pair_t pr = p.pairs[idx];
    const uint4 *const arena = p.arena + (size_t)pos * p.arena_units;
    const int32_t *const lo_tab = p.band_lo + (size_t)pos * p.band_lo_words;
    const int dist = res.distance;
    const uint32_t nw_max = ((2u * (uint32_t)dist + 15u) >> 4) + 1u;       /* at most 2 ops per score */
    const uint32_t ops_off = atomicAdd(p.ops_pool_head, nw_max);
    bool bad = ops_off + nw_max > p.ops_pool_words;
    uint32_t *const ops = p.ops_pool + ops_off;
    int cd = dist, ck = (int)pr.tlen - (int)pr.plen, comp = 0;
    uint32_t word = 0, n_ops = 0;
    auto resolveM = [&](int dd) { while (dd > 0 && p.steps[dd].kind == WFAGPU_STEP_NULL) dd -= A; return dd; };
    auto resolveG = [&](int dd) { while (dd > 0 && p.steps[dd].kind != WFAGPU_STEP_MDI) dd -= A; return dd; };
    while (!bad && !(comp == 0 && cd == 0)) {
        if (cd < 0) { bad = true; break; }
        const wfagpu_step_t st = p.steps[cd];
        uint32_t op;
        if (comp == 0 && st.kind == WFAGPU_STEP_M) {
            op = OP_SUB;
            cd = resolveM(cd - x);
        } else {
            if (st.kind != WFAGPU_STEP_MDI) { bad = true; break; }
            const int ii = ck - lo_tab[cd];
            if (ii < 0 || ii >= RW) { bad = true; break; }
            const uint32_t dec = reinterpret_cast<const uint8_t *>(arena + st.row_off)[ii];
            if (comp == 0) {
                op = OP_SUB;
                const int mop = (int)(dec >> 2) & 3;
                if (mop == OP_SUB) cd = resolveM(cd - x);
                else if (mop == OP_INS) comp = 1;
                else comp = 2;
            } else if (comp == 1) {
                op = OP_INS;
                ck -= 1;
                if (dec & 1u) cd = resolveG(cd - e); else { cd = resolveM(cd - oe); comp = 0; }
            } else {
                op = OP_DEL;
                ck += 1;
                if (dec & 2u) cd = resolveG(cd - e); else { cd = resolveM(cd - oe); comp = 0; }
            }
        }
        word |= op << (2 * (n_ops & 15u));
        ++n_ops;
        if ((n_ops & 15u) == 0) { ops[(n_ops >> 4) - 1] = word; word = 0; }
        if (n_ops >= 16u * nw_max) { bad = true; break; }                  /* never: at most 2 ops per score */
    }
    if (bad) {
        /* cannot happen for a finished pair; handled like a pair that ran out of budget */
        res.status = WFAGPU_ST_OVERBUDGET;
        res.distance = 0;
        res.ops_off = 0;
        res.n_ops = 0;
        p.retry_list[atomicAdd(p.retry_count, 1u)] = idx;
    } else {
        if (n_ops & 15u) ops[n_ops >> 4] = word;
        res.ops_off = ops_off;
        res.n_ops = n_ops;
    }
    p.out[idx] = res;
}

cudaError_t launch_band_traceback(const KernelParams &p, cudaStream_t s)
{
    if (p.n_items == 0) return cudaSuccess;
    wfa_band_traceback_kernel<<<(p.n_items + 127u) / 128u, 128, 0, s>>>(p);
    return cudaGetLastError();
}

size_t bandq_smem_bytes(int A, int win, int seq_words, int stages)
{
    const size_t rw = (size_t)((win + 3) & ~3) + 8;
    const size_t row_bytes = (rw * 2 + 15) & ~(size_t)15;
    const size_t ring_bytes = 3 * (size_t)A * row_bytes;
    const size_t win_bytes = 2 * (size_t)A * 16;
    return ring_bytes + win_bytes + 2 * (size_t)stages * seq_words * 4 + sizeof(BandQCtl) + 16;
}

/* ======================================================================== */
/*                       CIGAR text emission on the device                  */
/* ======================================================================== */
/*
 * Replaces the host stage recover_cigar_affine + insert_ops (utils/cigar.c:31-61,
 * 96-272; OpenMP loop of utils/wfa_cpu.c:88-107): one thread per pair walks its
 * op stream oldest first, re-derives the match runs on the ASCII copy that is
 * already in HBM, and prints the run-length text ("%d%c", no '=') into a slot of
 * the text pool.  Byte-for-byte the reference's output: X inside a gap is the
 * gap-close delimiter and prints nothing, equal ops merge unless a delimiter or a
 * match run separates them, score 0 prints "<tlen>M".  A second kernel compacts
 * the slots so that only the text itself crosses PCIe.
 */
__device__ __forceinline__ uint32_t put_run(char *dst, uint32_t pos, uint32_t rep, char op)
{
    /* "%d%c" (insert_ops, utils/cigar.c:31-61); nothing for an empty run */
    if (rep == 0) return pos;
    if (rep < 10u) {                                   /* almost every op run, half of the match runs */
        dst[pos++] = (char)('0' + rep);
    } else if (rep < 100u) {                           /* constant divisors: multiply-shift, no division */
        const uint32_t q = rep / 10u;
        dst[pos++] = (char)('0' + q);
        dst[pos++] = (char)('0' + (rep - 10u * q));
    } else if (rep < 1000u) {
        const uint32_t h = rep / 100u, r = rep - 100u * h, q = r / 10u;
        dst[pos++] = (char)('0' + h);
        dst[pos++] = (char)('0' + q);
        dst[pos++] = (char)('0' + (r - 10u * q));
    } else {
        uint32_t div = 1000u;
        while (rep / div >= 10u) div *= 10u;
        for (; div; div /= 10u) dst[pos++] = (char)('0' + (rep / div) % 10u);
    }
    dst[pos++] = op;
    return pos;
}

/* Match run from (v, h), found by the whole warp: 32 bases per round, ballot + ffs. */
__device__ __forceinline__ uint32_t match_run_warp(const char *__restrict__ P, const char *__restrict__ T,
                                                   int plen, int tlen, int v, int h, int lane)
{
    if (v < 0 || h < 0) return 0;
    const int room = min(plen - v, tlen - h);
    int n = 0;
    while (n < room) {
        const int j = n + lane;
        const bool diff = (j >= room) || (P[v + j] != T[h + j]);
        const uint32_t m = __ballot_sync(0xffffffffu, diff);
        if (m) return (uint32_t)(n + (__ffs((int)m) - 1));
        n += 32;
    }
    return (uint32_t)room;
}

/* One warp per pair.  The op walk is sequential; the warp shares the match-run scans
 * (coalesced 32-byte reads of both sequences) and lane 0 prints.
 * EF (ends-free, p.ends): the walk starts at (max(0, -k0), max(0, k0)) behind a leading I / D run of |k0| and ends
 * with the trailing I / D run to the end of both sequences; a free run joins the gap run of the same letter next to
 * it (wfagpu_ops_to_cigar_span prints the same text on the host). */
template <bool EF>
__global__ void __launch_bounds__(256) cigar_text_kernel(CigarParams p)
{
    const uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= p.n_pairs) return;
    const wfagpu_pair_out_t o = p.out[i];
    wfagpu_cigar_ref_t ref = {0u, 0u};
    if (!(o.status & WFAGPU_ST_FINISHED)) { if (lane == 0) p.refs[i] = ref; return; }
    const wfagpu_pair_t pr = p.pairs[i];
    const char *P = p.ascii + pr.p_ascii, *T = p.ascii + pr.t_ascii;
    const int plen = (int)pr.plen, tlen = (int)pr.tlen;
    if constexpr (EF) {
        /* every op prints at most 10 characters; plus the leading, last match and trailing runs (11 each) */
        const uint32_t cap = (10u * o.n_ops + 40u + 7u) & ~7u;
        unsigned long long slot = 0;
        if (lane == 0) slot = atomicAdd(p.slot_head, (unsigned long long)cap);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot + cap > p.slot_bytes) {
            if (lane == 0) { p.refs[i] = ref; atomicOr(p.overflow, 1u); }
            return;
        }
        char *dst = p.slots + slot;
        uint32_t pos = 0;
        const int k0 = p.ends[i].x;
        const uint32_t *ops = p.ops_pool + o.ops_off;
        int k = k0, off = max(0, k0);
        bool in_gap = false;
        uint32_t run_op = k0 > 0 ? OP_INS : (k0 < 0 ? OP_DEL : OP_NOOP), run_len = (uint32_t)abs(k0);
        uint32_t word = 0;
        for (uint32_t j = o.n_ops; j-- > 0;) {
            if ((j & 15u) == 15u || j == o.n_ops - 1) word = ops[j >> 4];
            uint32_t op = (word >> (2u * (j & 15u))) & 3u;
            /* the newest op closing a gap: hold the gap run, the trailing run may join it */
            const bool hold = j == 0 && in_gap && op == OP_SUB;
            if (op != run_op && run_len && !hold) { if (lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]); run_len = 0; }
            if (!in_gap) {
                const uint32_t m = match_run_warp(P, T, plen, tlen, off - k, off, lane);
                if (m) {
                    if (run_len) { if (lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]); run_len = 0; }
                    if (lane == 0) pos = put_run(dst, pos, m, 'M');
                    off += (int)m;
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
        const uint32_t m = in_gap ? 0u : match_run_warp(P, T, plen, tlen, off - k, off, lane);
        if (m) {
            if (run_len && lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]);
            run_len = 0;
            if (lane == 0) pos = put_run(dst, pos, m, 'M');
            off += (int)m;
        }
        const uint32_t tail_i = (uint32_t)(tlen - off), tail_d = (uint32_t)(plen - (off - k));
        const uint32_t tail = tail_i ? tail_i : tail_d, tail_op = tail_i ? OP_INS : OP_DEL;
        if (tail) {
            if (run_len && run_op == tail_op) run_len += tail;
            else {
                if (run_len && lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]);
                run_op = tail_op; run_len = tail;
            }
        }
        if (run_len && lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]);
        if (lane == 0) {
            ref.off = (uint32_t)(slot >> 3);
            ref.len = pos;
            p.refs[i] = ref;
        }
        return;
    }
    /* every op prints at most "1X" + "NNNNNNNM": 10 characters; plus the leading/trailing run */
    const uint32_t cap = (10u * o.n_ops + 24u + 7u) & ~7u;
    unsigned long long slot = 0;
    if (lane == 0) slot = atomicAdd(p.slot_head, (unsigned long long)cap);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    if (slot + cap > p.slot_bytes) {
        if (lane == 0) { p.refs[i] = ref; atomicOr(p.overflow, 1u); }
        return;
    }
    char *dst = p.slots + slot;
    uint32_t pos = 0;                                   /* meaningful in lane 0 only */
    if (o.distance == 0) {
        if (lane == 0) pos = put_run(dst, pos, (uint32_t)tlen, 'M');
    } else {
        const uint32_t *ops = p.ops_pool + o.ops_off;
        int k = 0, off = 0;
        bool in_gap = false;
        uint32_t run_op = OP_NOOP, run_len = 0;
        uint32_t word = 0;
        for (uint32_t j = o.n_ops; j-- > 0;) {
            if ((j & 15u) == 15u || j == o.n_ops - 1) word = ops[j >> 4];
            uint32_t op = (word >> (2u * (j & 15u))) & 3u;
            if (op != run_op && run_len) { if (lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]); run_len = 0; }
            if (!in_gap) {
                const uint32_t m = match_run_warp(P, T, plen, tlen, off - k, off, lane);
                if (m) {
                    if (run_len) { if (lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]); run_len = 0; }
                    if (lane == 0) pos = put_run(dst, pos, m, 'M');
                    off += (int)m;
                }
            }
            if (op == OP_DEL) { in_gap = true; --k; ++run_len; }
            else if (op == OP_INS) { in_gap = true; ++k; ++off; ++run_len; }
            else if (op == OP_SUB) {
                if (in_gap) { in_gap = false; op = OP_NOOP; }
                else { ++off; ++run_len; }
            }
            run_op = op;
        }
        if (run_len && lane == 0) pos = put_run(dst, pos, run_len, "?IXD"[run_op]);
        if (!in_gap) {
            const uint32_t m = match_run_warp(P, T, plen, tlen, off - k, off, lane);
            if (lane == 0) pos = put_run(dst, pos, m, 'M');
        }
    }
    if (lane == 0) {
        ref.off = (uint32_t)(slot >> 3);          /* slots are 8-byte aligned */
        ref.len = pos;
        p.refs[i] = ref;
    }
}

/* One warp per pair: move the text from its slack slot to a dense pool. */
__global__ void __launch_bounds__(256) cigar_compact_kernel(CigarParams p)
{
    const uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= p.n_pairs) return;
    wfagpu_cigar_ref_t ref = p.refs[i];
    if (ref.len == 0) return;
    uint32_t dst_off = 0;
    if (lane == 0) dst_off = (uint32_t)atomicAdd(p.text_head, (unsigned long long)ref.len);
    dst_off = __shfl_sync(0xffffffffu, dst_off, 0);
    const char *src = p.slots + ((unsigned long long)ref.off << 3);
    for (uint32_t j = lane; j < ref.len; j += 32) p.text[dst_off + j] = src[j];
    if (lane == 0) { ref.off = dst_off; p.refs[i] = ref; }
}

void launch_cigar_text(const CigarParams &p, cudaStream_t s)
{
    if (p.n_pairs == 0) return;
    if (p.ends) cigar_text_kernel<true><<<(p.n_pairs + 7) / 8, 256, 0, s>>>(p);
    else cigar_text_kernel<false><<<(p.n_pairs + 7) / 8, 256, 0, s>>>(p);
    cigar_compact_kernel<<<(p.n_pairs + 7) / 8, 256, 0, s>>>(p);
}

/* ---- host-side launch helpers ---------------------------------------------- */

cudaError_t launch(kernel_fn kfn, const KernelParams &p, int ctas, int threads, size_t smem, cudaStream_t s)
{
    if (!kfn) return cudaErrorInvalidValue;
    cudaError_t err = allow_max_smem(kfn);
    if (err != cudaSuccess) return err;
    kfn<<<ctas, threads, smem, s>>>(p);
    return cudaGetLastError();
}

int max_ctas_per_sm(kernel_fn kfn, int threads, size_t smem)
{
    int n = 0;
    if (!kfn || allow_max_smem(kfn) != cudaSuccess || occupancy_of(&n, kfn, threads, smem) != cudaSuccess) return 0;
    return n;
}

size_t exact_smem_bytes(int A, int E1, int row_stride, int seq_words, int groups_per_cta, int stages, bool sched, int E2,
                        bool org)
{
    const int rows = (A + 2 * E1 + 2 * E2) * (org ? 2 : 1);
    const size_t ring_bytes = ((size_t)rows * row_stride * sizeof(int16_t) + 15) & ~(size_t)15;
    const size_t seq_bytes = (size_t)seq_words * 4;
    const size_t group_bytes = (ring_bytes + 2 * (size_t)stages * seq_bytes + sizeof(GroupCtl) + (sched ? kSchedBytes : 0) + 15) & ~(size_t)15;
    return group_bytes * (size_t)groups_per_cta;
}

size_t bound_smem_bytes(int A, int E1, int warps) { return (size_t)warps * (size_t)(A + 2 * E1) * 32 * sizeof(int); }

cudaError_t launch_bound(const KernelParams &p, int ctas, int warps, cudaStream_t s)
{
    return launch(wfa_bound_kernel, p, ctas, 32 * warps, bound_smem_bytes(p.A, p.E1, warps), s);
}

int bound_max_ctas_per_sm(int A, int E1, int warps)
{
    return max_ctas_per_sm(wfa_bound_kernel, 32 * warps, bound_smem_bytes(A, E1, warps));
}

size_t traceback_smem_bytes(int A, int period, int warps)
{
    const size_t per_warp = ((size_t)3 * (period + A - 1) * (2 * period + 1) * 2 + 15) & ~(size_t)15;
    return per_warp * (size_t)warps;
}

static kernel_fn traceback_fn(bool ascii, int period)
{
    switch (period) {
    /* 2P + 1 diagonals at the base of a cone: 15 and 31 keep a level within one and two warp passes */
    case 7: return ascii ? wfa_traceback_kernel<true, 7> : wfa_traceback_kernel<false, 7>;
    case 15: return ascii ? wfa_traceback_kernel<true, 15> : wfa_traceback_kernel<false, 15>;
    case 31: return ascii ? wfa_traceback_kernel<true, 31> : wfa_traceback_kernel<false, 31>;
    default: return nullptr;
    }
}

cudaError_t launch_traceback(const KernelParams &p, int ctas, int warps, bool ascii, cudaStream_t s)
{
    return launch(traceback_fn(ascii, p.ck_period), p, ctas, 32 * warps, traceback_smem_bytes(p.A, p.ck_period, warps), s);
}

int traceback_max_ctas_per_sm(int A, int period, int warps, bool ascii)
{
    return max_ctas_per_sm(traceback_fn(ascii, period), 32 * warps, traceback_smem_bytes(A, period, warps));
}

/* wfa_exact_kernel of one tier (WARP, Ring) in the batch's mode: ends-free (score only: with or without origins),
 * 2-piece or single-piece global */
template <bool WARP, bool ASCII, bool BT, typename R>
static kernel_fn exact_mode(const KernelChoice &k)
{
    if (k.org) {
        if constexpr (!BT) {
            if (k.ef && !k.p2) return wfa_exact_kernel<WARP, ASCII, false, R, false, true, false, true>;
        }
        return nullptr;
    }
    if (k.ef) return wfa_exact_kernel<WARP, ASCII, BT, R, false, true>;
    if (k.p2) return wfa_exact_kernel<WARP, ASCII, BT, R, false, false, true>;
    return wfa_exact_kernel<WARP, ASCII, BT, R, false>;
}

template <bool ASCII, bool BT>
static kernel_fn exact_fn(const KernelChoice &k)
{
    if (k.ckpt) {
        /* ring snapshots: CTA per pair, shared-memory rings, CIGAR wanted, single-piece global alignment */
        if (k.warp || !BT || k.gring || k.ef || k.p2) return nullptr;
        return wfa_exact_kernel<false, ASCII, true, RingS16, true>;
    }
    if (k.gring) return exact_mode<false, ASCII, BT, RingG32>(k);     /* large tier: CTA per pair, int32 rings in HBM */
    return k.warp ? exact_mode<true, ASCII, BT, RingS16>(k) : exact_mode<false, ASCII, BT, RingS16>(k);
}

kernel_fn wavefront_kernel(const KernelChoice &k, bool count_cells)
{
    if (k.org && (k.family != Family::Exact || k.ckpt)) return nullptr;    /* origins: the exact kernel's ends-free rings */
    switch (k.family) {
    case Family::Exact:
        if (k.ascii) return k.bt ? exact_fn<true, true>(k) : exact_fn<true, false>(k);
        return k.bt ? exact_fn<false, true>(k) : exact_fn<false, false>(k);
    case Family::Quad:
        if (k.bt && !k.ckpt) return nullptr;               /* with backtrace: ring snapshots only */
        if (count_cells)   /* instrumented build of the same kernel: counts the cells of every window */
            return k.bt ? wfa_quad_kernel<true, true> : wfa_quad_kernel<false, true>;
        return k.bt ? wfa_quad_kernel<true, false> : wfa_quad_kernel<false, false>;
    case Family::QuadG:
        if (!k.gring) return nullptr;
        /* three register budgets: <= 512 threads (107 registers), <= 768 (85), <= 1024 (64) */
        if (k.threads <= 512) return k.bt ? wfa_quadg_kernel<true, 512> : wfa_quadg_kernel<false, 512>;
        if (k.threads <= 768) return k.bt ? wfa_quadg_kernel<true, 768> : wfa_quadg_kernel<false, 768>;
        return k.bt ? wfa_quadg_kernel<true, 1024> : wfa_quadg_kernel<false, 1024>;
    case Family::Banded:
        if (k.ascii) return k.bt ? wfa_banded_kernel<true, true> : wfa_banded_kernel<true, false>;
        return k.bt ? wfa_banded_kernel<false, true> : wfa_banded_kernel<false, false>;
    case Family::BandQ:
        return k.bt ? wfa_bandq_kernel<true> : wfa_bandq_kernel<false>;
    }
    return nullptr;
}

} // namespace wfagpu
