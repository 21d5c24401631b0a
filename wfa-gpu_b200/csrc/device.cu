/*
 * device.cu -- per-GPU context behind the C-ABI of include/wfagpu_b200.h.
 *
 * Replaces the launch glue of the reference (lib/sequence_alignment.cu:31-470,
 * lib/sequence_packing.cu:96-116 and the device half of lib/align.cu:42-481):
 * buffers are grow-only and cached per device, nothing is memset per batch, the
 * snapshot / decision arenas are sized by the step table, rings and launch shape
 * are provisioned from the scores of the previous batch, pairs that outgrow the
 * provision or the budget are re-dispatched on the GPU with a budget picked from
 * their score bounds, and pairs with an 'N' run through the byte-compare kernels.
 * There is no CPU path.
 */
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "wfa_kernels.cuh"

using namespace wfagpu;

#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            fprintf(stderr, "[wfagpu] CUDA error %s at %s:%d: %s\n", cudaGetErrorName(e_),        \
                    __FILE__, __LINE__, cudaGetErrorString(e_));                                  \
            return -1;                                                                            \
        }                                                                                         \
    } while (0)

namespace {

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    int ensure(size_t n, bool keep = false, cudaStream_t s = 0)
    {
        if (n <= cap) return 0;
        /* geometric growth for small buffers only: a 40 GB arena that has to hold 41 GB must not become 60 GB */
        size_t ncap = (n * sizeof(T) > ((size_t)256 << 20)) ? n : std::max(n, cap + cap / 2);
        T *np = nullptr;
        if (!keep && p) {                      /* nothing to carry over: give the old buffer back first */
            cudaFree(p);
            p = nullptr;
            cap = 0;
        }
        CK(cudaMalloc(&np, ncap * sizeof(T)));
        if (keep && p && cap) CK(cudaMemcpyAsync(np, p, cap * sizeof(T), cudaMemcpyDeviceToDevice, s));
        if (keep) CK(cudaStreamSynchronize(s));
        if (p) cudaFree(p);
        p = np;
        cap = ncap;
        return 0;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

template <typename T>
struct PinBuf {
    T *p = nullptr;
    size_t cap = 0;
    int ensure(size_t n)
    {
        if (n <= cap) return 0;
        size_t ncap = std::max(n, cap + cap / 2);
        T *np = nullptr;
        CK(cudaMallocHost(&np, ncap * sizeof(T)));
        if (p) cudaFreeHost(p);
        p = np;
        cap = ncap;
        return 0;
    }
    void release()
    {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

/* WFAGPU_TRACE=1: host-side time stamps of a pass (where does the launching thread spend its time) */
struct HostTrace {
    bool on;
    std::chrono::steady_clock::time_point t0;
    char buf[512];
    int len = 0;
    HostTrace() : on(getenv("WFAGPU_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) { buf[0] = 0; }
    void mark(const char *what)
    {
        if (!on) return;
        const double us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
        len += snprintf(buf + len, sizeof(buf) - (size_t)len > 0 ? sizeof(buf) - (size_t)len : 0, " %s=%.0fus", what, us);
        if (len > (int)sizeof(buf) - 1) len = (int)sizeof(buf) - 1;
    }
    ~HostTrace() { if (on) fprintf(stderr, "[wfagpu trace]%s\n", buf); }
};

enum { CTR_QUEUE = 0, CTR_POOL = 1, CTR_RETRY = 2, CTR_ASCII = 3, CTR_TBQ = 4, CTR_BQ = 5, CTR_WORDS = 8 };

struct LaunchCfg {
    KernelChoice k;       /* the wavefront kernel: the occupancy questions and the launch ask with this value */
    int group_threads;   /* 32 = warp per pair */
    int groups_per_cta;
    int ctas;
    int stages;
    int n_cap;
    int row_stride, center;
    int seq_words;
    size_t smem;
    int A, E1, G;
    int E2;               /* gap-affine 2-piece: depth of the I2 / D2 rings (0: one piece) */
    bool quad_pairs;      /* wfa_quad_kernel: two scores per barrier interval, rings one row deeper */
    int ring_m, ring_g;   /* rows of the M ring / of the I and D rings */
    int win;              /* adaptive band: window width in diagonals (0: exact) */
};

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool wf_timed = false;             /* ev[6], ev[7] bracket the first pass's wavefront kernel */
    cudaEvent_t ev_tab = nullptr;      /* after the last upload of a host-built table (step table, snapshot offsets) */
    bool tab_inflight = false;
    std::vector<int32_t> bound_sorted; /* scratch of the bound-first provisioning */
    std::vector<uint32_t> bound_count;
    int first_steps = 0;               /* wavefront-step budget the first pass of this batch ran with (>= plan.max_steps) */
    DevBuf<char> ascii;
    DevBuf<uint32_t> packed;
    DevBuf<wfagpu_pair_t> pairs;
    DevBuf<uint32_t> order, retry[2], ascii_list;
    DevBuf<wfagpu_pair_out_t> out;
    DevBuf<uint32_t> pool;
    DevBuf<uint32_t> counters;
    DevBuf<unsigned long long> cells;
    DevBuf<uint4> arena;
    DevBuf<uint32_t> scratch;
    DevBuf<int32_t> band_lo;
    DevBuf<int32_t> gring;
    DevBuf<char> slots, text;
    DevBuf<wfagpu_cigar_ref_t> refs;
    DevBuf<unsigned long long> heads;
    PinBuf<char> h_ascii;              /* staging for callers whose sequence buffer is pageable */
    PinBuf<char> h_text;
    PinBuf<wfagpu_cigar_ref_t> h_refs;
    PinBuf<unsigned long long> h_heads;
    DevBuf<wfagpu_step_t> steps;
    DevBuf<int32_t> bound;             /* per pair: score upper bound for the pruning */
    DevBuf<uint32_t> ck_off;           /* arena offset of every ring snapshot (checkpointed traceback) */
    std::vector<uint64_t> h_ck_off;    /* [j] = units used by the snapshots of scores < j * period */
    PinBuf<uint32_t> h_ck32;
    PinBuf<int32_t> h_bound;           /* re-dispatch: bounds and the retry list on the host */
    PinBuf<uint32_t> h_retry;
    int ck_key[1] = {-1};              /* period the offsets were built for */
    PinBuf<wfagpu_pair_t> h_pairs;
    PinBuf<uint32_t> h_order;
    PinBuf<uint32_t> h_seed;           /* one word: the re-dispatch counter a first pass starts from */
    PinBuf<wfagpu_pair_out_t> h_out;
    PinBuf<uint32_t> h_pool;
    PinBuf<uint32_t> h_counters;
    PinBuf<unsigned long long> h_cells;
    PinBuf<wfagpu_step_t> h_steps;
    int tab_key[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
    int tab_d_end = 0;
    uint64_t tab_arena_units = 0;
    size_t n = 0;
    size_t ascii_bytes = 0;
    size_t packed_words = 0;
    uint32_t max_len = 0;
    uint32_t kt_max = 0;               /* largest |tlen - plen| of the batch */
    uint32_t minlen_max = 0;           /* largest min(plen, tlen) of the batch */
    /* ends-free batch (wfagpu_device_align_span(s) with a non-zero span for some pair) */
    bool ef = false;
    DevBuf<int4> spans;                /* per pair {pb, pe, tb, te}, each clamped to the sequence it applies to */
    PinBuf<int4> h_spans;
    int ef_w = 0;                      /* half width of the start row: max(pb, tb), at most the longest sequence */
    int ef_ext = 0;                    /* widest end of the target range: max(pe, te), likewise */
    bool plain = true;                 /* global single-piece batch (neither ends-free nor 2-piece): it reads and learns the
                                        * provisioning hint, runs the packed-SIMD kernels and ring snapshots */
    DevBuf<int2> ends;                 /* per pair {k_begin, k_end} */
    PinBuf<int2> h_ends;
    size_t budget_cache = 0;           /* arena budget from the last cudaMemGetInfo (0 = ask again) */
    wfagpu_plan_t plan{};
    wfagpu_batch_stats_t stats{};
    bool have_events = false;
    bool text_queued = false; /* cigar_text kernels already follow the last alignment pass */
    int last_d_end = 0;
    bool capped = false;      /* the first pass provisioned fewer diagonals than the budget allows */
};

} // namespace

struct wfagpu_device {
    int dev = 0;
    cudaDeviceProp prop{};
    Slot slots[2];
    bool count_cells = false;
    int force_threads = 0, force_stages = 0, force_ctas_per_sm = 0, force_warp = -1;
    bool no_ckpt = false, no_bound = false, force_bound = false, no_quad = false, no_quad_pairs = false, no_band_tb = false, no_prebound = false, no_bound_order = false, no_skip_open = false;
    int force_period = 0;
    int arena_mb = 0;
    /* largest score seen in the last batch, per penalty set: sizes the rings of the next first pass */
    int hint_dist = 0;
    double hint_mean = 0;              /* mean score of the finished pairs of that batch */
    int hint_key[4] = {-1, -1, -1, -1};   /* x, o, e, length class (log2 of the longest sequence) */
    bool use_hint = true;
    bool force_large = false;
    bool device_text = true;   /* WFAGPU_HOST_CIGAR=1 leaves the text to the host */
    bool leased = false;       /* handed out by wfagpu_device_open and not released yet */
    bool independent = false;  /* wfagpu_device_rescore in progress: do not learn hints from it */
    int quad_min = 256;        /* smallest ring half width that runs the four-diagonals-per-thread kernel */
    int hint_margin_pm = 83, hint_min_pm = 31;   /* provisioning margins over the last batch's largest score, per mille */
    int hint_lift_pm = 250;    /* the first pass may exceed the -e budget by this much when the last batch needed it (0 = never) */
    int max_steps_cap = 60000; /* most wavefront steps a pair may take (WFAGPU_MAX_STEPS_CAP lowers it: tests) */
};

/* Contexts are leased: wfagpu_device_open hands out an idle context of that GPU (or makes a new one), so two
 * host threads -- or two workers of one call on the same GPU ("0,0") -- never share streams, slots or staging
 * buffers; wfagpu_device_release returns it to the pool with its grown buffers.  Only the provisioning hint
 * (largest / mean score of the last batch per penalty set) is shared per GPU, under g_mu. */
struct DevShared {
    int dev = -1;
    int hint_dist = 0;
    double hint_mean = 0;
    int hint_key[4] = {-1, -1, -1, -1};
};
static std::mutex g_mu;
static std::vector<wfagpu_device *> g_devices;
static std::vector<DevShared> g_shared;

/* a hint learnt on 150 bp reads says nothing about 10 kbp reads: hints are only used within a length class */
static int length_class(uint32_t max_len)
{
    int c = 0;
    while (max_len > 1) { max_len >>= 1; ++c; }
    return c;
}

static DevShared &shared_of(int dev)          /* g_mu held */
{
    for (auto &h : g_shared) if (h.dev == dev) return h;
    DevShared h;
    h.dev = dev;
    g_shared.push_back(h);
    return g_shared.back();
}
static void pull_hint(wfagpu_device *d)
{
    std::lock_guard<std::mutex> lk(g_mu);
    const DevShared &h = shared_of(d->dev);
    d->hint_dist = d->use_hint ? h.hint_dist : 0;
    d->hint_mean = h.hint_mean;
    for (int i = 0; i < 4; ++i) d->hint_key[i] = h.hint_key[i];
}
static void push_hint(wfagpu_device *d)
{
    std::lock_guard<std::mutex> lk(g_mu);
    DevShared &h = shared_of(d->dev);
    h.hint_dist = d->hint_dist;
    h.hint_mean = d->hint_mean;
    for (int i = 0; i < 4; ++i) h.hint_key[i] = d->hint_key[i];
}

static int env_int(const char *name, int dflt)
{
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

extern "C" wfagpu_device_t *wfagpu_device_open(int dev)
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto *d : g_devices)
        if (d->dev == dev && !d->leased) {
            cudaSetDevice(dev);
            d->leased = true;
            return d;
        }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || dev < 0 || dev >= count) {
        fprintf(stderr, "[wfagpu] CUDA device %d is not available (%s); this library has no CPU fallback\n", dev,
                e != cudaSuccess ? cudaGetErrorString(e) : "out of range");
        return nullptr;
    }
    if (cudaSetDevice(dev) != cudaSuccess) return nullptr;
    wfagpu_device *d = new wfagpu_device();
    d->dev = dev;
    if (cudaGetDeviceProperties(&d->prop, dev) != cudaSuccess) {
        delete d;
        return nullptr;
    }
    if (d->prop.major < 10) {
        fprintf(stderr, "[wfagpu] device %d is sm_%d%d; this build carries sm_100a code only\n", dev, d->prop.major,
                d->prop.minor);
        delete d;
        return nullptr;
    }
    for (auto &s : d->slots) {
        if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete d;
            return nullptr;
        }
        for (auto &ev : s.ev) cudaEventCreate(&ev);
        cudaEventCreateWithFlags(&s.ev_tab, cudaEventDisableTiming);
    }
    d->count_cells = env_int("WFAGPU_COUNT_CELLS", 0) != 0;
    d->force_threads = env_int("WFAGPU_THREADS", 0);
    d->force_stages = env_int("WFAGPU_STAGES", 0);
    d->force_ctas_per_sm = env_int("WFAGPU_CTAS_PER_SM", 0);
    d->force_warp = env_int("WFAGPU_WARP_KERNEL", -1);
    d->no_ckpt = env_int("WFAGPU_NO_CKPT", 0) != 0;
    d->no_bound = env_int("WFAGPU_NO_BOUND", 0) != 0;
    d->no_quad = env_int("WFAGPU_NO_QUAD", 0) != 0;
    d->no_band_tb = env_int("WFAGPU_NO_BAND_TB", 0) != 0;
    d->no_prebound = env_int("WFAGPU_NO_PREBOUND", 0) != 0;
    d->no_bound_order = env_int("WFAGPU_NO_BOUND_ORDER", 0) != 0;
    d->no_skip_open = env_int("WFAGPU_NO_SKIP_OPEN", 0) != 0;
    /* two scores per barrier interval: measured equal to one (22.9 vs 22.8 ms per 8192 x 10 kbp pairs) because the deeper
     * rings cost the fifth resident CTA; opt-in */
    d->no_quad_pairs = env_int("WFAGPU_QUAD_PAIRS", 0) == 0;
    d->force_bound = env_int("WFAGPU_FORCE_BOUND", 0) != 0;
    d->arena_mb = env_int("WFAGPU_ARENA_MB", 0);
    d->force_period = env_int("WFAGPU_CK_PERIOD", 0);
    if (d->force_period != 7 && d->force_period != 15 && d->force_period != 31) d->force_period = 0;
    d->use_hint = env_int("WFAGPU_NO_HINT", 0) == 0;
    d->force_large = env_int("WFAGPU_FORCE_LARGE", 0) != 0;
    d->device_text = env_int("WFAGPU_HOST_CIGAR", 0) == 0;
    d->quad_min = std::max(1, env_int("WFAGPU_QUAD_MIN", 256));
    d->hint_margin_pm = std::max(0, env_int("WFAGPU_HINT_MARGIN_PM", 83));
    d->hint_min_pm = std::min(d->hint_margin_pm, std::max(0, env_int("WFAGPU_HINT_MIN_PM", 31)));
    d->hint_lift_pm = std::max(0, env_int("WFAGPU_HINT_LIFT_PM", 250));
    d->max_steps_cap = std::min(60000, std::max(16, env_int("WFAGPU_MAX_STEPS_CAP", 60000)));
    d->leased = true;
    g_devices.push_back(d);
    return d;
}

extern "C" void wfagpu_device_release(wfagpu_device_t *d)
{
    if (!d) return;
    std::lock_guard<std::mutex> lk(g_mu);
    d->leased = false;
}

extern "C" void wfagpu_device_close_all(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto *d : g_devices) {
        cudaSetDevice(d->dev);
        for (auto &s : d->slots) {
            if (s.stream) cudaStreamSynchronize(s.stream);
            s.ascii.release(); s.packed.release(); s.pairs.release(); s.order.release();
            s.retry[0].release(); s.retry[1].release(); s.ascii_list.release(); s.out.release();
            s.pool.release(); s.counters.release(); s.cells.release(); s.arena.release(); s.bound.release(); s.ck_off.release(); s.h_ck32.release(); s.h_bound.release(); s.h_retry.release();
            s.scratch.release(); s.steps.release(); s.band_lo.release(); s.gring.release(); s.slots.release(); s.text.release(); s.refs.release(); s.heads.release();
            s.h_text.release(); s.h_refs.release(); s.h_heads.release(); s.h_ascii.release();
            s.h_pairs.release(); s.h_order.release(); s.h_seed.release(); s.h_out.release(); s.h_pool.release();
            s.h_counters.release(); s.h_cells.release(); s.h_steps.release(); s.ends.release(); s.h_ends.release();
            s.spans.release(); s.h_spans.release();
            for (auto &ev : s.ev) if (ev) cudaEventDestroy(ev);
            if (s.ev_tab) cudaEventDestroy(s.ev_tab);
            if (s.stream) cudaStreamDestroy(s.stream);
        }
        delete d;
    }
    g_devices.clear();
    g_shared.clear();
}

extern "C" int wfagpu_device_sm_count(wfagpu_device_t *d) { return d ? d->prop.multiProcessorCount : 0; }

static inline uint32_t packed_words_for(uint32_t len) { return ((((len + 7u) >> 3) + 1u) + 3u) & ~3u; }

extern "C" int wfagpu_device_upload(wfagpu_device_t *d, int slot, const char *ascii, size_t ascii_bytes,
                                    const wfagpu_pair_t *pairs, size_t n)
{
    if (!d || slot < 0 || slot > 1) return -1;
    CK(cudaSetDevice(d->dev));
    Slot &s = d->slots[slot];
    s.n = n;
    s.ascii_bytes = ascii_bytes;
    memset(&s.stats, 0, sizeof(s.stats));
    if (n == 0) return 0;
    if (s.h_pairs.ensure(n) || s.h_order.ensure(n)) return -1;
    /* packed layout + longest-first schedule */
    size_t words = 0;
    uint32_t max_len = 0, kt_max = 0, minlen_max = 0;
    uint64_t min_sum = ~0ull, max_sum = 0;
    for (size_t i = 0; i < n; ++i) {
        wfagpu_pair_t p = pairs[i];
        const uint64_t sum = (uint64_t)p.plen + p.tlen;
        kt_max = std::max(kt_max, p.plen > p.tlen ? p.plen - p.tlen : p.tlen - p.plen);
        minlen_max = std::max(minlen_max, std::min(p.plen, p.tlen));
        min_sum = std::min(min_sum, sum);
        max_sum = std::max(max_sum, sum);
        p.p_word = (uint32_t)words;
        words += packed_words_for(p.plen);
        p.t_word = (uint32_t)words;
        words += packed_words_for(p.tlen);
        p.flags = 0;
        s.h_pairs.p[i] = p;
        s.h_order.p[i] = (uint32_t)i;
        max_len = std::max(max_len, std::max(p.plen, p.tlen));
    }
    if (words >= (1ull << 32)) {
        fprintf(stderr, "[wfagpu] batch too large for 32-bit packed offsets; use a smaller batch_size\n");
        return -1;
    }
    s.packed_words = words;
    s.max_len = max_len;
    s.kt_max = kt_max;
    s.minlen_max = minlen_max;
    if ((uint64_t)min_sum * 8 < (uint64_t)max_sum * 7) {
        /* longest first only pays when the lengths differ by more than ~12 %: for uniform
         * reads the queue order is irrelevant and the sort would dominate the host time */
        const wfagpu_pair_t *hp = s.h_pairs.p;
        std::stable_sort(s.h_order.p, s.h_order.p + n, [hp](uint32_t a, uint32_t b) {
            return (uint64_t)hp[a].plen + hp[a].tlen > (uint64_t)hp[b].plen + hp[b].tlen;
        });
    }
    if (s.ascii.ensure(ascii_bytes + 64) || s.packed.ensure(words + 16) || s.pairs.ensure(n) || s.order.ensure(n) ||
        s.retry[0].ensure(n) || s.retry[1].ensure(n) || s.ascii_list.ensure(n) || s.out.ensure(n) ||
        s.counters.ensure(CTR_WORDS) || s.h_counters.ensure(CTR_WORDS) || s.cells.ensure(1) || s.h_cells.ensure(1))
        return -1;
    CK(cudaEventRecord(s.ev[0], s.stream));
    CK(cudaMemcpyAsync(s.ascii.p, ascii, ascii_bytes, cudaMemcpyHostToDevice, s.stream));
    CK(cudaMemsetAsync(s.ascii.p + ascii_bytes, 0, 64, s.stream));
    CK(cudaMemcpyAsync(s.pairs.p, s.h_pairs.p, n * sizeof(wfagpu_pair_t), cudaMemcpyHostToDevice, s.stream));
    CK(cudaMemcpyAsync(s.order.p, s.h_order.p, n * sizeof(uint32_t), cudaMemcpyHostToDevice, s.stream));
    CK(cudaEventRecord(s.ev[1], s.stream));
    s.stats.h2d_bytes += ascii_bytes + n * (sizeof(wfagpu_pair_t) + sizeof(uint32_t));
    s.have_events = true;
    return 0;
}

/* Ring depths of a plan: M (A, also the guard width G), I / D (E1), I2 / D2 of a 2-piece plan (E2; 0 for one piece). */
struct RingDepths {
    int A, E1, E2;
};
static RingDepths ring_depths(const wfagpu_plan_t &plan)
{
    const bool p2 = plan.e2 > 0;
    return {std::max(std::max(plan.o + plan.e, plan.x), p2 ? plan.o2 + plan.e2 : 0) + 1, plan.e + 1, p2 ? plan.e2 + 1 : 0};
}

/* Ring row geometry for a half width `ncap` and guard width G.  Aligned rows (snapshots copy 16-byte units, the quad
 * kernels load 8 or 16 bytes): diagonal 0 sits on an 8-element boundary and a row has 8 spare cells on both sides. */
static int ring_center(int ncap, int G, bool aligned) { return aligned ? ((ncap + 2 * G + 8 + 7) & ~7) : ncap + 2 * G + 1; }
static int ring_stride(int ncap, int G, bool aligned)
{
    return aligned ? 2 * ring_center(ncap, G, true) : 2 * (ncap + 2 * G + 1) + 2;
}

static int occupancy(const KernelChoice &k, size_t smem) { return max_ctas_per_sm(wavefront_kernel(k), k.threads, smem); }

/* Large tier (long sequences, or rings that do not fit one CTA's shared memory even single-buffered): a CTA per pair,
 * int32 rings in global memory. */
static int choose_large_cfg(wfagpu_device *d, const Slot &s, int n_want, size_t n_items, LaunchCfg *c)
{
    KernelChoice &kc = c->k;
    kc.gring = true;
    c->groups_per_cta = 1;
    c->stages = 1;
    c->n_cap = n_want;
    /* packed pairs: four diagonals per thread with 128-bit loads (wfa_quadg_kernel): rows 16-byte aligned */
    const bool quad = !kc.ascii && !d->no_quad && s.plain;       /* ends-free, 2-piece: one diagonal per thread */
    kc.family = quad ? Family::QuadG : Family::Exact;
    c->row_stride = ring_stride(n_want, c->G, quad);
    c->center = ring_center(n_want, c->G, quad);
    c->smem = exact_smem_bytes(c->A, c->E1, 0, c->seq_words, 1, 1, quad);     /* sequences + control (+ schedule records) only */
    if (!kc.ascii && c->smem > d->prop.sharedMemPerBlockOptin) {
        fprintf(stderr, "[wfagpu] sequences of %u bases do not fit in shared memory; not supported yet\n", s.max_len);
        return -2;
    }
    int most;
    if (quad) {
        /* one CTA per SM -- 148 x 0.7 MB of rings stay resident in the 126 MB L2 (two per SM: 681 instead of 902 pairs/s
         * at 50 kbp / 15 %); measured on B200, 592 pairs: 512 threads 1030, 768 1077, 1024 (64 registers) 1098 pairs/s */
        c->group_threads = d->force_threads ? d->force_threads : (n_want >= 2048 ? 1024 : (n_want >= 512 ? 512 : 256));
        most = 1;
    } else {
        /* wide wavefronts (50 kbp / 15 %: ~10 k diagonals per score) keep 1024 threads busy: 581 vs 416
         * pairs/s against 512 threads on B200 */
        c->group_threads = d->force_threads ? d->force_threads : (n_want >= 2048 ? 1024 : 512);
        most = 2;
    }
    kc.threads = c->group_threads;
    int occ = occupancy(kc, c->smem);
    if (occ < 1) return -1;
    occ = std::min(occ, d->force_ctas_per_sm ? d->force_ctas_per_sm : most);
    c->ctas = (int)std::max<size_t>(1, std::min<size_t>((size_t)occ * d->prop.multiProcessorCount, n_items));
    return 0;
}

/* Shared-memory / launch-shape policy of the exact kernels (replaces available_shared_mem_per_block and
 * the <<<num_workers, tpb>>> choice of lib/sequence_alignment.cu:81-108,211-330).
 *
 * The wavefront rings live in shared memory, so their width decides how many CTAs
 * share an SM.  Measured on B200 (10 kbp / 5 %): 1 CTA x 1024 threads 62 k pairs/s,
 * 2 x 512 95 k, 3 x 384 109 k -- more, smaller CTAs hide the per-score barrier.
 * `n_want` is the half width the launch should be able to hold. */
static int choose_cfg(wfagpu_device *d, const Slot &s, const wfagpu_plan_t &plan, int n_want, int n_min, size_t n_items,
                      bool ascii, LaunchCfg *c)
{
    /* 2-piece: one diagonal per thread, decision bytes, no schedule records; two more rings of e2 + 1 rows.  Score-only
     * ends-free with coordinates: an origin row beside every ring row */
    const bool p2 = plan.e2 > 0, sched = !p2, bt = plan.with_cigar != 0;
    const RingDepths rd = ring_depths(plan);
    const int A = rd.A, E1 = rd.E1, G = A, E2 = rd.E2;
    const size_t smem_max = d->prop.sharedMemPerBlockOptin;        /* 227 KB on B200 */
    const size_t smem_sm = d->prop.sharedMemPerMultiprocessor;     /* 228 KB */
    const int seq_words = (int)packed_words_for(s.max_len);
    c->A = A; c->E1 = E1; c->G = G; c->E2 = E2; c->seq_words = seq_words;
    c->ring_m = A; c->ring_g = E1;
    KernelChoice &kc = c->k;
    kc.ascii = ascii; kc.bt = bt; kc.ef = s.ef; kc.p2 = p2; kc.org = s.ef && !bt && plan.with_ends;
    n_want = std::max(1, n_want);
    if (d->force_large || s.max_len >= (1u << 15) ||
        exact_smem_bytes(A, E1, ring_stride(n_want, G, false), seq_words, 1, 1, sched, E2, kc.org) > smem_max)
        return choose_large_cfg(d, s, n_want, n_items, c);
    bool warp = (ring_stride(n_want, G, false) <= 400) && s.max_len <= 1024;
    if (d->force_warp >= 0) warp = d->force_warp != 0;

    if (warp) {
        c->group_threads = 32;
        c->groups_per_cta = 8;
        c->stages = 2;
        c->n_cap = n_want;
        c->row_stride = ring_stride(c->n_cap, G, false);
        c->center = ring_center(c->n_cap, G, false);
        c->smem = exact_smem_bytes(A, E1, c->row_stride, seq_words, c->groups_per_cta, c->stages, false, E2, kc.org);
        while (c->smem > smem_max && c->groups_per_cta > 1) {
            c->groups_per_cta >>= 1;
            c->smem = exact_smem_bytes(A, E1, c->row_stride, seq_words, c->groups_per_cta, c->stages, false, E2, kc.org);
        }
        if (c->smem > smem_max) warp = false;
    }
    if (!warp) {
        c->groups_per_cta = 1;
        kc.ckpt = bt && !d->no_ckpt && s.plain;     /* ends-free, 2-piece: decision bytes */
        /* packed pairs on shared-memory rings run four diagonals per thread (with backtrace: snapshots only) */
        /* (measured on B200: 1 kbp / 10 %, ring half width 196: 9.5 ms per 50 k pairs with one diagonal per thread and 16 CTAs per
         * SM against 11.0 ms; from a half width of ~300 on the four-diagonal kernel wins) */
        const bool quad = !ascii && !d->no_quad && s.plain && (!bt || kc.ckpt) && n_want >= d->quad_min;
        kc.family = quad ? Family::Quad : Family::Exact;
        /* two scores per barrier: score d + 1 must not read the extended M of score d (x >= 2, o + e >= 2) and takes
         * its extend sources from registers (e == 1); costs one more row per ring */
        c->quad_pairs = quad && !d->no_quad_pairs && plan.x >= 2 && plan.o + plan.e >= 2 && plan.e == 1;
        const bool ck = kc.ckpt || quad;       /* aligned row geometry */
        auto rs = [&](int ncap) { return ring_stride(ncap, G, ck); };
        const int RA = A + (c->quad_pairs ? 1 : 0), RE = E1 + (c->quad_pairs ? 1 : 0);
        c->ring_m = RA; c->ring_g = RE;
        int best_k = 0, stages = 1, n_cap = n_want;
        size_t smem = 0;
        /* CTA size follows the average width of the pruned wavefront (~ n_want): a quarter of it, 64..192
         * threads, and as many CTAs per SM as give ~960 threads (measured on B200: 10 kbp / 5 % is flat from
         * 128 to 192 threads at 5 CTAs; 1 kbp / 10 % runs 17.2 ms with 6 x 160 and 13.1 ms with 15 x 64) */
        const int t_pref = std::min(192, std::max(64, (((n_want + 3) / 4) + 31) & ~31));
        const int kmax = d->force_ctas_per_sm ? d->force_ctas_per_sm : std::min(16, std::max(1, 960 / t_pref));
        /* n_min <= n_want: the rings may be provisioned below n_want (down to n_min) when that buys
         * another resident CTA -- the few pairs that then outgrow them are re-dispatched */
        n_min = std::max(1, std::min(n_min, n_want));
        auto occ_at = [&](int threads, size_t bytes) {
            KernelChoice probe = kc;
            probe.threads = threads;
            return occupancy(probe, bytes);
        };
        /* do k CTAs of the smallest shape really fit with this much dynamic shared memory?  The arithmetic budget below is
         * a first filter; the runtime's occupancy calculator decides (allocation granularity: a ring 6 diagonals wider than
         * the arithmetic allowed cost rank 3 of an 8-GPU run its fifth CTA per SM, 33.4 instead of 29.2 ms per step) */
        auto fits = [&](int k, size_t bytes, size_t budget) { return bytes <= budget && occ_at(64, bytes) >= k; };
        for (int k = kmax; k >= 1 && !best_k; --k) {
            /* every resident CTA also reserves 1 KB of system shared memory */
            const size_t budget = std::min(smem_max, smem_sm / k - 1024);
            for (int st = 2; st >= 1; --st) {
                if (d->force_stages && st != d->force_stages) continue;
                if (!fits(k, exact_smem_bytes(RA, RE, rs(n_min), seq_words, 1, st, sched, E2, kc.org), budget)) continue;
                int lo = n_min, hi = n_want;             /* widest rings that still fit k CTAs */
                while (lo < hi) {
                    const int mid = (lo + hi + 1) / 2;
                    if (fits(k, exact_smem_bytes(RA, RE, rs(mid), seq_words, 1, st, sched, E2, kc.org), budget)) lo = mid; else hi = mid - 1;
                }
                best_k = k; stages = st; n_cap = lo;
                smem = exact_smem_bytes(RA, RE, rs(n_cap), seq_words, 1, st, sched, E2, kc.org);
                break;
            }
        }
        if (!best_k) {
            /* does not fit even alone: hold as many diagonals as one CTA can */
            stages = 1;
            const size_t fixed = exact_smem_bytes(RA, RE, 0, seq_words, 1, stages, sched, E2, kc.org);
            const int rows_q = (RA + 2 * RE + 2 * E2) * (kc.org ? 2 : 1);
            if (fixed + (size_t)rows_q * rs(1) * 2 > smem_max) return -2;   /* the sequences alone do not fit */
            n_cap = (int)((smem_max - fixed - 64) / ((size_t)rows_q * 4)) - 2 * G - (ck ? 16 : 2);
            if (n_cap < 1) return -2;
            smem = exact_smem_bytes(RA, RE, rs(n_cap), seq_words, 1, stages, sched, E2, kc.org);
            best_k = 1;
        }
        c->stages = stages;
        c->n_cap = n_cap;
        c->row_stride = rs(n_cap);
        c->center = ring_center(n_cap, G, ck);
        c->smem = smem;
        /* about 1152 threads per SM in total, never more threads than half the widest wavefront */
        /* (measured on B200: 3 x 384, 5 x 192 -- the per-score overhead is paid per warp) */
        int t = best_k == 1 ? 1024 : (best_k == 2 ? 512 : (best_k == 3 ? 384 : ((960 / best_k) / 32) * 32));
        const int width = 2 * n_cap + 1;
        if (quad) {
            /* a thread covers four diagonals per trip: one to two trips over the average window (~ n_cap);
             * the kernel needs ~80 registers: never so many threads that the registers cost a resident CTA */
            t = std::min(std::min(t, 512), std::max(64, ((n_cap / 6) + 31) & ~31));
            while (t > 64 && !d->force_threads && occ_at(t, smem) < best_k) t -= 32;
        } else {
            while (t > 64 && t * 2 > width) t -= 32;
        }
        t = std::max(64, t);
        if (d->force_threads) t = d->force_threads;
        c->group_threads = t;
    }
    kc.warp = c->group_threads == 32;     /* 32 threads per group run the warp kernel, also when WFAGPU_THREADS=32 */
    kc.threads = kc.warp ? 32 * c->groups_per_cta : c->group_threads;
    int occ = occupancy(kc, c->smem);
    if (occ < 1) {
        fprintf(stderr, "[wfagpu] kernel configuration does not fit (threads=%d smem=%zu)\n", kc.threads, c->smem);
        return -1;
    }
    if (d->force_ctas_per_sm) occ = std::min(occ, d->force_ctas_per_sm);
    size_t ctas = (size_t)occ * d->prop.multiProcessorCount;
    const size_t need = (n_items + c->groups_per_cta - 1) / c->groups_per_cta;
    c->ctas = (int)std::max<size_t>(1, std::min(ctas, need));
    return 0;
}

/* Launch shape of the adaptive band: window = the reference's threads_per_block (lib/sequence_alignment.cu:270-277). */
static int choose_band_cfg(wfagpu_device *d, const Slot &s, const wfagpu_plan_t &plan, size_t n_items, bool ascii,
                           LaunchCfg *c)
{
    const int win = plan.band_width > 0 ? plan.band_width : 512;
    const int d_full = s.tab_d_end;
    int n_full = 0;
    for (int dd = d_full - 1; dd >= 0 && dd >= d_full - 4; --dd) n_full = std::max(n_full, (int)s.h_steps.p[dd].n);
    c->win = win;
    c->A = ring_depths(plan).A; c->E1 = plan.e + 1; c->G = c->A;
    c->seq_words = (int)packed_words_for(s.max_len);
    c->groups_per_cta = 1;
    /* a few diagonals per thread: the per-score overhead (window bookkeeping, barrier) is paid
     * per thread, and small CTAs let more pairs share an SM (measured on B200, W = 512:
     * 512 threads 114 k, 256 threads 165 k, 128 threads 189 k pairs/s at 10 kbp / 5 %) */
    c->group_threads = std::min(1024, std::max(64, ((win / 4) + 31) & ~31));
    /* packed pairs: four diagonals per thread (wfa_bandq_kernel), one quad per thread and score */
    const bool quad = !ascii && !d->no_quad;
    c->k.family = quad ? Family::BandQ : Family::Banded;
    c->k.ascii = ascii;
    c->k.bt = plan.with_cigar != 0;
    /* a window spans win / 4 + 1 quads: two trips of half of them (measured on B200, W = 512, 10 kbp / 5 %:
     * 64 threads 32.5 ms, 96 threads 31.4 ms, 128 threads 33.0 ms per 8192 pairs end to end) */
    if (quad) c->group_threads = std::min(512, std::max(64, (((win / 4 + 2) / 2) + 31) & ~31));
    if (d->force_threads) c->group_threads = d->force_threads;
    auto band_smem = [&](int stages) {
        return quad ? bandq_smem_bytes(c->A, win, c->seq_words, stages) : banded_smem_bytes(c->A, win, c->seq_words, stages);
    };
    c->stages = 2;
    c->smem = band_smem(c->stages);
    if (c->smem > d->prop.sharedMemPerBlockOptin) {
        c->stages = 1;
        c->smem = band_smem(c->stages);
    }
    if (c->smem > d->prop.sharedMemPerBlockOptin) {
        fprintf(stderr, "[wfagpu] band of %d diagonals does not fit in shared memory\n", win);
        return -2;
    }
    c->n_cap = n_full; c->row_stride = win; c->center = 0;
    c->k.threads = c->group_threads;
    const int occ = occupancy(c->k, c->smem);
    if (occ < 1) return -1;
    c->ctas = (int)std::max<size_t>(1, std::min<size_t>((size_t)occ * d->prop.multiProcessorCount, n_items));
    return 0;
}

/* Remember the largest score of the batch whose results sit in s.h_out: the next first
 * pass with the same penalties provisions its rings for that (plus a margin). */
static void learn_hint(wfagpu_device *d, Slot &s, size_t n)
{
    int dmax = 0;
    double sum = 0;
    size_t cnt = 0;
    for (size_t i = 0; i < n; ++i)
        if (s.h_out.p[i].status & WFAGPU_ST_FINISHED) {
            dmax = std::max(dmax, s.h_out.p[i].distance);
            sum += s.h_out.p[i].distance;
            ++cnt;
        }
    d->hint_dist = d->use_hint ? dmax : 0;
    d->hint_mean = cnt ? sum / (double)cnt : 0;
    d->hint_key[0] = s.plan.x; d->hint_key[1] = s.plan.o; d->hint_key[2] = s.plan.e; d->hint_key[3] = length_class(s.max_len);
    push_hint(d);
}

/* the hint was learnt on a batch like this one: exact alignment, same penalties, same length class */
static bool hint_applies(const wfagpu_device *d, const Slot &s, const wfagpu_plan_t &plan)
{
    return plan.band <= 0 && d->hint_dist > 0 && d->hint_key[0] == plan.x && d->hint_key[1] == plan.o &&
           d->hint_key[2] == plan.e && d->hint_key[3] == length_class(s.max_len);
}

/* the hint's largest score plus `pm` per mille plus `k` */
static long long hint_plus(const wfagpu_device *d, int pm, int k)
{
    return (long long)d->hint_dist + (long long)d->hint_dist * pm / 1000 + k;
}

/* Does bounding every pair pay?  With D = d_end - 1 and a typical score m (the hint's mean score, or D / 2 when `m_hint`
 * is 0), the launch bound leaves cells(D/m) * m^2 cells per pair (cells(r) = r^2/4 + (1.5r - 1)(1 - r/2), 1 from r = 2 on),
 * the pair's own bound 0.5 * m^2; the bound pass costs ~32 cells per score at ~3x the cost per cell (measured on B200:
 * ~240 against ~2.75 warp instructions). */
static bool bound_pays(int d_end, double m_hint)
{
    const double m = m_hint > 0 ? m_hint : 0.5 * (d_end - 1);
    const double r = std::min(2.0, std::max(1.0, (d_end - 1) / std::max(1.0, m)));
    const double cells = r * r / 4 + (1.5 * r - 1) * (1 - r / 2);
    return (cells - 0.5) * m > 130.0;
}

/* The host-built tables are uploaded from pinned memory that the next pass rewrites.  Waiting for the last such upload
 * (an event) is enough; waiting for the whole stream would also wait for the chunk's own sequence upload and pack, which
 * a first pass has just queued (0.5 ms per 12500 x 1 kbp chunk whenever first pass and re-dispatch budgets alternate). */
static int tables_idle(Slot &s)
{
    if (!s.tab_inflight) return 0;
    if (s.ev_tab) CK(cudaEventSynchronize(s.ev_tab)); else CK(cudaStreamSynchronize(s.stream));
    s.tab_inflight = false;
    return 0;
}
static int tables_sent(Slot &s)
{
    if (s.ev_tab) CK(cudaEventRecord(s.ev_tab, s.stream));
    s.tab_inflight = true;
    return 0;
}

/* Ring-snapshot layout of the checkpointed traceback for period P: snapshot j (score j * P) holds
 * (A-1) + 2e rows of the 16-byte units that cover [-n, n] at that score.  h_ck_off[j] = units used
 * by the snapshots before j. */
static int ensure_ck_table(Slot &s, const wfagpu_plan_t &plan, int period)
{
    if (s.ck_key[0] == period) return 0;
    const int de = s.tab_d_end;
    const uint64_t rows_ck = (uint64_t)(ring_depths(plan).A - 1 + 2 * plan.e);
    const int n_ck = (de - 1) / period + 2;
    s.h_ck_off.assign((size_t)n_ck + 1, 0);
    if (s.h_ck32.ensure((size_t)n_ck + 1)) return -1;
    if (tables_idle(s)) return -1;            /* an earlier pass may still be reading the pinned copy */
    uint64_t acc = 0;
    s.h_ck32.p[0] = 0;
    for (int j = 1; j <= n_ck; ++j) {
        s.h_ck_off[j] = acc;
        s.h_ck32.p[j] = (uint32_t)std::min<uint64_t>(acc, 0xffffffffu);
        const long long dj = (long long)j * period;
        if (dj < de) {
            const int n = s.h_steps.p[dj].n;
            acc += rows_ck * (uint64_t)((((n + 7) & ~7) + ((n + 8) & ~7)) >> 3);
        }
    }
    if (s.ck_off.ensure((size_t)n_ck + 1)) return -1;
    CK(cudaMemcpyAsync(s.ck_off.p, s.h_ck32.p, ((size_t)n_ck + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, s.stream));
    if (tables_sent(s)) return -1;
    s.ck_key[0] = period;
    return 0;
}

/* Step table for a budget of `max_steps` wavefront steps (cached per slot; host copy in s.h_steps). */
static int ensure_step_table(Slot &s, const wfagpu_plan_t &plan, int max_steps)
{
    const bool p2 = plan.e2 > 0;
    const int widest = ring_depths(plan).A - 1;
    const int max_dist = std::min<long long>((long long)max_steps * (widest + 1) + 16, 1 << 30);
    const int tab_win = plan.band > 0 ? (plan.band_width > 0 ? plan.band_width : 512) : 0;
    const int extra = s.ef ? s.ef_w : 0;   /* ends-free: the start row widens every score's range */
    const int o2 = p2 ? plan.o2 : 0, e2 = p2 ? plan.e2 : 0;
    if (s.tab_key[0] == plan.x && s.tab_key[1] == plan.o && s.tab_key[2] == plan.e && s.tab_key[3] == max_steps &&
        s.tab_key[4] == tab_win && s.tab_key[5] == extra && s.tab_key[6] == o2 && s.tab_key[7] == e2)
        return 0;
    if (s.h_steps.ensure((size_t)max_dist + 1)) return -1;
    if (tables_idle(s)) return -1;        /* a previous pass may still be reading the pinned table */
    uint64_t units = 0;
    const int de = p2 ? wfagpu_build_step_table_affine2p(plan.x, plan.o, plan.e, o2, e2, max_steps, max_dist, s.h_steps.p, &units)
                 : extra ? wfagpu_build_step_table_span(plan.x, plan.o, plan.e, max_steps, max_dist, extra, s.h_steps.p, &units)
                         : wfagpu_build_step_table(plan.x, plan.o, plan.e, max_steps, max_dist, tab_win, s.h_steps.p, &units);
    if (de < 1) return -1;
    if (s.steps.ensure((size_t)de + 1)) return -1;
    CK(cudaMemcpyAsync(s.steps.p, s.h_steps.p, (size_t)de * sizeof(wfagpu_step_t), cudaMemcpyHostToDevice, s.stream));
    if (tables_sent(s)) return -1;
    s.tab_key[0] = plan.x; s.tab_key[1] = plan.o; s.tab_key[2] = plan.e; s.tab_key[3] = max_steps; s.tab_key[4] = tab_win;
    s.tab_key[5] = extra; s.tab_key[6] = o2; s.tab_key[7] = e2;
    s.tab_d_end = de;
    s.tab_arena_units = units;
    s.ck_key[0] = -1;     /* snapshot offsets follow the table */
    return 0;
}

/* Score upper bounds only (wfa_bound_kernel) for `n_items` entries of `order_dev`, with a budget of `max_steps`, queued for the
 * host: s.h_bound (indexed by pair) holds them after the next stream sync.  The first pass sizes its rings from them; the
 * re-dispatch loop picks a budget that is enough in one go and prunes that pass per pair.  -2: the bound kernel does not serve
 * these penalties.  Leaves the step table of `max_steps` cached. */
static int bounds_to_host(wfagpu_device *d, Slot &s, const wfagpu_plan_t &plan, int max_steps, const uint32_t *order_dev,
                          size_t n_items)
{
    if (plan.e2 > 0) return -2;           /* the bound kernel and its step table are single-piece */
    if (ensure_step_table(s, plan, max_steps)) return -1;
    if (s.bound.ensure(s.n + 1)) return -1;
    KernelParams kp{};
    kp.packed = s.packed.p;
    kp.pairs = s.pairs.p;
    kp.order = order_dev;
    kp.n_items = (uint32_t)n_items;
    kp.steps = s.steps.p;
    kp.d_end = s.tab_d_end;
    kp.x = plan.x; kp.o = plan.o; kp.e = plan.e;
    kp.A = ring_depths(plan).A;
    kp.E1 = plan.e + 1;
    kp.bound = s.bound.p;
    kp.bound_queue = s.counters.p + CTR_BQ;
    constexpr int kWarps = 8;
    const int occ = bound_max_ctas_per_sm(kp.A, kp.E1, kWarps);
    if (occ < 1) return -2;
    CK(cudaMemsetAsync(s.counters.p + CTR_BQ, 0, sizeof(uint32_t), s.stream));
    const int ctas = (int)std::min<size_t>((size_t)occ * d->prop.multiProcessorCount, (n_items + kWarps - 1) / kWarps);
    cudaError_t e = launch_bound(kp, std::max(1, ctas), kWarps, s.stream);
    if (e != cudaSuccess) {
        fprintf(stderr, "[wfagpu] bound kernel launch failed: %s\n", cudaGetErrorString(e));
        return -1;
    }
    s.stats.launches += 1;
    if (s.h_bound.ensure(s.n + 1)) return -1;
    CK(cudaMemcpyAsync(s.h_bound.p, s.bound.p, s.n * sizeof(int32_t), cudaMemcpyDeviceToHost, s.stream));
    return 0;
}

/* What one pass aligns. */
struct PassRequest {
    const uint32_t *order;      /* device list of pair indices */
    size_t n_items;             /* entries of `order` this pass aligns */
    uint32_t *retry;            /* device list the pass appends the pairs it does not finish to */
    int max_steps;              /* wavefront-step budget */
    bool ascii = false;         /* byte-compare kernels on the ASCII copy (pairs with non-ACGT bytes) */
    bool first_pass = false;    /* the batch's first pass: hints, bound pre-pass, wavefront timing, launch-shape stats */
    bool have_bounds = false;   /* s.bound already holds the bounds of these pairs */
    size_t n_seed = 0;          /* bound pre-pass: entries after the first n_items that skip this pass (straight to `retry`) */
};

/* Scores a pass provisions for. */
struct Scores {
    int d_full = 0;             /* the full budget: the step table's d_end */
    int d_reach = 0;            /* scores beyond this cannot occur in this batch */
    int d_want = 0;             /* scores the rings are provisioned for */
    bool hinted = false;        /* d_want comes from the hint */
    int d_p99 = 0;              /* 99 % of the bounded pairs finish below this score (0 = unknown) */
    int n_want = 0;             /* exact: ring half width for d_want */
};

/* Ring half width for scores below d_end.  The kernel prunes every cell that cannot reach the target diagonal within
 * d_end - 1 (score-bound pruning), so the rings only have to hold max_d min(n_d, kt_max + (d_end - 1 - d) / e). */
static int n_need(const Slot &s, const wfagpu_plan_t &plan, int d_end)
{
    const wfagpu_step_t *tab = s.h_steps.p;
    const int pen_e = plan.e2 > 0 ? std::min(plan.e, plan.e2) : plan.e;     /* 2-piece: the pruning's min(e1, e2) */
    const long long kt_max = s.kt_max;
    /* n_d grows, kt + (Dmax - d) / e shrinks: the largest min sits where they cross.  A global pair with |kt| > Dmax / e
     * cannot finish; an ends-free one can (the start row and the target range may meet at no cost), and its window
     * reaches max(pe, te) beyond kt: no clamp, n_d bounds it */
    const long long Dmax = d_end - 1;
    const long long ktm = s.ef ? kt_max + s.ef_ext : std::min<long long>(kt_max, Dmax / pen_e);
    int lo = 0, hi = d_end;                      /* first d with n_d >= ktm + (Dmax - d) / e */
    while (lo < hi) {
        const int mid = (lo + hi) / 2;
        if ((long long)tab[mid].n >= ktm + (Dmax - mid) / pen_e) hi = mid; else lo = mid + 1;
    }
    long long best = 1;
    for (int dd = std::max(0, lo - 2); dd < std::min(d_end, lo + 3); ++dd)
        best = std::max(best, std::min<long long>(tab[dd].n, ktm + (Dmax - dd) / pen_e));
    return (int)best;
}

/* Stage 1: the full budget, or (first pass only) what recent batches with these penalties needed plus a margin -- pairs
 * that outgrow it are re-dispatched.  No pair of the batch can score more than substitutions all along the shorter
 * sequence plus one gap for the length difference: a generous -e (or a stale hint) does not widen the rings. */
static Scores provision_scores(const wfagpu_device *d, const Slot &s, const wfagpu_plan_t &plan, bool first_pass)
{
    Scores sc;
    sc.d_full = s.tab_d_end;
    sc.d_want = sc.d_full;
    if (first_pass && hint_applies(d, s, plan)) {
        sc.d_want = (int)std::min<long long>(hint_plus(d, d->hint_margin_pm, 8), sc.d_full - 1) + 1;
        sc.hinted = sc.d_want < sc.d_full;
    }
    sc.d_reach = sc.d_full;
    if (plan.band <= 0) {
        long long cap = (long long)plan.x * s.minlen_max + plan.o + (long long)plan.e * s.kt_max + 2;
        if (plan.e2 > 0) cap = std::min(cap, (long long)plan.x * s.minlen_max + plan.o2 + (long long)plan.e2 * s.kt_max + 2);   /* the cheaper piece */
        if (cap < sc.d_reach) sc.d_reach = (int)std::max<long long>(cap, 2);
        if (sc.d_reach < sc.d_want) sc.d_want = sc.d_reach;
    }
    return sc;
}

/* Stage 2, the first pass of a packed exact batch where the per-pair score bounds pay (long reads): the bound kernel runs
 * first and its largest bound sizes the rings -- what this batch needs, not what the last one needed, so a first call, a
 * call without hints and a call after a batch of another kind all run at the speed of a well-hinted one.  Costs one host
 * round trip per pass (bounds back: 4 bytes per pair); the only stage that waits for the GPU. */
static int bound_prepass(wfagpu_device *d, Slot &s, const wfagpu_plan_t &plan, PassRequest &r, Scores &sc)
{
    if (!r.first_pass || r.have_bounds || plan.band > 0 || r.ascii || plan.e2 > 0 || d->no_bound || d->no_prebound ||
        r.n_items != s.n || bound_max_ctas_per_sm(ring_depths(plan).A, plan.e + 1, 8) < 1)   /* penalties whose rings fit the bound kernel */
        return 0;
    const int d_full = sc.d_full;
    bool pays = d->force_bound ||
                bound_pays(sc.d_want, (sc.d_want < d_full && d->hint_mean > 0 && d->hint_dist > 0) ? d->hint_mean : 0);
    if (!pays && sc.d_want < d_full && d->hint_dist > 0 && s.max_len >= 2000 && r.n_items >= 1024 && r.order == s.order.p) {
        /* a hint tight enough that bounding every pair does not pay: is it still true for this batch?  Bound the first
         * 128 pairs of the queue; if they already outgrow the hint (every pair would be re-dispatched) or stay far
         * below it (rings wider than needed), provision from this batch's own bounds after all */
        constexpr size_t kSample = 128;
        if (int rc = bounds_to_host(d, s, plan, r.max_steps, r.order, kSample)) return rc;
        CK(cudaStreamSynchronize(s.stream));
        long long smax = 0;
        for (size_t i = 0; i < kSample; ++i) {
            const uint32_t idx = s.h_order.p[i];
            if (idx < s.n) smax = std::max<long long>(smax, std::min<int32_t>(s.h_bound.p[idx], d_full));
        }
        const long long covered = hint_plus(d, d->hint_min_pm, 0);
        pays = smax > covered || smax * 13 < (long long)d->hint_dist * 10;
    }
    if (!pays) return 0;
    if (int rc = bounds_to_host(d, s, plan, r.max_steps, r.order, r.n_items)) return rc;
    CK(cudaStreamSynchronize(s.stream));
    std::vector<int32_t> &bv = s.bound_sorted;
    bv.clear();
    for (size_t i = 0; i < s.n; ++i)
        if (s.h_bound.p[i] < d_full - 1) bv.push_back(s.h_bound.p[i]);
    r.have_bounds = true;
    if (r.order == s.order.p && !d->no_bound_order) {
        /* longest first by the pair's own bound (work ~ bound^2): the queue's tail is made of the cheapest pairs
         * (counting sort, descending).  Pairs the bound pass could not bound within this budget go to the end of
         * the list and straight to the re-dispatch tier: their first pass would run to the end of the budget for
         * nothing (a pair flagged for the byte-compare kernel stays: the wavefront kernel routes it).
         * The order list was uploaded before the sync. */
        std::vector<uint32_t> &cnt = s.bound_count;
        cnt.assign((size_t)d_full + 2, 0u);
        auto key_of = [&](int32_t b) -> size_t {
            if (b == 0x7fffffff) return (size_t)d_full;              /* flagged: first */
            if (b >= d_full - 1) return (size_t)d_full + 1;          /* open: last (descending order below) */
            return (size_t)std::max(b, 0);
        };
        size_t n_open = 0;
        for (size_t i = 0; i < s.n; ++i) {
            const size_t k = key_of(s.h_bound.p[i]);
            cnt[k] += 1;
            n_open += (k == (size_t)d_full + 1);
        }
        uint32_t acc = 0;
        for (int b = d_full; b >= 0; --b) { const uint32_t c0 = cnt[(size_t)b]; cnt[(size_t)b] = acc; acc += c0; }
        cnt[(size_t)d_full + 1] = acc;
        for (size_t i = 0; i < s.n; ++i) s.h_order.p[cnt[key_of(s.h_bound.p[i])]++] = (uint32_t)i;
        CK(cudaMemcpyAsync(s.order.p, s.h_order.p, s.n * sizeof(uint32_t), cudaMemcpyHostToDevice, s.stream));
        if (n_open > 0 && !d->no_skip_open) {
            r.n_seed = n_open;
            r.n_items = s.n - n_open;
        }
    }
    if (!bv.empty()) {
        const size_t k99 = (bv.size() - 1) - (bv.size() - 1) / 100;
        std::nth_element(bv.begin(), bv.begin() + (long)k99, bv.end());
        const int b99 = bv[k99];
        const int bmax = *std::max_element(bv.begin() + (long)k99, bv.end());
        sc.d_want = std::min(d_full, bmax + 2);
        sc.d_want = std::min(sc.d_want, sc.d_reach);
        sc.d_p99 = std::min(sc.d_want, b99 + 2);
        sc.hinted = false;
    }
    return 0;
}

/* What a launch computes and where its backtrace state goes. */
struct Arenas {
    int d_end = 0;                /* scores 1 .. d_end - 1 may be computed */
    int period = 0;               /* ring-snapshot period (0: no snapshots) */
    bool band_tb = false;         /* adaptive band on packed pairs: decision rows walked by a traceback kernel after the launch */
    uint64_t arena_units = 0;     /* uint4 units per arena */
    size_t arenas = 0;            /* snapshots, band_tb: one per pair of a sub-launch; else one per resident group */
    size_t items_per_launch = 0;
    uint64_t gring_elems = 0;     /* large tier: ring elements per group */
    uint32_t scratch_words = 0, band_lo_words = 0;
};

/* Stage 4: the scores the launch can reach, the snapshot period, the arenas within a third of the free device memory, and
 * every buffer the launch writes. */
static int size_arenas(wfagpu_device *d, Slot &s, const wfagpu_plan_t &plan, const PassRequest &r, const Scores &sc,
                       LaunchCfg &c, Arenas &a, HostTrace &tr)
{
    const bool banded = plan.band > 0;
    const size_t n_items = r.n_items;
    /* scores this launch can reach and the decision units they need */
    a.d_end = banded ? sc.d_full : sc.d_want;
    uint64_t arena_units = s.tab_arena_units;
    if (!banded) {
        if (c.n_cap < sc.n_want) {
            int lo = 1, hi = sc.d_want;              /* largest d_end whose pruned wavefronts fit the rings */
            while (lo < hi) {
                const int mid = (lo + hi + 1) / 2;
                if (n_need(s, plan, mid) <= c.n_cap) lo = mid; else hi = mid - 1;
            }
            a.d_end = lo;
        }
        arena_units = a.d_end < sc.d_full ? s.h_steps.p[a.d_end].row_off : s.tab_arena_units;
    }

    /* memory budget of the arenas: a third of the free device memory.  cudaMemGetInfo takes 0.2 - 15 ms on a busy box and
     * would leave the GPU idle between the pack kernel and this pass: ask only when the answer can have changed (first use,
     * arena grew) */
    if (d->arena_mb > 0) {
        s.budget_cache = (size_t)d->arena_mb << 20;          /* WFAGPU_ARENA_MB: fixed budget (tests) */
    } else if (s.budget_cache == 0) {
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        s.budget_cache = std::max<size_t>((free_b + s.arena.cap * sizeof(uint4)) / 3, (size_t)64 << 20);
    }
    size_t arena_budget = s.budget_cache;
    tr.mark("meminfo");
    if (c.k.ckpt) {
        /* Snapshot period: the traceback recomputes ~ score * P cells per pair against ~ score^2 in
         * the forward pass, the snapshots take ~ 1/P of the cells: short periods for low scores,
         * longer ones when memory is tight. */
        const int d_expect = sc.hinted ? std::min(a.d_end, d->hint_dist + 1) : a.d_end;
        int period = d->force_period ? d->force_period : (d_expect >= 3000 ? 31 : 15);   /* measured on B200: shorter never wins */
        for (;;) {
            if (ensure_ck_table(s, plan, period)) return -1;
            arena_units = s.h_ck_off[(size_t)(a.d_end - 1) / period + 1];      /* snapshots of scores j * P < d_end */
            if (period >= 31 || d->force_period || (arena_units * sizeof(uint4) + 1) * n_items <= arena_budget) break;
            period = 2 * period + 1;
        }
        if (arena_units >= 0xffffffffull) { fprintf(stderr, "[wfagpu] snapshot arena exceeds 32-bit offsets\n"); return -1; }
        a.period = period;
    }

    if (!plan.with_cigar) arena_units = 0;
    a.arena_units = arena_units;
    /* adaptive band on packed pairs: decision rows per pair, walked by a traceback kernel after the launch */
    a.band_tb = banded && c.k.quad() && plan.with_cigar && !d->no_band_tb;
    const bool per_pair = c.k.ckpt || a.band_tb;
    /* keep the arenas within a third of the free device memory: fewer, not smaller, groups
     * (decision bytes: one arena per resident group; snapshots: one per pair of a sub-launch) */
    a.items_per_launch = n_items;
    for (int attempt = 0;; ++attempt) {
        const size_t budget = arena_budget;
        if (per_pair) {
            const size_t per_item = (size_t)arena_units * sizeof(uint4) + (a.band_tb ? ((size_t)a.d_end + 1) * sizeof(int32_t) : 0) + 1;
            a.items_per_launch = std::max<size_t>(1, std::min<size_t>(n_items, budget / per_item));
            c.ctas = (int)std::min<size_t>((size_t)c.ctas, a.items_per_launch);
        } else {
            const size_t per_group = (size_t)arena_units * sizeof(uint4) * (size_t)c.groups_per_cta + 1;
            const size_t max_ctas = std::max<size_t>(1, budget / per_group);
            if ((size_t)c.ctas > max_ctas) c.ctas = (int)max_ctas;
        }
        /* an arena that has to grow is checked against the memory that is free right now (the budget may date from an
         * emptier device: other slots, contexts and processes allocate too); the old arena is given back first */
        const size_t want = ((per_pair ? a.items_per_launch : (size_t)c.ctas * c.groups_per_cta) * arena_units + 1);
        if (want <= s.arena.cap || d->arena_mb > 0 || attempt >= 4) break;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); break; }
        const size_t avail = free_b + s.arena.cap * sizeof(uint4);
        const size_t spare = (size_t)2 << 30;                    /* text slots, op pool, staging of this pass */
        if (want * sizeof(uint4) + spare <= avail) break;
        arena_budget = std::max<size_t>((size_t)64 << 20, std::min(arena_budget / 2, avail > spare ? (avail - spare) / 2 : (size_t)0));
        s.budget_cache = arena_budget;
    }
    const size_t groups = (size_t)c.ctas * c.groups_per_cta;
    a.gring_elems = c.k.gring ? (uint64_t)(c.A + 2 * c.E1 + 2 * c.E2) * (c.k.org ? 2u : 1u) * (uint64_t)c.row_stride : 0;
    if (s.gring.ensure(groups * a.gring_elems + 1)) return -1;
    a.scratch_words = plan.with_cigar ? (uint32_t)((2 * (size_t)a.d_end + 31) / 16 + 2) : 1;
    a.arenas = per_pair ? a.items_per_launch : groups;
    if (a.arenas * arena_units + 1 > s.arena.cap) s.budget_cache = 0;      /* the arena grows: re-read the free memory next time */
    if (s.arena.ensure(a.arenas * arena_units + 1) || s.scratch.ensure(groups * a.scratch_words + 1)) return -1;
    a.band_lo_words = (banded && plan.with_cigar) ? (uint32_t)a.d_end + 1 : 0;
    if (s.band_lo.ensure((a.band_tb ? a.items_per_launch : groups) * (size_t)a.band_lo_words + 1)) return -1;
    /* op pool: worst case for this pass on top of what is already used */
    /* later passes run after read_counters(): the host copy of the pool head is current */
    const uint32_t pool_used = r.first_pass ? 0u : s.h_counters.p[CTR_POOL];
    const size_t pool_need = (size_t)pool_used + (plan.with_cigar ? n_items * (size_t)a.scratch_words : 0) + 16;
    if (pool_need >= (1ull << 32)) {
        fprintf(stderr, "[wfagpu] op pool exceeds 32-bit offsets; use a smaller batch_size\n");
        return -1;
    }
    if (s.pool.ensure(pool_need, true, s.stream)) return -1;
    tr.mark("buffers");
    return 0;
}

/* Stage 5: the retry list's seed, the kernel parameters, and the sub-launches (bound, wavefront and traceback kernels). */
static int enqueue_pass(wfagpu_device *d, Slot &s, const wfagpu_plan_t &plan, const PassRequest &r, const Scores &sc,
                        const LaunchCfg &c, const Arenas &a, HostTrace &tr)
{
    const bool banded = plan.band > 0;
    const size_t n_items = r.n_items;
    if (r.n_seed > 0) {
        /* the re-dispatch list starts with the pairs that skip this pass */
        if (s.h_seed.ensure(1)) return -1;
        s.h_seed.p[0] = (uint32_t)r.n_seed;
        CK(cudaMemcpyAsync(s.counters.p + CTR_RETRY, s.h_seed.p, sizeof(uint32_t), cudaMemcpyHostToDevice, s.stream));
        CK(cudaMemcpyAsync(r.retry, s.order.p + n_items, r.n_seed * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s.stream));
    } else {
        CK(cudaMemsetAsync(s.counters.p + CTR_RETRY, 0, sizeof(uint32_t), s.stream));
    }

    KernelParams kp{};
    kp.packed = s.packed.p;
    kp.ascii = s.ascii.p;
    kp.pairs = s.pairs.p;
    kp.order = r.order;
    kp.n_items = (uint32_t)n_items;
    kp.queue = s.counters.p + CTR_QUEUE;
    kp.tb_queue = s.counters.p + CTR_TBQ;
    kp.bound_queue = s.counters.p + CTR_BQ;
    /* per-pair bounds: first pass of the packed exact path only (a re-dispatched pair never depends on them), or the
     * bounds s.bound already holds (bounds_to_host) */
    bool use_bound = !banded && !r.ascii && plan.e2 <= 0 && (r.first_pass || r.have_bounds) && !d->no_bound;
    if (use_bound && !d->force_bound && !r.have_bounds) use_bound = bound_pays(a.d_end, sc.hinted ? d->hint_mean : 0);
    if (use_bound && s.bound.ensure(s.n + 1)) return -1;
    kp.bound = use_bound ? s.bound.p : nullptr;
    kp.steps = s.steps.p;
    kp.d_end = a.d_end;
    kp.n_cap = c.n_cap;
    kp.x = plan.x; kp.o = plan.o; kp.e = plan.e;
    kp.A = c.A; kp.E1 = c.E1; kp.G = c.G;
    kp.row_stride = c.row_stride;
    kp.center = c.center;
    kp.seq_words = c.seq_words;
    kp.with_bt = plan.with_cigar;
    kp.stages = c.stages;
    kp.quad_pairs = c.quad_pairs ? 1 : 0;
    kp.ring_m = c.ring_m; kp.ring_g = c.ring_g;
    kp.band = plan.band;
    kp.win = c.win;
    kp.band_lo = s.band_lo.p;
    kp.band_lo_words = a.band_lo_words;
    kp.band_tb = a.band_tb ? 1 : 0;
    kp.gring = c.k.gring ? s.gring.p : nullptr;
    kp.gring_elems = a.gring_elems;
    kp.arena = s.arena.p;
    kp.arena_units = a.arena_units;
    kp.ck_off = c.k.ckpt ? s.ck_off.p : nullptr;
    kp.ck_period = a.period;
    kp.ops_scratch = s.scratch.p;
    kp.ops_scratch_words = a.scratch_words;
    kp.ops_pool = s.pool.p;
    kp.ops_pool_head = s.counters.p + CTR_POOL;
    kp.ops_pool_words = (uint32_t)std::min<size_t>(s.pool.cap, 0xffffffffu);
    kp.out = s.out.p;
    kp.retry_list = r.retry;
    kp.retry_count = s.counters.p + CTR_RETRY;
    kp.ascii_list = s.ascii_list.p;
    kp.ascii_count = s.counters.p + CTR_ASCII;
    kp.cells = d->count_cells ? s.cells.p : nullptr;
    if (s.ef) {
        kp.spans = s.spans.p;
        kp.ends = s.ends.p;
    }
    if (plan.e2 > 0) { kp.o2 = plan.o2; kp.e2 = plan.e2; kp.E2 = c.E2; }
    if (env_int("WFAGPU_VERBOSE", 0)) {
        const bool quad = c.k.quad(), ckpt = c.k.ckpt;
        fprintf(stderr, "[wfagpu] pass: items=%zu max_steps=%d n_cap=%d d_end=%d group=%d x%d ctas=%d stages=%d smem=%zu ascii=%d band=%d tier=%s period=%d arena=%.1f MB\n",
                n_items, r.max_steps, c.n_cap, a.d_end, c.group_threads, c.groups_per_cta, c.ctas, c.stages, c.smem,
                (int)r.ascii, c.win, c.k.gring ? (quad ? "global-int32x4" : "global-int32") : (quad ? (c.quad_pairs ? (ckpt ? "smem-int16x4x2+ckpt" : "smem-int16x4x2") : (ckpt ? "smem-int16x4+ckpt" : "smem-int16x4")) : (ckpt ? "smem-int16+ckpt" : "smem-int16")), a.period, a.arenas * a.arena_units * 16.0 / 1e6);
    }
    int tb_ctas = 0;
    constexpr int kTbWarps = 8;
    if (c.k.ckpt) {
        const int occ = traceback_max_ctas_per_sm(c.A, a.period, kTbWarps, r.ascii);
        if (occ < 1) { fprintf(stderr, "[wfagpu] traceback kernel does not fit\n"); return -1; }
        tb_ctas = occ * d->prop.multiProcessorCount;
    }
    int bound_ctas = 0;
    constexpr int kBoundWarps = 8;
    if (use_bound && !r.have_bounds) {
        const int occ = bound_max_ctas_per_sm(c.A, c.E1, kBoundWarps);
        if (occ < 1) kp.bound = nullptr; else bound_ctas = occ * d->prop.multiProcessorCount;
    }
    const kernel_fn wavefront = wavefront_kernel(c.k, d->count_cells);
    tr.mark("occ");
    for (size_t off = 0; off < n_items; off += a.items_per_launch) {
        const size_t cnt = std::min(a.items_per_launch, n_items - off);
        kp.order = r.order + off;
        kp.n_items = (uint32_t)cnt;
        if (kp.bound && !r.have_bounds) {
            CK(cudaMemsetAsync(s.counters.p + CTR_BQ, 0, sizeof(uint32_t), s.stream));
            const int ctas = (int)std::min<size_t>((size_t)bound_ctas, (cnt + kBoundWarps - 1) / kBoundWarps);
            cudaError_t eb = launch_bound(kp, ctas, kBoundWarps, s.stream);
            if (eb != cudaSuccess) {
                fprintf(stderr, "[wfagpu] bound kernel launch failed: %s\n", cudaGetErrorString(eb));
                return -1;
            }
            s.stats.launches += 1;
        }
        CK(cudaMemsetAsync(s.counters.p + CTR_QUEUE, 0, sizeof(uint32_t), s.stream));
        const bool time_it = r.first_pass && a.items_per_launch >= n_items && s.ev[6] && s.ev[7];
        if (time_it) CK(cudaEventRecord(s.ev[6], s.stream));
        /* the banded kernels always launch the full shape */
        const int ctas = banded ? c.ctas : (int)std::min<size_t>(c.ctas, cnt);
        cudaError_t e = launch(wavefront, kp, ctas, c.k.threads, c.smem, s.stream);
        if (e != cudaSuccess) {
            fprintf(stderr, "[wfagpu] alignment kernel launch failed: %s\n", cudaGetErrorString(e));
            return -1;
        }
        if (time_it) { CK(cudaEventRecord(s.ev[7], s.stream)); s.wf_timed = true; }
        tr.mark("fwd");
        s.stats.launches += 1;
        if (a.band_tb) {
            e = launch_band_traceback(kp, s.stream);
            if (e != cudaSuccess) {
                fprintf(stderr, "[wfagpu] band traceback kernel launch failed: %s\n", cudaGetErrorString(e));
                return -1;
            }
            s.stats.launches += 1;
        }
        if (c.k.ckpt) {
            /* ring snapshots -> 2-bit ops, a warp per pair */
            CK(cudaMemsetAsync(s.counters.p + CTR_TBQ, 0, sizeof(uint32_t), s.stream));
            const int ctas_tb = (int)std::min<size_t>((size_t)tb_ctas, (cnt + kTbWarps - 1) / kTbWarps);
            e = launch_traceback(kp, ctas_tb, kTbWarps, r.ascii, s.stream);
            if (e != cudaSuccess) {
                fprintf(stderr, "[wfagpu] traceback kernel launch failed: %s\n", cudaGetErrorString(e));
                return -1;
            }
            s.stats.launches += 1;
        }
    }
    tr.mark("tb");
    if (r.first_pass) {
        s.stats.n_cap = (uint32_t)c.n_cap;
        s.stats.cta_threads = (uint32_t)c.k.threads;
        s.stats.ctas = (uint32_t)c.ctas;
        s.stats.d_end = (uint32_t)a.d_end;
    }
    s.last_d_end = std::max(s.last_d_end, a.d_end);
    s.text_queued = false;
    return 0;
}

/* One pass over a request's pairs, in five stages: the scores to provision for, the bound pre-pass (first pass only), the
 * launch shape, the scores and arenas, the launches.  Returns < 0 on error, else 1 if the pass was capped: provisioned
 * for fewer scores than the budget and the lengths allow (the pairs it leaves over may only need wider rings), else 0. */
static int launch_pass(wfagpu_device *d, Slot &s, const wfagpu_plan_t &plan, PassRequest r)
{
    HostTrace tr;
    if (r.first_pass) {
        pull_hint(d);                        /* what the last batch on this GPU needed (any context) */
        if (!s.plain) { d->hint_dist = 0; d->hint_mean = 0; }   /* hints are learnt on global single-piece batches */
    }
    if (ensure_step_table(s, plan, r.max_steps)) return -1;
    Scores sc = provision_scores(d, s, plan, r.first_pass);
    if (int rc = bound_prepass(d, s, plan, r, sc)) return rc;
    LaunchCfg c{};
    int rc;
    if (plan.band > 0) {
        rc = choose_band_cfg(d, s, plan, r.n_items, r.ascii, &c);
    } else {
        sc.n_want = n_need(s, plan, sc.d_want);
        /* with a hint, rings for hint + 3 % are enough for (almost) every pair; with bounds, rings for 99 % of the pairs
         * when that buys a resident CTA */
        int n_min = sc.n_want;
        if (sc.hinted)
            n_min = std::min(sc.n_want, n_need(s, plan, (int)std::min<long long>(hint_plus(d, d->hint_min_pm, 4), sc.d_full - 1) + 1));
        if (sc.d_p99 > 0) n_min = std::min(sc.n_want, n_need(s, plan, sc.d_p99));
        rc = choose_cfg(d, s, plan, sc.n_want, n_min, r.n_items, r.ascii, &c);
    }
    if (rc) return rc;
    tr.mark("cfg");
    Arenas a;
    if (size_arenas(d, s, plan, r, sc, c, a, tr) || enqueue_pass(d, s, plan, r, sc, c, a, tr)) return -1;
    return a.d_end < sc.d_reach ? 1 : 0;
}

/* CIGAR text on the device: queued right behind the alignment kernel so that it overlaps with
 * the host's work on the previous chunk; redone by download() if pairs had to be re-dispatched. */
static int enqueue_text(wfagpu_device *d, Slot &s, size_t n, int d_end_bound)
{
    (void)d;
    /* slack slots: 10 characters per op, at most 2 ops per score */
    const size_t slot_bytes = n * ((size_t)20 * (size_t)d_end_bound + 64) + 64;
    if (s.slots.ensure(slot_bytes) || s.text.ensure(slot_bytes) || s.refs.ensure(n) || s.heads.ensure(4) ||
        s.h_refs.ensure(n) || s.h_heads.ensure(4))
        return -1;
    CK(cudaMemsetAsync(s.heads.p, 0, 4 * sizeof(unsigned long long), s.stream));
    CigarParams cp{};
    cp.ascii = s.ascii.p;
    cp.pairs = s.pairs.p;
    cp.out = s.out.p;
    cp.ops_pool = s.pool.p;
    cp.n_pairs = (uint32_t)n;
    cp.slots = s.slots.p;
    cp.slot_bytes = slot_bytes;
    cp.slot_head = s.heads.p;
    cp.text = s.text.p;
    cp.text_head = s.heads.p + 1;
    cp.refs = s.refs.p;
    cp.overflow = reinterpret_cast<uint32_t *>(s.heads.p + 2);
    cp.ends = s.ef ? s.ends.p : nullptr;
    launch_cigar_text(cp, s.stream);
    CK(cudaGetLastError());
    s.stats.launches += 2;
    CK(cudaMemcpyAsync(s.h_heads.p, s.heads.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaMemcpyAsync(s.h_refs.p, s.refs.p, n * sizeof(wfagpu_cigar_ref_t), cudaMemcpyDeviceToHost, s.stream));
    s.text_queued = true;
    return 0;
}

extern "C" int wfagpu_device_align(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int resident)
{
    return wfagpu_device_align_span(d, slot, n, plan, resident, nullptr);
}

/* The span of pair i is spans[i * stride] (stride 0: one span for the batch); spans = NULL: global. */
static int align_spans(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, const wfagpu_span_t *spans,
                       size_t stride)
{
    if (!d || slot < 0 || slot > 1 || !plan) return -1;
    bool ef = false;
    for (size_t i = 0; spans && i < (stride ? n : 1); ++i) {
        const wfagpu_span_t &sp = spans[i * stride];
        if (sp.pattern_begin_free < 0 || sp.pattern_end_free < 0 || sp.text_begin_free < 0 || sp.text_end_free < 0) {
            fprintf(stderr, "[wfagpu] ends-free span values must be >= 0 (got %d,%d,%d,%d for pair %zu)\n",
                    sp.pattern_begin_free, sp.pattern_end_free, sp.text_begin_free, sp.text_end_free, i);
            return -3;
        }
        ef = ef || sp.pattern_begin_free || sp.pattern_end_free || sp.text_begin_free || sp.text_end_free;
    }
    if (ef && plan->band > 0) {
        fprintf(stderr, "[wfagpu] ends-free alignment is exact only: it cannot be combined with the adaptive band\n");
        return -3;
    }
    if (plan->o2 < 0 || plan->e2 < 0) {
        fprintf(stderr, "[wfagpu] gap-affine 2-piece penalties must be >= 0 (got o2=%d e2=%d)\n", plan->o2, plan->e2);
        return -3;
    }
    const bool p2 = plan->e2 > 0;
    if (p2 && (plan->band > 0 || ef)) {
        fprintf(stderr, "[wfagpu] gap-affine 2-piece alignment is global and exact only: it cannot be combined with %s\n",
                ef ? "an ends-free span" : "the adaptive band");
        return -3;
    }
    if (plan->x < 1 || plan->e < 1 || plan->o < 0) {
        /* x = 0 or e = 0 make a wavefront its own source (and divide by zero in the pruning quotient) */
        fprintf(stderr, "[wfagpu] penalties must satisfy x >= 1, e >= 1, o >= 0 (got %d,%d,%d)\n", plan->x, plan->o, plan->e);
        return -3;
    }
    CK(cudaSetDevice(d->dev));
    Slot &s = d->slots[slot];
    if (n != s.n) return -1;
    s.plan = *plan;
    s.ef = ef;
    s.plain = !ef && !p2;
    /* the span of every pair clamped to that pair (the kernels read it by pair index, on every pass), then the widest of
     * the batch: the start row's half width and the reach of the target range beyond kt (the step table and the rings
     * are shared by the pairs of a batch) */
    s.ef_w = 0;
    s.ef_ext = 0;
    if (ef && n > 0) {
        if (s.spans.ensure(n) || s.h_spans.ensure(n)) return -1;
        for (size_t i = 0; i < n; ++i) {
            const wfagpu_span_t &sp = spans[i * stride];
            const int pl = (int)s.h_pairs.p[i].plen, tl = (int)s.h_pairs.p[i].tlen;
            const int4 c = make_int4(std::min(sp.pattern_begin_free, pl), std::min(sp.pattern_end_free, pl),
                                     std::min(sp.text_begin_free, tl), std::min(sp.text_end_free, tl));
            s.h_spans.p[i] = c;
            s.ef_w = std::max(s.ef_w, std::max(c.x, c.z));
            s.ef_ext = std::max(s.ef_ext, std::max(c.y, c.w));
        }
        CK(cudaMemcpyAsync(s.spans.p, s.h_spans.p, n * sizeof(int4), cudaMemcpyHostToDevice, s.stream));
    }
    if (n == 0) return 0;
    if (ef && (s.ends.ensure(n) || s.h_ends.ensure(n))) return -1;
    /* the batch may be re-aligned while it stays resident: start from clean counters */
    s.stats.launches = 0;
    s.stats.redispatched = 0;
    s.stats.ascii_pairs = 0;
    CK(cudaMemsetAsync(s.counters.p, 0, CTR_WORDS * sizeof(uint32_t), s.stream));
    CK(cudaMemsetAsync(s.cells.p, 0, sizeof(unsigned long long), s.stream));
    CK(cudaMemsetAsync(s.out.p, 0, n * sizeof(wfagpu_pair_out_t), s.stream));   /* a pair may skip the first pass: no stale record */
    CK(cudaEventRecord(s.ev[2], s.stream));
    PackParams pp{s.ascii.p, s.packed.p, s.pairs.p, (uint32_t)n};
    launch_pack(pp, s.stream);
    CK(cudaGetLastError());
    s.stats.launches += 1;
    CK(cudaEventRecord(s.ev[3], s.stream));
    s.last_d_end = 0;
    s.wf_timed = false;
    /* -e is where the reference hands a pair to its CPU aligner (lib/align.cu:237); here such pairs cost a second pass on the
     * GPU.  When the last batch of this kind needed scores a little beyond -e (at most a quarter more), the first pass is
     * given that budget straight away: 100 k x 1 kbp / 10 % with -e 300 re-dispatched 4.4 % of its pairs in every chunk. */
    int first_steps = plan->max_steps;
    pull_hint(d);
    if (s.plain && d->hint_lift_pm > 0 && hint_applies(d, s, *plan)) {
        const long long want = hint_plus(d, d->hint_margin_pm, 12);
        const long long most = (long long)plan->max_steps + (long long)plan->max_steps * d->hint_lift_pm / 1000;
        if (want > first_steps && d->hint_dist <= most) first_steps = (int)std::min<long long>(want, d->max_steps_cap);
    }
    s.first_steps = first_steps;
    PassRequest first{s.order.p, n, s.retry[0].p, first_steps};
    first.first_pass = true;
    const int rc = launch_pass(d, s, *plan, first);
    if (rc < 0) return rc;
    s.capped = rc > 0;
    d->device_text = env_int("WFAGPU_HOST_CIGAR", 0) == 0;   /* re-read: tests flip it between runs */
    if (plan->with_cigar && d->device_text && enqueue_text(d, s, n, s.last_d_end)) return -1;
    CK(cudaEventRecord(s.ev[4], s.stream));                  /* align time = bound + wavefronts + traceback + CIGAR text */
    return 0;
}

extern "C" int wfagpu_device_align_span(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int resident,
                                        const wfagpu_span_t *span)
{
    (void)resident;
    return align_spans(d, slot, n, plan, span, 0);
}

extern "C" int wfagpu_device_align_spans(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int resident,
                                         const wfagpu_span_t *spans)
{
    (void)resident;
    return align_spans(d, slot, n, plan, spans, 1);
}

extern "C" int wfagpu_device_download(wfagpu_device_t *d, int slot, size_t n, wfagpu_pair_out_t *out, uint32_t **ops,
                                      size_t *ops_used, uint32_t *pair_flags)
{
    if (!d || slot < 0 || slot > 1) return -1;
    CK(cudaSetDevice(d->dev));
    Slot &s = d->slots[slot];
    if (n != s.n) return -1;
    if (ops) *ops = nullptr;
    if (ops_used) *ops_used = 0;
    if (n == 0) return 0;
    const wfagpu_plan_t plan = s.plan;

    auto read_counters = [&]() -> int {
        CK(cudaMemcpyAsync(s.h_counters.p, s.counters.p, CTR_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
        return 0;
    };
    if (read_counters()) return -1;

    /* Re-dispatched pairs always run the exact kernels: a band that lost the alignment does not find it
     * again with a larger budget (the reference hands such pairs to the CPU WFA, utils/wfa_cpu.c:30-86). */
    wfagpu_plan_t replan = plan;
    replan.band = 0;

    /* Budget oracle: score upper bounds of the pending pairs (bound kernel with the largest budget)
     * -> the number of wavefront steps that is enough for all of them, 0 if one has no bound. */
    auto bound_budget = [&](int cur, uint32_t pending, long long *need) -> int {
        *need = 0;
        if (s.h_retry.ensure(pending + 1)) return -1;
        int rc = bounds_to_host(d, s, replan, d->max_steps_cap, s.retry[cur].p, pending);
        if (rc == -2) return 0;                     /* the bound kernel does not fit these penalties: keep doubling */
        if (rc) return rc;
        CK(cudaMemcpyAsync(s.h_retry.p, s.retry[cur].p, pending * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
        const int d_big = s.tab_d_end;
        int maxb = 0;
        for (uint32_t i = 0; i < pending; ++i) {
            const uint32_t idx = s.h_retry.p[i];
            if (idx >= s.n) return -1;
            const int b = s.h_bound.p[idx];
            if (b >= d_big - 1) return 0;           /* not found within the largest budget: keep doubling */
            maxb = std::max(maxb, b);
        }
        long long steps_needed = 1;                 /* the reference counts the score-0 wavefront as step 1 */
        for (int dd = 1; dd <= maxb; ++dd) steps_needed += (s.h_steps.p[dd].kind == WFAGPU_STEP_MDI);
        *need = std::max<long long>(steps_needed + 3, 8);
        return 0;
    };

    /* ---- re-dispatch tier: pairs that outgrew the provisioned rings or the budget get, in one go,
     * the budget their score bounds call for (and are pruned by them); without bounds (banded,
     * byte-compare pairs) first the full budget, then the budget doubles until everything finishes ---- */
    /* pairs the GPU cannot finish (more than 60000 wavefront steps, or wavefronts wider than one CTA can hold):
     * their indices, taken from a device retry list */
    std::vector<uint32_t> failed;
    auto fail_pending = [&](int buf, uint32_t count) -> int {
        if (count == 0) return 0;
        if (s.h_retry.ensure((size_t)count + 1)) return -1;
        CK(cudaMemcpyAsync(s.h_retry.p, s.retry[buf].p, (size_t)count * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
        for (uint32_t i = 0; i < count; ++i)
            if (s.h_retry.p[i] < s.n) failed.push_back(s.h_retry.p[i]);
        return 0;
    };
    auto redispatch = [&](bool ascii, int start_steps, bool capped) -> int {
        int cur = 0;
        long long steps = start_steps;
        uint32_t pending = s.h_counters.p[CTR_RETRY];
        bool oracle_tried = false;
        while (pending > 0) {
            s.stats.redispatched += pending;
            long long next = capped ? steps : std::max<long long>(steps * 2, 64);
            bool have_bounds = false;
            if (!oracle_tried && !ascii && !d->no_bound) {
                oracle_tried = true;
                long long need = 0;
                int rcb = bound_budget(cur, pending, &need);
                if (rcb < 0) return rcb;
                if (rcb == 0 && need > 0) { next = need; have_bounds = true; }
            }
            if (next > d->max_steps_cap) {
                /* per pair, not per job: these pairs are reported as failed, everything else keeps its result */
                fprintf(stderr, "[wfagpu] %u pairs need more than %lld wavefront steps; reported as failed\n", pending, steps);
                return fail_pending(cur, pending);
            }
            steps = next;
            PassRequest r{s.retry[cur].p, pending, s.retry[cur ^ 1].p, (int)steps};
            r.ascii = ascii;
            r.have_bounds = have_bounds;
            const int rc = launch_pass(d, s, replan, r);
            if (rc < 0) return rc;
            if (read_counters()) return -1;
            if (rc > 0 && s.h_counters.p[CTR_RETRY] > 0) {
                fprintf(stderr, "[wfagpu] %u pairs exceed the wavefront capacity of one CTA; reported as failed\n",
                        s.h_counters.p[CTR_RETRY]);
                return fail_pending(cur ^ 1, s.h_counters.p[CTR_RETRY]);
            }
            capped = false;
            pending = s.h_counters.p[CTR_RETRY];
            cur ^= 1;
        }
        return 0;
    };
    int rc = redispatch(false, std::max(plan.max_steps, s.first_steps), s.capped);
    if (rc) return rc;

    /* ---- pairs with non-ACGT bytes: byte-compare kernel on the ASCII copy ---- */
    const uint32_t n_ascii = s.h_counters.p[CTR_ASCII];
    if (n_ascii > 0) {
        s.stats.ascii_pairs = n_ascii;
        PassRequest r{s.ascii_list.p, n_ascii, s.retry[0].p, plan.max_steps};
        r.ascii = true;
        rc = launch_pass(d, s, plan, r);
        if (rc < 0) return rc;
        if (read_counters()) return -1;
        rc = redispatch(true, plan.max_steps, rc > 0);
        if (rc) return rc;
    }
    CK(cudaEventRecord(s.ev[5], s.stream));

    /* ---- results back to the host ---- */
    if (s.h_out.ensure(n)) return -1;
    const uint32_t pool_used = s.h_counters.p[CTR_POOL];
    if (s.h_pool.ensure((size_t)pool_used + 1)) return -1;
    CK(cudaMemcpyAsync(s.h_out.p, s.out.p, n * sizeof(wfagpu_pair_out_t), cudaMemcpyDeviceToHost, s.stream));
    if (pool_used)
        CK(cudaMemcpyAsync(s.h_pool.p, s.pool.p, (size_t)pool_used * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    if (pair_flags) CK(cudaMemcpyAsync(s.h_pairs.p, s.pairs.p, n * sizeof(wfagpu_pair_t), cudaMemcpyDeviceToHost, s.stream));
    if (d->count_cells) CK(cudaMemcpyAsync(s.h_cells.p, s.cells.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    for (uint32_t idx : failed) {
        s.h_out.p[idx].status = WFAGPU_ST_FAILED;
        s.h_out.p[idx].distance = -1;
        s.h_out.p[idx].n_ops = 0;
    }
    s.stats.failed_pairs = (uint32_t)failed.size();
    memcpy(out, s.h_out.p, n * sizeof(wfagpu_pair_out_t));
    if (!d->independent && s.plain) learn_hint(d, s, n);
    if (pair_flags)
        for (size_t i = 0; i < n; ++i) pair_flags[i] = s.h_pairs.p[i].flags;
    if (ops) *ops = s.h_pool.p;
    if (ops_used) *ops_used = pool_used;
    s.stats.d2h_bytes += n * sizeof(wfagpu_pair_out_t) + (size_t)pool_used * 4;
    if (d->count_cells) s.stats.cells = s.h_cells.p[0];
    if (s.have_events) {
        cudaEventElapsedTime(&s.stats.ms_h2d, s.ev[0], s.ev[1]);
        cudaEventElapsedTime(&s.stats.ms_pack, s.ev[2], s.ev[3]);
        cudaEventElapsedTime(&s.stats.ms_align, s.ev[3], s.ev[5]);
        cudaEventElapsedTime(&s.stats.ms_total, s.ev[0], s.ev[5]);
    }
    return 0;
}

extern "C" int wfagpu_device_rescore(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, int32_t *scores)
{
    return wfagpu_device_rescore_span(d, slot, n, plan, nullptr, scores);
}

static int rescore_spans(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan, const wfagpu_span_t *spans,
                         size_t stride, int32_t *scores)
{
    if (!d || !plan || !scores || slot < 0 || slot > 1) return -1;
    if (n != d->slots[slot].n) return -1;
    /* a different code path on purpose: what it shares with the production path is the packing, the step table
     * and the extend */
    const bool nb = d->no_bound, nq = d->no_quad, uh = d->use_hint;
    const int fw = d->force_warp;
    d->no_bound = true; d->no_quad = true; d->use_hint = false; d->force_warp = 0; d->independent = true;
    wfagpu_plan_t p2 = *plan;
    p2.with_cigar = 0;
    p2.with_ends = 0;
    std::vector<wfagpu_pair_out_t> out(n);
    int rc = align_spans(d, slot, n, &p2, spans, stride);
    if (!rc) rc = wfagpu_device_download(d, slot, n, out.data(), nullptr, nullptr, nullptr);
    d->no_bound = nb; d->no_quad = nq; d->use_hint = uh; d->force_warp = fw; d->independent = false;
    if (rc) return rc;
    for (size_t i = 0; i < n; ++i) scores[i] = (out[i].status & WFAGPU_ST_FINISHED) ? out[i].distance : -1;
    return 0;
}

extern "C" int wfagpu_device_rescore_span(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan,
                                          const wfagpu_span_t *span, int32_t *scores)
{
    return rescore_spans(d, slot, n, plan, span, 0, scores);
}

extern "C" int wfagpu_device_rescore_spans(wfagpu_device_t *d, int slot, size_t n, const wfagpu_plan_t *plan,
                                           const wfagpu_span_t *spans, int32_t *scores)
{
    return rescore_spans(d, slot, n, plan, spans, 1, scores);
}

extern "C" int wfagpu_device_download_ends(wfagpu_device_t *d, int slot, size_t n, int32_t *ends)
{
    if (!d || slot < 0 || slot > 1 || (!ends && n)) return -1;
    CK(cudaSetDevice(d->dev));
    Slot &s = d->slots[slot];
    if (n != s.n || !s.ef) return -1;
    if (n == 0) return 0;
    CK(cudaMemcpyAsync(s.h_ends.p, s.ends.p, n * sizeof(int2), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    memcpy(ends, s.h_ends.p, n * sizeof(int2));
    return 0;
}

extern "C" int wfagpu_device_wait(wfagpu_device_t *d, int slot, float *ms_pack, float *ms_align)
{
    if (!d || slot < 0 || slot > 1) return -1;
    CK(cudaSetDevice(d->dev));
    Slot &s = d->slots[slot];
    CK(cudaStreamSynchronize(s.stream));
    if (ms_pack) cudaEventElapsedTime(ms_pack, s.ev[2], s.ev[3]);
    if (ms_align) cudaEventElapsedTime(ms_align, s.ev[3], s.ev[4]);
    s.stats.ms_wavefront = 0;
    if (s.wf_timed) cudaEventElapsedTime(&s.stats.ms_wavefront, s.ev[6], s.ev[7]);
    /* pairs the timed pass left for the re-dispatch tier / the byte-compare kernel (both run in download()) */
    if (s.n) {
        CK(cudaMemcpyAsync(s.h_counters.p, s.counters.p, CTR_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
        s.stats.pending_pairs = s.h_counters.p[CTR_RETRY] + s.h_counters.p[CTR_ASCII];
    }
    if (s.n && d->use_hint && s.plain) {
        /* read the result records back (16 B per pair) so that a re-run of the resident
         * batch is provisioned like the next batch of a stream would be */
        if (s.h_out.ensure(s.n)) return -1;
        CK(cudaMemcpyAsync(s.h_out.p, s.out.p, s.n * sizeof(wfagpu_pair_out_t), cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
        learn_hint(d, s, s.n);
    }
    return 0;
}

/* 1 if `ptr` is page-locked (cudaHostAlloc / cudaHostRegister), 0 if pageable or unknown */
extern "C" int wfagpu_host_is_pinned(const void *ptr)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { cudaGetLastError(); return 0; }
    return at.type == cudaMemoryTypeHost ? 1 : 0;
}

/* Page-locked staging area of a slot (grow-only): a caller with a pageable sequence buffer copies the batch here
 * (with its own threads) and uploads from it, so that the H2D copy is asynchronous DMA like for pinned callers.
 * The previous upload from this slot must have been waited for (download). */
extern "C" char *wfagpu_device_staging(wfagpu_device_t *d, int slot, size_t bytes)
{
    if (!d || slot < 0 || slot > 1) return nullptr;
    if (cudaSetDevice(d->dev) != cudaSuccess) return nullptr;
    Slot &s = d->slots[slot];
    if (s.h_ascii.ensure(bytes + 64)) return nullptr;
    return s.h_ascii.p;
}

/* Page-locked host memory for the aligner's own buffers (the reference's TODO, utils/sequence_reader.c:73):
 * NULL when no CUDA device / driver is usable -- the caller then falls back to plain calloc. */
extern "C" void *wfagpu_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    memset(p, 0, bytes);
    return p;
}
extern "C" void wfagpu_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

extern "C" int wfagpu_host_register(void *ptr, size_t bytes)
{
    cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        fprintf(stderr, "[wfagpu] cudaHostRegister failed: %s\n", cudaGetErrorString(e));
        return -1;
    }
    return 0;
}

extern "C" int wfagpu_host_unregister(void *ptr)
{
    return cudaHostUnregister(ptr) == cudaSuccess ? 0 : -1;
}

extern "C" int wfagpu_device_download_text(wfagpu_device_t *d, int slot, size_t n, const char **text, size_t *text_bytes,
                                           const wfagpu_cigar_ref_t **refs)
{
    if (!d || slot < 0 || slot > 1 || !text || !text_bytes || !refs) return -1;
    CK(cudaSetDevice(d->dev));
    Slot &s = d->slots[slot];
    if (n != s.n) return -1;
    *text = nullptr; *text_bytes = 0; *refs = nullptr;
    if (n == 0) return 0;
    if (!s.text_queued && enqueue_text(d, s, n, s.last_d_end)) return -1;
    CK(cudaStreamSynchronize(s.stream));
    if (s.h_heads.p[2] != 0) {
        fprintf(stderr, "[wfagpu] CIGAR text pool overflow\n");
        return -1;
    }
    const size_t used = (size_t)s.h_heads.p[1];
    if (s.h_text.ensure(used + 1)) return -1;
    if (used) CK(cudaMemcpyAsync(s.h_text.p, s.text.p, used, cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    s.stats.d2h_bytes += used + n * sizeof(wfagpu_cigar_ref_t);
    *text = s.h_text.p;
    *text_bytes = used;
    *refs = s.h_refs.p;
    return 0;
}

extern "C" void wfagpu_device_last_stats(wfagpu_device_t *d, int slot, wfagpu_batch_stats_t *st)
{
    if (!d || !st || slot < 0 || slot > 1) return;
    *st = d->slots[slot].stats;
}

extern "C" int wfagpu_device_pack_only(wfagpu_device_t *d, const char *ascii, size_t ascii_bytes, wfagpu_pair_t *pairs,
                                       size_t n, uint32_t *packed_out, size_t packed_words)
{
    if (!d) return -1;
    if (wfagpu_device_upload(d, 0, ascii, ascii_bytes, pairs, n)) return -1;
    Slot &s = d->slots[0];
    PackParams pp{s.ascii.p, s.packed.p, s.pairs.p, (uint32_t)n};
    launch_pack(pp, s.stream);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s.stream));
    if (packed_words < s.packed_words) return -1;
    CK(cudaMemcpy(packed_out, s.packed.p, s.packed_words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(pairs, s.pairs.p, n * sizeof(wfagpu_pair_t), cudaMemcpyDeviceToHost));
    return 0;
}

/* ------------------------------------------------------------------------ */
/* utils/device_query.cu:27-54 equivalents                                   */
extern "C" void get_num_cuda_devices(int *n)
{
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) c = 0;
    if (n) *n = c;
}

extern "C" char *get_cuda_dev_name(int dev)
{
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return nullptr;
    return strdup(prop.name);
}

extern "C" int get_cuda_SM_count(int dev)
{
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    return v;
}

extern "C" void get_cuda_capability(int dev, int *major, int *minor)
{
    int a = 0, b = 0;
    cudaDeviceGetAttribute(&a, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMinor, dev);
    if (major) *major = a;
    if (minor) *minor = b;
}
