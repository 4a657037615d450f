// urlgpu.cu — C ABI (include/urlgpu.h) and host-side orchestration of the sm_100a kernels.
//
// One context owns one device and one stream.  Per-variable results are dense tables indexed by the COMPACT
// parent-set mask (bit i = i-th candidate of the variable in ascending variable index, the child itself
// removed — score_calculator.cpp:65-74,100), which makes subset look-ups (accept / prune DPs) a single XOR.
#include "../../include/urlgpu.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <ctime>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "bic_kernels.cuh"
#include "tree_kernels.cuh"
#include "cbic_kernels.cuh"
#include "rank_kernels.cuh"
#include "spg_kernels.cuh"
#include "order_kernels.cuh"
#include "regret.hpp"

using namespace urlgpu;

static inline bool is_discrete(int score_type) { return score_type == URLGPU_BIC || score_type == URLGPU_FNML || score_type == URLGPU_BDEU; }

namespace {

thread_local std::string g_create_error;
std::atomic<int> g_ctx_on_device[64];   // live contexts per device: each budgets its share of the free memory

enum Family { F_COUNT = 0, F_CUBE, F_CBIC, F_ACCEPT, F_PRUNE, F_GRAM, F_OTHER, F_STD, F_ORDER_TABLES, F_ORDER_LAYERS, F_N };

struct EvPair { cudaEvent_t a, b; int fam; };

} // namespace

struct urlgpu_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // device->host copies of fetched results: not ordered behind later scoring work
    std::vector<unsigned long long *> free_pinned; // 33-counter blocks of pinned host memory (urlgpu_result::h_counts)
    // scratch of the copy stream (expanded masks of the range being fetched).  NOT from the pool: pool blocks are recycled in
    // the order of the scoring stream, the copy stream runs concurrently with it
    uint64_t *d_fetch_wide = nullptr; size_t fetch_wide_cap = 0; int *d_fetch_cand = nullptr;
    std::string err;
    int sm_count = 148;
    size_t smem_optin = 0;

    // discrete data
    int64_t n = 0, n_stride = 0;
    int p = 0;
    std::vector<int32_t> card;
    uint8_t *d_codes = nullptr;
    long long *d_qlog = nullptr;
    float base = 0.f;
    bool have_discrete = false;
    // the discrete score the next K1 launches compute (select_discrete_score): per-configuration table, the smallest
    // configuration count that contributes, the penalty constant
    const long long *ds_qcfg = nullptr; int ds_cfg_min = 1; float ds_base = 0.f;
    float ds_ess = 0.f; double ds_scale = 1.0 / 8388608.0;   // BDeu: equivalent sample size (> 0) and the 2^-30 accumulator unit
    std::map<int, long long *> d_qfnml;   // fNML: arity -> qlog + log-regret table [n+2] (built on first use, owned by this context)
    std::set<int> t16_overflowed;         // variables whose speculative 16-bit tables overflowed once: scored with 32-bit tables from then on
    bool borrowed_discrete = false; // d_codes/d_qlog belong to another context on the same device (urlgpu_share_discrete)

    // continuous data
    int64_t cn = 0;
    int cp = 0;
    double *d_z = nullptr;
    double *d_zcache = nullptr; size_t zcache_cap = 0;
    double *d_x = nullptr; const double *d_x_view = nullptr; int64_t shard_n = 0; bool borrow_device_x = false; // attached raw rows (sharded protocol)
    int64_t shard_stride = 0;   // row pitch of d_x_view: shard_n for a borrowed buffer, shard_n rounded up to kGramKC for the engine's own copy
    std::vector<double> h_gram;
    double *d_gram = nullptr;   // device copy of h_gram (urlgpu_score_sets gathers each set's sub-Gram from it)
    double gram_dmax = 0;   // largest diagonal entry of the Gram: scale of the pivot guard (CbicParams::piv_tol)
    bool have_gram = false;

    // scratch
    int *d_tables = nullptr; size_t tables_cap = 0;          // int32 elements
    void *d_misc = nullptr; size_t misc_cap = 0;
    int *d_cubeA = nullptr, *d_cubeB = nullptr; size_t cubeA_cap = 0, cubeB_cap = 0; // ping-pong layer buffers of the cube path
    size_t mem_free_sample = 0;  // free device memory (plus the cube buffers) when the current data set was installed
    uint32_t *d_high_sorted = nullptr; int high_bits = -1; std::vector<int> high_off;   // segment DP lists (accept / prune)
    uint16_t *d_low_sorted = nullptr; int low_bits = -1; std::vector<int> low_off;
    bool use_slice_count = true; // cube path: count big roots in shared-memory slices (URLGPU_SLICE_COUNT=0 disables)
    bool fuse_roots = true;      // cube path: ancestor-only roots hand their children straight to HBM (URLGPU_FUSE_ROOTS=0 disables)
    // cube path: tables of layers >= table16_min_layer are written with uint16 cells, speculatively (URLGPU_TABLE16=0 disables,
    // URLGPU_TABLE16_MINLAYER sets the layer); a count that does not fit flags the call and the variable is recomputed in 32 bits
    bool table16 = true;
    int table16_min_layer = 8;
    uint32_t root_budget = 24 * 1024; // cells of a root slice (URLGPU_ROOT_BUDGET): 96 KB + segment tables, two 512-thread CTAs per SM
    uint32_t root_seg_cap = 1024;     // row segments of a slice kept in shared memory (URLGPU_ROOT_SEGS)
    int root_warps = 16;              // warps per CTA of bic_root_kernel (URLGPU_ROOT_WARPS = 8, 12 or 16)
    // K1 strategy: the cube path (roots counted in shared-memory slices, the rest marginalised through HBM), or, with
    // URLGPU_BIC_MODE=direct, direct counting of every set from the rows
    bool bic_direct = false;

    // rank-space layout: binomial tables [256][K + 2] per parent limit K (tiny; kept for the life of the context so kernels in
    // flight never lose theirs), and the layout policy (URLGPU_LAYOUT=dense|rank|auto)
    uint32_t *d_binom[kMaxRankLayers + 1] = {nullptr};
    int layout_policy = 0;       // 0 auto, 1 dense whenever possible, 2 rank whenever possible

    // pinned staging arena for host->device descriptor uploads (pageable cudaMemcpyAsync would sync the stream)
    // two arenas used alternately per call, each guarded by an event recorded when its call has been enqueued, so the
    // host can plan and upload call k+1 while the GPU still executes call k
    char *h_stage[2] = {nullptr, nullptr}; size_t stage_cap[2] = {0, 0}; size_t stage_used = 0;
    cudaEvent_t stage_ev[2] = {nullptr, nullptr}; int stage_cur = 0;

    // caching device allocator: cudaMalloc/cudaFree of multi-GB tables cost tens of ms each
    struct PoolBlock { void *p; size_t bytes; bool used; };
    std::vector<PoolBlock> pool;

    // URLGPU_DEBUG_TIMING: wall time the host spends blocked in (0) staging-arena waits, (1) cudaMemGetInfo, (2) cudaMalloc of
    // pool blocks, (3) pinned-arena copies, (4) arena growth, printed by urlgpu_destroy
    double dbg_wall[8] = {0}; uint64_t dbg_n[8] = {0};

    // stats
    urlgpu_stats st{};
    bool timing = false;
    std::vector<EvPair> pending;
    std::vector<cudaEvent_t> free_events;

    int fail(int code, const std::string &m) { err = m; return code; }
    int cuda_fail(cudaError_t e, const char *what, int line) {
        err = std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what + " (urlgpu.cu:" + std::to_string(line) + ")";
        return URLGPU_ERR_CUDA;
    }
};

#define CK(call)                                                            \
    do {                                                                    \
        cudaError_t e_ = (call);                                            \
        if (e_ != cudaSuccess) return ctx->cuda_fail(e_, #call, __LINE__);  \
    } while (0)

namespace {

struct DbgTimer {
    urlgpu_ctx *c; int k; std::chrono::steady_clock::time_point t0;
    DbgTimer(urlgpu_ctx *ctx, int kind) : c(ctx), k(kind), t0(std::chrono::steady_clock::now()) {}
    ~DbgTimer() { c->dbg_wall[k] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); c->dbg_n[k]++; }
};

// size classes: powers of two up to 64 MB, multiples of 64 MB above.  Requests of any size then find a cached block after
// the first few calls (per-variable tables differ in size from variable to variable; exact-size caching never converged)
size_t pool_class(size_t bytes) {
    bytes = std::max<size_t>(bytes, 256);
    const size_t big = (size_t)64 << 20;
    if (bytes > big) return (bytes + big - 1) / big * big;
    size_t c = 256;
    while (c < bytes) c <<= 1;
    return c;
}

cudaError_t pool_alloc(urlgpu_ctx *ctx, void **out, size_t bytes) {
    bytes = pool_class(bytes);
    int best = -1;
    for (size_t i = 0; i < ctx->pool.size(); i++) {
        auto &b = ctx->pool[i];
        if (!b.used && b.bytes >= bytes && b.bytes <= bytes + bytes / 4 && (best < 0 || b.bytes < ctx->pool[best].bytes)) best = (int)i;
    }
    if (best >= 0) { ctx->pool[best].used = true; *out = ctx->pool[best].p; return cudaSuccess; }
    DbgTimer dt(ctx, 2);
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) { // release every cached block and retry once
        cudaGetLastError();
        for (size_t i = 0; i < ctx->pool.size();) {
            if (!ctx->pool[i].used) { cudaFree(ctx->pool[i].p); ctx->pool.erase(ctx->pool.begin() + i); } else i++;
        }
        e = cudaMalloc(out, bytes);
        if (e != cudaSuccess) return e;
    }
    ctx->pool.push_back({*out, bytes, true});
    return cudaSuccess;
}
void pool_free(urlgpu_ctx *ctx, void *p) {
    if (!p) return;
    for (size_t i = 0; i < ctx->pool.size(); i++)
        if (ctx->pool[i].p == p) {
            if (ctx->pool[i].bytes > ((size_t)4 << 30)) { cudaFree(p); ctx->pool.erase(ctx->pool.begin() + i); } // do not hoard huge blocks
            else ctx->pool[i].used = false;
            return;
        }
    cudaFree(p);
}
void pool_destroy(urlgpu_ctx *ctx) {
    for (auto &b : ctx->pool) cudaFree(b.p);
    ctx->pool.clear();
}

struct DevBuf { // RAII device allocation from the context's pool.  Released blocks are only ever handed to later work on the SAME stream
                // (the context's scoring stream), so kernels still in flight keep their buffers without a synchronisation
    urlgpu_ctx *ctx;
    void *p = nullptr;
    explicit DevBuf(urlgpu_ctx *c) : ctx(c) {}
    ~DevBuf() { pool_free(ctx, p); }
    cudaError_t alloc(size_t bytes) { pool_free(ctx, p); p = nullptr; return pool_alloc(ctx, &p, bytes); }
    template <typename T> T *as() { return static_cast<T *>(p); }
};

cudaEvent_t get_event(urlgpu_ctx *ctx) {
    if (!ctx->free_events.empty()) { cudaEvent_t e = ctx->free_events.back(); ctx->free_events.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

void fold_events(urlgpu_ctx *ctx) {
    if (ctx->pending.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (auto &ep : ctx->pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ep.a, ep.b) == cudaSuccess) {
            double *dst = ep.fam == F_COUNT ? &ctx->st.ms_count : ep.fam == F_CUBE ? &ctx->st.ms_cube : ep.fam == F_CBIC ? &ctx->st.ms_cbic
                        : ep.fam == F_ACCEPT ? &ctx->st.ms_accept : ep.fam == F_PRUNE ? &ctx->st.ms_prune : ep.fam == F_GRAM ? &ctx->st.ms_gram
                        : ep.fam == F_STD ? &ctx->st.ms_standardise : ep.fam == F_ORDER_TABLES ? &ctx->st.ms_order_tables
                        : ep.fam == F_ORDER_LAYERS ? &ctx->st.ms_order_layers : nullptr;
            if (dst) *dst += ms;
        }
        ctx->free_events.push_back(ep.a);
        ctx->free_events.push_back(ep.b);
    }
    ctx->pending.clear();
}

// Brackets a group of launches of one kernel family with CUDA events on the context's stream.
struct Region {
    urlgpu_ctx *ctx; int fam; EvPair ep{};
    bool on;
    Region(urlgpu_ctx *c, int f, uint64_t launches) : ctx(c), fam(f), on(c->timing) {
        c->st.launches_total += launches;
        uint64_t *cnt = f == F_COUNT ? &c->st.launches_count : f == F_CUBE ? &c->st.launches_cube : f == F_CBIC ? &c->st.launches_cbic
                      : f == F_ACCEPT ? &c->st.launches_accept : f == F_PRUNE ? &c->st.launches_prune : &c->st.launches_other;
        *cnt += launches;
        if (on) { ep.a = get_event(c); ep.b = get_event(c); ep.fam = f; cudaEventRecord(ep.a, c->stream); }
    }
    ~Region() {
        if (on) {
            cudaEventRecord(ep.b, ctx->stream);
            ctx->pending.push_back(ep);
            if (ctx->pending.size() > 4096) fold_events(ctx);
        }
    }
};

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// binomial sums (host)
uint64_t family_size(int c, int K) {
    uint64_t total = 0, b = 1;
    for (int l = 0; l <= K && l <= c; l++) {
        total += b;
        b = b * (uint64_t)(c - l) / (uint64_t)(l + 1);
    }
    return total;
}

// C(b, i) saturating at 2^32 - 1
uint32_t binom_sat(int b, int i) {
    if (i < 0 || i > b) return 0;
    unsigned __int128 r = 1;
    for (int k = 1; k <= i; k++) {
        r = r * (unsigned)(b - i + k) / (unsigned)k;
        if (r > 0xFFFFFFFFull) return 0xFFFFFFFFu;
    }
    return (uint32_t)r;
}

} // namespace

struct urlgpu_result {
    urlgpu_ctx *ctx = nullptr;
    int variable = 0, c = 0, max_parents = 0, mask_words = 1;
    std::vector<int> cand;          // compact bit -> variable index
    float *d_table = nullptr;       // dense layout: 2^c floats by compact mask; rank layout: rs.layer_base[K+1] floats by colex index
    bool rank_layout = false;
    RankSpace rs{};
    // speculative 16-bit tables (cube path): d_ovf is raised by a count that did not fit; checked when the result is first
    // read (the flag travels with the compaction counters), and the variable is then recomputed with 32-bit tables
    int *d_ovf = nullptr;
    bool is_bic = false;
    int score_type = URLGPU_BIC;
    unsigned filter_flags = 0;
    uint64_t n_masks = 0, n_scored = 0;   // n_masks = entries of d_table
    // compaction into canonical order (|S|, mask): enqueued on the context's stream by urlgpu_result_prefetch, no host sync
    bool prefetched = false, counted = false;
    uint32_t *d_masks = nullptr;    // dense: compact masks, rank: indices; canonical order (capacity n_scored)
    float *d_vals = nullptr;
    uint32_t *d_segcnt = nullptr;   // [32 layers][segments] stored entries, then their exclusive prefix
    unsigned long long *d_counts = nullptr;  // [33]: stored entries per layer, total
    unsigned long long *h_counts = nullptr;  // pinned copy
    cudaEvent_t ready = nullptr;    // compaction + the copy of the counts have completed
    uint64_t n_stored = 0; uint64_t layer_count[32] = {0};
};

// ============================================================================================ context

extern "C" int urlgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int urlgpu_create(urlgpu_ctx **out, int device_id) {
    if (!out) return URLGPU_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        g_create_error = std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                         "); urlgpu has no CPU fallback";
        return URLGPU_ERR_CUDA;
    }
    if (device_id < 0 || device_id >= ndev) { g_create_error = "device_id out of range"; return URLGPU_ERR_ARG; }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return URLGPU_ERR_CUDA; }
    if (prop.major != 10) {
        g_create_error = "device " + std::to_string(device_id) + " (" + prop.name + ", sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                         ") is not a Blackwell sm_100 device; this library carries sm_100a code only";
        return URLGPU_ERR_CUDA;
    }
    auto *ctx = new urlgpu_ctx();
    ctx->device = device_id;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if ((e = cudaSetDevice(device_id)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete ctx;
        return URLGPU_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    if (const char *m = getenv("URLGPU_SLICE_COUNT")) ctx->use_slice_count = atoi(m) != 0;
    if (const char *m = getenv("URLGPU_FUSE_ROOTS")) ctx->fuse_roots = atoi(m) != 0;
    if (const char *m = getenv("URLGPU_TABLE16")) ctx->table16 = atoi(m) != 0;
    if (const char *m = getenv("URLGPU_TABLE16_MINLAYER")) ctx->table16_min_layer = std::max(1, atoi(m));
    if (const char *m = getenv("URLGPU_ROOT_BUDGET")) ctx->root_budget = (uint32_t)std::max(1024, std::min(atoi(m), 48 * 1024)) / 4 * 4;
    if (const char *m = getenv("URLGPU_ROOT_SEGS")) ctx->root_seg_cap = (uint32_t)std::max(32, std::min(atoi(m), 8192));
    if (const char *m = getenv("URLGPU_ROOT_WARPS")) ctx->root_warps = atoi(m) == 8 ? 8 : atoi(m) == 12 ? 12 : 16;
    if (const char *m = getenv("URLGPU_LAYOUT")) ctx->layout_policy = strcmp(m, "dense") == 0 ? 1 : strcmp(m, "rank") == 0 ? 2 : 0;
    if (const char *m = getenv("URLGPU_BIC_MODE")) ctx->bic_direct = strcmp(m, "direct") == 0;
    // the large dynamic shared-memory opt-ins are per device: every context sets them for its own.  A refused opt-in fails
    // the creation here; unchecked, it would surface as a stale error of some later, unrelated call
    {
        auto refuse = [&](const std::string &m) {
            cudaGetLastError();
            g_create_error = m + ": " + cudaGetErrorString(e);
            cudaStreamDestroy(ctx->copy_stream);
            cudaStreamDestroy(ctx->own_stream);
            delete ctx;
            return URLGPU_ERR_CUDA;
        };
        const void *roots[] = {(const void *)bic_root_kernel<0, 8>, (const void *)bic_root_kernel<2, 8>, (const void *)bic_root_kernel<3, 8>,
                               (const void *)bic_root_kernel<4, 8>, (const void *)bic_root_kernel<0, 12>, (const void *)bic_root_kernel<2, 12>,
                               (const void *)bic_root_kernel<3, 12>, (const void *)bic_root_kernel<4, 12>, (const void *)bic_root_kernel<0, 16>,
                               (const void *)bic_root_kernel<2, 16>, (const void *)bic_root_kernel<3, 16>, (const void *)bic_root_kernel<4, 16>};
        // bic_root_kernel holds the slice (root_budget cells), two segment tables (root_seg_cap each) and one counter in
        // dynamic shared memory, next to its static shared memory (the byte look-up tables, the root descriptor).  Both
        // switches at the top of their ranges ask for more than a block may opt into: the segment cap gives way first (slices
        // with more segments take the kernel's fragmented path), then the budget
        size_t root_static = 0;
        for (const void *f : roots) {
            cudaFuncAttributes fa{};
            if ((e = cudaFuncGetAttributes(&fa, f)) != cudaSuccess) return refuse("cannot read the root kernel's attributes");
            root_static = std::max(root_static, fa.sharedSizeBytes);
        }
        const int64_t cap = ((int64_t)ctx->smem_optin - (int64_t)root_static) / (int64_t)sizeof(int) - 1;   // budget + 2 * segments
        if ((int64_t)ctx->root_budget + 2 * (int64_t)ctx->root_seg_cap > cap)
            ctx->root_seg_cap = (uint32_t)std::max<int64_t>(32, (cap - (int64_t)ctx->root_budget) / 2);
        if ((int64_t)ctx->root_budget + 2 * (int64_t)ctx->root_seg_cap > cap)
            ctx->root_budget = (uint32_t)std::max<int64_t>(0, (cap - 2 * (int64_t)ctx->root_seg_cap) / 4 * 4);
        const int smem = (int)((ctx->root_budget + 2 * ctx->root_seg_cap + 1) * sizeof(int));
        const int big = (int)ctx->smem_optin - 2048;
        std::vector<std::pair<const void *, int>> attrs;
        for (const void *f : roots) attrs.push_back({f, smem});
        attrs.push_back({(const void *)bic_count_smem_kernel<MaskSets>, big});
        attrs.push_back({(const void *)bic_count_smem_kernel<RankSets>, big});
        attrs.push_back({(const void *)bic_count_smem_kernel<ListSets>, big});
        attrs.push_back({(const void *)cbic_sets_kernel, big});
        attrs.push_back({(const void *)gram_partial_kernel, (int)kGramSmemBytes});
        attrs.push_back({(const void *)order_layer_rank_kernel, (int)order_rank_smem_bytes(kOrderRankMaxVars)});
        attrs.push_back({(const void *)order_climb_kernel<ClimbTable>, (int)order_climb_smem_bytes(kClimbMaxVars)});
        attrs.push_back({(const void *)order_climb_kernel<ClimbList>, (int)order_climb_smem_bytes(kClimbMaxVars)});
        for (const auto &a : attrs)
            if ((e = cudaFuncSetAttribute(a.first, cudaFuncAttributeMaxDynamicSharedMemorySize, a.second)) != cudaSuccess)
                return refuse("cannot opt a kernel into " + std::to_string(a.second) + " bytes of dynamic shared memory (the device allows " +
                              std::to_string(ctx->smem_optin) + " bytes per block, static shared memory included)");
    }
    if (device_id < 64) g_ctx_on_device[device_id]++;
    *out = ctx;
    return URLGPU_OK;
}

static void free_discrete(urlgpu_ctx *ctx) {
    if (!ctx->borrowed_discrete) {
        if (ctx->d_codes) cudaFree(ctx->d_codes);
        if (ctx->d_qlog) cudaFree(ctx->d_qlog);
    }
    for (auto &kv : ctx->d_qfnml) cudaFree(kv.second);
    ctx->d_qfnml.clear();
    ctx->d_codes = nullptr; ctx->d_qlog = nullptr; ctx->have_discrete = false; ctx->borrowed_discrete = false;
}
static void free_continuous(urlgpu_ctx *ctx) {
    if (ctx->d_z) cudaFree(ctx->d_z);
    if (ctx->d_x) cudaFree(ctx->d_x);
    if (ctx->d_gram) cudaFree(ctx->d_gram);
    ctx->d_x = nullptr; ctx->d_x_view = nullptr; ctx->d_gram = nullptr;
    ctx->d_z = nullptr; ctx->have_gram = false;
}

extern "C" int urlgpu_destroy(urlgpu_ctx *ctx) {
    if (!ctx) return URLGPU_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    fold_events(ctx);
    if (getenv("URLGPU_DEBUG_TIMING"))
        fprintf(stderr, "[urlgpu host waits] arena wait %.1f ms (%llu), cudaMemGetInfo %.1f ms (%llu), pool cudaMalloc %.1f ms (%llu), arena copies %.1f ms (%llu), arena growth %.1f ms (%llu)\n",
                ctx->dbg_wall[0], (unsigned long long)ctx->dbg_n[0], ctx->dbg_wall[1], (unsigned long long)ctx->dbg_n[1], ctx->dbg_wall[2], (unsigned long long)ctx->dbg_n[2],
                ctx->dbg_wall[3], (unsigned long long)ctx->dbg_n[3], ctx->dbg_wall[4], (unsigned long long)ctx->dbg_n[4]);
    for (auto e : ctx->free_events) cudaEventDestroy(e);
    free_discrete(ctx);
    free_continuous(ctx);
    if (ctx->d_tables) cudaFree(ctx->d_tables);
    if (ctx->d_zcache) cudaFree(ctx->d_zcache);
    if (ctx->d_misc) cudaFree(ctx->d_misc);
    if (ctx->d_cubeA) cudaFree(ctx->d_cubeA);
    if (ctx->d_high_sorted) cudaFree(ctx->d_high_sorted);
    if (ctx->d_low_sorted) cudaFree(ctx->d_low_sorted);
    if (ctx->d_cubeB) cudaFree(ctx->d_cubeB);
    pool_destroy(ctx);
    for (int k = 0; k < 2; k++) { if (ctx->h_stage[k]) cudaFreeHost(ctx->h_stage[k]); if (ctx->stage_ev[k]) cudaEventDestroy(ctx->stage_ev[k]); }
    for (auto *hp : ctx->free_pinned) cudaFreeHost(hp);
    if (ctx->d_fetch_wide) cudaFree(ctx->d_fetch_wide);
    if (ctx->d_fetch_cand) cudaFree(ctx->d_fetch_cand);
    for (auto *b : ctx->d_binom) if (b) cudaFree(b);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->device < 64) g_ctx_on_device[ctx->device]--;
    delete ctx;
    return URLGPU_OK;
}

extern "C" const char *urlgpu_last_error(urlgpu_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int urlgpu_set_stream(urlgpu_ctx *ctx, void *s) {
    if (!ctx) return URLGPU_ERR_ARG;
    fold_events(ctx);
    // pooled device blocks are recycled in stream order: drain the old stream before work is enqueued on another one
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return URLGPU_OK;
}

extern "C" int urlgpu_synchronize(urlgpu_ctx *ctx) {
    if (!ctx) return URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return URLGPU_OK;
}

extern "C" int urlgpu_stats_reset(urlgpu_ctx *ctx) {
    if (!ctx) return URLGPU_ERR_ARG;
    fold_events(ctx);
    ctx->st = urlgpu_stats{};
    return URLGPU_OK;
}
extern "C" int urlgpu_stats_get(urlgpu_ctx *ctx, urlgpu_stats *out) {
    if (!ctx || !out) return URLGPU_ERR_ARG;
    fold_events(ctx);
    *out = ctx->st;
    return URLGPU_OK;
}
extern "C" int urlgpu_stats_enable_timing(urlgpu_ctx *ctx, int on) {
    if (!ctx) return URLGPU_ERR_ARG;
    fold_events(ctx);
    ctx->timing = on != 0;
    return URLGPU_OK;
}

// ============================================================================================ data upload

static int set_discrete_common(urlgpu_ctx *ctx, const uint8_t *src, bool src_on_device, int64_t n, int p, const int32_t *cardinality) {
    if (!ctx || !src || !cardinality || n < 1 || p < 1) return ctx ? ctx->fail(URLGPU_ERR_ARG, "set_discrete: bad arguments") : URLGPU_ERR_ARG;
    if (n > (int64_t)2000000000) return ctx->fail(URLGPU_ERR_LIMIT, "set_discrete: more than 2e9 records");
    CK(cudaSetDevice(ctx->device));
    for (int i = 0; i < p; i++)
        if (cardinality[i] < 1 || cardinality[i] > 256) return ctx->fail(URLGPU_ERR_ARG, "set_discrete: cardinality must be in 1..256");
    // a data set of the same shape re-uses the device buffers, and the log table depends on n only
    const bool same_shape = ctx->have_discrete && !ctx->borrowed_discrete && ctx->n == n && ctx->p == p;
    if (!same_shape) { free_discrete(ctx); ctx->t16_overflowed.clear(); }
    ctx->have_discrete = false;
    ctx->n = n; ctx->p = p;
    ctx->n_stride = (n + 15) / 16 * 16;
    ctx->card.assign(cardinality, cardinality + p);
    if (!same_shape) {
        CK(cudaMalloc(&ctx->d_codes, (size_t)ctx->n_stride * p));
        CK(cudaMemsetAsync(ctx->d_codes, 0, (size_t)ctx->n_stride * p, ctx->stream));
    }
    CK(cudaMemcpy2DAsync(ctx->d_codes, (size_t)ctx->n_stride, src, (size_t)n, (size_t)n, (size_t)p,
                         src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    if (!same_shape) {
        // the reference's float table ilogi[i] = (float)(i*log(i)) (log_likelihood_calculator.h:30-38), as exact
        // int64 multiples of 2^-23.  Built on the host with libm's log so it is the same table the reference builds.
        std::vector<long long> q((size_t)n + 2);
        q[0] = 0;
        for (int64_t i = 1; i < n + 2; i++) {
            const float l = (float)((int)i * std::log((double)(int)i));
            q[i] = (long long)std::ldexp((double)l, 23);
        }
        CK(cudaMalloc(&ctx->d_qlog, q.size() * sizeof(long long)));
        CK(cudaMemcpyAsync(ctx->d_qlog, q.data(), q.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream)); // q goes out of scope
    } else CK(cudaStreamSynchronize(ctx->stream)); // the caller may reuse its buffer
    ctx->base = (float)(std::log((double)(int)n) / 2); // bic_scoring_function.cpp:13
    ctx->ds_qcfg = ctx->d_qlog; ctx->ds_cfg_min = 1; ctx->ds_base = ctx->base;
    ctx->have_discrete = true;
    ctx->mem_free_sample = 0;
    return URLGPU_OK;
}

extern "C" int urlgpu_share_discrete(urlgpu_ctx *ctx, urlgpu_ctx *owner) {
    if (!ctx || !owner || ctx == owner) return ctx ? ctx->fail(URLGPU_ERR_ARG, "share_discrete: bad arguments") : URLGPU_ERR_ARG;
    if (ctx->device != owner->device) return ctx->fail(URLGPU_ERR_ARG, "share_discrete: the contexts are on different devices");
    if (!owner->have_discrete || owner->borrowed_discrete) return ctx->fail(URLGPU_ERR_ARG, "share_discrete: the owner holds no data set of its own");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(owner->stream)); // the owner's upload has landed
    free_discrete(ctx);
    ctx->n = owner->n; ctx->p = owner->p; ctx->n_stride = owner->n_stride; ctx->card = owner->card;
    ctx->d_codes = owner->d_codes; ctx->d_qlog = owner->d_qlog; ctx->base = owner->base;
    ctx->ds_qcfg = ctx->d_qlog; ctx->ds_cfg_min = 1; ctx->ds_base = ctx->base;
    ctx->have_discrete = true; ctx->borrowed_discrete = true;
    ctx->mem_free_sample = 0;
    return URLGPU_OK;
}

constexpr int64_t kFnmlMaxRecords = 238609293;   // 9 * (n + 1) <= INT_MAX: the largest fNML data set of a child of arity >= 2

// Chooses what the K1 kernels compute for `variable`: BIC (log_likelihood - tVal * ln(N)/2, bic_scoring_function.cpp:73) or
// fNML (log_likelihood - sum_j log C(N_ij, r_v), fnml_scoring_function.cpp:28-74).  The fNML per-configuration table is
// qlog[N] + round(2^23 * (float)log C(N, r_v)): the exact-integer contract of bic_kernels.cuh extended by one more float
// table of the reference, so an fNML score is again independent of summation order, path and GPU count.
static int select_discrete_score(urlgpu_ctx *ctx, int score_type, int variable, double param) {
    ctx->ds_ess = 0.f; ctx->ds_scale = 1.0 / 8388608.0;
    if (score_type == URLGPU_BDEU) {
        // BDeu (bdeu_scoring_function.cpp): lgamma terms evaluated in the direct-counting kernels (score_configs_bdeu); `param` = ess
        if (!(param > 0) || !std::isfinite(param)) return ctx->fail(URLGPU_ERR_ARG, "BDeu: the equivalent sample size (the lambda argument) must be positive");
        if (ctx->n > 100000000) return ctx->fail(URLGPU_ERR_LIMIT, "BDeu: more than 1e8 records overflow the 2^-30 fixed-point accumulator");
        ctx->ds_qcfg = ctx->d_qlog; ctx->ds_cfg_min = 1; ctx->ds_base = 0.f;
        ctx->ds_ess = (float)param; ctx->ds_scale = 1.0 / 1073741824.0;
        return URLGPU_OK;
    }
    if (score_type != URLGPU_FNML) {
        ctx->ds_qcfg = ctx->d_qlog; ctx->ds_cfg_min = 1; ctx->ds_base = ctx->base;
        return URLGPU_OK;
    }
    const int r = ctx->card[variable];
    // the table covers N = 0..n+1, and for r >= 2 every entry goes through regret::r2, whose Szpankowski branch evaluates
    // 9 * N in int exactly as the reference writes it: that wraps from N = 238 609 295 on (NaN, then wrong values)
    if (r >= 2 && ctx->n > kFnmlMaxRecords)
        return ctx->fail(URLGPU_ERR_LIMIT, "fNML: more than " + std::to_string(kFnmlMaxRecords) + " records with a child of arity " + std::to_string(r) +
                                               ": the regret C(N, 2) of the reference computes 9 * N in int, which overflows at N = " +
                                               std::to_string(kFnmlMaxRecords + 2));
    auto it = ctx->d_qfnml.find(r);
    if (it == ctx->d_qfnml.end()) {
        const int64_t n = ctx->n;
        std::vector<float> lr = regret::log_regret(n + 1, r);
        std::vector<long long> q((size_t)n + 2);
        q[0] = 0;
        for (int64_t i = 0; i < n + 2; i++) {
            if (!std::isfinite(lr[(size_t)i]))
                return ctx->fail(URLGPU_ERR_LIMIT, "fNML: the regret C(N, r) of arity " + std::to_string(r) + " overflows float32 at N = " + std::to_string(i) +
                                                   " (the reference would store -inf)");
            long long ql = 0;
            if (i > 0) { const float l = (float)((int)i * std::log((double)(int)i)); ql = (long long)std::ldexp((double)l, 23); }
            q[(size_t)i] = ql + std::llrint(std::ldexp((double)lr[(size_t)i], 23));
        }
        long long *d = nullptr;
        CK(cudaMalloc(&d, q.size() * sizeof(long long)));
        CK(cudaMemcpyAsync(d, q.data(), q.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        it = ctx->d_qfnml.emplace(r, d).first;
    }
    ctx->ds_qcfg = it->second; ctx->ds_cfg_min = 0; ctx->ds_base = 0.f;
    return URLGPU_OK;
}

extern "C" int urlgpu_set_discrete(urlgpu_ctx *ctx, const uint8_t *codes, int64_t n, int p, const int32_t *cardinality) {
    return set_discrete_common(ctx, codes, false, n, p, cardinality);
}
extern "C" int urlgpu_set_discrete_device(urlgpu_ctx *ctx, const uint8_t *d_codes, int64_t n, int p, const int32_t *cardinality) {
    return set_discrete_common(ctx, d_codes, true, n, p, cardinality);
}

// ---- continuous data: the pieces below are the single-GPU urlgpu_set_continuous and, called separately, the
// row-sharded multi-GPU protocol (urlgpu_shard_begin / _moments / _finish, see include/urlgpu.h) ----

static int shard_begin_impl(urlgpu_ctx *ctx, const double *src, bool src_on_device, int64_t n_local, int p) {
    if (!ctx || !src || n_local < 1 || p < 1) return ctx ? ctx->fail(URLGPU_ERR_ARG, "continuous data: bad arguments") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    free_continuous(ctx);
    if (ctx->d_x) { cudaFree(ctx->d_x); ctx->d_x = nullptr; }
    ctx->shard_n = n_local; ctx->cp = p;
    if (src_on_device && ctx->borrow_device_x) { ctx->d_x_view = src; ctx->shard_stride = n_local; } // no copy: the caller keeps the buffer alive until shard_finish
    else { // the engine's own copy has the padded row pitch of the Gram kernel, so it can be standardised in place
        const int64_t pitch = (n_local + kGramKC - 1) / kGramKC * kGramKC;
        CK(cudaMalloc(&ctx->d_x, (size_t)pitch * p * sizeof(double)));
        CK(cudaMemcpy2DAsync(ctx->d_x, (size_t)pitch * sizeof(double), src, (size_t)n_local * sizeof(double), (size_t)n_local * sizeof(double), (size_t)p,
                             src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
        ctx->d_x_view = ctx->d_x;
        ctx->shard_stride = pitch;
    }
    return URLGPU_OK;
}

// sum1[c] = sum_r (x[c][r] - shift[c]), sum2[c] = sum_r (x[c][r] - shift[c])^2 over the attached rows (fixed order)
static int shard_moments_impl(urlgpu_ctx *ctx, const double *shift_host, double *sum1, double *sum2) {
    if (!ctx || !ctx->d_x_view) return ctx ? ctx->fail(URLGPU_ERR_ARG, "shard_moments: call urlgpu_shard_begin first") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int p = ctx->cp;
    const int64_t n = ctx->shard_n;
    DevBuf part(ctx), out(ctx), shift(ctx);
    CK(part.alloc((size_t)p * kRedBlocks * sizeof(double)));
    CK(out.alloc((size_t)2 * p * sizeof(double)));
    if (shift_host) {
        CK(shift.alloc(p * sizeof(double)));
        CK(cudaMemcpyAsync(shift.p, shift_host, p * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    {
        Region rg(ctx, F_STD, 4);
        const dim3 rgrid(kRedBlocks, p);
        const unsigned pb = blocks_for(p, 128);
        for (int mode = 0; mode < 2; mode++) {
            if ((mode == 0 && !sum1) || (mode == 1 && !sum2)) continue;
            col_partial_kernel<<<rgrid, kRedThreads, 0, s>>>(ctx->d_x_view, n, ctx->shard_stride, shift_host ? shift.as<double>() : nullptr, mode, part.as<double>());
            col_combine_kernel<<<pb, 128, 0, s>>>(part.as<double>(), p, out.as<double>() + (size_t)mode * p);
        }
    }
    if (sum1) CK(cudaMemcpyAsync(sum1, out.as<double>(), p * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (sum2) CK(cudaMemcpyAsync(sum2, out.as<double>() + p, p * sizeof(double), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// z = (x - mean)/dev on the attached rows (BIC_OLS.cpp:76-77), partial Gram of these rows; n_total = rows of the whole data set
static int shard_finish_impl(urlgpu_ctx *ctx, const double *mean_host, const double *dev_host, int64_t n_total, bool keep_z) {
    if (!ctx || !ctx->d_x_view || !mean_host || !dev_host) return ctx ? ctx->fail(URLGPU_ERR_ARG, "shard_finish: call urlgpu_shard_begin first") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int p = ctx->cp;
    const int64_t n = ctx->shard_n;
    DevBuf md(ctx), gpart(ctx), g(ctx);
    CK(md.alloc((size_t)2 * p * sizeof(double)));
    CK(cudaMemcpyAsync(md.p, mean_host, p * sizeof(double), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(md.as<double>() + p, dev_host, p * sizeof(double), cudaMemcpyHostToDevice, s));
    // standardise in place when the engine owns the (padded) copy, else into a cached padded buffer
    const int64_t z_stride = (n + kGramKC - 1) / kGramKC * kGramKC;
    double *zbuf = ctx->d_x;
    const bool borrowed = zbuf == nullptr;
    if (borrowed) { // caller's device buffer is left untouched
        const size_t need = (size_t)z_stride * p * sizeof(double);
        if (ctx->zcache_cap < need) { if (ctx->d_zcache) cudaFree(ctx->d_zcache); ctx->d_zcache = nullptr; ctx->zcache_cap = 0; CK(cudaMalloc(&ctx->d_zcache, need)); ctx->zcache_cap = need; }
        zbuf = ctx->d_zcache;
    }
    {
        Region rg(ctx, F_STD, 1);
        standardise_kernel<<<dim3(ctx->sm_count * 2, p), 256, 0, s>>>(ctx->d_x_view, n, ctx->shard_stride, md.as<double>(), md.as<double>() + p, zbuf, z_stride);
    }
    {
        Region rg(ctx, F_GRAM, 2);
        const int tiles = (p + kGramTile - 1) / kGramTile;
        const int pairs = tiles * (tiles + 1) / 2;
        // row slices (multiples of the chunk): enough CTAs to fill the machine several times over, at least 1024 records each
        // (beyond 65 535 * 8192 records the slices grow instead: gridDim.y holds at most 65 535)
        int64_t rps = std::max<int64_t>(1024, std::min<int64_t>(8192, z_stride * pairs / ((int64_t)ctx->sm_count * 8)));
        rps = std::max<int64_t>(rps, (z_stride + 65534) / 65535);
        rps = (rps + kGramKC - 1) / kGramKC * kGramKC;
        const int slices = (int)((z_stride + rps - 1) / rps);
        CK(gpart.alloc((size_t)slices * p * p * sizeof(double)));
        CK(g.alloc((size_t)p * p * sizeof(double)));
        gram_partial_kernel<<<dim3(pairs, slices), kGramThreads, kGramSmemBytes, s>>>(zbuf, z_stride, p, rps, tiles, gpart.as<double>());
        gram_combine_kernel<<<blocks_for((uint64_t)p * p, 256), 256, 0, s>>>(gpart.as<double>(), p, slices, g.as<double>());
        ctx->st.gram_flops += 2.0 * (double)n * p * p;
    }
    ctx->h_gram.resize((size_t)p * p);
    CK(cudaMemcpyAsync(ctx->h_gram.data(), g.p, (size_t)p * p * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (ctx->d_gram) { cudaFree(ctx->d_gram); ctx->d_gram = nullptr; }
    CK(cudaMalloc(&ctx->d_gram, (size_t)p * p * sizeof(double)));
    CK(cudaMemcpyAsync(ctx->d_gram, g.p, (size_t)p * p * sizeof(double), cudaMemcpyDeviceToDevice, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    if (!borrowed) { if (keep_z) ctx->d_z = zbuf; else cudaFree(zbuf); }
    ctx->d_x = nullptr; ctx->d_x_view = nullptr;
    ctx->cn = n_total;
    ctx->gram_dmax = 0;
    for (int i = 0; i < p; i++) ctx->gram_dmax = std::max(ctx->gram_dmax, ctx->h_gram[(size_t)i * p + i]);
    ctx->have_gram = true;
    return URLGPU_OK;
}

static int set_continuous_common(urlgpu_ctx *ctx, const double *src, bool src_on_device, int64_t n, int p) {
    if (!ctx || !src || n < 2 || p < 1) return ctx ? ctx->fail(URLGPU_ERR_ARG, "set_continuous: bad arguments") : URLGPU_ERR_ARG;
    ctx->borrow_device_x = false;
    int rc = shard_begin_impl(ctx, src, src_on_device, n, p);
    if (rc) return rc;
    std::vector<double> s1(p), s2(p), mean(p), dev(p);
    // mean_x = sum/n (BIC_OLS.cpp:69); dev_x = sqrt(var(x - mean_x)), Armadillo's variance with N-1 (:70-71)
    rc = shard_moments_impl(ctx, nullptr, s1.data(), nullptr);
    if (rc) return rc;
    for (int c = 0; c < p; c++) mean[c] = s1[c] / (double)n;
    rc = shard_moments_impl(ctx, mean.data(), s1.data(), s2.data());
    if (rc) return rc;
    for (int c = 0; c < p; c++) dev[c] = std::sqrt((s2[c] - s1[c] * s1[c] / (double)n) / ((double)n - 1.0));
    return shard_finish_impl(ctx, mean.data(), dev.data(), n, false);
}

extern "C" int urlgpu_set_continuous(urlgpu_ctx *ctx, const double *x, int64_t n, int p) { return set_continuous_common(ctx, x, false, n, p); }
extern "C" int urlgpu_set_continuous_device(urlgpu_ctx *ctx, const double *x, int64_t n, int p) { return set_continuous_common(ctx, x, true, n, p); }

extern "C" int urlgpu_shard_begin(urlgpu_ctx *ctx, const double *x_colmajor, int64_t n_local, int p, int on_device) {
    if (ctx) ctx->borrow_device_x = on_device != 0;
    return shard_begin_impl(ctx, x_colmajor, on_device != 0, n_local, p);
}
extern "C" int urlgpu_shard_moments(urlgpu_ctx *ctx, const double *shift, double *sum1, double *sum2) { return shard_moments_impl(ctx, shift, sum1, sum2); }
extern "C" int urlgpu_shard_finish(urlgpu_ctx *ctx, const double *mean, const double *dev, int64_t n_total) { return shard_finish_impl(ctx, mean, dev, n_total, false); }

extern "C" int urlgpu_get_gram(urlgpu_ctx *ctx, double *g) {
    if (!ctx || !g) return URLGPU_ERR_ARG;
    if (!ctx->have_gram) return ctx->fail(URLGPU_ERR_ARG, "get_gram: no continuous data set");
    memcpy(g, ctx->h_gram.data(), ctx->h_gram.size() * sizeof(double));
    return URLGPU_OK;
}
extern "C" int urlgpu_set_gram(urlgpu_ctx *ctx, const double *g, int64_t n_total, int p) {
    if (!ctx || !g || p < 1 || n_total < 2) return ctx ? ctx->fail(URLGPU_ERR_ARG, "set_gram: bad arguments") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    free_continuous(ctx);
    ctx->cn = n_total; ctx->cp = p;
    CK(cudaMalloc(&ctx->d_gram, (size_t)p * p * sizeof(double)));
    CK(cudaMemcpyAsync(ctx->d_gram, g, (size_t)p * p * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream)); // the caller may reuse its buffer
    ctx->h_gram.assign(g, g + (size_t)p * p);
    ctx->gram_dmax = 0;
    for (int i = 0; i < p; i++) ctx->gram_dmax = std::max(ctx->gram_dmax, g[(size_t)i * p + i]);
    ctx->have_gram = true;
    return URLGPU_OK;
}

// Measured FP64 issue rates of this device (TFLOP/s): plain DFMA and the DMMA (mma.sync.m8n8k4.f64) tensor path.
// Best of three timed launches after one warm-up, CUDA events on the context's stream.
extern "C" int urlgpu_probe_fp64(urlgpu_ctx *ctx, double *dfma_tflops, double *dmma_tflops) {
    if (!ctx) return URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    DevBuf out(ctx);
    CK(out.alloc(64));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const int iters = 1 << 14, threads = 256;
    const unsigned grid = (unsigned)ctx->sm_count * 8;
    double best[2] = {0, 0};
    for (int kind = 0; kind < 2; kind++)
        for (int rep = 0; rep < 4; rep++) {
            CK(cudaEventRecord(e0, s));
            if (kind == 0) probe_dfma_kernel<<<grid, threads, 0, s>>>(out.as<double>(), iters, 0.999999, 1e-9);
            else probe_dmma_kernel<<<grid, threads, 0, s>>>(out.as<double>(), iters, 0.999999, 1e-9);
            CK(cudaEventRecord(e1, s));
            CK(cudaEventSynchronize(e1));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            // dfma: 2 flop x 8 chains per thread and iteration; dmma: 8 tiles x (8*8*4*2 = 512 flop) per warp and iteration
            const double flop = kind == 0 ? 2.0 * 8 * iters * (double)threads * grid : 512.0 * 8 * iters * (double)(threads / 32) * grid;
            if (rep > 0) best[kind] = std::max(best[kind], flop / (ms * 1e-3) / 1e12);
        }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    CK(cudaGetLastError());
    ctx->st.launches_total += 8; ctx->st.launches_other += 8;
    if (dfma_tflops) *dfma_tflops = best[0];
    if (dmma_tflops) *dmma_tflops = best[1];
    return URLGPU_OK;
}

// ============================================================================================ scoring

static int candidates_from_mask(urlgpu_ctx *ctx, int p, int variable, const uint64_t *neighbors, int mask_words, std::vector<int> &cand) {
    if (mask_words < 1 || (int64_t)mask_words * 64 < p) return ctx->fail(URLGPU_ERR_ARG, "mask_words too small for the variable count");
    cand.clear();
    for (int i = 0; i < p; i++)
        if (i != variable && ((neighbors[i >> 6] >> (i & 63)) & 1)) cand.push_back(i);
    for (int w = 0; w < mask_words; w++)
        for (int b = 0; b < 64; b++)
            if (w * 64 + b >= p && ((neighbors[w] >> b) & 1)) return ctx->fail(URLGPU_ERR_ARG, "mask names a variable >= p");
    return URLGPU_OK;
}

static int ensure_tables(urlgpu_ctx *ctx, size_t elems) {
    if (ctx->tables_cap >= elems) return URLGPU_OK;
    if (ctx->d_tables) cudaFree(ctx->d_tables);
    ctx->d_tables = nullptr; ctx->tables_cap = 0;
    CK(cudaMalloc(&ctx->d_tables, elems * sizeof(int)));
    ctx->tables_cap = elems;
    return URLGPU_OK;
}

namespace {
constexpr uint32_t kTier0Cells = 12 * 1024;                 // 48 KB of shared memory, several CTAs per SM
constexpr uint64_t kCellLimit = (uint64_t)1 << 30;          // 4 GB table
constexpr size_t kBatchTableElems = (size_t)12 << 20;       // 48 MB of tables per batch: stays L2 resident
}

static CandInfo make_candinfo(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, int K) {
    CandInfo ci{};
    ci.c = (int)cand.size(); ci.v = variable; ci.rv = ctx->card[variable]; ci.max_parents = K;
    for (int i = 0; i < ci.c; i++) { ci.var[i] = cand[i]; ci.card[i] = ctx->card[cand[i]]; }
    return ci;
}

// A batch of B global-tier tables (zeroed, at their table_off in `tables`): count the rows of every set in row slices,
// then score the tables into acc[set] in configuration chunks; both grids hold ~8 CTAs per SM over the batch.
template <class Sets>
static void launch_count_global(urlgpu_ctx *ctx, const BicData &bd, const Sets &fam, const GlobalSet *d_sets, size_t B, int *tables) {
    const int threads = 256;
    int64_t R = std::max<int64_t>(1, (int64_t)(ctx->sm_count * 8 + B - 1) / (int64_t)B);
    int64_t rps = (bd.n + R - 1) / R;
    rps = std::max<int64_t>((rps + 15) / 16 * 16, 16 * threads);
    R = (bd.n + rps - 1) / rps;
    bic_count_global_kernel<<<dim3((unsigned)B, (unsigned)R), threads, 0, ctx->stream>>>(bd, fam, d_sets, tables, rps);
}
static void launch_score_tables(urlgpu_ctx *ctx, const BicData &bd, int rv, const GlobalSet *d_sets, size_t B, uint32_t max_cells, const int *tables, long long *acc) {
    const int threads = 256;
    const int64_t nconf = max_cells / rv;
    const int64_t chunks = std::max<int64_t>(1, std::min<int64_t>((nconf + threads * 4 - 1) / (threads * 4), (ctx->sm_count * 8 + (int64_t)B - 1) / (int64_t)B));
    const int64_t cpc = (nconf + chunks - 1) / chunks;
    bic_score_tables_kernel<<<dim3((unsigned)B, (unsigned)chunks), threads, 0, ctx->stream>>>(bd, rv, d_sets, tables, acc, cpc);
}

// ------------------------------------------------------------------------------------------------------------
// Cube path: count only the root tables from the rows, derive every other table of the family by summing one
// digit out of a table one variable larger (cube_derive_kernel).  Candidates are re-ordered by ascending arity
// ("cube bits"); the parent of a set is the set plus its lowest missing cube bit, so the digit that is summed
// out always has the smallest arity available and sits right after the child digit.  Layers above max_parents
// exist only as ancestors (they contain the lowest cube bits), which cuts the number of row-counting passes:
// with c=16, K=11 the 4368 sets of layer 11 are derived from 1365 roots of layer 12.
// ------------------------------------------------------------------------------------------------------------
namespace {
struct CubeSet {
    uint32_t cube_mask, res_mask;
    uint64_t cells, off;
    int parent;       // index in the layer above
    int leaf_child;   // a set that holds cube bit 0: index of its leaf child (the set without bit 0) in the layer below, or -1
    uint32_t Bc, r;
    bool t16;         // the table is stored with uint16 cells
};
inline uint32_t gosper_next(uint32_t v) {
    const uint32_t t = (v | (v - 1)) + 1;
    return t | ((((t & (~t + 1)) / (v & (~v + 1))) >> 1) - 1);
}
} // namespace


// Truly asynchronous H2D upload of a host array: the bytes are copied into one of the context's two pinned arenas
// (bump allocated) and sent with cudaMemcpyAsync.  stage_begin() switches to the other arena and waits only for the
// call that used it two calls ago; stage_end() marks the end of the current call.
static int stage_begin(urlgpu_ctx *ctx) {
    ctx->stage_cur ^= 1;
    const int k = ctx->stage_cur;
    DbgTimer dt(ctx, 0);
    if (!ctx->stage_ev[k]) CK(cudaEventCreateWithFlags(&ctx->stage_ev[k], cudaEventDisableTiming));
    else CK(cudaEventSynchronize(ctx->stage_ev[k]));
    ctx->stage_used = 0;
    return URLGPU_OK;
}
static int stage_end(urlgpu_ctx *ctx) {
    const int k = ctx->stage_cur;
    if (ctx->stage_ev[k]) CK(cudaEventRecord(ctx->stage_ev[k], ctx->stream));
    return URLGPU_OK;
}
static int h2d_async(urlgpu_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (bytes == 0) return URLGPU_OK;
    const int k = ctx->stage_cur;
    const size_t need = (ctx->stage_used + 255) / 256 * 256 + bytes;
    if (need > ctx->stage_cap[k]) {
        DbgTimer dt(ctx, 4);
        // the arena is full: drain the stream (pending copies read from it), then grow
        CK(cudaStreamSynchronize(ctx->stream));
        if (bytes > ctx->stage_cap[k]) {
            if (ctx->h_stage[k]) cudaFreeHost(ctx->h_stage[k]);
            ctx->h_stage[k] = nullptr; ctx->stage_cap[k] = 0;
            const size_t cap = std::max<size_t>(bytes * 2, (size_t)32 << 20);
            CK(cudaHostAlloc(reinterpret_cast<void **>(&ctx->h_stage[k]), cap, cudaHostAllocDefault));
            ctx->stage_cap[k] = cap;
        }
        ctx->stage_used = 0;
    }
    const size_t off = (ctx->stage_used + 255) / 256 * 256;
    DbgTimer dt(ctx, 3);
    memcpy(ctx->h_stage[k] + off, src, bytes);
    ctx->stage_used = off + bytes;
    CK(cudaMemcpyAsync(dst, ctx->h_stage[k] + off, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return URLGPU_OK;
}

// part / parts: score only the sub-forest of the roots i with i % parts == part (and everything derived from them); the parts
// are disjoint and cover the family (urlgpu_score_part: one variable's K1 work split over several GPUs)
static int bic_score_family_cube(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, int K, float *d_table, uint64_t *n_scored, bool *used, const RankSpace &om, int part = 0, int parts = 1, int *d_ovf = nullptr) {
    *used = false;
    cudaStream_t s = ctx->stream;
    { int rc_ = stage_begin(ctx); if (rc_) return rc_; }
    static const bool dbg = getenv("URLGPU_DEBUG_TIMING") != nullptr;
    auto cpu_ms = [] { timespec ts; clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    const double C0 = dbg ? cpu_ms() : 0.0;
    auto tnow = [] { return std::chrono::steady_clock::now(); };
    auto tms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    const auto T0 = tnow();
    const int c = (int)cand.size();
    const int Kc = std::min(K, c);
    const int rv = ctx->card[variable];
    const uint64_t n = (uint64_t)ctx->n;
    if (c == 0) return URLGPU_OK; // only the empty set: the direct path handles it
    // cube order: ascending arity, ties by variable index
    std::vector<int> perm(c);
    for (int i = 0; i < c; i++) perm[i] = i;
    std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return ctx->card[cand[a]] < ctx->card[cand[b]]; });
    std::vector<int> cube_vars(c);
    std::vector<uint64_t> ccard(c), prefix(c + 1, 1);
    for (int i = 0; i < c; i++) { cube_vars[i] = cand[perm[i]]; ccard[i] = (uint64_t)ctx->card[cube_vars[i]]; }
    for (int i = 0; i < c; i++) prefix[i + 1] = std::min<uint64_t>(prefix[i] * ccard[i], (uint64_t)1 << 40);
    CandInfo ci_cube = make_candinfo(ctx, variable, cube_vars, K);
    CandInfo ci_res = make_candinfo(ctx, variable, cand, K);
    BicData bd{ctx->d_codes, ctx->n, ctx->n_stride, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, ctx->ds_base, ctx->ds_ess, ctx->ds_scale};
    const uint32_t tier1_cells = (uint32_t)((ctx->smem_optin - 2048) / sizeof(int));

    // ---- enumerate layers 0..Lmax (layers above Kc: only sets containing the lowest l-Kc cube bits) ----
    const int Lmax = std::min(Kc + 2, c);
    std::vector<std::vector<CubeSet>> layers(Lmax + 1);
    // per-byte lookup tables: cells factor and result-order mask of every 8-bit group of cube bits
    std::vector<uint64_t> cellsT(4 * 256, 1);
    std::vector<uint32_t> resT(4 * 256, 0);
    for (int g = 0; g < 4; g++)
        for (int m = 0; m < 256; m++) {
            uint64_t f = 1; uint32_t rm = 0;
            for (int b = 0; b < 8; b++) {
                const int i = g * 8 + b;
                if (i < c && ((m >> b) & 1)) { f *= ccard[i]; rm |= 1u << perm[i]; }
            }
            cellsT[g * 256 + m] = f; resT[g * 256 + m] = rm;
        }
    auto make_set = [&](uint32_t cm) {
        CubeSet cs{};
        cs.cube_mask = cm;
        const uint32_t b0 = cm & 255, b1 = (cm >> 8) & 255, b2 = (cm >> 16) & 255, b3 = cm >> 24;
        __uint128_t cells = (__uint128_t)rv * cellsT[b0] * cellsT[256 + b1];
        cells = std::min<__uint128_t>(cells, kCellLimit + 1) * cellsT[512 + b2];
        cells = std::min<__uint128_t>(cells, kCellLimit + 1) * cellsT[768 + b3];
        cs.cells = (uint64_t)std::min<__uint128_t>(cells, kCellLimit + 1);
        cs.res_mask = resT[b0] | resT[256 + b1] | resT[512 + b2] | resT[768 + b3];
        cs.parent = -1;
        cs.leaf_child = -1;
        return cs;
    };
    for (int l = 0; l <= Lmax; l++) {
        const int j = std::max(0, l - Kc);      // forced low bits
        const int free_bits = c - j, pick = l - j;
        const uint32_t lowmask = (j ? ((1u << j) - 1) : 0);
        auto &L = layers[l];
        if (pick == 0) { L.push_back(make_set(lowmask)); continue; }
        uint32_t v = (1u << pick) - 1;
        const uint64_t lim = (uint64_t)1 << free_bits;
        while ((uint64_t)v < lim) {
            L.push_back(make_set((v << j) | lowmask));
            if (pick == free_bits) break;
            v = gosper_next(v);
        }
    }
    // ---- choose the root layer by a simple cost model (seconds) ----
    auto root_cost = [&](const CubeSet &cs, int l) {
        if (cs.cells > kCellLimit) return 1e30;
        if (cs.cells <= tier1_cells) return (double)n * (l + 1) / 6e12 + 2e-7;
        return 6.5e-6 + (double)cs.cells * 1.95e-12; // fitted to the slice-count kernel on B200 (n = 1e6)
    };
    auto derive_cost = [&](const CubeSet &cs, int /*l*/, uint64_t rdrop) { return (double)cs.cells * 4.0 * (double)(rdrop + 1) / 5e12 + 1e-7; };
    // free device memory is sampled once per data set: cudaMemGetInfo blocks for ~1.5 ms while the GPU is busy (measured)
    if (ctx->mem_free_sample == 0) {
        size_t free_b = 0, total_b = 0;
        DbgTimer dt(ctx, 1);
        CK(cudaMemGetInfo(&free_b, &total_b));
        ctx->mem_free_sample = free_b + (ctx->cubeA_cap + ctx->cubeB_cap) * sizeof(int);
    }
    // The test below is deliberately generous: it counts every table of a layer, although fused roots and leaf sets are never
    // materialised (the buffers that are really allocated, needA / needB further down, are several times smaller), and several
    // contexts on one device (EnginePool, `score -t T`) each see the whole free memory.  Dividing the budget by the number of
    // contexts pushed big families to root layer K (3x the row counting; measured 314 -> 716 ms per step at configs[3]).  An
    // allocation that does fail is handled where it happens: cached pool blocks are released, and if that is not enough
    // the family takes the direct path.
    const double mem_budget = (double)ctx->mem_free_sample * 0.7;
    std::vector<double> layer_cells(Lmax + 1, 0.0);
    for (int l = 0; l <= Lmax; l++)
        for (auto &cs : layers[l]) layer_cells[l] += (double)((cs.cells + 3) / 4 * 4);
    int Lstar = -1;
    double best = 1e300;
    for (int Ls = Kc; Ls <= Lmax; Ls++) {
        double cost = 0, maxl = 0;
        for (auto &cs : layers[Ls]) cost += root_cost(cs, Ls);
        if (cost >= 1e29) continue; // a root table above the 2^30-cell limit
        for (int l = Kc; l < Ls; l++)
            for (auto &cs : layers[l]) {
                const int z = __builtin_ctz(~cs.cube_mask);
                cost += derive_cost(cs, l, ccard[z]);
            }
        for (int l = 0; l <= Ls; l++) maxl = std::max(maxl, layer_cells[l]);
        if (2.0 * maxl * 4.0 > mem_budget) continue;
        if (cost < best) { best = cost; Lstar = Ls; }
    }
    if (Lstar < 0) return URLGPU_OK; // does not fit: caller falls back to the direct path
    // ---- which roots go through bic_root_kernel, and which of those are fused (decided before the offsets: a fused root's
    // table is never materialised, so it takes no room in the layer buffer) ----
    const bool score_roots = Lstar <= Kc;
    TreeVar tv{};
    const uint32_t RB = ctx->root_budget, seg_cap = ctx->root_seg_cap;
    bool packed_ok = ctx->n >= 65536 && ctx->use_slice_count;
    uint64_t Pd = 1;
    int dmax = 0;
    if (packed_ok) {
        uint64_t maxr = (uint64_t)rv;
        for (int i = 0; i < c; i++) maxr = std::max(maxr, ccard[i]);
        tv.c = c; tv.rv = rv;
        tv.w = maxr <= 4 ? 2 : maxr <= 16 ? 4 : 8;
        if ((c + 1) * tv.w > 64) packed_ok = false;
        for (int i = 0; i < c; i++) tv.card[i] = (uint16_t)ccard[i];
        tv.pre[0] = 1;
        for (int b = 0; b < kPreMax; b++) tv.pre[b + 1] = (uint32_t)std::min<uint64_t>((uint64_t)tv.pre[b] * (b < c ? ccard[b] : 1), (uint64_t)1 << 31);
        for (int b = 0; b <= kPreMax; b++) tv.magic[b] = tv.pre[b] > 1 ? 0xFFFFFFFFu / tv.pre[b] : 0;
        for (int b = 0; b < kPreMax; b++) tv.cmagic[b] = b < c && ccard[b] > 1 ? (uint32_t)(0xFFFFFFFFull / ccard[b]) : 0;
        while (dmax < c && dmax < kTreeMaxZone && Pd * ccard[c - 1 - dmax] <= kTreeMaxBuckets) { Pd *= ccard[c - 1 - dmax]; dmax++; }
        tv.dmax = dmax; tv.P_dmax = (uint32_t)Pd;
    }
    // slicing of root P along its top digits until the slice fits the budget; the `zf` lowest digits stay inside the slice
    auto slice_root = [&](uint32_t P, int zf, TreeRoot &r) {
        uint64_t H = 1;
        for (int b = zf; b < c; b++) if ((P >> b) & 1) { H *= ccard[b]; if (H > ((uint64_t)1 << 40)) H = (uint64_t)1 << 40; }
        const uint64_t U0 = (uint64_t)rv * tv.pre[zf];
        if (U0 > RB) return false;
        int depth = 0;
        uint64_t nslices = 1, nseg = 1;
        while (U0 * H > RB) {
            const int b = c - 1 - depth;
            if (depth == dmax || b < zf) return false;
            depth++;
            if ((P >> b) & 1) { H /= ccard[b]; nslices *= ccard[b]; } else nseg *= ccard[b];
            if (nseg > ((uint64_t)1 << 22)) return false;
        }
        if (nslices > 0x3fffffffull) return false;
        r = TreeRoot{};
        r.mask = P; r.nslices = (uint32_t)nslices; r.H = (uint32_t)H; r.nseg = (uint32_t)nseg; r.z = (uint8_t)zf;
        r.fstride[0] = 1;
        for (int b = 0; b < zf; b++) r.fstride[b + 1] = (uint16_t)((uint32_t)rv * tv.pre[b]);
        uint32_t hs = (uint32_t)U0;
        for (int b = zf; b < c - depth; b++)
            if ((P >> b) & 1) { r.fstride[b + 1] = (uint16_t)hs; hs *= (uint32_t)ccard[b]; }
        for (int f = 0; f <= c; f++)
            if (r.fstride[f]) r.gmask |= (uint8_t)(1u << (f * tv.w / 8));
        for (int g = 0; g < 8; g++) if ((r.gmask >> g) & 1) r.glist[r.ng++] = (uint8_t)g;
        uint64_t w = 1;
        for (int b = c - depth; b < c; b++) {
            const uint32_t mg = ccard[b] > 1 ? (uint32_t)(0xFFFFFFFFull / ccard[b]) : 0;
            if ((P >> b) & 1) { r.pres_card[r.npres] = (uint16_t)ccard[b]; r.pres_weight[r.npres] = (uint32_t)w; r.pres_magic[r.npres] = mg; r.npres++; }
            else { r.abs_card[r.nabs] = (uint16_t)ccard[b]; r.abs_weight[r.nabs] = (uint32_t)w; r.abs_magic[r.nabs] = mg; r.nabs++; }
            w *= ccard[b];
        }
        r.q_stride = (uint32_t)(Pd / w);
        return true;
    };
    std::vector<char> root_kind(layers[Lstar].size(), 0); // 0: small table or RED path, 1: plain root of bic_root_kernel, 2: fused
    std::vector<std::vector<char>> mine(Lstar + 1);        // sets of this call's sub-forest (all of them when parts == 1)
    mine[Lstar].assign(layers[Lstar].size(), 1);
    if (parts > 1) for (size_t i = 0; i < layers[Lstar].size(); i++) mine[Lstar][i] = (int)(i % (size_t)parts) == part;
    if (packed_ok) {
        uint64_t total_slices = 0;
        auto &R = layers[Lstar];
        for (size_t i = 0; i < R.size(); i++) {
            if (!mine[Lstar][i]) continue;
            if (R[i].cells <= tier1_cells) continue;
            const uint32_t P = R[i].cube_mask;
            const int run = std::min(c, (int)__builtin_ctz(~P));
            TreeRoot r{};
            // layers above Kc hold only sets with their lowest bits forced: the droppable bits of P start at bfirst
            const int bfirst = std::max(0, Lstar - 1 - Kc);
            if (!score_roots && ctx->fuse_roots && Lstar >= 1 && run > bfirst && run <= kRootMaxChild && run <= kPreMax && slice_root(P, run, r)) root_kind[i] = 2;
            else if (slice_root(P, 0, r)) root_kind[i] = 1;
            if (root_kind[i]) total_slices += r.nslices;
        }
        if (total_slices < (uint64_t)std::max(1, 128 / parts) || total_slices > 0x7fffffffull) std::fill(root_kind.begin(), root_kind.end(), 0); // too few CTAs to fill the machine
    }
    // ---- offsets and parent links ----
    // Layer Lstar lives in buffer A, Lstar-1 in B, Lstar-2 in A again, ...: each buffer is sized for its own layers only.
    // Tables that are never materialised take no room: fused roots, and below the root layer every set without cube
    // bit 0 (nothing is derived from it, its table is only scored on the fly).
    const bool use16 = ctx->table16 && d_ovf != nullptr;
    size_t needA = 0, needB = 0;
    for (int l = 0; l <= Lstar; l++) {
        uint64_t off = 0;
        for (size_t i = 0; i < layers[l].size(); i++) {
            auto &cs = layers[l][i];
            cs.off = off;
            cs.t16 = false;
            if (l == Lstar && root_kind[i] == 2) continue;          // fused root
            if (l < Lstar && (cs.cube_mask & 1u) == 0) continue;    // leaf
            cs.t16 = use16 && l < Lstar && l >= ctx->table16_min_layer;   // root tables stay int32 (several kernels write them)
            off += cs.t16 ? ((cs.cells + 1) / 2 + 3) / 4 * 4 : (cs.cells + 3) / 4 * 4;
        }
        if (((Lstar - l) & 1) == 0) needA = std::max<size_t>(needA, off); else needB = std::max<size_t>(needB, off);
        if (l < Lstar) {
            auto &P = layers[l + 1];
            for (size_t i = 0; i < layers[l].size(); i++) {
                auto &cs = layers[l][i];
                const int z = __builtin_ctz(~cs.cube_mask); // lowest missing cube bit (< c because l < Lstar <= c)
                const uint32_t pm = cs.cube_mask | (1u << z);
                auto it = std::lower_bound(P.begin(), P.end(), pm, [](const CubeSet &a, uint32_t m) { return a.cube_mask < m; });
                if (it == P.end() || it->cube_mask != pm) return ctx->fail(URLGPU_ERR_INTERNAL, "cube: parent set missing");
                cs.parent = (int)(it - P.begin());
                cs.Bc = (uint32_t)prefix[z];
                cs.r = (uint32_t)ccard[z];
                if (z == 0) it->leaf_child = (int)i;   // a leaf: its parent is the set plus bit 0
            }
        }
    }
    for (int l = Lstar - 1; l >= 0; l--) { // a set belongs to the sub-forest of its parent
        mine[l].resize(layers[l].size());
        for (size_t i = 0; i < layers[l].size(); i++) mine[l][i] = mine[l + 1][layers[l][i].parent];
    }
    needA = std::max<size_t>(needA, 4); needB = std::max<size_t>(needB, 4);
    // layer buffers: on an allocation failure give the pool's cached blocks back to the driver and retry once; if the device
    // still cannot hold them (other contexts took the memory since the sample) the family goes through the direct path
    auto grow = [&](int *&buf, size_t &cap, size_t need) -> bool {
        if (cap >= need) return true;
        if (buf) cudaFree(buf);
        buf = nullptr; cap = 0;
        if (cudaMalloc(&buf, need * sizeof(int)) != cudaSuccess) {
            cudaGetLastError();
            for (size_t i = 0; i < ctx->pool.size();) {
                if (!ctx->pool[i].used) { cudaFree(ctx->pool[i].p); ctx->pool.erase(ctx->pool.begin() + i); } else i++;
            }
            if (cudaMalloc(&buf, need * sizeof(int)) != cudaSuccess) { cudaGetLastError(); buf = nullptr; return false; }
        }
        cap = need;
        return true;
    };
    if (!grow(ctx->d_cubeA, ctx->cubeA_cap, needA) || !grow(ctx->d_cubeB, ctx->cubeB_cap, needB)) {
        ctx->mem_free_sample = 0; // re-sample next time
        { int rc_ = stage_end(ctx); if (rc_) return rc_; }
        return URLGPU_OK;          // *used stays false: the caller takes the direct path
    }
    int *bufP = ctx->d_cubeA, *bufC = ctx->d_cubeB;
    const auto T1 = tnow();
    const double C1 = dbg ? cpu_ms() : 0.0;

    size_t max_sets = 0;
    for (int l = 0; l <= Lstar; l++) max_sets = std::max(max_sets, layers[l].size());
    DevBuf dacc(ctx), dres(ctx), dpairs(ctx), dwork(ctx), doffs(ctx), dgsets(ctx);
    // one exact accumulator per set of every layer (a pass over layer l+1 may already score sets of layer l)
    std::vector<size_t> acc_off(Lstar + 2, 0);
    for (int l = 0; l <= Lstar; l++) acc_off[l + 1] = acc_off[l] + layers[l].size();
    CK(dacc.alloc(acc_off[Lstar + 1] * sizeof(long long)));
    CK(cudaMemsetAsync(dacc.p, 0, acc_off[Lstar + 1] * sizeof(long long), s));
    CK(dres.alloc(max_sets * sizeof(uint32_t)));
    CK(dpairs.alloc(max_sets * sizeof(CubePair)));
    std::vector<uint32_t> hres;
    auto finalize_layer = [&](int l) -> int {
        auto &L = layers[l];
        hres.resize(L.size());
        for (size_t i = 0; i < L.size(); i++) hres[i] = mine[l][i] ? L[i].res_mask : 0xffffffffu; // 0xffffffff: not this call's set
        { int rc_ = h2d_async(ctx, dres.p, hres.data(), L.size() * sizeof(uint32_t)); if (rc_) return rc_; }
        Region rg(ctx, F_OTHER, 1);
        cube_finalize_kernel<<<blocks_for(L.size(), 256), 256, 0, s>>>(bd, ci_res, dres.as<uint32_t>(), dacc.as<long long>() + acc_off[l], (int)L.size(), d_table, om);
        return URLGPU_OK;
    };

    // ---- roots: counted from the rows ----
    std::vector<char> fused_root(layers[Lstar].size(), 0); // root tables that never reach HBM: their children come out of the root kernel
    bool fused_any = false;
    {
        auto &R = layers[Lstar];
        std::vector<uint32_t> small_m; std::vector<uint64_t> small_off; std::vector<size_t> small_idx;
        std::vector<GlobalSet> big; std::vector<size_t> big_idx;
        for (size_t i = 0; i < R.size(); i++) {
            if (!mine[Lstar][i]) continue;
            ctx->st.k1_bytes_read += 8.0 * (double)n;  // one packed row word per record and root (L2 resident)
            if (R[i].cells <= tier1_cells) { small_m.push_back(R[i].cube_mask); small_off.push_back(R[i].off); small_idx.push_back(i); }
            else { big.push_back(GlobalSet{R[i].cube_mask, (uint32_t)R[i].cells, R[i].off}); big_idx.push_back(i); }
        }
        // acc of roots is indexed by position in R: small roots are scattered through an index-ordered launch, so
        // split the accumulator ranges: [0, small) in launch order then copy back by index on the host if scoring.
        DevBuf dacc_small(ctx), dacc_big(ctx);
        if (!small_m.empty()) {
            CK(dwork.alloc(small_m.size() * sizeof(uint32_t)));
            CK(doffs.alloc(small_off.size() * sizeof(uint64_t)));
            CK(dacc_small.alloc(small_m.size() * sizeof(long long)));
            { int rc_ = h2d_async(ctx, dwork.p, small_m.data(), small_m.size() * sizeof(uint32_t)); if (rc_) return rc_; }
            { int rc_ = h2d_async(ctx, doffs.p, small_off.data(), small_off.size() * sizeof(uint64_t)); if (rc_) return rc_; }
            // two launches by table size so that small tables get several CTAs per SM
            std::vector<size_t> order(small_m.size());
            Region rg(ctx, F_COUNT, 1);
            uint32_t maxc = 0;
            for (size_t i : small_idx) maxc = std::max<uint32_t>(maxc, (uint32_t)R[i].cells);
            const bool tiny = maxc <= kTier0Cells;
            const int threads = tiny ? (ctx->n >= 65536 ? 256 : 128) : 1024;
            const size_t smem = (tiny ? (size_t)kTier0Cells : (size_t)tier1_cells) * sizeof(int);
            bic_count_smem_kernel<<<(unsigned)small_m.size(), threads, smem, s>>>(bd, MaskSets{ci_cube}, dwork.as<uint32_t>(), nullptr, doffs.as<uint64_t>(), bufP,
                                                                               score_roots ? dacc_small.as<long long>() : nullptr);
        }
        if (!big.empty()) {
            CK(dgsets.alloc(big.size() * sizeof(GlobalSet)));
            CK(dacc_big.alloc(big.size() * sizeof(long long)));
            CK(cudaMemsetAsync(dacc_big.p, 0, big.size() * sizeof(long long), s));
            { int rc_ = h2d_async(ctx, dgsets.p, big.data(), big.size() * sizeof(GlobalSet)); if (rc_) return rc_; }
            // (1) roots whose table can be cut along its top digits are counted in shared-memory slices of the bucketed
            //     packed rows (bic_root_kernel, tree_kernels.cuh).  A root that is only an ancestor (layer K+1) and whose
            //     run of low digits fits one slice is FUSED: its children are marginalised, scored and written by the
            //     same CTA and the root table never reaches HBM.  (2) The rest use global RED atomics.
            std::vector<char> sliced(big.size(), 0);
            std::vector<CubeRoot> croots;
            DevBuf dkeys(ctx), dhist(ctx), doffp(ctx), dcursor(ctx), drows(ctx), dcroots(ctx), dmap(ctx), dtmp(ctx);
            uint64_t rchunk = 0;
            {
                auto &Lc = layers[Lstar > 0 ? Lstar - 1 : 0];
                for (size_t i = 0; i < big.size(); i++) {
                    const int kind = root_kind[big_idx[i]];
                    if (!kind) continue; // RED path below
                    const uint32_t P = big[i].key;
                    const int run = std::min(c, (int)__builtin_ctz(~P));
                    CubeRoot cr{};
                    if (!slice_root(P, kind == 2 ? run : 0, cr.t)) return ctx->fail(URLGPU_ERR_INTERNAL, "cube: root slicing is not reproducible");
                    if (kind == 2) {
                        cr.nchild = (uint32_t)run;
                        cr.bfirst = (uint16_t)std::max(0, Lstar - 1 - Kc);
                        // children b >= 1 hold bit 0: the root kernel also scores their leaves root \ {b, 0} (layer Lstar - 2 <= Kc)
                        cr.score = (Lstar - 1 <= Kc ? 1 : 0) | (run > std::max<int>(cr.bfirst, 1) ? 2 : 0);
                        for (int b = cr.bfirst; b < run; b++) {
                            const uint32_t cm = P & ~(1u << b);
                            auto it = std::lower_bound(Lc.begin(), Lc.end(), cm, [](const CubeSet &a, uint32_t m) { return a.cube_mask < m; });
                            if (it == Lc.end() || it->cube_mask != cm) return ctx->fail(URLGPU_ERR_INTERNAL, "cube: child of a fused root missing");
                            cr.child_off[b] = it->off;
                            cr.child_acc[b] = (uint32_t)(acc_off[Lstar - 1] + (it - Lc.begin()));
                            if (b > 0) {
                                if (it->leaf_child < 0) return ctx->fail(URLGPU_ERR_INTERNAL, "cube: leaf of a fused root's child missing");
                                cr.leaf_acc[b] = (uint32_t)(acc_off[Lstar - 2] + it->leaf_child);
                            }
                            if (it->t16) cr.child16 |= 1u << b;
                            if (b > 0) ctx->st.k1_bytes_written += (it->t16 ? 2.0 : 4.0) * (double)it->cells; // only children that have children of their own are stored
                        }
                        fused_root[big_idx[i]] = 1;
                    } else cr.table_off = big[i].table_off;
                    cr.t.chunk0 = (uint32_t)rchunk;
                    rchunk += cr.t.nslices;
                    croots.push_back(cr);
                    sliced[i] = 1;
                }
            }
            if (!croots.empty()) {
                bool any_fused = false;
                for (auto &cr : croots) any_fused |= cr.nchild > 0;
                if (any_fused) fused_any = true;
                CK(dkeys.alloc(n * sizeof(uint32_t)));
                CK(dhist.alloc(((size_t)Pd + 1) * sizeof(uint32_t)));
                CK(doffp.alloc(((size_t)Pd + 1) * sizeof(uint32_t)));
                CK(dcursor.alloc(((size_t)Pd + 1) * sizeof(uint32_t)));
                CK(drows.alloc(n * sizeof(unsigned long long)));
                CK(dcroots.alloc(croots.size() * sizeof(CubeRoot)));
                CK(dmap.alloc(rchunk * sizeof(uint32_t)));
                { int rc_ = h2d_async(ctx, dcroots.p, croots.data(), croots.size() * sizeof(CubeRoot)); if (rc_) return rc_; }
                tv.rows = drows.as<unsigned long long>();
                tv.prefix_off = doffp.as<uint32_t>();
                Region rg(ctx, F_COUNT, 8);
                CK(cudaMemsetAsync(dhist.p, 0, ((size_t)Pd + 1) * sizeof(uint32_t), s));
                tree_key_kernel<<<blocks_for(n, 256), 256, 0, s>>>(bd, ci_cube, tv.dmax, dkeys.as<uint32_t>(), dhist.as<uint32_t>());
                {
                    const uint32_t nscan = (uint32_t)(Pd + 1), ntiles = (nscan + kScanTile - 1) / kScanTile;   // <= 257 tiles
                    CK(dtmp.alloc(1024 * sizeof(uint32_t)));
                    bucket_scan_sums_kernel<<<ntiles, kScanThreads, 0, s>>>(dhist.as<uint32_t>(), nscan, dtmp.as<uint32_t>());
                    bucket_scan_tiles_kernel<<<1, 1024, 0, s>>>(dtmp.as<uint32_t>(), ntiles);
                    bucket_scan_final_kernel<<<ntiles, kScanThreads, 0, s>>>(dhist.as<uint32_t>(), nscan, dtmp.as<uint32_t>(), doffp.as<uint32_t>());
                }
                CK(cudaMemcpyAsync(dcursor.p, doffp.p, ((size_t)Pd + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
                tree_scatter_kernel<<<blocks_for(n, 256), 256, 0, s>>>(bd, ci_cube, tv, dkeys.as<uint32_t>(), dcursor.as<uint32_t>(), drows.as<unsigned long long>());
                root_map_kernel<<<blocks_for(rchunk, 256), 256, 0, s>>>(dcroots.as<CubeRoot>(), (int)croots.size(), (uint32_t)rchunk, dmap.as<uint32_t>());
                const size_t smem = ((size_t)RB + 2 * seg_cap + 1) * sizeof(int);
                const unsigned grid = (unsigned)rchunk;
                switch (rv) {
#define URLGPU_ROOT_ARGS tv, dcroots.as<CubeRoot>(), dmap.as<uint32_t>(), ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, bufP, bufC, dacc.as<long long>(), RB, seg_cap, d_ovf, (int)std::min<int64_t>(ctx->n + 2, 1 << 30)
#define URLGPU_ROOT(RVV)                                                                             \
    do {                                                                                             \
        if (ctx->root_warps == 8) bic_root_kernel<RVV, 8><<<grid, 256, smem, s>>>(URLGPU_ROOT_ARGS); \
        else if (ctx->root_warps == 12) bic_root_kernel<RVV, 12><<<grid, 384, smem, s>>>(URLGPU_ROOT_ARGS); \
        else bic_root_kernel<RVV, 16><<<grid, 512, smem, s>>>(URLGPU_ROOT_ARGS);                     \
    } while (0)
                case 2: URLGPU_ROOT(2); break;
                case 3: URLGPU_ROOT(3); break;
                case 4: URLGPU_ROOT(4); break;
                default: URLGPU_ROOT(0); break;
#undef URLGPU_ROOT
#undef URLGPU_ROOT_ARGS
                }
            }
            size_t i0 = 0;
            while (i0 < big.size()) { // RED batches whose tables stay L2 resident; sliced roots only need scoring
                size_t i1 = i0;
                uint64_t bytes = 0;
                while (i1 < big.size() && (i1 == i0 || bytes + big[i1].cells * 4 <= kBatchTableElems * 4) && i1 - i0 < 65535 && sliced[i1] == sliced[i0]) { bytes += (big[i1].cells + 3) / 4 * 16; i1++; }
                const size_t B = i1 - i0;
                const bool red = !sliced[i0];
                if (red || score_roots) {
                    Region rg(ctx, F_COUNT, (red ? 2 : 0) + (score_roots ? 1 : 0));
                    if (red) {
                        for (size_t i = i0; i < i1; i++) CK(cudaMemsetAsync(bufP + big[i].table_off, 0, big[i].cells * sizeof(int), s));
                        launch_count_global(ctx, bd, MaskSets{ci_cube}, dgsets.as<GlobalSet>() + i0, B, bufP);
                    }
                    if (score_roots) {
                        uint32_t maxc = 0;
                        for (size_t i = i0; i < i1; i++) maxc = std::max(maxc, big[i].cells);
                        launch_score_tables(ctx, bd, rv, dgsets.as<GlobalSet>() + i0, B, maxc, bufP, dacc_big.as<long long>() + i0);
                    }
                }
                i0 = i1;
            }
        }
        if (score_roots) { // gather the two accumulator arrays into layer order
            std::vector<long long> ha(R.size(), 0), hs(small_m.size()), hb(big.size());
            if (!hs.empty()) CK(cudaMemcpyAsync(hs.data(), dacc_small.p, hs.size() * sizeof(long long), cudaMemcpyDeviceToHost, s));
            if (!hb.empty()) CK(cudaMemcpyAsync(hb.data(), dacc_big.p, hb.size() * sizeof(long long), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            for (size_t i = 0; i < hs.size(); i++) ha[small_idx[i]] = hs[i];
            for (size_t i = 0; i < hb.size(); i++) ha[big_idx[i]] = hb[i];
            { int rc_ = h2d_async(ctx, dacc.as<long long>() + acc_off[Lstar], ha.data(), ha.size() * sizeof(long long)); if (rc_) return rc_; }
            CK(cudaStreamSynchronize(s));
            int rc = finalize_layer(Lstar);
            if (rc) return rc;
        }
    }
    const auto T2 = tnow();
    // ---- derived layers ----
    // Pairs are emitted grouped by PARENT: blocks are dispatched in launch order, so the children of one parent run
    // back to back and all but the first read the parent table from L2 (126 MB) instead of HBM.
    std::vector<CubePair> hp;
    DevBuf dcmap(ctx);
    for (int l = Lstar - 1; l >= 0; l--) {
        auto &L = layers[l];
        auto &P = layers[l + 1];
        if (L.empty()) break;
        if (l == Lstar - 1)
            for (size_t i = 0; i < P.size(); i++) if (!fused_root[i] && mine[l + 1][i]) ctx->st.k1_bytes_written += 4.0 * (double)P[i].cells; // root tables that were written
        const bool top = l == Lstar - 1 && fused_any; // children of fused roots were produced by the root kernel
        std::vector<uint32_t> first(P.size() + 1, 0), order;
        auto skip = [&](const CubeSet &cs) {
            if (!mine[l + 1][cs.parent]) return true;   // outside this call's sub-forest
            // a leaf of a derived table was scored by the pass that derived its parent (the derive or the root kernel); only
            // leaves of root tables, which come from kernels that do not build digit-0 groups, are derived on their own
            if ((cs.cube_mask & 1u) == 0 && l + 1 < Lstar) return true;
            return top && fused_root[cs.parent] != 0;
        };
        for (auto &cs : L) if (!skip(cs)) first[cs.parent + 1]++;
        for (size_t i = 0; i < P.size(); i++) first[i + 1] += first[i];
        order.resize(first[P.size()]);
        {
            std::vector<uint32_t> pos(first.begin(), first.end() - 1);
            for (size_t i = 0; i < L.size(); i++) if (!skip(L[i])) order[pos[L[i].parent]++] = (uint32_t)i;
        }
        hp.resize(order.size());
        uint64_t chunk = 0;
        for (size_t k = 0; k < order.size(); k++) {
            const CubeSet &cs = L[order[k]];
            CubePair pr{};
            const bool leaf = (cs.cube_mask & 1u) == 0; // lowest missing bit is 0: nothing is derived from this set
            pr.parent_off = P[cs.parent].off; pr.child_off = cs.off;
            pr.r0 = leaf ? 1u : (uint32_t)ccard[0];
            pr.groups = (uint32_t)(cs.cells / rv / pr.r0);
            pr.Bc = cs.Bc; pr.r = cs.r; pr.chunk0 = (uint32_t)chunk;
            pr.acc_index = (uint32_t)(acc_off[l] + order[k]);
            pr.flags = (leaf ? 0u : kCubeStore) | (l <= Kc ? kCubeScoreChild : 0u);
            if (!leaf) { // l >= 1 and l - 1 <= Kc: the leaf child exists and is scored from this pair's groups
                if (cs.leaf_child < 0) return ctx->fail(URLGPU_ERR_INTERNAL, "cube: leaf child missing");
                pr.leaf_acc = (uint32_t)(acc_off[l - 1] + cs.leaf_child);
                pr.flags |= kCubeScoreLeaf;
            }
            pr.fmt = (P[cs.parent].t16 ? 1u : 0u) | (cs.t16 ? 2u : 0u);
            pr.magic = pr.Bc > 1 ? 0xFFFFFFFFu / pr.Bc : 0;
            ctx->st.k1_bytes_read += (P[cs.parent].t16 ? 2.0 : 4.0) * (double)cs.cells * (double)cs.r;
            if (!leaf) ctx->st.k1_bytes_written += (cs.t16 ? 2.0 : 4.0) * (double)cs.cells;
            const uint32_t gpb = kCubeConfigsPerBlock / pr.r0;
            chunk += (pr.groups + gpb - 1) / gpb;
            hp[k] = pr;
        }
        if (chunk > 0x7fffffffull) return ctx->fail(URLGPU_ERR_LIMIT, "cube: too many blocks in one layer");
        const bool score = l <= Kc;
        { int rc_ = h2d_async(ctx, dpairs.p, hp.data(), hp.size() * sizeof(CubePair)); if (rc_) return rc_; }
        if (chunk > 0) {
            CK(dcmap.alloc(chunk * sizeof(uint32_t)));
            Region rg(ctx, F_CUBE, 2);
            const unsigned grid = (unsigned)chunk;
            cube_map_kernel<<<blocks_for(chunk, 256), 256, 0, s>>>(dpairs.as<CubePair>(), (int)hp.size(), grid, dcmap.as<uint32_t>());
            switch (rv) {
            case 2: cube_derive_kernel<2><<<grid, kCubeThreads, 0, s>>>(dpairs.as<CubePair>(), dcmap.as<uint32_t>(), bufP, bufC, rv, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, dacc.as<long long>(), d_ovf, (int)std::min<int64_t>(ctx->n + 2, 1 << 30)); break;
            case 3: cube_derive_kernel<3><<<grid, kCubeThreads, 0, s>>>(dpairs.as<CubePair>(), dcmap.as<uint32_t>(), bufP, bufC, rv, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, dacc.as<long long>(), d_ovf, (int)std::min<int64_t>(ctx->n + 2, 1 << 30)); break;
            case 4: cube_derive_kernel<4><<<grid, kCubeThreads, 0, s>>>(dpairs.as<CubePair>(), dcmap.as<uint32_t>(), bufP, bufC, rv, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, dacc.as<long long>(), d_ovf, (int)std::min<int64_t>(ctx->n + 2, 1 << 30)); break;
            default: cube_derive_kernel<0><<<grid, kCubeThreads, 0, s>>>(dpairs.as<CubePair>(), dcmap.as<uint32_t>(), bufP, bufC, rv, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, dacc.as<long long>(), d_ovf, (int)std::min<int64_t>(ctx->n + 2, 1 << 30)); break;
            }
        }
        if (score) { int rc = finalize_layer(l); if (rc) return rc; }
        std::swap(bufP, bufC);
    }
    CK(cudaGetLastError());
    { int rc_ = stage_end(ctx); if (rc_) return rc_; }
    if (dbg) fprintf(stderr, "[urlgpu cube] v=%d c=%d K=%d L*=%d roots=%zu plan+alloc %.2f ms (cpu %.2f), roots %.2f ms, derive %.2f ms, cpu total %.2f\n", variable, c, K, Lstar,
                     layers[Lstar].size(), tms(T0, T1), C1 - C0, tms(T1, T2), tms(T2, tnow()), cpu_ms() - C0);
    *n_scored = family_size(c, K);
    {
        double bytes = 0;
        uint64_t cnt = 0;
        for (int l = 0; l <= Kc; l++)
            for (size_t i = 0; i < layers[l].size(); i++) if (mine[l][i]) { bytes += (double)ctx->n * (l + 1); cnt++; }
        ctx->st.algorithmic_bytes += bytes;
        ctx->st.sets_scored += cnt;
        if (parts > 1) *n_scored = cnt;
    }
    *used = true;
    return URLGPU_OK;
}

// the K3 parameter block of a family scored with sets of at most K parents and penalty weight lambda
static CbicParams cbic_params(const urlgpu_ctx *ctx, int K, double lambda) {
    CbicParams prm{};
    prm.max_parents = K;
    prm.n = (double)(int)ctx->cn;
    prm.lam_logn = lambda * std::log((double)(int)ctx->cn);
    prm.log_n = std::log((double)(int)ctx->cn);
    prm.piv_tol = 1e-10 * ctx->gram_dmax;
    return prm;
}

// the candidate Gram: packed lower triangle over (v, cand_0, cand_1, ...), indexed by tri()
static std::vector<double> cbic_sub_gram(const urlgpu_ctx *ctx, int variable, const std::vector<int> &cand) {
    const int c = (int)cand.size();
    std::vector<int> order(1, variable);
    order.insert(order.end(), cand.begin(), cand.end());
    std::vector<double> sub((size_t)(c + 1) * (c + 2) / 2);
    for (int a = 0; a <= c; a++)
        for (int b = 0; b <= a; b++) sub[tri(a, b)] = ctx->h_gram[(size_t)order[a] * ctx->cp + order[b]];
    return sub;
}

// level B over the J low candidate bits: one thread per prefix (J <= 4), or one CTA per prefix with the upper levels in
// shared memory (J >= 7)
template <int J>
static void launch_level_b(const double *roots, const CbicParams &prm, uint32_t n_prefix, float *ts, cudaStream_t s) {
    if constexpr (J >= 7) cbic_tree_kernel<J><<<n_prefix, 1 << (J - kTreeJB), 0, s>>>(roots, prm, n_prefix, ts);
    else cbic_dfs_kernel<J><<<blocks_for(n_prefix, 128), 128, 0, s>>>(roots, prm, n_prefix, ts);
}

static int cbic_score_family(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, int K, double lambda, float *d_table, uint64_t *n_scored) {
    cudaStream_t s = ctx->stream;
    const int c = (int)cand.size();
    *n_scored = family_size(c, K);
    const std::vector<double> sub = cbic_sub_gram(ctx, variable, cand);
    const CbicParams prm = cbic_params(ctx, K, lambda);
    // low bits walked in level B: the per-thread DFS keeps all its matrices in registers up to J = 4, the CTA tree takes
    // J = 7..11; the FMA sequence of a set does not depend on where the split falls
    const int J = c <= 13 ? std::min(c, 3) : c <= 16 ? 4 : std::min(11, c - 10);
    const uint32_t n_prefix = 1u << (c - J);
    const int outsz = (J + 1) * (J + 2) / 2;
    const bool use_tree = J >= 7;
    DevBuf dsub(ctx), droots(ctx), dmid(ctx), dmid2(ctx);
    CK(dsub.alloc(sub.size() * sizeof(double)));
    CK(droots.alloc((size_t)outsz * n_prefix * sizeof(double)));
    // the sub-Gram travels through the pinned staging arena: truly asynchronous, `sub` may go out of scope, and the call
    // returns without a stream synchronisation (variable v + 1 is planned and enqueued while v still runs)
    { int rc_ = stage_begin(ctx); if (rc_) return rc_; }
    { int rc_ = h2d_async(ctx, dsub.p, sub.data(), sub.size() * sizeof(double)); if (rc_) return rc_; }
    {
        Region rg(ctx, F_CBIC, 4);
        const int warps = 8;
        // level A in stages of <= 7 bits: the sweeps of the higher bits are shared by all the prefixes below them
        const int hbits = c - J;
        const int nstages = std::max(1, (hbits + 6) / 7);
        const double *src = dsub.as<double>();
        size_t src_stride = 0;
        int c_in = c, done = 0;
        DevBuf *mids[2] = {&dmid, &dmid2};
        for (int st = 0; st < nstages; st++) {
            const int bits = (hbits - done) / (nstages - st); // even split of what is left
            const bool last = st == nstages - 1;
            const int c_out = c_in - bits;
            const size_t insz = (size_t)(c_in + 1) * (c_in + 2) / 2, osz = (size_t)(c_out + 1) * (c_out + 2) / 2;
            const uint32_t n_out = 1u << (done + bits);
            double *dst = droots.as<double>();
            if (!last) {
                CK(mids[st & 1]->alloc(osz * n_out * sizeof(double)));
                dst = mids[st & 1]->as<double>();
            }
            cbic_roots_kernel<<<blocks_for(n_out, warps), warps * 32, (size_t)warps * insz * sizeof(double), s>>>(src, src_stride, c_in, bits, K, n_out, dst, last && !use_tree ? 1 : 0, prm.piv_tol);
            src = dst; src_stride = osz; c_in = c_out; done += bits;
        }
        switch (J) {
#define URLGPU_LEVEL_B(JJ) case JJ: launch_level_b<JJ>(droots.as<double>(), prm, n_prefix, d_table, s); break;
            URLGPU_LEVEL_B(0) URLGPU_LEVEL_B(1) URLGPU_LEVEL_B(2) URLGPU_LEVEL_B(3) URLGPU_LEVEL_B(4)
            URLGPU_LEVEL_B(7) URLGPU_LEVEL_B(8) URLGPU_LEVEL_B(9) URLGPU_LEVEL_B(10) URLGPU_LEVEL_B(11)
#undef URLGPU_LEVEL_B
        default: return ctx->fail(URLGPU_ERR_INTERNAL, "bad J");
        }
    }
    {
        double flops = 0, b = 1;
        for (int l = 0; l <= K && l <= c; l++) { flops += b * ((double)l * l * l / 3.0 + 2.0 * l * l + 2.0 * l); b = b * (c - l) / (l + 1); }
        ctx->st.algorithmic_flops += flops;
        ctx->st.sets_scored += *n_scored;
    }
    { int rc_ = stage_end(ctx); if (rc_) return rc_; }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// popcount-sorted lists of the high and low mask parts, cached per (hb, lb)
static int ensure_seg_lists(urlgpu_ctx *ctx, int hb, int lb) {
    auto build = [](int bits, std::vector<uint32_t> &sorted, std::vector<int> &off) {
        const uint32_t n = 1u << bits;
        sorted.resize(n);
        off.assign(bits + 2, 0);
        for (uint32_t m = 0; m < n; m++) off[__builtin_popcount(m) + 1]++;
        for (int i = 0; i <= bits; i++) off[i + 1] += off[i];
        std::vector<int> pos(off.begin(), off.end() - 1);
        for (uint32_t m = 0; m < n; m++) sorted[pos[__builtin_popcount(m)]++] = m;
    };
    if (ctx->high_bits != hb) {
        std::vector<uint32_t> sorted;
        build(hb, sorted, ctx->high_off);
        if (ctx->d_high_sorted) cudaFree(ctx->d_high_sorted);
        ctx->d_high_sorted = nullptr; ctx->high_bits = -1;
        CK(cudaMalloc(&ctx->d_high_sorted, sorted.size() * sizeof(uint32_t)));
        CK(cudaMemcpy(ctx->d_high_sorted, sorted.data(), sorted.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        ctx->high_bits = hb;
    }
    if (ctx->low_bits != lb) {
        std::vector<uint32_t> sorted;
        build(lb, sorted, ctx->low_off);
        std::vector<uint16_t> s16(sorted.begin(), sorted.end());
        if (ctx->d_low_sorted) cudaFree(ctx->d_low_sorted);
        ctx->d_low_sorted = nullptr; ctx->low_bits = -1;
        CK(cudaMalloc(&ctx->d_low_sorted, s16.size() * sizeof(uint16_t)));
        CK(cudaMemcpy(ctx->d_low_sorted, s16.data(), s16.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
        ctx->low_bits = lb;
    }
    return URLGPU_OK;
}

// MODE 0 = cBIC acceptance DP (K4), MODE 1 = subset-dominance prune (K5); one launch per popcount of the high part
template <int MODE>
static int run_segment_dp(urlgpu_ctx *ctx, float *d_table, int c, int K) {
    cudaStream_t s = ctx->stream;
    const uint64_t n_masks = (uint64_t)1 << c;
    const int lb = std::min(c, kSegMaxLb), hb = c - lb;
    int rc = ensure_seg_lists(ctx, hb, lb);
    if (rc) return rc;
    DevBuf aux(ctx);
    CK(aux.alloc(n_masks * sizeof(float)));
    SegLists sl{};
    sl.high_sorted = ctx->d_high_sorted; sl.low_sorted = ctx->d_low_sorted;
    for (int i = 0; i <= lb + 1; i++) sl.low_off[i] = ctx->low_off[i];
    {
        Region rg(ctx, MODE == 0 ? F_ACCEPT : F_PRUNE, std::min(hb, K) + 1);
        for (int a = 0; a <= hb && a <= K; a++) {
            const int begin = ctx->high_off[a], count = ctx->high_off[a + 1] - begin;
            segment_dp_kernel<MODE><<<count, 256, 0, s>>>(d_table, aux.as<float>(), sl, begin, lb, a, K);
        }
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}
static int run_accept(urlgpu_ctx *ctx, float *d_table, int c, int K) { return run_segment_dp<0>(ctx, d_table, c, K); }
static int run_prune(urlgpu_ctx *ctx, float *d_table, int c, int K) { return run_segment_dp<1>(ctx, d_table, c, K); }

// ============================================================================================ rank-space layout
// (rank_kernels.cuh)  index(S) = layer_base[|S|] + colex rank of S among the |S|-subsets of the c candidates.

static int ensure_binom(urlgpu_ctx *ctx, int K, const uint32_t **out) {
    if (K < 0 || K > kMaxRankLayers) return ctx->fail(URLGPU_ERR_LIMIT, "rank layout: parent limit above " + std::to_string(kMaxRankLayers));
    if (!ctx->d_binom[K]) {
        const int bs = K + 2;
        std::vector<uint32_t> h((size_t)(kMaxRankCand + 1) * bs);
        for (int b = 0; b <= kMaxRankCand; b++)
            for (int i = 0; i < bs; i++) h[(size_t)b * bs + i] = binom_sat(b, i);
        CK(cudaMalloc(reinterpret_cast<void **>(&ctx->d_binom[K]), h.size() * sizeof(uint32_t)));
        CK(cudaMemcpy(ctx->d_binom[K], h.data(), h.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    *out = ctx->d_binom[K];
    return URLGPU_OK;
}

// fills rs for (c, K); URLGPU_ERR_LIMIT when the family does not fit 32-bit indices
static int make_rank_space(urlgpu_ctx *ctx, int c, int K, RankSpace &rs) {
    if (c > kMaxRankCand) return ctx->fail(URLGPU_ERR_LIMIT, std::to_string(c) + " candidate parents; at most " + std::to_string(kMaxRankCand) + " are supported");
    K = std::min(K, c);
    rs = RankSpace{};
    rs.c = c; rs.K = K; rs.bstride = K + 2;
    uint64_t base = 0;
    for (int l = 0; l <= K; l++) {
        rs.layer_base[l] = (uint32_t)base;
        const uint32_t b = binom_sat(c, l);
        base += b;
        if (b == 0xFFFFFFFFu || base > 0xFFFFFFF0ull)
            return ctx->fail(URLGPU_ERR_LIMIT, "the candidate family (" + std::to_string(c) + " candidates, sets of up to " + std::to_string(K) +
                                                   " parents) has more than 2^32 parent sets");
    }
    for (int l = K + 1; l < kMaxRankLayers + 2; l++) rs.layer_base[l] = (uint32_t)base;
    return ensure_binom(ctx, K, &rs.binom);
}

// ---- K3 in rank space: per-set Schur sweeps, one launch per layer, entries [first, first + count) of the index space
// `who` names the caller in the refusal of more than kRankGenericMaxL parents.  urlgpu_score_variable comes here only for
// families over more than 30 candidates; the range entry points come here for every family, and for one over at most 30
// candidates urlgpu_score_variable is the route that scores larger parent limits.
static int cbic_score_rank(urlgpu_ctx *ctx, const char *who, int variable, const std::vector<int> &cand, const RankSpace &rs, double lambda, uint32_t first,
                           uint32_t count, float *d_scores /*indexed by global index*/) {
    cudaStream_t s = ctx->stream;
    const int c = rs.c;
    if (rs.K > kRankGenericMaxL)
        return ctx->fail(URLGPU_ERR_LIMIT, std::string(who) + ": cBIC scored set by set handles sets of at most " + std::to_string(kRankGenericMaxL) + " parents" +
                                               (c > kMaxDenseCand ? " (no other cBIC route takes a family over more than 30 candidates)"
                                                                  : " (urlgpu_score_variable scores this family, over at most 30 candidates, whole)"));
    const std::vector<double> g = cbic_sub_gram(ctx, variable, cand);
    DevBuf dg(ctx);
    CK(dg.alloc(g.size() * sizeof(double)));
    { int rc_ = stage_begin(ctx); if (rc_) return rc_; }
    { int rc_ = h2d_async(ctx, dg.p, g.data(), g.size() * sizeof(double)); if (rc_) return rc_; }
    const CbicParams prm = cbic_params(ctx, rs.K, lambda);
    const size_t smem = rs_binom_bytes(rs);
    // each layer's part of [first, first + count)
    struct Span { int l; uint32_t b0, cnt; };
    std::vector<Span> spans;
    for (int l = 0; l <= rs.K; l++) {
        const uint64_t b0 = std::max<uint64_t>(rs.layer_base[l], first), b1 = std::min<uint64_t>(rs.layer_base[l + 1], (uint64_t)first + count);
        if (b0 < b1) spans.push_back({l, (uint32_t)b0, (uint32_t)(b1 - b0)});
    }
    {
        Region rg(ctx, F_CBIC, (int)spans.size());
        for (const Span &sp : spans) {
            const unsigned grid = blocks_for(((uint64_t)sp.cnt + kRankRun - 1) / kRankRun, 128);
#define URLGPU_RANK_CBIC(LL) rank_cbic_kernel<LL><<<grid, 128, smem, s>>>(rs, dg.as<double>(), prm, sp.l, sp.b0, sp.cnt, d_scores)
            switch (sp.l) {
            case 1: URLGPU_RANK_CBIC(1); break;
            case 2: URLGPU_RANK_CBIC(2); break;
            case 3: URLGPU_RANK_CBIC(3); break;
            case 4: URLGPU_RANK_CBIC(4); break;
            case 5: URLGPU_RANK_CBIC(5); break;
            case 6: URLGPU_RANK_CBIC(6); break;
            case 7: URLGPU_RANK_CBIC(7); break;
            case 8: URLGPU_RANK_CBIC(8); break;
            default: URLGPU_RANK_CBIC(0); break;   // layer 0 (the empty set: the_score 0) and layers above 8
            }
#undef URLGPU_RANK_CBIC
        }
    }
    { int rc_ = stage_end(ctx); if (rc_) return rc_; }
    {
        double flops = 0;
        for (const Span &sp : spans) flops += (double)sp.cnt * ((double)sp.l * sp.l * sp.l / 3.0 + 2.0 * sp.l * sp.l + 2.0 * sp.l);
        ctx->st.algorithmic_flops += flops;
        ctx->st.sets_scored += count;
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// ---- K1 by direct counting: every set of [first, first + count) of the rank space is counted from the rows.  The sets
// are named by their index (RankSets); a score goes to its index, or to its compact mask when by_mask (dense layout).
// Sets are classified by table size: two shared-memory tiers (one CTA per set) and the global tier below.

// The global tier: tables in an L2-resident scratch batch, RED atomics.  Scores (and, optionally, the fixed-point
// log-likelihoods) go to d_scores at each set's output index; counts_out, if given, receives the table of sets[0].
template <class Sets>
static int direct_global_tier(urlgpu_ctx *ctx, const BicData &bd, const Sets &fam, std::vector<GlobalSet> &sets, float *d_scores,
                              long long *d_llfixed, int32_t *counts_out, int64_t n_cells) {
    cudaStream_t s = ctx->stream;
    size_t max_cells = 0;
    for (auto &g : sets) max_cells = std::max<size_t>(max_cells, g.cells);
    int rc = ensure_tables(ctx, std::max(kBatchTableElems, max_cells));
    if (rc) return rc;
    std::vector<std::pair<size_t, size_t>> batches;
    for (size_t i0 = 0; i0 < sets.size();) {
        size_t used = 0, i1 = i0;
        while (i1 < sets.size() && (i1 == i0 || used + sets[i1].cells <= ctx->tables_cap) && i1 - i0 < 65535) {
            sets[i1].table_off = used;
            used += (sets[i1].cells + 3) / 4 * 4;
            i1++;
        }
        batches.push_back({i0, i1});
        i0 = i1;
    }
    DevBuf dsets(ctx), dacc(ctx);
    CK(dsets.alloc(sets.size() * sizeof(GlobalSet)));
    CK(dacc.alloc(sets.size() * sizeof(long long)));
    CK(cudaMemsetAsync(dacc.p, 0, sets.size() * sizeof(long long), s));
    CK(cudaMemcpyAsync(dsets.p, sets.data(), sets.size() * sizeof(GlobalSet), cudaMemcpyHostToDevice, s));
    for (auto &bt : batches) {
        const size_t B = bt.second - bt.first;
        const size_t used = sets[bt.second - 1].table_off + sets[bt.second - 1].cells;
        uint32_t maxc = 0;
        for (size_t i = bt.first; i < bt.second; i++) maxc = std::max(maxc, sets[i].cells);
        Region rg(ctx, F_COUNT, 3);
        CK(cudaMemsetAsync(ctx->d_tables, 0, used * sizeof(int), s));
        launch_count_global(ctx, bd, fam, dsets.as<GlobalSet>() + bt.first, B, ctx->d_tables);
        launch_score_tables(ctx, bd, fam.rv(), dsets.as<GlobalSet>() + bt.first, B, maxc, ctx->d_tables, dacc.as<long long>() + bt.first);
        if (counts_out && bt.first == 0) {
            CK(cudaMemcpyAsync(counts_out, ctx->d_tables, (size_t)n_cells * sizeof(int), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
        }
    }
    if (d_scores) {
        Region rg(ctx, F_OTHER, 1);
        bic_finalize_kernel<<<blocks_for(sets.size(), 256), 256, 0, s>>>(bd, fam, dsets.as<GlobalSet>(), dacc.as<long long>(), (int)sets.size(), d_scores, d_llfixed);
    }
    CK(cudaStreamSynchronize(s)); // dsets/dacc are freed on return
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// the candidates' variables and arities on the device (dcand, uploaded from hv, which the caller keeps until its stream has
// been synchronised), and the key space of the direct-counting kernels over them
static int make_rank_sets(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, const RankSpace &rs, bool by_mask, std::vector<int> &hv, DevBuf &dcand,
                          RankSets &fam) {
    const int c = (int)cand.size();
    hv.assign(2 * (size_t)std::max(c, 1), 0);
    for (int i = 0; i < c; i++) { hv[i] = cand[i]; hv[c + i] = ctx->card[cand[i]]; }
    CK(dcand.alloc(hv.size() * sizeof(int)));
    CK(cudaMemcpyAsync(dcand.p, hv.data(), hv.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    fam = RankSets{rs, RankCand{variable, ctx->card[variable], dcand.as<int>(), dcand.as<int>() + c}, by_mask ? 1 : 0};
    return URLGPU_OK;
}

static int bic_score_direct(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, const RankSpace &rs, uint32_t first, uint32_t count, float *d_scores,
                            bool by_mask) {
    cudaStream_t s = ctx->stream;
    if (rs.K + 1 > kMaxCols) return ctx->fail(URLGPU_ERR_LIMIT, "BIC: more than 31 parents in one set");
    BicData bd{ctx->d_codes, ctx->n, ctx->n_stride, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, ctx->ds_base, ctx->ds_ess, ctx->ds_scale};
    const uint32_t tier1_cells = (uint32_t)((ctx->smem_optin - 2048) / sizeof(int));
    std::vector<int> hv;
    DevBuf dcand(ctx), lists(ctx), counters(ctx);
    RankSets fam{};
    int rc = make_rank_sets(ctx, variable, cand, rs, by_mask, hv, dcand, fam);
    if (rc) return rc;
    CK(lists.alloc((size_t)count * (sizeof(GlobalSet) + 2 * sizeof(uint32_t))));
    CK(counters.alloc(4 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(counters.p, 0, 4 * sizeof(unsigned long long), s));
    GlobalSet *l2 = lists.as<GlobalSet>();
    uint32_t *l0 = reinterpret_cast<uint32_t *>(l2 + count), *l1 = l0 + count;
    {
        Region rg(ctx, F_OTHER, 1);
        bic_classify_kernel<<<blocks_for(count, 256), 256, rs_binom_bytes(rs), s>>>(fam, first, count, kTier0Cells, tier1_cells, kCellLimit, l0, l1, l2,
                                                                                    counters.as<unsigned long long>());
    }
    unsigned long long hc[4];
    CK(cudaMemcpyAsync(hc, counters.p, sizeof hc, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (hc[3]) return ctx->fail(URLGPU_ERR_LIMIT, "a contingency table of this family has more than 2^30 cells");
    if (hc[0]) {
        Region rg(ctx, F_COUNT, 1);
        const int threads = ctx->n >= 65536 ? 256 : 128;
        bic_count_smem_kernel<<<(unsigned)hc[0], threads, kTier0Cells * sizeof(int), s>>>(bd, fam, l0, d_scores, nullptr, nullptr, nullptr);
    }
    if (hc[1]) {
        Region rg(ctx, F_COUNT, 1);
        bic_count_smem_kernel<<<(unsigned)hc[1], 1024, (size_t)tier1_cells * sizeof(int), s>>>(bd, fam, l1, d_scores, nullptr, nullptr, nullptr);
    }
    if (hc[2]) {
        std::vector<GlobalSet> sets(hc[2]);
        CK(cudaMemcpyAsync(sets.data(), l2, hc[2] * sizeof(GlobalSet), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        std::sort(sets.begin(), sets.end(), [](const GlobalSet &a, const GlobalSet &b) { return a.key < b.key; });
        rc = direct_global_tier(ctx, bd, fam, sets, d_scores, nullptr, nullptr, 0);
        if (rc) return rc;
    }
    {   // algorithmic bytes: n*(k+1) per set (SURVEY.md §8d)
        double bytes = 0;
        const uint64_t last = (uint64_t)first + count;
        for (int l = 0; l <= rs.K; l++) {
            const uint64_t b0 = std::max<uint64_t>(rs.layer_base[l], first), b1 = std::min<uint64_t>(rs.layer_base[l + 1], last);
            if (b0 < b1) bytes += (double)(b1 - b0) * (double)ctx->n * (l + 1);
        }
        ctx->st.algorithmic_bytes += bytes;
        ctx->st.sets_scored += count;
    }
    CK(cudaStreamSynchronize(s)); // hv / dcand / lists / counters are freed on return
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// K1 for a whole family: the cube path (c <= 30, BIC / fNML), else, or when the cube path cannot lay the family out, direct
// counting of every set.  `om` says where a set's score goes: dense by compact mask (om.binom == nullptr), or rank space.
static int bic_score_family(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, int K, float *d_table, uint64_t *n_scored, const RankSpace &om,
                            int *d_ovf = nullptr) {
    if (ctx->ds_ess == 0.f && !ctx->bic_direct && (int)cand.size() <= kMaxDenseCand) {
        bool used = false;
        int rc = bic_score_family_cube(ctx, variable, cand, K, d_table, n_scored, &used, om, 0, 1, d_ovf);
        if (rc || used) return rc;
    }
    RankSpace rs = om;
    if (!om.binom) { int rc = make_rank_space(ctx, (int)cand.size(), K, rs); if (rc) return rc; }
    *n_scored = rs.layer_base[rs.K + 1];
    return bic_score_direct(ctx, variable, cand, rs, 0, (uint32_t)*n_scored, d_table, om.binom == nullptr);
}

// K4 (MODE 0) / K5 (MODE 1) in rank space: one launch per layer, ascending
template <int MODE>
static int run_rank_dp(urlgpu_ctx *ctx, const RankSpace &rs, float *d_scores) {
    cudaStream_t s = ctx->stream;
    const uint32_t total = rs.layer_base[rs.K + 1];
    DevBuf aux(ctx);
    CK(aux.alloc((size_t)total * sizeof(float)));
    const size_t smem = rs_binom_bytes(rs);
    {
        Region rg(ctx, MODE == 0 ? F_ACCEPT : F_PRUNE, rs.K + 1);
        for (int l = 0; l <= rs.K; l++) {
            const uint32_t nl = rs.layer_base[l + 1] - rs.layer_base[l];
            if (nl == 0) continue;
            rank_dp_kernel<MODE><<<blocks_for(nl, 256), 256, smem, s>>>(rs, l, d_scores, aux.as<float>());
        }
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// dense (2^c floats by compact mask) or rank layout for this family?
static bool choose_rank_layout(urlgpu_ctx *ctx, int c, int K, bool bic) {
    if (c > kMaxDenseCand) return true;
    const int Kc = std::min(K, c);
    if (ctx->layout_policy == 1) return false;
    if (!bic && Kc > kRankGenericMaxL) return false;            // cBIC per-set sweeps hold up to 16 parents; larger limits are the DFS's domain
    if (Kc > kMaxRankLayers - 1) return false;
    if (ctx->layout_policy == 2) return true;
    // auto: rank space when the family is a small part of the 2^c lattice (the dense DPs and the compaction walk all 2^c entries)
    return c >= 16 && (double)family_size(c, Kc) * 8.0 < std::ldexp(1.0, c);
}

// K4 as written (URLGPU_CBIC_ACCEPT_LITERAL): accept_literal_kernel, layer by layer, two launches per layer when variable 0
// is a candidate (rank_kernels.cuh)
static int run_accept_literal(urlgpu_ctx *ctx, urlgpu_result *res) {
    cudaStream_t s = ctx->stream;
    const int c = res->c, K = res->max_parents;
    if (K > kLiteralMaxK) return ctx->fail(URLGPU_ERR_LIMIT, "literal-zero acceptance emulates the reference's recursion per parent set and handles sets of at most " +
                                                              std::to_string(kLiteralMaxK) + " parents");
    if (c > 62) return ctx->fail(URLGPU_ERR_LIMIT, "literal-zero acceptance handles at most 62 candidates");
    RankSpace enumr{};
    int rc = make_rank_space(ctx, c, K, enumr);
    if (rc) return rc;
    const RankSpace lay = res->rank_layout ? res->rs : RankSpace{};
    uint32_t widest = 0;
    for (int l = 0; l <= K; l++) widest = std::max(widest, enumr.layer_base[l + 1] - enumr.layer_base[l]);
    if ((uint64_t)widest * (sizeof(LiteralFrame) * (kLiteralMaxK + 1) + 1024) > ((uint64_t)16 << 30))
        return ctx->fail(URLGPU_ERR_LIMIT, "literal-zero acceptance: the widest layer of this family needs more than 16 GB of per-set recursion state");
    DevBuf frames(ctx), checked(ctx);
    CK(frames.alloc((size_t)widest * (kLiteralMaxK + 1) * sizeof(LiteralFrame)));
    CK(checked.alloc((size_t)widest * 256 * sizeof(uint32_t)));
    const int zero_cand = (!res->cand.empty() && res->cand[0] == 0) ? 0 : -1;
    {
        Region rg(ctx, F_ACCEPT, (zero_cand >= 0 ? 2 : 1) * (K + 1));
        for (int l = 0; l <= K; l++) {
            const uint32_t nl = enumr.layer_base[l + 1] - enumr.layer_base[l];
            if (nl == 0) continue;
            for (int phase = (zero_cand >= 0 ? 0 : 2); phase <= (zero_cand >= 0 ? 1 : 2); phase++)
                accept_literal_kernel<<<blocks_for(nl, 128), 128, 0, s>>>(enumr, lay, l, zero_cand, phase, res->d_table, frames.as<LiteralFrame>(), checked.as<uint32_t>());
        }
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// store rule / acceptance and the optional prune on a table of RAW scores (BIC: the score, cBIC: the_score)
static int apply_filters(urlgpu_ctx *ctx, urlgpu_result *res, bool bic, unsigned filter_flags) {
    cudaStream_t s = ctx->stream;
    const int c = res->c, K = res->max_parents;
    int rc = URLGPU_OK;
    if (!bic && (filter_flags & URLGPU_CBIC_ACCEPT_LITERAL) && !(filter_flags & URLGPU_CBIC_NO_ACCEPT)) {
        if ((rc = run_accept_literal(ctx, res))) return rc;
        if (filter_flags & URLGPU_PRUNE_DOMINATED) rc = res->rank_layout ? run_rank_dp<1>(ctx, res->rs, res->d_table) : run_prune(ctx, res->d_table, c, K);
        return rc;
    }
    if (res->rank_layout) {
        const RankSpace &rs = res->rs;
        const uint32_t total = (uint32_t)res->n_masks;
        if (bic) {
            Region rg(ctx, F_OTHER, 1);
            rank_store_rule_kernel<<<blocks_for(total, 256), 256, 0, s>>>(res->d_table, total);
        } else if (filter_flags & URLGPU_CBIC_NO_ACCEPT) {
            Region rg(ctx, F_OTHER, 1);
            cbic_negate_kernel<<<blocks_for(total, 256), 256, 0, s>>>(res->d_table, total);
        } else if ((rc = run_rank_dp<0>(ctx, rs, res->d_table))) return rc;
        if (filter_flags & URLGPU_PRUNE_DOMINATED) rc = run_rank_dp<1>(ctx, rs, res->d_table);
    } else {
        if (bic) {
            Region rg(ctx, F_OTHER, 1);
            bic_store_rule_kernel<<<blocks_for(res->n_masks, 256), 256, 0, s>>>(res->d_table, res->n_masks, K);
        } else if (filter_flags & URLGPU_CBIC_NO_ACCEPT) {
            Region rg(ctx, F_OTHER, 1);
            cbic_negate_kernel<<<blocks_for(res->n_masks, 256), 256, 0, s>>>(res->d_table, res->n_masks);
        } else if ((rc = run_accept(ctx, res->d_table, c, K))) return rc;
        if (filter_flags & URLGPU_PRUNE_DOMINATED) rc = run_prune(ctx, res->d_table, c, K);
    }
    return rc;
}

static int check_score_args(urlgpu_ctx *ctx, const char *who, int variable, const uint64_t *neighbors, int mask_words, int score_type, std::vector<int> &cand,
                            double param = 1.0) {
    const bool bic = is_discrete(score_type);
    if (!bic && score_type != URLGPU_CBIC) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": unknown score type");
    if (bic && !ctx->have_discrete) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": BIC / fNML need urlgpu_set_discrete first");
    if (!bic && !ctx->have_gram) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": cBIC needs urlgpu_set_continuous first");
    const int p = bic ? ctx->p : ctx->cp;
    if (variable < 0 || variable >= p) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": variable out of range");
    if (bic) { const int rc = select_discrete_score(ctx, score_type, variable, param); if (rc) return rc; }
    return candidates_from_mask(ctx, p, variable, neighbors, mask_words, cand);
}

extern "C" int urlgpu_score_variable(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type,
                                     double lambda, unsigned filter_flags, urlgpu_result **out) {
    if (!ctx || !neighbors || !out) return ctx ? ctx->fail(URLGPU_ERR_ARG, "score_variable: null argument") : URLGPU_ERR_ARG;
    *out = nullptr;
    static const bool dbg = getenv("URLGPU_DEBUG_TIMING") != nullptr;
    const auto T0 = std::chrono::steady_clock::now();
    auto since = [&](std::chrono::steady_clock::time_point a) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count(); };
    CK(cudaSetDevice(ctx->device));
    const bool bic = is_discrete(score_type);
    std::vector<int> cand;
    int rc = check_score_args(ctx, "score_variable", variable, neighbors, mask_words, score_type, cand, lambda);
    if (rc) return rc;
    const int c = (int)cand.size();
    int K = std::max(0, std::min(max_parents, c));
    const bool rank = choose_rank_layout(ctx, c, K, bic);
    auto *res = new urlgpu_result();
    res->ctx = ctx; res->variable = variable; res->c = c; res->max_parents = K; res->mask_words = mask_words; res->cand = cand;
    res->rank_layout = rank;
    if (rank) {
        rc = make_rank_space(ctx, c, K, res->rs);
        if (rc) { delete res; return rc; }
        res->n_masks = res->rs.layer_base[K + 1];
    } else res->n_masks = (uint64_t)1 << c;
    cudaError_t e = pool_alloc(ctx, reinterpret_cast<void **>(&res->d_table), res->n_masks * sizeof(float));
    if (e != cudaSuccess) { delete res; return ctx->cuda_fail(e, "cudaMalloc(score table)", __LINE__); }
    cudaStream_t s = ctx->stream;
    auto cleanup = [&](int code) { pool_free(ctx, res->d_table); if (res->d_ovf) pool_free(ctx, res->d_ovf); delete res; return code; };
    res->is_bic = bic; res->score_type = score_type; res->filter_flags = filter_flags;
    if (bic && ctx->ds_ess == 0.f && ctx->table16 && c <= kMaxDenseCand && !ctx->bic_direct && !ctx->t16_overflowed.count(variable)) {
        e = pool_alloc(ctx, reinterpret_cast<void **>(&res->d_ovf), sizeof(int));
        if (e != cudaSuccess) return cleanup(ctx->cuda_fail(e, "cudaMalloc(flag)", __LINE__));
        cudaMemsetAsync(res->d_ovf, 0, sizeof(int), s);
    }
    const double t_alloc = since(T0);
    if (rank) {
        const uint32_t total = (uint32_t)res->n_masks;
        res->n_scored = total;
        if (bic) {
            fill_u32_kernel<<<blocks_for(total, 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(res->d_table), total, kSentinelBits);
            rc = bic_score_family(ctx, variable, cand, K, res->d_table, &res->n_scored, res->rs, res->d_ovf);
        } else rc = cbic_score_rank(ctx, "score_variable", variable, cand, res->rs, lambda, 0, total, res->d_table);
    } else {
        fill_u32_kernel<<<blocks_for(res->n_masks, 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(res->d_table), res->n_masks, kSentinelBits);
        if (bic) rc = bic_score_family(ctx, variable, cand, K, res->d_table, &res->n_scored, RankSpace{}, res->d_ovf);
        else rc = cbic_score_family(ctx, variable, cand, K, lambda, res->d_table, &res->n_scored);
    }
    if (rc) return cleanup(rc);
    const double t_score = since(T0);
    rc = apply_filters(ctx, res, bic, filter_flags);
    if (rc) return cleanup(rc);
    if (dbg) fprintf(stderr, "[urlgpu score_variable] v=%d alloc %.2f ms, score %.2f ms, filters %.2f ms\n", variable, t_alloc, t_score - t_alloc, since(T0) - t_score);
    e = cudaGetLastError();
    if (e != cudaSuccess) return cleanup(ctx->cuda_fail(e, "score_variable", __LINE__));
    *out = res;
    return URLGPU_OK;
}

// ---- (variable, parent-set range) shards: SURVEY.md 8(e), BASELINE.json north_star -------------------------------------
// A family's canonical order IS the rank-space index order, so a contiguous index range is a self-contained unit of
// scoring work: N ranks score N ranges of one variable (or a deal of ranges over many variables), the raw scores are
// exchanged (NCCL all-gather / all-to-all of float arrays, urlearning-cpp_b200/distributed.py) and the variable's owner
// applies the filters, which need the whole subset-closed family, with urlgpu_result_from_scores.

extern "C" int urlgpu_family_size(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type, uint64_t *n) {
    if (!ctx || !neighbors || !n) return ctx ? ctx->fail(URLGPU_ERR_ARG, "family_size: null argument") : URLGPU_ERR_ARG;
    std::vector<int> cand;
    int rc = check_score_args(ctx, "family_size", variable, neighbors, mask_words, score_type, cand);
    if (rc) return rc;
    RankSpace rs{};
    rc = make_rank_space(ctx, (int)cand.size(), std::max(0, max_parents), rs);
    if (rc) return rc;
    *n = rs.layer_base[rs.K + 1];
    return URLGPU_OK;
}

extern "C" int urlgpu_score_range(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type, double lambda,
                                  uint64_t first, uint64_t count, float *scores, int on_device) {
    if (!ctx || !neighbors || !scores) return ctx ? ctx->fail(URLGPU_ERR_ARG, "score_range: null argument") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const bool bic = is_discrete(score_type);
    std::vector<int> cand;
    int rc = check_score_args(ctx, "score_range", variable, neighbors, mask_words, score_type, cand, lambda);
    if (rc) return rc;
    RankSpace rs{};
    rc = make_rank_space(ctx, (int)cand.size(), std::max(0, max_parents), rs);
    if (rc) return rc;
    const uint64_t total = rs.layer_base[rs.K + 1];
    if (first + count > total) return ctx->fail(URLGPU_ERR_ARG, "score_range: the range exceeds the family (" + std::to_string(total) + " sets)");
    if (count == 0) return URLGPU_OK;
    cudaStream_t s = ctx->stream;
    DevBuf tmp(ctx);
    float *d_out = scores;
    if (!on_device) { CK(tmp.alloc(count * sizeof(float))); d_out = tmp.as<float>(); }
    // the kernels index by global family index: shift the base so that entry `first` lands on d_out[0]
    float *d_base = d_out - first;
    if (bic) rc = bic_score_direct(ctx, variable, cand, rs, (uint32_t)first, (uint32_t)count, d_base, false);
    else rc = cbic_score_rank(ctx, "score_range", variable, cand, rs, lambda, (uint32_t)first, (uint32_t)count, d_base);
    if (rc) return rc;
    if (!on_device) {
        CK(cudaMemcpyAsync(scores, d_out, count * sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

extern "C" int urlgpu_score_part(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type, double lambda,
                                 int part, int parts, float *scores, int on_device) {
    if (!ctx || !neighbors || !scores || parts < 1 || part < 0 || part >= parts) return ctx ? ctx->fail(URLGPU_ERR_ARG, "score_part: bad argument") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const bool bic = is_discrete(score_type);
    std::vector<int> cand;
    int rc = check_score_args(ctx, "score_part", variable, neighbors, mask_words, score_type, cand, lambda);
    if (rc) return rc;
    const int c = (int)cand.size();
    const int K = std::max(0, std::min(max_parents, c));
    RankSpace rs{};
    rc = make_rank_space(ctx, c, K, rs);
    if (rc) return rc;
    const uint32_t total = rs.layer_base[rs.K + 1];
    cudaStream_t s = ctx->stream;
    DevBuf tmp(ctx);
    float *d_out = scores;
    if (!on_device) { CK(tmp.alloc((size_t)total * sizeof(float))); d_out = tmp.as<float>(); }
    fill_u32_kernel<<<blocks_for(total, 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(d_out), total, kSentinelBits);
    bool done = false;
    if (bic && ctx->ds_ess == 0.f && c <= kMaxDenseCand && !ctx->bic_direct) { // the cube path: part = a sub-forest of the root tables
        uint64_t ns = 0;
        DevBuf flag(ctx);
        if (ctx->table16) { CK(flag.alloc(sizeof(int))); CK(cudaMemsetAsync(flag.p, 0, sizeof(int), s)); }
        rc = bic_score_family_cube(ctx, variable, cand, K, d_out, &ns, &done, rs, part, parts, flag.as<int>());
        if (rc) return rc;
        if (done && flag.p) { // 16-bit tables are speculative: check now (this entry point hands raw scores out)
            int h = 0;
            CK(cudaMemcpyAsync(&h, flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            if (h) {
                ctx->st.table16_fallbacks++;
                fill_u32_kernel<<<blocks_for(total, 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(d_out), total, kSentinelBits);
                rc = bic_score_family_cube(ctx, variable, cand, K, d_out, &ns, &done, rs, part, parts, nullptr);
                if (rc) return rc;
            }
        }
    }
    if (!done) { // a contiguous range of the canonical numbering
        const uint64_t b0 = (uint64_t)total * part / parts, b1 = (uint64_t)total * (part + 1) / parts;
        if (b1 > b0) {
            if (bic) rc = bic_score_direct(ctx, variable, cand, rs, (uint32_t)b0, (uint32_t)(b1 - b0), d_out, false);
            else rc = cbic_score_rank(ctx, "score_part", variable, cand, rs, lambda, (uint32_t)b0, (uint32_t)(b1 - b0), d_out);
            if (rc) return rc;
        }
    }
    if (!on_device) {
        CK(cudaMemcpyAsync(scores, d_out, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

extern "C" int urlgpu_result_from_scores(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type,
                                         const float *scores, uint64_t n, int on_device, unsigned filter_flags, urlgpu_result **out) {
    if (!ctx || !neighbors || !scores || !out) return ctx ? ctx->fail(URLGPU_ERR_ARG, "result_from_scores: null argument") : URLGPU_ERR_ARG;
    *out = nullptr;
    CK(cudaSetDevice(ctx->device));
    const bool bic = is_discrete(score_type);
    std::vector<int> cand;
    int rc = check_score_args(ctx, "result_from_scores", variable, neighbors, mask_words, score_type, cand);
    if (rc) return rc;
    const int c = (int)cand.size();
    const int K = std::max(0, std::min(max_parents, c));
    auto *res = new urlgpu_result();
    res->ctx = ctx; res->variable = variable; res->c = c; res->max_parents = K; res->mask_words = mask_words; res->cand = cand;
    res->rank_layout = true;
    rc = make_rank_space(ctx, c, K, res->rs);
    if (rc) { delete res; return rc; }
    res->n_masks = res->rs.layer_base[K + 1];
    res->n_scored = res->n_masks;
    if (n != res->n_masks) { delete res; return ctx->fail(URLGPU_ERR_ARG, "result_from_scores: expected " + std::to_string(res->n_masks) + " scores"); }
    cudaError_t e = pool_alloc(ctx, reinterpret_cast<void **>(&res->d_table), res->n_masks * sizeof(float));
    if (e != cudaSuccess) { delete res; return ctx->cuda_fail(e, "cudaMalloc(score table)", __LINE__); }
    auto cleanup = [&](int code) { pool_free(ctx, res->d_table); delete res; return code; };
    e = cudaMemcpyAsync(res->d_table, scores, n * sizeof(float), on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) return cleanup(ctx->cuda_fail(e, "copy of the scores", __LINE__));
    if (!on_device) { e = cudaStreamSynchronize(ctx->stream); if (e != cudaSuccess) return cleanup(ctx->cuda_fail(e, "copy of the scores", __LINE__)); }
    rc = apply_filters(ctx, res, bic, filter_flags);
    if (rc) return cleanup(rc);
    *out = res;
    return URLGPU_OK;
}

// ============================================================================================ results
//
// The stored entries of a variable's dense table are compacted ON THE DEVICE into the canonical order (|S| ascending,
// mask ascending) by three kernels with no host round trip: per-(layer, 2048-mask segment) counts, an exclusive scan
// per layer plus the layer bases, and an order-preserving write.  urlgpu_result_prefetch enqueues them (and a copy of
// the 33 counters into pinned memory) on the context's stream right behind the scoring kernels, so a caller that
// scores variable v+1 before fetching v never stalls the GPU; the payload is then copied on a second stream.

namespace {
constexpr int kCompactSeg = 2048;      // masks per CTA
constexpr int kCompactThreads = 256;   // 8 consecutive masks per thread

__global__ void __launch_bounds__(kCompactThreads) compact_count_kernel(const float *__restrict__ table, uint64_t n_masks, uint32_t nseg,
                                                                        uint32_t *__restrict__ segcnt /*[32][nseg]*/) {
    __shared__ unsigned int sh[32];
    if (threadIdx.x < 32) sh[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t m0 = (uint64_t)blockIdx.x * kCompactSeg + (uint64_t)threadIdx.x * 8;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint64_t m = m0 + k;
        if (m < n_masks && !is_sentinel(table[m])) atomicAdd(&sh[__popcll(m)], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 32) segcnt[(size_t)threadIdx.x * nseg + blockIdx.x] = sh[threadIdx.x];
}

// one CTA per layer: exclusive scan of its segment counts in place; totals to counts[layer]
__global__ void __launch_bounds__(1024) compact_scan_kernel(uint32_t *__restrict__ segcnt, uint32_t nseg, unsigned long long *__restrict__ counts) {
    __shared__ unsigned long long part[1024];
    uint32_t *row = segcnt + (size_t)blockIdx.x * nseg;
    const uint32_t per = (nseg + blockDim.x - 1) / blockDim.x;
    const uint32_t b = min(nseg, threadIdx.x * per), e = min(nseg, b + per);
    unsigned long long sum = 0;
    for (uint32_t i = b; i < e; i++) sum += row[i];
    part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (uint32_t i = 0; i < blockDim.x; i++) { const unsigned long long t = part[i]; part[i] = run; run += t; }
        counts[blockIdx.x] = run;
    }
    __syncthreads();
    unsigned long long run = part[threadIdx.x];
    for (uint32_t i = b; i < e; i++) { const uint32_t t = row[i]; row[i] = (uint32_t)run; run += t; } // a layer holds < 2^32 entries (c <= 30)
}

__global__ void compact_bases_kernel(unsigned long long *__restrict__ counts /*[33]*/, unsigned long long *__restrict__ bases /*[32]*/) {
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int l = 0; l < 32; l++) { bases[l] = run; run += counts[l]; }
        counts[32] = run;
    }
}

__global__ void __launch_bounds__(kCompactThreads) compact_write_kernel(const float *__restrict__ table, uint64_t n_masks, uint32_t nseg,
                                                                        const uint32_t *__restrict__ segoff, const unsigned long long *__restrict__ bases,
                                                                        uint32_t *__restrict__ out_masks, float *__restrict__ out_vals) {
    __shared__ uint8_t cnt[32][kCompactThreads];   // stored entries of layer l among thread t's 8 masks
    __shared__ uint16_t excl[32][kCompactThreads]; // exclusive prefix over the threads
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int i = t; i < 32 * kCompactThreads; i += kCompactThreads) (&cnt[0][0])[i] = 0;
    __syncthreads();
    const uint64_t m0 = (uint64_t)blockIdx.x * kCompactSeg + (uint64_t)t * 8;
    float v[8];
    unsigned stored = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint64_t m = m0 + k;
        v[k] = m < n_masks ? table[m] : sentinel();
        if (!is_sentinel(v[k])) { stored |= 1u << k; cnt[__popcll(m)][t]++; }
    }
    __syncthreads();
    for (int l = warp; l < 32; l += kCompactThreads / 32) { // warp `warp` scans layers warp, warp + 8, ...
        unsigned carry = 0;
        for (int b0 = 0; b0 < kCompactThreads; b0 += 32) {
            const unsigned c0 = cnt[l][b0 + lane];
            unsigned x = c0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
            excl[l][b0 + lane] = (uint16_t)(carry + x - c0);
            carry += __shfl_sync(0xffffffffu, x, 31);
        }
    }
    __syncthreads();
    if (!stored) return;
    unsigned seen[4] = {0, 0, 0, 0}; // per-layer entries already written by this thread: its 8 masks span <= 4 distinct popcounts
    const int pc0 = __popcll(m0 >> 3);  // popcount of the shared high part; the low 3 bits add 0..3
#pragma unroll
    for (int k = 0; k < 8; k++) {
        if (!((stored >> k) & 1)) continue;
        const int dl = __popc(k), l = pc0 + dl;
        const unsigned long long pos = bases[l] + segoff[(size_t)l * nseg + blockIdx.x] + excl[l][t] + seen[dl];
        seen[dl]++;
        out_masks[pos] = (uint32_t)(m0 + k);
        out_vals[pos] = v[k];
    }
}

// compact mask -> the caller's multi-word varsets
__global__ void expand_masks_kernel(const uint32_t *__restrict__ masks, uint64_t n, const int *__restrict__ cand, int c, int words, uint64_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t cm = masks[i];
    for (int w = 0; w < words; w++) {
        uint64_t x = 0;
        for (int b = 0; b < c; b++)
            if (((cm >> b) & 1) && (cand[b] >> 6) == w) x |= (uint64_t)1 << (cand[b] & 63);
        out[i * (uint64_t)words + w] = x;
    }
}
} // namespace

static int result_prefetch_impl(urlgpu_result *res) {
    urlgpu_ctx *ctx = res->ctx;
    if (res->prefetched) return URLGPU_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const uint32_t nseg = res->rank_layout ? (uint32_t)((res->n_masks + kRankCompactSeg - 1) / kRankCompactSeg) : (uint32_t)((res->n_masks + kCompactSeg - 1) / kCompactSeg);
    const uint64_t cap = std::max<uint64_t>(1, std::min<uint64_t>(res->n_scored, res->n_masks));
    CK(pool_alloc(ctx, reinterpret_cast<void **>(&res->d_masks), cap * sizeof(uint32_t)));
    CK(pool_alloc(ctx, reinterpret_cast<void **>(&res->d_vals), cap * sizeof(float)));
    CK(pool_alloc(ctx, reinterpret_cast<void **>(&res->d_segcnt), (size_t)(res->rank_layout ? 1 : 32) * nseg * sizeof(uint32_t)));
    CK(pool_alloc(ctx, reinterpret_cast<void **>(&res->d_counts), (33 + 32) * sizeof(unsigned long long)));
    if (!ctx->free_pinned.empty()) { res->h_counts = ctx->free_pinned.back(); ctx->free_pinned.pop_back(); }
    else CK(cudaHostAlloc(reinterpret_cast<void **>(&res->h_counts), 34 * sizeof(unsigned long long), cudaHostAllocDefault));
    res->h_counts[33] = 0;
    res->ready = get_event(ctx);
    if (res->rank_layout) { // index order is the canonical order: one order-preserving compaction of the whole table
        Region rg(ctx, F_OTHER, 3);
        const uint32_t total = (uint32_t)res->n_masks;
        CK(cudaMemsetAsync(res->d_counts, 0, 33 * sizeof(unsigned long long), s));
        rank_compact_count_kernel<<<nseg, kRankCompactThreads, 0, s>>>(res->d_table, total, res->d_segcnt);
        rank_compact_scan_kernel<<<1, 1024, 0, s>>>(res->d_segcnt, nseg, res->d_counts);
        rank_compact_write_kernel<<<nseg, kRankCompactThreads, 0, s>>>(res->d_table, total, res->d_segcnt, res->d_masks, res->d_vals);
    } else {
        Region rg(ctx, F_OTHER, 4);
        compact_count_kernel<<<nseg, kCompactThreads, 0, s>>>(res->d_table, res->n_masks, nseg, res->d_segcnt);
        compact_scan_kernel<<<32, 1024, 0, s>>>(res->d_segcnt, nseg, res->d_counts);
        compact_bases_kernel<<<1, 32, 0, s>>>(res->d_counts, res->d_counts + 33);
        compact_write_kernel<<<nseg, kCompactThreads, 0, s>>>(res->d_table, res->n_masks, nseg, res->d_segcnt, res->d_counts + 33, res->d_masks, res->d_vals);
    }
    CK(cudaMemcpyAsync(res->h_counts, res->d_counts, 33 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    if (res->d_ovf) CK(cudaMemcpyAsync(&res->h_counts[33], res->d_ovf, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(res->ready, s));
    CK(cudaGetLastError());
    res->prefetched = true;
    return URLGPU_OK;
}

static int result_wait_counts(urlgpu_result *res) {
    urlgpu_ctx *ctx = res->ctx;
    if (res->counted) return URLGPU_OK;
    int rc = result_prefetch_impl(res);
    if (rc) return rc;
    CK(cudaEventSynchronize(res->ready));
    if (res->d_ovf && (res->h_counts[33] & 0xffffffffull) != 0) {
        // a cell count did not fit 16 bits somewhere in this variable's tables: the scores are discarded and the family is
        // recomputed with 32-bit tables on the result's own table, then filtered and compacted again
        ctx->st.table16_fallbacks++;
        ctx->t16_overflowed.insert(res->variable);   // a hint only (32-bit tables are always right): kept while the data set keeps its shape
        pool_free(ctx, res->d_ovf);
        res->d_ovf = nullptr;
        res->h_counts[33] = 0;
        pool_free(ctx, res->d_masks); pool_free(ctx, res->d_vals); pool_free(ctx, res->d_segcnt); pool_free(ctx, res->d_counts);
        res->d_masks = nullptr; res->d_vals = nullptr; res->d_segcnt = nullptr; res->d_counts = nullptr;
        ctx->free_events.push_back(res->ready);
        res->ready = nullptr;
        ctx->free_pinned.push_back(res->h_counts);
        res->h_counts = nullptr;
        cudaStream_t s = ctx->stream;
        fill_u32_kernel<<<blocks_for(res->n_masks, 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(res->d_table), res->n_masks, kSentinelBits);
        uint64_t ns = 0;
        rc = select_discrete_score(ctx, res->score_type, res->variable, 1.0);   // a later call may have selected another score / arity (never BDeu: no cube path)
        if (rc) return rc;
        rc = bic_score_family(ctx, res->variable, res->cand, res->max_parents, res->d_table, &ns, res->rank_layout ? res->rs : RankSpace{}, nullptr);
        if (rc) return rc;
        rc = apply_filters(ctx, res, true, res->filter_flags);
        if (rc) return rc;
        res->prefetched = false;
        rc = result_prefetch_impl(res);
        if (rc) return rc;
        CK(cudaEventSynchronize(res->ready));
    }
    res->n_stored = res->h_counts[32];
    for (int l = 0; l < 32; l++) res->layer_count[l] = res->h_counts[l];
    if (res->n_stored > std::min<uint64_t>(res->n_scored, res->n_masks)) return ctx->fail(URLGPU_ERR_INTERNAL, "result: more stored entries than scored sets");
    res->counted = true;
    return URLGPU_OK;
}

extern "C" int urlgpu_result_prefetch(urlgpu_result *res) {
    if (!res) return URLGPU_ERR_ARG;
    return result_prefetch_impl(res);
}

extern "C" int urlgpu_result_count(urlgpu_result *res, uint64_t *n) {
    if (!res || !n) return URLGPU_ERR_ARG;
    int rc = result_wait_counts(res);
    if (rc) return rc;
    *n = res->n_stored;
    return URLGPU_OK;
}
extern "C" int urlgpu_result_scored(urlgpu_result *res, uint64_t *n) {
    if (!res || !n) return URLGPU_ERR_ARG;
    *n = res->n_scored;
    return URLGPU_OK;
}

extern "C" int urlgpu_result_fetch(urlgpu_result *res, uint64_t offset, uint64_t n, uint64_t *masks, float *scores) {
    if (!res) return URLGPU_ERR_ARG;
    urlgpu_ctx *ctx = res->ctx;
    CK(cudaSetDevice(ctx->device));
    int rc = result_wait_counts(res);
    if (rc) return rc;
    if (offset + n > res->n_stored) return ctx->fail(URLGPU_ERR_ARG, "result_fetch: range exceeds the stored count");
    if (n == 0) return URLGPU_OK;
    cudaStream_t cs = ctx->copy_stream; // the compaction has completed (ready event): nothing here waits for later scoring work
    if (masks) {
        const size_t need = n * (size_t)res->mask_words * sizeof(uint64_t);
        if (ctx->fetch_wide_cap < need) {
            if (ctx->d_fetch_wide) cudaFree(ctx->d_fetch_wide);
            ctx->d_fetch_wide = nullptr; ctx->fetch_wide_cap = 0;
            const size_t cap = std::max<size_t>(need + need / 2, (size_t)1 << 20);
            CK(cudaMalloc(reinterpret_cast<void **>(&ctx->d_fetch_wide), cap));
            ctx->fetch_wide_cap = cap;
        }
        if (!ctx->d_fetch_cand) CK(cudaMalloc(reinterpret_cast<void **>(&ctx->d_fetch_cand), (kMaxRankCand + 2) * sizeof(int)));
        if (!res->cand.empty()) CK(cudaMemcpyAsync(ctx->d_fetch_cand, res->cand.data(), res->cand.size() * sizeof(int), cudaMemcpyHostToDevice, cs));
        if (res->rank_layout)
            rank_expand_kernel<<<blocks_for(n, 256), 256, rs_binom_bytes(res->rs), cs>>>(res->rs, res->d_masks + offset, n, ctx->d_fetch_cand, res->mask_words, ctx->d_fetch_wide);
        else
            expand_masks_kernel<<<blocks_for(n, 256), 256, 0, cs>>>(res->d_masks + offset, n, ctx->d_fetch_cand, res->c, res->mask_words, ctx->d_fetch_wide);
        CK(cudaMemcpyAsync(masks, ctx->d_fetch_wide, need, cudaMemcpyDeviceToHost, cs));
    }
    if (scores) CK(cudaMemcpyAsync(scores, res->d_vals + offset, n * sizeof(float), cudaMemcpyDeviceToHost, cs));
    CK(cudaStreamSynchronize(cs));
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// The same entries into DEVICE memory — this device's or a peer-mapped buffer on another GPU (urlgpu_peer_open): the expansion
// kernel writes the wide masks straight to the destination, the scores follow with one device-to-device copy.  Masks are
// written with `mask_words_out` words and every variable index shifted up by `variable_shift` (a data set that is one block
// of a larger one: the gathered cache then names the global variables).
extern "C" int urlgpu_result_fetch_device(urlgpu_result *res, uint64_t offset, uint64_t n, int mask_words_out, int variable_shift, uint64_t *d_masks, float *d_scores) {
    if (!res) return URLGPU_ERR_ARG;
    urlgpu_ctx *ctx = res->ctx;
    CK(cudaSetDevice(ctx->device));
    int rc = result_wait_counts(res);
    if (rc) return rc;
    if (offset + n > res->n_stored) return ctx->fail(URLGPU_ERR_ARG, "result_fetch_device: range exceeds the stored count");
    if (variable_shift < 0 || mask_words_out < 1) return ctx->fail(URLGPU_ERR_ARG, "result_fetch_device: bad mask width or shift");
    for (int v : res->cand)
        if ((v + variable_shift) / 64 >= mask_words_out) return ctx->fail(URLGPU_ERR_ARG, "result_fetch_device: mask_words_out is too small for the shifted variables");
    if (n == 0) return URLGPU_OK;
    cudaStream_t cs = ctx->copy_stream;
    if (d_masks) {
        if (!ctx->d_fetch_cand) CK(cudaMalloc(reinterpret_cast<void **>(&ctx->d_fetch_cand), (kMaxRankCand + 2) * sizeof(int)));
        std::vector<int> shifted(res->cand);
        for (int &v : shifted) v += variable_shift;
        if (!shifted.empty()) CK(cudaMemcpyAsync(ctx->d_fetch_cand, shifted.data(), shifted.size() * sizeof(int), cudaMemcpyHostToDevice, cs));
        if (res->rank_layout)
            rank_expand_kernel<<<blocks_for(n, 256), 256, rs_binom_bytes(res->rs), cs>>>(res->rs, res->d_masks + offset, n, ctx->d_fetch_cand, mask_words_out, d_masks);
        else
            expand_masks_kernel<<<blocks_for(n, 256), 256, 0, cs>>>(res->d_masks + offset, n, ctx->d_fetch_cand, res->c, mask_words_out, d_masks);
    }
    if (d_scores) CK(cudaMemcpyAsync(d_scores, res->d_vals + offset, n * sizeof(float), cudaMemcpyDefault, cs));
    CK(cudaStreamSynchronize(cs));   // `shifted` goes out of scope; the caller may publish the destination after this returns
    CK(cudaGetLastError());
    return URLGPU_OK;
}
// plain copy out of a device buffer named by address (e.g. a score board others filled): the binding has no other way to read one
extern "C" int urlgpu_copy_to_host(urlgpu_ctx *ctx, void *dst_host, const void *src_device, uint64_t bytes) {
    if (!ctx || (bytes && (!dst_host || !src_device))) return ctx ? ctx->fail(URLGPU_ERR_ARG, "copy_to_host: null argument") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (bytes) {
        CK(cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
        CK(cudaStreamSynchronize(ctx->copy_stream));
    }
    return URLGPU_OK;
}

// page-locked host memory for result payloads: device->host copies into it run at PCIe speed and need no staging copy
extern "C" void *urlgpu_host_alloc(uint64_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void urlgpu_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// ---- peer memory (include/urlgpu.h): score boards that other ranks' kernels write through NVLink ---------------------
extern "C" int urlgpu_peer_alloc(urlgpu_ctx *ctx, uint64_t bytes, void **dev_ptr, unsigned char handle[URLGPU_PEER_HANDLE_BYTES]) {
    if (!ctx || !dev_ptr || !handle) return ctx ? ctx->fail(URLGPU_ERR_ARG, "peer_alloc: null argument") : URLGPU_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == URLGPU_PEER_HANDLE_BYTES, "CUDA IPC handle size");
    CK(cudaSetDevice(ctx->device));
    void *p = nullptr;
    CK(cudaMalloc(&p, bytes ? bytes : 1));     // its own allocation: an IPC handle names a whole cudaMalloc block
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return ctx->cuda_fail(e, "cudaIpcGetMemHandle", __LINE__); }
    memcpy(handle, &h, sizeof h);
    *dev_ptr = p;
    return URLGPU_OK;
}
extern "C" int urlgpu_peer_open(urlgpu_ctx *ctx, const unsigned char handle[URLGPU_PEER_HANDLE_BYTES], void **dev_ptr) {
    if (!ctx || !dev_ptr || !handle) return ctx ? ctx->fail(URLGPU_ERR_ARG, "peer_open: null argument") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    void *p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *dev_ptr = p;
    return URLGPU_OK;
}
extern "C" int urlgpu_peer_close(urlgpu_ctx *ctx, void *dev_ptr) {
    if (!ctx) return URLGPU_ERR_ARG;
    if (!dev_ptr) return URLGPU_OK;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaIpcCloseMemHandle(dev_ptr));
    return URLGPU_OK;
}
extern "C" int urlgpu_peer_free(urlgpu_ctx *ctx, void *dev_ptr) {
    if (!ctx) return URLGPU_ERR_ARG;
    if (!dev_ptr) return URLGPU_OK;
    CK(cudaSetDevice(ctx->device));
    CK(cudaFree(dev_ptr));
    return URLGPU_OK;
}

extern "C" int urlgpu_result_free(urlgpu_result *res) {
    if (!res) return URLGPU_OK;
    urlgpu_ctx *ctx = res->ctx;
    cudaSetDevice(ctx->device);
    // stream-ordered reuse: the pool hands these blocks to later work on the same stream, no sync needed
    if (res->d_table) pool_free(ctx, res->d_table);
    if (res->d_ovf) pool_free(ctx, res->d_ovf);
    if (res->d_masks) pool_free(ctx, res->d_masks);
    if (res->d_vals) pool_free(ctx, res->d_vals);
    if (res->d_segcnt) pool_free(ctx, res->d_segcnt);
    if (res->d_counts) pool_free(ctx, res->d_counts);
    if (res->h_counts) {
        if (res->ready) cudaEventSynchronize(res->ready); // the pinned block must not be recycled while its copy is in flight
        ctx->free_pinned.push_back(res->h_counts);
    }
    if (res->ready) ctx->free_events.push_back(res->ready);
    delete res;
    return URLGPU_OK;
}

// ============================================================================================ sparse parent graph (device query structure)

struct urlgpu_spg {
    urlgpu_ctx *ctx = nullptr;
    uint64_t n = 0, bw = 0;
    int words = 1, variable_count = 0;
    uint64_t *d_masks = nullptr;
    float *d_scores = nullptr;
    uint64_t *d_not_used = nullptr;
    std::vector<uint64_t> h_masks;   // sorted order, for best_parents
};

extern "C" int urlgpu_spg_build(urlgpu_ctx *ctx, const uint64_t *masks, const float *scores, uint64_t n, int mask_words, int variable_count, urlgpu_spg **out) {
    if (!ctx || !out || (n && (!masks || !scores)) || mask_words < 1 || mask_words > kSpgMaxWords || variable_count < 1 || variable_count > mask_words * 64)
        return ctx ? ctx->fail(URLGPU_ERR_ARG, "spg_build: bad argument") : URLGPU_ERR_ARG;
    *out = nullptr;
    CK(cudaSetDevice(ctx->device));
    // sorted by (score ascending, |S|, mask): sparse_parent_bitwise.cpp:33-46 sorts by score; ties get a deterministic order
    std::vector<uint64_t> order(n);
    for (uint64_t i = 0; i < n; i++) order[i] = i;
    auto card = [&](uint64_t i) { int c = 0; for (int w = 0; w < mask_words; w++) c += __builtin_popcountll(masks[i * mask_words + w]); return c; };
    std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) {
        if (scores[a] != scores[b]) return scores[a] < scores[b];
        const int ca = card(a), cb = card(b);
        if (ca != cb) return ca < cb;
        for (int w = mask_words - 1; w >= 0; w--)
            if (masks[a * mask_words + w] != masks[b * mask_words + w]) return masks[a * mask_words + w] < masks[b * mask_words + w];
        return a < b;
    });
    auto *sp = new urlgpu_spg();
    sp->ctx = ctx; sp->n = n; sp->words = mask_words; sp->variable_count = variable_count; sp->bw = (n + 63) / 64;
    sp->h_masks.resize(n * mask_words);
    std::vector<float> hs(n);
    for (uint64_t i = 0; i < n; i++) {
        memcpy(&sp->h_masks[i * mask_words], &masks[order[i] * mask_words], mask_words * sizeof(uint64_t));
        hs[i] = scores[order[i]];
    }
    cudaStream_t s = ctx->stream;
    auto fail = [&](cudaError_t e, int line) { if (sp->d_masks) cudaFree(sp->d_masks); if (sp->d_scores) cudaFree(sp->d_scores); if (sp->d_not_used) cudaFree(sp->d_not_used); delete sp; return ctx->cuda_fail(e, "spg_build", line); };
    cudaError_t e;
    if ((e = cudaMalloc(reinterpret_cast<void **>(&sp->d_masks), std::max<size_t>(8, n * mask_words * sizeof(uint64_t)))) != cudaSuccess) return fail(e, __LINE__);
    if ((e = cudaMalloc(reinterpret_cast<void **>(&sp->d_scores), std::max<size_t>(4, n * sizeof(float)))) != cudaSuccess) return fail(e, __LINE__);
    if ((e = cudaMalloc(reinterpret_cast<void **>(&sp->d_not_used), std::max<size_t>(8, sp->bw * variable_count * sizeof(uint64_t)))) != cudaSuccess) return fail(e, __LINE__);
    if (n) {
        if ((e = cudaMemcpyAsync(sp->d_masks, sp->h_masks.data(), n * mask_words * sizeof(uint64_t), cudaMemcpyHostToDevice, s)) != cudaSuccess) return fail(e, __LINE__);
        if ((e = cudaMemcpyAsync(sp->d_scores, hs.data(), n * sizeof(float), cudaMemcpyHostToDevice, s)) != cudaSuccess) return fail(e, __LINE__);
        {
            Region rg(ctx, F_OTHER, 1);
            spg_build_kernel<<<blocks_for(sp->bw * variable_count, 256), 256, 0, s>>>(sp->d_masks, n, mask_words, variable_count, sp->bw, sp->d_not_used);
        }
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail(e, __LINE__); // hs goes out of scope
    }
    *out = sp;
    return URLGPU_OK;
}

extern "C" int urlgpu_spg_query(urlgpu_spg *sp, const uint64_t *allowed, uint64_t nq, float *best_scores, uint64_t *best_parents, int64_t *best_index) {
    if (!sp) return URLGPU_ERR_ARG;
    urlgpu_ctx *ctx = sp->ctx;
    if (!allowed || !best_scores) return ctx->fail(URLGPU_ERR_ARG, "spg_query: null argument");
    if (nq == 0) return URLGPU_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    DevBuf dq(ctx), db(ctx), di(ctx);
    CK(dq.alloc(nq * sp->words * sizeof(uint64_t)));
    CK(db.alloc(nq * sizeof(float)));
    CK(di.alloc(nq * sizeof(long long)));
    CK(cudaMemcpyAsync(dq.p, allowed, nq * sp->words * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    {
        Region rg(ctx, F_OTHER, 1);
        spg_query_kernel<<<blocks_for(nq * 32, 256), 256, 0, s>>>(sp->d_not_used, sp->d_scores, sp->n, sp->bw, sp->variable_count, sp->words, dq.as<uint64_t>(), nq,
                                                                 db.as<float>(), di.as<long long>());
    }
    std::vector<long long> hi(nq);
    CK(cudaMemcpyAsync(best_scores, db.p, nq * sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(hi.data(), di.p, nq * sizeof(long long), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    for (uint64_t i = 0; i < nq; i++) {
        if (best_index) best_index[i] = hi[i];
        if (best_parents)
            for (int w = 0; w < sp->words; w++) best_parents[i * sp->words + w] = hi[i] >= 0 ? sp->h_masks[(uint64_t)hi[i] * sp->words + w] : 0;
    }
    return URLGPU_OK;
}

extern "C" int urlgpu_spg_free(urlgpu_spg *sp) {
    if (!sp) return URLGPU_OK;
    cudaSetDevice(sp->ctx->device);
    cudaStreamSynchronize(sp->ctx->stream);
    cudaFree(sp->d_masks); cudaFree(sp->d_scores); cudaFree(sp->d_not_used);
    delete sp;
    return URLGPU_OK;
}

// ============================================================================================ order-graph search
// urlgpu_order_search, urlgpu_order_search_layered, urlgpu_order_local_search and urlgpu_order_local_search_sparse
// (order_kernels.cuh).  order_prepare validates everything on the host, keeps the component's qualifying entries, sorts each
// variable's list in the (score, |S|, mask) order of SortedEntries::build and lays out the best-parent tables, compacting each
// entry straight from its variable-space mask onto cand_v's bits; the sparse form has no tables and gets each entry's parent set
// over C's positions instead.  order_tables uploads the entries and builds the tables.  Each entry point sizes its call before
// any allocation; the host maps each chosen sorted position back to its parent mask.
struct OrderPrep {
    std::vector<int> vars;                       // position j of C -> variable
    std::vector<std::vector<uint64_t>> ent;      // per position: indices into masks/scores, sorted
    std::vector<std::vector<int>> cand;          // per position: cand_j as positions in C, ascending
    std::vector<uint64_t> table;                 // per position: offset of T_j (uint32 elements), 2^c_j of them
    std::vector<uint32_t> score;                 // per position: offset of j's sorted entries
    std::vector<unsigned long long> where;       // per sorted entry: its slot in the tables
    std::vector<uint32_t> epos;                  // per sorted entry: its position in its variable's list
    std::vector<float> escore;                   // per sorted entry: its score
    std::vector<unsigned long long> ewords;      // sparse: word w of sorted entry e's parent set over C at [w * n_ent + e]
    int words = 0;                               // sparse: ceil(k / 64)
    uint64_t n_ent = 0, table_elems = 0;
};

// every check and translation the four entry points share; `who` prefixes the messages.  Components of more than max_k
// variables and variables with more than max_cand candidate parents inside the component are refused.  sparse: no table
// layout (2^c_v would overflow past 63 candidates), the entries' words over C instead
static int order_prepare(urlgpu_ctx *ctx, const std::string &who, int max_k, int max_cand, bool sparse, int p, int mask_words, const uint64_t *offsets,
                         const uint64_t *masks, const float *scores, const uint64_t *component, OrderPrep &P) {
    auto refuse = [&](int code, const std::string &m) { return ctx->fail(code, who + m); };
    if (p < 1) return refuse(URLGPU_ERR_ARG, "p must be at least 1");
    if (mask_words < 1 || mask_words > kSpgMaxWords) return refuse(URLGPU_ERR_ARG, "mask_words must be in 1.." + std::to_string(kSpgMaxWords));
    if ((int64_t)mask_words * 64 < p) return refuse(URLGPU_ERR_ARG, "mask_words too small for the variable count");
    for (int v = 0; v < p; v++)
        if (offsets[v + 1] < offsets[v]) return refuse(URLGPU_ERR_ARG, "offsets decrease at variable " + std::to_string(v));
    if (offsets[p] > offsets[0] && (!masks || !scores)) return refuse(URLGPU_ERR_ARG, "null entries");
    auto bit = [&](const uint64_t *m, int v) { return (m[v >> 6] >> (v & 63)) & 1; };
    std::vector<int> pos_of(p, -1);
    for (int w = 0; w < mask_words; w++)
        for (int b = 0; b < 64; b++) {
            if (!((component[w] >> b) & 1)) continue;
            if (w * 64 + b >= p) return refuse(URLGPU_ERR_ARG, "the component names variable " + std::to_string(w * 64 + b) + " >= p");
            pos_of[w * 64 + b] = (int)P.vars.size();
            P.vars.push_back(w * 64 + b);
        }
    if (P.vars.empty()) return refuse(URLGPU_ERR_ARG, "empty component");
    for (int v = 0; v < p; v++)
        for (uint64_t e = offsets[v]; e < offsets[v + 1]; e++) {
            if (std::isnan(scores[e])) return refuse(URLGPU_ERR_ARG, "variable " + std::to_string(v) + ", entry " + std::to_string(e - offsets[v]) + ": NaN score");
            if (bit(masks + e * mask_words, v)) return refuse(URLGPU_ERR_ARG, "variable " + std::to_string(v) + ", entry " + std::to_string(e - offsets[v]) + ": the parent set contains the variable itself");
        }
    const int k = (int)P.vars.size();
    if (k > max_k) return refuse(URLGPU_ERR_LIMIT, std::to_string(k) + " variables in the component; at most " + std::to_string(max_k) + " are supported");

    // qualifying entries (all parents inside C), per-variable sort, cand_j, table layout
    P.ent.assign(k, {});
    P.cand.assign(k, {});
    P.table.assign(k, 0);
    P.score.assign(k, 0);
    for (int j = 0; j < k; j++) {
        const int v = P.vars[j];
        auto &E = P.ent[j];
        std::vector<uint64_t> cw(mask_words, 0);
        for (uint64_t e = offsets[v]; e < offsets[v + 1]; e++) {
            bool inside = true;
            for (int w = 0; w < mask_words && inside; w++) inside = (masks[e * mask_words + w] & ~component[w]) == 0;
            if (!inside) continue;
            E.push_back(e);
            for (int w = 0; w < mask_words; w++) cw[w] |= masks[e * mask_words + w];
        }
        auto card = [&](uint64_t i) { int c = 0; for (int w = 0; w < mask_words; w++) c += __builtin_popcountll(masks[i * mask_words + w]); return c; };
        std::sort(E.begin(), E.end(), [&](uint64_t a, uint64_t b) {   // as urlgpu_spg_build (sparse_parent_list.cpp:7-9, ties by |S|, mask)
            if (scores[a] != scores[b]) return scores[a] < scores[b];
            const int ca = card(a), cb = card(b);
            if (ca != cb) return ca < cb;
            for (int w = mask_words - 1; w >= 0; w--)
                if (masks[a * mask_words + w] != masks[b * mask_words + w]) return masks[a * mask_words + w] < masks[b * mask_words + w];
            return a < b;
        });
        if (E.size() > 0xFFFFFFFEull) return refuse(URLGPU_ERR_LIMIT, "variable " + std::to_string(v) + " has 2^32 or more entries inside the component");
        for (int u = 0; u < p; u++) if (bit(cw.data(), u)) P.cand[j].push_back(pos_of[u]);
        if (P.cand[j].size() > (size_t)max_cand)
            return refuse(URLGPU_ERR_LIMIT, "variable " + std::to_string(v) + " has " + std::to_string(P.cand[j].size()) +
                                                " candidate parents inside the component; at most " + std::to_string(max_cand) + " are supported");
        P.table[j] = P.table_elems;
        P.score[j] = (uint32_t)P.n_ent;
        if (!sparse) P.table_elems += (uint64_t)1 << P.cand[j].size();
        P.n_ent += E.size();
    }
    if (P.n_ent > 0xFFFFFFFFull) return refuse(URLGPU_ERR_LIMIT, "2^32 or more entries inside the component");
    P.escore.resize(P.n_ent);
    if (sparse) {
        P.words = (k + 63) / 64;
        P.ewords.assign((size_t)P.words * P.n_ent, 0);
    } else {
        P.where.resize(P.n_ent);
        P.epos.resize(P.n_ent);
    }
    for (int j = 0; j < k; j++)
        for (size_t i = 0; i < P.ent[j].size(); i++) {
            const uint64_t *m = masks + P.ent[j][i] * mask_words;
            const uint64_t e = P.score[j] + i;
            P.escore[e] = scores[P.ent[j][i]];
            if (sparse) {                                      // the entry over C's positions
                for (int q : P.cand[j]) if (bit(m, P.vars[q])) P.ewords[(size_t)(q >> 6) * P.n_ent + e] |= 1ull << (q & 63);
                continue;
            }
            uint64_t idx = 0;                                  // the entry over cand_j's bits
            for (size_t q = 0; q < P.cand[j].size(); q++) if (bit(m, P.vars[P.cand[j][q]])) idx |= 1ull << q;
            P.where[e] = P.table[j] + idx;
            P.epos[e] = (uint32_t)i;
        }
    return URLGPU_OK;
}

// d_ent = where | pos | score (16 bytes an entry); T = every T_j: fill, scatter, subset-min transform, under ms_order_tables
static int order_tables(urlgpu_ctx *ctx, const OrderPrep &P, void *d_ent, uint32_t *T) {
    cudaStream_t s = ctx->stream;
    const uint64_t n_ent = P.n_ent;
    unsigned long long *dw = static_cast<unsigned long long *>(d_ent);
    uint32_t *dp = reinterpret_cast<uint32_t *>(dw + n_ent);
    float *ds = reinterpret_cast<float *>(dp + n_ent);
    if (n_ent) {
        CK(cudaMemcpyAsync(dw, P.where.data(), n_ent * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dp, P.epos.data(), n_ent * 4, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ds, P.escore.data(), n_ent * 4, cudaMemcpyHostToDevice, s));
    }
    const int k = (int)P.vars.size();
    uint64_t launches = 1;
    for (int j = 0; j < k; j++) launches += 1 + std::max(0, (int)P.cand[j].size() - kOrderSegBits);
    Region rg(ctx, F_ORDER_TABLES, launches);
    CK(cudaMemsetAsync(T, 0xFF, P.table_elems * 4, s));
    if (n_ent) order_scatter_kernel<<<blocks_for(n_ent, 256), 256, 0, s>>>(dw, dp, n_ent, T);
    for (int j = 0; j < k; j++) {
        const int c = (int)P.cand[j].size(), lb = std::min(c, kOrderSegBits);
        uint32_t *Tj = T + P.table[j];
        if (lb) order_table_low_kernel<<<(unsigned)(1u << (c - lb)), std::min(1024, std::max(32, 1 << (lb - 1))), 0, s>>>(Tj, lb);
        for (int b = lb; b < c; b++) order_table_high_kernel<<<blocks_for((uint64_t)1 << (c - 1), 256), 256, 0, s>>>(Tj, b, (uint64_t)1 << (c - 1));
    }
    CK(cudaGetLastError());
    return URLGPU_OK;
}

// the device's free memory plus the allocator's idle blocks
static int order_free_bytes(urlgpu_ctx *ctx, size_t *free_b) {
    CK(cudaSetDevice(ctx->device));
    size_t total_b = 0;
    CK(cudaMemGetInfo(free_b, &total_b));
    for (auto &b : ctx->pool) if (!b.used) *free_b += b.bytes;      // cached blocks the allocator can hand out or release
    return URLGPU_OK;
}

static int order_search_impl(urlgpu_ctx *ctx, bool layered, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                             const float *scores, const uint64_t *edges, const uint64_t *component, float *cost, int32_t *order,
                             uint64_t *parents) {
    if (!ctx) return URLGPU_ERR_ARG;
    const std::string who = layered ? "order_search_layered: " : "order_search: ";
    auto refuse = [&](int code, const std::string &m) { return ctx->fail(code, who + m); };
    if (!offsets || !component || !cost || !order || !parents) return refuse(URLGPU_ERR_ARG, "null argument");
    OrderPrep P;
    const int max_k = layered ? kOrderRankMaxVars : kOrderMaxVars;        // c_v < k, so max_k - 1 never refuses a variable
    if (int rc = order_prepare(ctx, who, max_k, max_k - 1, false, p, mask_words, offsets, masks, scores, component, P)) return rc;
    const int k = (int)P.vars.size();
    const uint64_t n_ent = P.n_ent, table_elems = P.table_elems;
    std::vector<OrderVarRank> hv(k);
    for (int j = 0; j < k; j++) {
        uint64_t cand = 0;
        for (int q : P.cand[j]) cand |= 1ull << q;
        hv[j].table = P.table[j];
        hv[j].score = P.score[j];
        hv[j].cand = cand;
        hv[j].adj = ~0ull;
        if (edges) {
            hv[j].adj = 0;
            for (int i = 0; i < k; i++) if ((edges[(size_t)P.vars[j] * mask_words + (P.vars[i] >> 6)] >> (P.vars[i] & 63)) & 1) hv[j].adj |= 1ull << i;
        }
        for (int b = 0; b < kOrderRankLut; b++) hv[j].shift[b] = (uint8_t)__builtin_popcountll(cand & ((1ull << (8 * b)) - 1));
    }

    // binomials: C(b, i) for b, i <= kOrderRankMaxVars (the dense kernels take the uint32 corner b, i <= kOrderMaxVars)
    std::vector<unsigned long long> binom(kOrderRankBinom * kOrderRankBinom, 0);
    for (int b = 0; b < kOrderRankBinom; b++)
        for (int i = 0; i <= b; i++) binom[b * kOrderRankBinom + i] = i == 0 || i == b ? 1ull : binom[(b - 1) * kOrderRankBinom + i - 1] + binom[(b - 1) * kOrderRankBinom + i];
    std::vector<uint32_t> binom32(kOrderBinom * kOrderBinom);
    for (int b = 0; b < kOrderBinom; b++)
        for (int i = 0; i < kOrderBinom; i++) binom32[b * kOrderBinom + i] = (uint32_t)binom[b * kOrderRankBinom + i];

    // the device memory of the call, before anything is allocated.  Dense: a cost and a leaf for each of the 2^k nodes.
    // Layered: a leaf for each node and the costs of two layers, each at most C(k, k/2) nodes
    const int n_lut = layered ? kOrderRankLut : 4;
    const size_t var_bytes = layered ? sizeof(OrderVarRank) : sizeof(OrderVar);
    const size_t binom_bytes = layered ? binom.size() * 8 : binom32.size() * 4;
    const uint64_t nodes = (uint64_t)1 << k, widest = binom[k * kOrderRankBinom + k / 2];
    const size_t small_bytes = (size_t)k * var_bytes + (size_t)k * n_lut * 256 + binom_bytes + (2 + 2 * (size_t)k) * 4;
    const uint64_t node_bytes = layered ? nodes + 8 * widest : 5 * nodes;
    const size_t need = node_bytes + 4 * table_elems + n_ent * (8 + 4 + 4) + small_bytes;
    size_t free_b = 0;
    if (int rc = order_free_bytes(ctx, &free_b)) return rc;
    auto bytes_msg = [&]() {
        const std::string nodes_part = layered ? std::to_string(nodes) + " for the leaves of the 2^" + std::to_string(k) + " nodes, " +
                                                     std::to_string(8 * widest) + " for two cost layers of C(" + std::to_string(k) + ", " + std::to_string(k / 2) + ") nodes, "
                                               : std::to_string(5 * nodes) + " for the 2^" + std::to_string(k) + " nodes, ";
        return std::to_string(need) + " bytes of device memory (" + nodes_part + std::to_string(4 * table_elems) + " for the best-parent tables)";
    };
    if (need > free_b) return refuse(URLGPU_ERR_LIMIT, "the search needs " + bytes_msg() + ", " + std::to_string(free_b) + " are free");

    // host arrays: descriptors and byte look-up tables
    std::vector<OrderVar> hv32(layered ? 0 : k);
    for (int j = 0; j < (int)hv32.size(); j++) {
        hv32[j].table = hv[j].table;
        hv32[j].score = hv[j].score;
        hv32[j].adj = (uint32_t)hv[j].adj;
        hv32[j].cand = (uint32_t)hv[j].cand;
        for (int b = 0; b < 4; b++) hv32[j].shift[b] = hv[j].shift[b];
    }
    std::vector<uint8_t> lut((size_t)k * n_lut * 256);
    for (int j = 0; j < k; j++)
        for (int b = 0; b < n_lut; b++) {
            const uint32_t cb = (uint32_t)(hv[j].cand >> (8 * b)) & 255;
            for (uint32_t x = 0; x < 256; x++) {
                uint32_t c = 0; int q = 0;
                for (int i = 0; i < 8; i++) if ((cb >> i) & 1) { if ((x >> i) & 1) c |= 1u << q; q++; }
                lut[((size_t)j * n_lut + b) * 256 + x] = (uint8_t)c;
            }
        }

    cudaStream_t s = ctx->stream;
    DevBuf d_cost(ctx), d_leaf(ctx), d_tab(ctx), d_small(ctx), d_ent(ctx);
    auto alloc = [&](DevBuf &b, size_t bytes) {
        const cudaError_t e = b.alloc(bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return false; }
        return true;
    };
    const size_t ent_bytes = std::max<size_t>(16, n_ent * 16);
    const size_t cost_bytes = layered ? 8 * widest : 4 * nodes;
    if (!alloc(d_cost, cost_bytes) || !alloc(d_leaf, nodes) || !alloc(d_tab, table_elems * 4) || !alloc(d_small, small_bytes + 64) || !alloc(d_ent, ent_bytes))
        return refuse(URLGPU_ERR_LIMIT, "allocating " + bytes_msg() + " failed");
    // d_small: vars | lut | binom | out
    char *sm = d_small.as<char>();
    uint8_t *dl = reinterpret_cast<uint8_t *>(sm + k * var_bytes);
    char *db = reinterpret_cast<char *>(dl + lut.size());
    uint32_t *dout = reinterpret_cast<uint32_t *>(db + binom_bytes);
    CK(cudaMemcpyAsync(sm, layered ? (const void *)hv.data() : (const void *)hv32.data(), k * var_bytes, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(dl, lut.data(), lut.size(), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(db, layered ? (const void *)binom.data() : (const void *)binom32.data(), binom_bytes, cudaMemcpyHostToDevice, s));
    uint32_t *T = d_tab.as<uint32_t>();
    if (int rc = order_tables(ctx, P, d_ent.p, T)) return rc;
    const float *ds = reinterpret_cast<const float *>(reinterpret_cast<const uint32_t *>(d_ent.as<unsigned long long>() + n_ent) + n_ent);
    float *cst = d_cost.as<float>();
    uint8_t *lf = d_leaf.as<uint8_t>();
    {
        Region rg(ctx, F_ORDER_LAYERS, (uint64_t)k + 1);
        CK(cudaMemsetAsync(cst, 0, sizeof(float), s));            // cost(empty set) = 0
        int per_sm = 0;
        if (!layered) {
            const OrderVar *dv = reinterpret_cast<const OrderVar *>(sm);
            const uint32_t *db32 = reinterpret_cast<const uint32_t *>(db);
            const size_t smem = order_smem_bytes(k);
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, order_layer_kernel, 256, smem));
            const uint64_t grid_cap = (uint64_t)std::max(1, per_sm) * ctx->sm_count;
            for (int l = 1; l <= k; l++) {
                const uint32_t count = binom32[k * kOrderBinom + l];
                const uint64_t runs = (count + kOrderRun - 1) / kOrderRun;
                order_layer_kernel<<<(unsigned)std::min<uint64_t>(grid_cap, (runs + 255) / 256), 256, smem, s>>>(dv, dl, db32, T, ds, k, l, count, cst, lf);
            }
            order_backtrack_kernel<<<1, 32, 0, s>>>(dv, T, cst, lf, k, dout);
        } else {
            const OrderVarRank *dv = reinterpret_cast<const OrderVarRank *>(sm);
            const unsigned long long *db64 = reinterpret_cast<const unsigned long long *>(db);
            const size_t smem = order_rank_smem_bytes(k);
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, order_layer_rank_kernel, 256, smem));
            const uint64_t grid_cap = (uint64_t)std::max(1, per_sm) * ctx->sm_count;
            float *layer_cost[2] = {cst, cst + widest};          // layer l is written to layer_cost[l & 1]
            uint64_t base = 1;                                     // base_l = sum_{m<l} C(k, m)
            for (int l = 1; l <= k; l++) {
                const uint64_t count = binom[k * kOrderRankBinom + l];
                const uint64_t runs = (count + kOrderRun - 1) / kOrderRun;
                order_layer_rank_kernel<<<(unsigned)std::min<uint64_t>(grid_cap, (runs + 255) / 256), 256, smem, s>>>(
                    dv, dl, db64, T, ds, k, l, count, base, layer_cost[(l - 1) & 1], layer_cost[l & 1], lf);
                base += count;
            }
            order_backtrack_rank_kernel<<<1, 32, 0, s>>>(dv, db64, T, layer_cost[k & 1], lf, k, dout);
        }
        CK(cudaGetLastError());
    }
    std::vector<uint32_t> out(2 + 2 * (size_t)k);
    CK(cudaMemcpyAsync(out.data(), dout, out.size() * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    float c;
    memcpy(&c, &out[0], sizeof c);
    if (!out[1] || c == INFINITY) return ctx->fail(URLGPU_ERR_ARG, "No solution found.");   // search_capi.cpp:87
    *cost = c;
    for (int i = 0; i < k; i++) {
        const int j = (int)out[2 + i], v = P.vars[j];
        const uint32_t q = out[2 + k + i];
        order[i] = v;
        for (int w = 0; w < mask_words; w++) parents[(size_t)v * mask_words + w] = q == kOrderNone ? 0 : masks[P.ent[j][q] * mask_words + w];
    }
    return URLGPU_OK;
}

extern "C" int urlgpu_order_search(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks, const float *scores,
                                   const uint64_t *edges, const uint64_t *component, float *cost, int32_t *order, uint64_t *parents) {
    return order_search_impl(ctx, false, p, mask_words, offsets, masks, scores, edges, component, cost, order, parents);
}

extern "C" int urlgpu_order_search_layered(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                                           const float *scores, const uint64_t *edges, const uint64_t *component, float *cost,
                                           int32_t *order, uint64_t *parents) {
    return order_search_impl(ctx, true, p, mask_words, offsets, masks, scores, edges, component, cost, order, parents);
}

// Local search: the tables as above (sparse: the entries' words over C, no tables), then one order_climb_kernel launch over all
// restarts.  The host reads every restart's cost and move count, takes the least cost (ties: the smallest restart), and copies
// back that restart's order and family positions.
static int order_local_search_impl(urlgpu_ctx *ctx, bool sparse, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                                   const float *scores, const uint64_t *edges, const uint64_t *component, uint32_t restarts,
                                   uint64_t seed, float *cost, int32_t *order, uint64_t *parents, float *restart_costs,
                                   uint32_t *restart_moves) {
    if (!ctx) return URLGPU_ERR_ARG;
    const std::string who = sparse ? "order_local_search_sparse: " : "order_local_search: ";
    auto refuse = [&](int code, const std::string &m) { return ctx->fail(code, who + m); };
    if (!offsets || !component || !cost || !order || !parents) return refuse(URLGPU_ERR_ARG, "null argument");
    if (restarts < 1 || restarts > (1u << 20)) return refuse(URLGPU_ERR_ARG, "restarts must be in 1..2^20");
    OrderPrep P;
    if (int rc = order_prepare(ctx, who, kClimbMaxVars, sparse ? kClimbMaxVars - 1 : kClimbMaxCand, sparse, p, mask_words, offsets, masks, scores,
                               component, P))
        return rc;
    const int k = (int)P.vars.size();
    std::vector<OrderClimbVar> hv(k);
    for (int j = 0; j < k; j++) {
        OrderClimbVar &V = hv[j];
        memset(&V, 0, sizeof V);
        V.score = P.score[j];
        V.ncand = (uint32_t)P.cand[j].size();
        if (sparse) {
            V.nent = P.ent[j].size();
        } else {
            V.table = P.table[j];
            for (size_t q = 0; q < P.cand[j].size(); q++) V.cand[q] = (uint8_t)P.cand[j][q];
        }
        for (int i = 0; i < k; i++)
            if (!edges || ((edges[(size_t)P.vars[j] * mask_words + (P.vars[i] >> 6)] >> (P.vars[i] & 63)) & 1)) V.adj[i >> 6] |= 1ull << (i & 63);
    }

    // the device memory of the call: tables, entries (table form: where | position | score, sparse: W words | score), and per
    // restart a cost, a move count, the order and the family positions
    const uint64_t table_bytes = 4 * P.table_elems, ent_bytes = (sparse ? 8 * (uint64_t)P.words + 4 : 16) * P.n_ent;
    const uint64_t restart_bytes = (uint64_t)restarts * (8 + 5 * (uint64_t)k);
    const size_t var_bytes = (size_t)k * sizeof(OrderClimbVar);
    const size_t need = table_bytes + ent_bytes + restart_bytes + var_bytes;
    size_t free_b = 0;
    if (int rc = order_free_bytes(ctx, &free_b)) return rc;
    auto bytes_msg = [&]() {
        return std::to_string(need) + " bytes of device memory (" + (sparse ? "" : std::to_string(table_bytes) + " for the best-parent tables, ") +
               std::to_string(ent_bytes) + " for the entries, " + std::to_string(restart_bytes) + " for the state of " +
               std::to_string(restarts) + " restarts)";
    };
    if (need > free_b) return refuse(URLGPU_ERR_LIMIT, "the search needs " + bytes_msg() + ", " + std::to_string(free_b) + " are free");

    cudaStream_t s = ctx->stream;
    DevBuf d_tab(ctx), d_ent(ctx), d_var(ctx), d_res(ctx);
    auto alloc = [&](DevBuf &b, size_t bytes) {
        const cudaError_t e = b.alloc(bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return false; }
        return true;
    };
    if ((!sparse && !alloc(d_tab, table_bytes)) || !alloc(d_ent, std::max<uint64_t>(16, ent_bytes)) || !alloc(d_var, var_bytes) ||
        !alloc(d_res, restart_bytes))
        return refuse(URLGPU_ERR_LIMIT, "allocating " + bytes_msg() + " failed");
    // d_res: cost | moves | positions | order
    float *r_cost = d_res.as<float>();
    uint32_t *r_moves = reinterpret_cast<uint32_t *>(r_cost + restarts);
    uint32_t *r_pos = r_moves + restarts;
    uint8_t *r_order = reinterpret_cast<uint8_t *>(r_pos + (size_t)restarts * k);
    CK(cudaMemcpyAsync(d_var.p, hv.data(), var_bytes, cudaMemcpyHostToDevice, s));
    const float *ds;
    ClimbTable table{};
    ClimbList list{};
    if (sparse) {                                              // d_ent: words | score
        list.E = d_ent.as<unsigned long long>();
        list.stride = (uint32_t)P.n_ent;
        list.words = P.words;
        ds = reinterpret_cast<const float *>(list.E + P.ewords.size());
        if (P.n_ent) {
            CK(cudaMemcpyAsync(d_ent.p, P.ewords.data(), P.ewords.size() * 8, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(const_cast<float *>(ds), P.escore.data(), P.n_ent * 4, cudaMemcpyHostToDevice, s));
        }
    } else {
        table.T = d_tab.as<uint32_t>();
        if (int rc = order_tables(ctx, P, d_ent.p, d_tab.as<uint32_t>())) return rc;
        ds = reinterpret_cast<const float *>(reinterpret_cast<const uint32_t *>(d_ent.as<unsigned long long>() + P.n_ent) + P.n_ent);
    }
    {
        Region rg(ctx, F_ORDER_LAYERS, 1);
        const size_t smem = order_climb_smem_bytes(k);
        auto launch = [&](auto kernel, const auto &look) -> int {
            int per_sm = 0;
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kClimbThreads, smem));
            const uint64_t grid = std::min<uint64_t>(restarts, (uint64_t)std::max(1, per_sm) * ctx->sm_count);
            kernel<<<(unsigned)grid, kClimbThreads, smem, s>>>(d_var.as<OrderClimbVar>(), look, ds, k, restarts, seed, r_cost, r_moves, r_order, r_pos);
            CK(cudaGetLastError());
            return URLGPU_OK;
        };
        if (int rc = sparse ? launch(order_climb_kernel<ClimbList>, list) : launch(order_climb_kernel<ClimbTable>, table)) return rc;
    }
    std::vector<float> rc_h(restarts);
    std::vector<uint32_t> rm_h(restarts);
    CK(cudaMemcpyAsync(rc_h.data(), r_cost, (size_t)restarts * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rm_h.data(), r_moves, (size_t)restarts * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    uint32_t best = 0;
    for (uint32_t r = 1; r < restarts; r++) if (rc_h[r] < rc_h[best]) best = r;
    if (!(rc_h[best] < INFINITY)) return ctx->fail(URLGPU_ERR_ARG, "No solution found.");   // search_capi.cpp:87
    std::vector<uint8_t> ord(k);
    std::vector<uint32_t> pos(k);
    CK(cudaMemcpyAsync(ord.data(), r_order + (size_t)best * k, k, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(pos.data(), r_pos + (size_t)best * k, (size_t)k * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *cost = rc_h[best];
    for (int m = 0; m < k; m++) {
        const int j = ord[m], v = P.vars[j];
        order[m] = v;
        for (int w = 0; w < mask_words; w++) parents[(size_t)v * mask_words + w] = pos[m] == kOrderNone ? 0 : masks[P.ent[j][pos[m]] * mask_words + w];
    }
    if (restart_costs) memcpy(restart_costs, rc_h.data(), (size_t)restarts * 4);
    if (restart_moves) memcpy(restart_moves, rm_h.data(), (size_t)restarts * 4);
    return URLGPU_OK;
}

extern "C" int urlgpu_order_local_search(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                                         const float *scores, const uint64_t *edges, const uint64_t *component, uint32_t restarts,
                                         uint64_t seed, float *cost, int32_t *order, uint64_t *parents, float *restart_costs,
                                         uint32_t *restart_moves) {
    return order_local_search_impl(ctx, false, p, mask_words, offsets, masks, scores, edges, component, restarts, seed, cost, order, parents,
                                   restart_costs, restart_moves);
}

extern "C" int urlgpu_order_local_search_sparse(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                                                const float *scores, const uint64_t *edges, const uint64_t *component, uint32_t restarts,
                                                uint64_t seed, float *cost, int32_t *order, uint64_t *parents, float *restart_costs,
                                                uint32_t *restart_moves) {
    return order_local_search_impl(ctx, true, p, mask_words, offsets, masks, scores, edges, component, restarts, seed, cost, order, parents,
                                   restart_costs, restart_moves);
}

// ============================================================================================ listed sets
// urlgpu_score_sets, and urlgpu_score_one as a list of one.  The whole list is validated on the host first.  Discrete entries are
// then grouped by child arity (the fNML per-configuration table and bic_score_tables_kernel's rv are per launch) and, inside a
// group, sent to the direct-counting tiers by table size; cBIC entries are grouped by set size, one warp per set.  Every output
// goes to the entry's position in the list.  The launches depend on the groups and tiers present, not on the list's length.
static int score_sets_impl(urlgpu_ctx *ctx, const char *who, bool list, uint64_t n_sets, const int32_t *variables, const uint64_t *parents,
                           int mask_words, int score_type, double lambda, float *scores, double *values64) {
    auto refuse = [&](int code, uint64_t i, const std::string &m) {
        return ctx->fail(code, std::string(who) + ": " + (list ? "entry " + std::to_string(i) + ": " : "") + m);
    };
    CK(cudaSetDevice(ctx->device));
    if (n_sets >= ((uint64_t)1 << 32)) return ctx->fail(URLGPU_ERR_LIMIT, std::string(who) + ": 2^32 or more entries in one call");
    const bool bic = is_discrete(score_type);
    if (!bic && score_type != URLGPU_CBIC) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": unknown score type");
    if (bic && !ctx->have_discrete) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": BIC / fNML need urlgpu_set_discrete first");
    if (!bic && !ctx->have_gram) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": cBIC needs urlgpu_set_continuous first");
    const int p = bic ? ctx->p : ctx->cp;
    if (mask_words < 1 || (int64_t)mask_words * 64 < p) return ctx->fail(URLGPU_ERR_ARG, std::string(who) + ": mask_words too small for the variable count");
    if (score_type == URLGPU_BDEU) { const int rc = select_discrete_score(ctx, score_type, 0, lambda); if (rc) return rc; }   // the ESS and the record count
    const int max_k = bic ? kMaxDenseCand : 200;
    const uint32_t n = (uint32_t)n_sets;
    std::vector<ListEntry> ent(n);
    std::vector<int> par;
    std::vector<uint32_t> cells(bic ? n : 0);
    for (uint32_t i = 0; i < n; i++) {
        const int v = variables[i];
        if (v < 0 || v >= p) return refuse(URLGPU_ERR_ARG, i, "variable out of range");
        const uint64_t *row = parents + (uint64_t)i * mask_words;
        const uint32_t off = (uint32_t)par.size();
        for (int w = 0; w < mask_words; w++) {
            uint64_t x = row[w];
            if (w * 64 + 64 > p && (w * 64 >= p ? x : x >> (p - w * 64))) return refuse(URLGPU_ERR_ARG, i, "mask names a variable >= p");
            if (v >> 6 == w) x &= ~((uint64_t)1 << (v & 63));   // the child itself is not a parent
            for (; x; x &= x - 1) par.push_back(w * 64 + __builtin_ctzll(x));
        }
        const int k = (int)(par.size() - off);
        if (k > max_k) return refuse(URLGPU_ERR_LIMIT, i, "more than " + std::to_string(max_k) + " parents in one set");
        if (par.size() > 0xffffffffull) return refuse(URLGPU_ERR_LIMIT, i, "the list names more than 2^32 parents in all");   // ListEntry::off
        if (bic) {
            uint64_t c = (uint64_t)ctx->card[v];
            for (int j = 0; j < k; j++) { c *= (uint64_t)ctx->card[par[off + j]]; if (c > kCellLimit) return refuse(URLGPU_ERR_LIMIT, i, "contingency table exceeds 2^30 cells"); }
            cells[i] = (uint32_t)c;
        }
        ent[i] = ListEntry{v, k, off};
    }
    if (n == 0) return URLGPU_OK;
    cudaStream_t s = ctx->stream;
    // groups: by child arity (discrete) or by set size (cBIC), entries in list order inside a group
    std::map<int, std::vector<uint32_t>> groups;
    for (uint32_t i = 0; i < n; i++) groups[bic ? ctx->card[ent[i].v] : ent[i].k].push_back(i);
    if (score_type == URLGPU_FNML)   // build every arity's table before anything is launched
        for (auto &g : groups) { const int rc = select_discrete_score(ctx, score_type, ent[g.second[0]].v, lambda); if (rc) return refuse(rc, g.second[0], ctx->err); }
    // the device list: entries, parents, arities, then the keys in launch order (`work`)
    const uint32_t tier1_cells = (uint32_t)((ctx->smem_optin - 2048) / sizeof(int));
    std::vector<uint32_t> work;
    work.reserve(n);
    struct Launch { int group; uint32_t first, count; int tier; };
    std::vector<Launch> launches;
    std::vector<std::vector<GlobalSet>> global(groups.size());
    {
        int gi = 0;
        for (auto &g : groups) {
            if (!bic) { launches.push_back({g.first, (uint32_t)work.size(), (uint32_t)g.second.size(), 0}); work.insert(work.end(), g.second.begin(), g.second.end()); }
            else
                for (int t = 0; t < 2; t++) {
                    const uint32_t first = (uint32_t)work.size();
                    for (uint32_t i : g.second)
                        if (t == 0 ? cells[i] <= kTier0Cells : cells[i] > kTier0Cells && cells[i] <= tier1_cells) work.push_back(i);
                    if (work.size() > first) launches.push_back({gi, first, (uint32_t)work.size() - first, t});
                }
            if (bic)
                for (uint32_t i : g.second) if (cells[i] > tier1_cells) global[gi].push_back(GlobalSet{i, cells[i], 0});
            gi++;
        }
    }
    auto align = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t b_ent = align(n * sizeof(ListEntry)), b_par = align(std::max<size_t>(par.size(), 1) * sizeof(int)), b_card = align(ctx->card.size() * sizeof(int));
    const size_t b_work = align(std::max<size_t>(work.size(), 1) * sizeof(uint32_t)), b_sc = align(n * sizeof(float)), b_v64 = align(n * sizeof(double));
    DevBuf dl(ctx), dout(ctx);
    CK(dl.alloc(b_ent + b_par + b_card + b_work));
    CK(dout.alloc(b_sc + 2 * b_v64));   // scores by key; FP64 / fixed-point values by key; fixed-point values of the shared-memory tiers by work position
    char *base = dl.as<char>();
    const ListEntry *d_ent = reinterpret_cast<const ListEntry *>(base);
    const int *d_par = reinterpret_cast<const int *>(base + b_ent);
    const int *d_card = reinterpret_cast<const int *>(base + b_ent + b_par);
    const uint32_t *d_work = reinterpret_cast<const uint32_t *>(base + b_ent + b_par + b_card);
    float *d_sc = dout.as<float>();
    char *d_v64 = dout.as<char>() + b_sc, *d_pos = d_v64 + b_v64;
    CK(cudaMemcpyAsync(base, ent.data(), n * sizeof(ListEntry), cudaMemcpyHostToDevice, s));
    if (!par.empty()) CK(cudaMemcpyAsync(base + b_ent, par.data(), par.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    if (bic) CK(cudaMemcpyAsync(base + b_ent + b_par, ctx->card.data(), ctx->card.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    if (!work.empty()) CK(cudaMemcpyAsync(base + b_ent + b_par + b_card, work.data(), work.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    constexpr uint32_t kMaxGrid = 0x7fffffffu;
    if (bic) {
        int gi = 0;
        for (auto &g : groups) {
            int rc = select_discrete_score(ctx, score_type, ent[g.second[0]].v, lambda);
            if (rc) return rc;
            const BicData bd{ctx->d_codes, ctx->n, ctx->n_stride, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, ctx->ds_base, ctx->ds_ess, ctx->ds_scale};
            const ListSets fam{d_ent, d_par, d_card, g.first};
            for (const Launch &l : launches) {
                if (l.group != gi) continue;
                Region rg(ctx, F_COUNT, 1);
                for (uint32_t c0 = 0; c0 < l.count; c0 += kMaxGrid) {
                    const uint32_t cnt = std::min(kMaxGrid, l.count - c0);
                    long long *acc = reinterpret_cast<long long *>(d_pos) + l.first + c0;
                    if (l.tier == 0)
                        bic_count_smem_kernel<<<cnt, ctx->n >= 65536 ? 256 : 128, kTier0Cells * sizeof(int), s>>>(bd, fam, d_work + l.first + c0, d_sc, nullptr, nullptr, acc);
                    else
                        bic_count_smem_kernel<<<cnt, 1024, (size_t)tier1_cells * sizeof(int), s>>>(bd, fam, d_work + l.first + c0, d_sc, nullptr, nullptr, acc);
                }
            }
            if (!global[gi].empty()) {
                rc = direct_global_tier(ctx, bd, fam, global[gi], d_sc, reinterpret_cast<long long *>(d_v64), nullptr, 0);
                if (rc) return rc;
            }
            gi++;
        }
    } else {
        const CbicParams prm = cbic_params(ctx, 200, lambda);
        Region rg(ctx, F_CBIC, launches.size());
        for (const Launch &l : launches) {
            const int k = l.group;
            const size_t tsz = (size_t)(k + 1) * (k + 2) / 2;
            // small sets: up to 8 warps in 48 KB; from k = 78 on, one warp holds more than 48 KB (200 parents: 159 KB)
            const uint32_t warps = (uint32_t)std::max<size_t>(1, std::min<size_t>(8, (48 * 1024) / (tsz * sizeof(double))));
            for (uint32_t c0 = 0; c0 < l.count; c0 += kMaxGrid / 8 * warps) {
                const uint32_t cnt = std::min(kMaxGrid / 8 * warps, l.count - c0);
                cbic_sets_kernel<<<blocks_for(cnt, warps), warps * 32, warps * tsz * sizeof(double), s>>>(ctx->d_gram, p, d_ent, d_par, d_work + l.first + c0, cnt, k, prm,
                                                                                                           d_sc, reinterpret_cast<double *>(d_v64));
            }
        }
    }
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(scores, d_sc, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    std::vector<long long> fx, pos;
    if (values64) {
        if (bic) {
            fx.resize(n);
            pos.resize(work.size());
            CK(cudaMemcpyAsync(fx.data(), d_v64, n * sizeof(long long), cudaMemcpyDeviceToHost, s));
            if (!work.empty()) CK(cudaMemcpyAsync(pos.data(), d_pos, work.size() * sizeof(long long), cudaMemcpyDeviceToHost, s));
        } else CK(cudaMemcpyAsync(values64, d_v64, n * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    if (values64 && bic) {   // the shared-memory tiers wrote their fixed-point sums by position in `work`, the global tier by key
        for (size_t j = 0; j < work.size(); j++) fx[work[j]] = pos[j];
        for (uint32_t i = 0; i < n; i++) values64[i] = (double)fx[i] * ctx->ds_scale;
    }
    double work_units = 0;
    for (const ListEntry &e : ent)
        work_units += bic ? (double)ctx->n * (e.k + 1) : (double)e.k * e.k * e.k / 3.0 + 2.0 * e.k * e.k + 2.0 * e.k;
    (bic ? ctx->st.algorithmic_bytes : ctx->st.algorithmic_flops) += work_units;
    ctx->st.sets_scored += n;
    return URLGPU_OK;
}

extern "C" int urlgpu_score_sets(urlgpu_ctx *ctx, uint64_t n_sets, const int32_t *variables, const uint64_t *parents, int mask_words, int score_type,
                                 double lambda, float *scores, double *values64) {
    if (!ctx) return URLGPU_ERR_ARG;
    if (n_sets == 0) return URLGPU_OK;
    if (!variables || !parents || !scores) return ctx->fail(URLGPU_ERR_ARG, "score_sets: null argument");
    return score_sets_impl(ctx, "score_sets", true, n_sets, variables, parents, mask_words, score_type, lambda, scores, values64);
}

extern "C" int urlgpu_score_one(urlgpu_ctx *ctx, int variable, const uint64_t *parents, int mask_words, int score_type, double lambda, float *score,
                                double *value64) {
    if (!ctx || !parents || !score) return ctx ? ctx->fail(URLGPU_ERR_ARG, "score_one: null argument") : URLGPU_ERR_ARG;
    const int32_t v = variable;
    return score_sets_impl(ctx, "score_one", false, 1, &v, parents, mask_words, score_type, lambda, score, value64);
}

// ============================================================================================ counts / prune

// the set of all `cand` as the one entry of a global tier (key space: the family of cand with no parent limit)
static int single_set(urlgpu_ctx *ctx, int variable, const std::vector<int> &cand, std::vector<int> &hv, DevBuf &dcand, RankSets &fam,
                      std::vector<GlobalSet> &one) {
    const int c = (int)cand.size();
    uint64_t cells = (uint64_t)ctx->card[variable];
    for (int b = 0; b < c; b++) { cells *= (uint64_t)ctx->card[cand[b]]; if (cells > kCellLimit) return ctx->fail(URLGPU_ERR_LIMIT, "contingency table exceeds 2^30 cells"); }
    RankSpace rs{};
    int rc = make_rank_space(ctx, c, c, rs);
    if (rc) return rc;
    rc = make_rank_sets(ctx, variable, cand, rs, false, hv, dcand, fam);
    if (rc) return rc;
    one.assign(1, GlobalSet{rs.layer_base[c], (uint32_t)cells, 0});
    return URLGPU_OK;
}

extern "C" int urlgpu_contingency(urlgpu_ctx *ctx, int variable, const uint64_t *parents, int mask_words, int32_t *counts, int64_t n_cells) {
    if (!ctx || !parents || !counts) return ctx ? ctx->fail(URLGPU_ERR_ARG, "contingency: null argument") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_discrete) return ctx->fail(URLGPU_ERR_ARG, "contingency: needs urlgpu_set_discrete first");
    if (variable < 0 || variable >= ctx->p) return ctx->fail(URLGPU_ERR_ARG, "contingency: variable out of range");
    std::vector<int> cand;
    int rc = candidates_from_mask(ctx, ctx->p, variable, parents, mask_words, cand);
    if (rc) return rc;
    const int c = (int)cand.size();
    if (c > kMaxDenseCand) return ctx->fail(URLGPU_ERR_LIMIT, "contingency: more than 30 parents in one set");
    std::vector<int> hv;
    DevBuf dcand(ctx);
    RankSets fam{};
    std::vector<GlobalSet> one;
    rc = single_set(ctx, variable, cand, hv, dcand, fam, one);
    if (rc) return rc;
    if ((int64_t)one[0].cells != n_cells) return ctx->fail(URLGPU_ERR_ARG, "contingency: n_cells must be r_v * prod r_pa = " + std::to_string(one[0].cells));
    BicData bd{ctx->d_codes, ctx->n, ctx->n_stride, ctx->d_qlog, ctx->ds_qcfg, ctx->ds_cfg_min, ctx->ds_base, ctx->ds_ess, ctx->ds_scale};
    return direct_global_tier(ctx, bd, fam, one, nullptr, nullptr, counts, n_cells);
}

extern "C" int urlgpu_prune(urlgpu_ctx *ctx, const uint64_t *masks, const float *scores, uint64_t n, int mask_words, uint8_t *keep) {
    if (!ctx || !masks || !scores || !keep || mask_words < 1) return ctx ? ctx->fail(URLGPU_ERR_ARG, "prune: bad argument") : URLGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (n == 0) return URLGPU_OK;
    // compact the union of all masks to <= 30 bits
    std::vector<uint64_t> uni(mask_words, 0);
    for (uint64_t i = 0; i < n; i++)
        for (int w = 0; w < mask_words; w++) uni[w] |= masks[i * mask_words + w];
    std::vector<int> vars;
    for (int w = 0; w < mask_words; w++)
        for (int b = 0; b < 64; b++) if ((uni[w] >> b) & 1) vars.push_back(w * 64 + b);
    const int c = (int)vars.size();
    if (c > kMaxDenseCand) return ctx->fail(URLGPU_ERR_LIMIT, "prune: masks span more than 30 distinct variables");
    std::vector<int> pos(mask_words * 64, -1);
    for (int i = 0; i < c; i++) pos[vars[i]] = i;
    const uint64_t n_masks = (uint64_t)1 << c;
    std::vector<uint32_t> cm(n);
    int K = 0;
    for (uint64_t i = 0; i < n; i++) {
        uint32_t m = 0;
        for (int j = 0; j < c; j++) if ((masks[i * mask_words + (vars[j] >> 6)] >> (vars[j] & 63)) & 1) m |= 1u << j;
        cm[i] = m;
        K = std::max(K, __builtin_popcount(m));
    }
    cudaStream_t s = ctx->stream;
    DevBuf tab(ctx), dm(ctx), dv(ctx), dout(ctx);
    CK(tab.alloc(n_masks * sizeof(float)));
    CK(dm.alloc(n * sizeof(uint32_t))); CK(dv.alloc(n * sizeof(float))); CK(dout.alloc(n * sizeof(float)));
    fill_u32_kernel<<<blocks_for(n_masks, 256), 256, 0, s>>>(tab.as<uint32_t>(), n_masks, kSentinelBits);
    // scatter on the host side of a staging table would need 2^c floats; scatter on the device instead
    CK(cudaMemcpyAsync(dm.p, cm.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(dv.p, scores, n * sizeof(float), cudaMemcpyHostToDevice, s));
    extern __global__ void urlgpu_scatter_kernel(float *, const uint32_t *, const float *, uint64_t);
    extern __global__ void gather_scores_kernel(const float *, const uint32_t *, uint64_t, float *);
    urlgpu_scatter_kernel<<<blocks_for(n, 256), 256, 0, s>>>(tab.as<float>(), dm.as<uint32_t>(), dv.as<float>(), n);
    int rc = run_prune(ctx, tab.as<float>(), c, K);
    if (rc) return rc;
    gather_scores_kernel<<<blocks_for(n, 256), 256, 0, s>>>(tab.as<float>(), dm.as<uint32_t>(), n, dout.as<float>());
    std::vector<float> out(n);
    CK(cudaMemcpyAsync(out.data(), dout.p, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    for (uint64_t i = 0; i < n; i++) {
        uint32_t bits;
        memcpy(&bits, &out[i], 4);
        keep[i] = bits != kSentinelBits;
    }
    return URLGPU_OK;
}

__global__ void gather_scores_kernel(const float *__restrict__ table, const uint32_t *__restrict__ masks, uint64_t n, float *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = table[masks[i]];
}

__global__ void urlgpu_scatter_kernel(float *table, const uint32_t *masks, const float *vals, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) table[masks[i]] = vals[i];
}
