// rank_kernels.cuh — the RANK-SPACE layout of a variable's score cache and the kernels that work in it (sm_100a).
//
// The reference enumerates a variable's candidate family layer by layer, each layer in Gosper order = increasing compact
// mask = COLEX order of the index tuples (score_calculator.cpp:76-120, typedefs.h:692-697; SURVEY.md 7.1).  A set
// {e_1 < e_2 < ... < e_l} of compact candidate positions therefore has the dense index
//
//      index(S) = layer_base[l] + sum_i C(e_i, i)              (combinatorial number system)
//
// and the canonical output order (|S|, mask) IS the index order.  A table of  T = sum_{l<=K} C(c, l)  floats holds the
// whole family: no 2^c dense table, so the candidate count c is bounded by 255 instead of 30 and the per-set cost no
// longer depends on c - K.  Everything downstream of the scoring kernels has a rank-space form here:
//   * the store rule of the caller (score_calculator.cpp:59,111),
//   * the cBIC acceptance DP (BIC_OLS.cpp:125-276, "clean" recursion) and the subset-dominance prune
//     (score_calculator.cpp:150-197), layer by layer, a set looking its |S| immediate subsets up by rank,
//   * order-preserving compaction of the stored entries and expansion of ranks to the caller's multi-word varsets,
// plus the scoring kernels themselves: per-set Schur sweeps for cBIC (same FMA sequence per set as the dense-layout K3,
// so both layouts give bit-identical scores) and the key space of K1's direct row counting (RankSets).
#pragma once
#include "bic_kernels.cuh"
#include "cbic_kernels.cuh"

namespace urlgpu {

// ---- shared-memory copy of the binomial table (divergent look-ups; constant memory would serialise them) ----
__device__ __forceinline__ void rs_load_binom(const RankSpace &rs, uint32_t *s_binom) {
    const int n = (rs.c + 1) * rs.bstride;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_binom[i] = __ldg(rs.binom + i);
    __syncthreads();
}
__host__ __device__ __forceinline__ size_t rs_binom_bytes(const RankSpace &rs) { return (size_t)(rs.c + 1) * rs.bstride * sizeof(uint32_t); }

__device__ __forceinline__ int rs_layer_of(const RankSpace &rs, uint32_t idx) {
    int l = 0;
    while (l < rs.K && idx >= rs.layer_base[l + 1]) l++;
    return l;
}

// rank within layer l -> ascending positions e[0..l-1]
__device__ __forceinline__ void rs_unrank(const uint32_t *B, int bstride, int c, int l, uint32_t r, uint8_t *e) {
    int hi = c - 1;
    for (int i = l; i >= 1; i--) {
        int lo = i - 1, h = hi;                   // largest b in [i-1, hi] with C(b, i) <= r  (C(i-1, i) = 0)
        while (lo < h) {
            const int mid = (lo + h + 1) >> 1;
            if (B[mid * bstride + i] <= r) lo = mid; else h = mid - 1;
        }
        e[i - 1] = (uint8_t)lo;
        r -= B[lo * bstride + i];
        hi = lo - 1;
    }
}
// colex successor inside a layer
__device__ __forceinline__ void rs_next(int l, uint8_t *e) {
    int i = 0;
    while (i < l - 1 && e[i] + 1 == e[i + 1]) i++;
    e[i]++;
    for (int j = 0; j < i; j++) e[j] = (uint8_t)j;
}
// compact mask (c <= 64) -> index
__device__ __forceinline__ uint32_t rs_index_of_mask(const RankSpace &rs, const uint32_t *B, uint64_t mask) {
    uint32_t r = 0;
    int i = 0;
    for (uint64_t m = mask; m; m &= m - 1) { i++; r += B[(__ffsll((long long)m) - 1) * rs.bstride + i]; }
    return rs.layer_base[i] + r;
}

// ------------------------------------------------------------------------------------------------ store rule (BIC)
// empty set stored iff score < 1, others iff score < 0 (score_calculator.cpp:59,111); index 0 is the empty set
__global__ void rank_store_rule_kernel(float *__restrict__ scores, uint32_t total) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float s = scores[i];
    if (is_sentinel(s)) return;
    if (!(i == 0 ? s < 1.0f : s < 0.0f)) scores[i] = sentinel();
}

// ------------------------------------------------------------------------------------------------ K3 in rank space
// One thread scores kRankRun consecutive sets of layer L: unrank the first, colex successor for the rest.  The set's
// (L+1)x(L+1) sub-Gram over (v, e_1..e_L) is gathered from the candidate Gram (packed lower triangle over (v, cand_0, ..),
// indexed by tri(): members ascend, so every entry read is G[tri(pos[a], pos[b])] with pos[a] >= pos[b]) and the
// candidates are swept out highest first — the FMA sequence of cbic_roots_kernel / cbic_sweep / cbic_sets_kernel.
// Pivot guard: see CbicParams::piv_tol (cbic_kernels.cuh).
constexpr int kRankRun = 4;

template <int L>
__device__ __forceinline__ double rank_cbic_rss(const double *__restrict__ G, const uint8_t *e, double piv_tol) {
    double A[(L + 1) * (L + 2) / 2];
    int pos[L + 1];
    pos[0] = 0;
#pragma unroll
    for (int i = 0; i < L; i++) pos[i + 1] = (int)e[i] + 1;
#pragma unroll
    for (int a = 0; a <= L; a++)
#pragma unroll
        for (int b = 0; b <= a; b++) A[tri(a, b)] = __ldg(G + tri(pos[a], pos[b]));
#pragma unroll
    for (int piv = L; piv >= 1; piv--) {
        const double inv = guarded_inv(A[tri(piv, piv)], piv_tol);
#pragma unroll
        for (int a = 0; a < piv; a++) {
            const double f = -A[tri(piv, a)] * inv;
#pragma unroll
            for (int b = 0; b <= a; b++) A[tri(a, b)] = fma(f, A[tri(piv, b)], A[tri(a, b)]);
        }
    }
    return A[0];
}
// any L (matrix in local memory): layers above 8
__device__ __noinline__ double rank_cbic_rss_generic(const double *__restrict__ G, const uint8_t *e, int L, double piv_tol, double *A) {
    for (int a = 0; a <= L; a++) {
        const int pa = a ? (int)e[a - 1] + 1 : 0;
        for (int b = 0; b <= a; b++) A[tri(a, b)] = __ldg(G + tri(pa, b ? (int)e[b - 1] + 1 : 0));
    }
    for (int piv = L; piv >= 1; piv--) {
        const double inv = guarded_inv(A[tri(piv, piv)], piv_tol);
        for (int a = 0; a < piv; a++) {
            const double f = -A[tri(piv, a)] * inv;
            for (int b = 0; b <= a; b++) A[tri(a, b)] = fma(f, A[tri(piv, b)], A[tri(a, b)]);
        }
    }
    return A[0];
}

constexpr int kRankGenericMaxL = 16;

template <int L> // L = 0: generic (run-time layer `layer`)
__global__ void __launch_bounds__(128) rank_cbic_kernel(RankSpace rs, const double *__restrict__ G, CbicParams prm, int layer,
                                                        uint32_t first /*global index*/, uint32_t count, float *__restrict__ out) {
    extern __shared__ uint32_t s_binom[];
    rs_load_binom(rs, s_binom);
    const int l = L > 0 ? L : layer;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t i0 = (uint64_t)t * kRankRun;
    if (i0 >= count) return;
    const uint32_t idx0 = first + (uint32_t)i0;
    const uint32_t nrun = (uint32_t)min((uint64_t)kRankRun, (uint64_t)count - i0);
    uint8_t e[L > 0 ? L : kRankGenericMaxL];
    rs_unrank(s_binom, rs.bstride, rs.c, l, idx0 - rs.layer_base[l], e);
    for (uint32_t u = 0; u < nrun; u++) {
        double rss;
        if constexpr (L > 0) rss = rank_cbic_rss<L>(G, e, prm.piv_tol);
        else {
            double A[(kRankGenericMaxL + 1) * (kRankGenericMaxL + 2) / 2];
            rss = rank_cbic_rss_generic(G, e, l, prm.piv_tol, A);
        }
        out[idx0 + u] = (float)cbic_the_score64(rss, l, prm);
        if (u + 1 < nrun) rs_next(l, e);
    }
}

// ------------------------------------------------------------------------------------------------ K4 / K5 in rank space
// Layer l, one thread per set: the l immediate subsets S \ {e_i} are looked up by rank,
//     rank(S \ e_i) = sum_{j<i} C(e_j, j) + sum_{j>i} C(e_j, j-1)          (1-based j)
// MODE 0 — acceptance (rules as in cbic_kernels.cuh, K4): in val[] = the_score, out val[] = stored value or sentinel,
//          aux[] = g(S) = stored ? val : F(S).
// MODE 1 — prune (K5): aux[] = M(S) = max(val'(S), max_i M(S \ e_i)); S is dropped unless val(S) > max_i M(S \ e_i).
template <int MODE>
__global__ void __launch_bounds__(256) rank_dp_kernel(RankSpace rs, int layer, float *__restrict__ val, float *__restrict__ aux) {
    extern __shared__ uint32_t s_binom[];
    rs_load_binom(rs, s_binom);
    const uint32_t n_layer = rs.layer_base[layer + 1] - rs.layer_base[layer];
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_layer) return;
    const uint32_t idx = rs.layer_base[layer] + r;
    const float v = val[idx];
    if (layer == 0) {
        if (MODE == 0) { if (!is_sentinel(v)) { val[idx] = -v; aux[idx] = 0.0f; } else aux[idx] = 0.0f; }
        else aux[idx] = is_sentinel(v) ? -INFINITY : v;
        return;
    }
    if (MODE == 0 && is_sentinel(v)) { aux[idx] = 0.0f; return; }
    if (MODE == 0 && v > 0.0f) { val[idx] = -v; aux[idx] = -v; return; }
    uint8_t e[kMaxRankLayers];
    rs_unrank(s_binom, rs.bstride, rs.c, layer, r, e);
    // suffix sums with the subset's exponents: up[i] = sum_{j>i} C(e_j, j-1)
    float best = MODE == 0 ? 0.0f : -INFINITY;
    if (MODE == 1 || layer > 1) {
        uint32_t up = 0;
        for (int j = layer; j >= 2; j--) up += s_binom[e[j - 1] * rs.bstride + (j - 1)];   // subset without e_1
        uint32_t down = 0;
        const float *sub = aux + rs.layer_base[layer - 1];
        for (int i = 1; i <= layer; i++) {
            const float g = sub[down + up];
            if (MODE == 0) { if (g > best) best = g; } else best = fmaxf(best, g);
            if (i < layer) {
                down += s_binom[e[i - 1] * rs.bstride + i];
                up -= s_binom[e[i] * rs.bstride + i];
            }
        }
    }
    if (MODE == 0) {
        if (v == 0.0f) { val[idx] = sentinel(); aux[idx] = best; return; }
        const float nv = -v;
        if (best >= nv) { val[idx] = sentinel(); aux[idx] = best; }
        else { val[idx] = nv; aux[idx] = nv; }
    } else {
        const bool stored = !is_sentinel(v);
        if (stored && !(v > best)) val[idx] = sentinel();
        aux[idx] = stored ? fmaxf(best, v) : best;
    }
}

// ------------------------------------------------------------------------------------------------ compaction
// Stored entries in index order = canonical order.  Three kernels, no host round trip: per-block counts, a single-CTA
// exclusive scan, an order-preserving write of (index, value).
constexpr int kRankCompactThreads = 256;
constexpr int kRankCompactPer = 8;                                     // consecutive entries per thread
constexpr int kRankCompactSeg = kRankCompactThreads * kRankCompactPer;

__global__ void __launch_bounds__(kRankCompactThreads) rank_compact_count_kernel(const float *__restrict__ val, uint32_t total, uint32_t *__restrict__ blockcnt) {
    __shared__ unsigned int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    const uint64_t i0 = (uint64_t)blockIdx.x * kRankCompactSeg + (uint64_t)threadIdx.x * kRankCompactPer;
    unsigned mine = 0;
#pragma unroll
    for (int k = 0; k < kRankCompactPer; k++)
        if (i0 + k < total && !is_sentinel(val[i0 + k])) mine++;
    mine = __reduce_add_sync(0xffffffffu, mine);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&cnt, mine);
    __syncthreads();
    if (threadIdx.x == 0) blockcnt[blockIdx.x] = cnt;
}
__global__ void __launch_bounds__(1024) rank_compact_scan_kernel(uint32_t *__restrict__ blockcnt, uint32_t nblocks, unsigned long long *__restrict__ counts /*[33]: [32] = total*/) {
    __shared__ unsigned long long part[1024];
    const uint32_t per = (nblocks + blockDim.x - 1) / blockDim.x;
    const uint32_t b = min(nblocks, threadIdx.x * per), e = min(nblocks, b + per);
    unsigned long long sum = 0;
    for (uint32_t i = b; i < e; i++) sum += blockcnt[i];
    part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (uint32_t i = 0; i < blockDim.x; i++) { const unsigned long long t = part[i]; part[i] = run; run += t; }
        counts[32] = run;
    }
    __syncthreads();
    unsigned long long run = part[threadIdx.x];
    for (uint32_t i = b; i < e; i++) { const uint32_t t = blockcnt[i]; blockcnt[i] = (uint32_t)run; run += t; }
}
__global__ void __launch_bounds__(kRankCompactThreads) rank_compact_write_kernel(const float *__restrict__ val, uint32_t total, const uint32_t *__restrict__ blockoff,
                                                                                 uint32_t *__restrict__ out_idx, float *__restrict__ out_val) {
    __shared__ uint32_t warp_tot[kRankCompactThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t i0 = (uint64_t)blockIdx.x * kRankCompactSeg + (uint64_t)threadIdx.x * kRankCompactPer;
    float v[kRankCompactPer];
    unsigned mine = 0;
#pragma unroll
    for (int k = 0; k < kRankCompactPer; k++) {
        v[k] = i0 + k < total ? val[i0 + k] : sentinel();
        if (!is_sentinel(v[k])) mine++;
    }
    unsigned x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    uint32_t pos = blockoff[blockIdx.x] + x - mine;
    for (int w = 0; w < warp; w++) pos += warp_tot[w];
#pragma unroll
    for (int k = 0; k < kRankCompactPer; k++)
        if (!is_sentinel(v[k])) { out_idx[pos] = (uint32_t)(i0 + k); out_val[pos] = v[k]; pos++; }
}

// index -> the caller's multi-word varsets
__global__ void __launch_bounds__(256) rank_expand_kernel(RankSpace rs, const uint32_t *__restrict__ idx, uint64_t n, const int *__restrict__ cand, int words,
                                                          uint64_t *__restrict__ out) {
    extern __shared__ uint32_t s_binom[];
    rs_load_binom(rs, s_binom);
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t ix = idx[i];
    const int l = rs_layer_of(rs, ix);
    uint8_t e[kMaxRankLayers];
    rs_unrank(s_binom, rs.bstride, rs.c, l, ix - rs.layer_base[l], e);
    for (int w = 0; w < words; w++) {
        uint64_t x = 0;
        for (int j = 0; j < l; j++) {
            const int var = cand[e[j]];
            if ((var >> 6) == w) x |= (uint64_t)1 << (var & 63);
        }
        out[i * (uint64_t)words + w] = x;
    }
}

// ------------------------------------------------------------------------------------------------ K1, direct counting
// Sets named by their index (bic_kernels.cuh, "How the direct-counting kernels name a set"): every direct count goes
// through this key space, whatever the layout of the result and up to 255 candidates.  Candidate variables and arities
// live in device arrays.  The score goes to the set's index, or, for a dense result (c <= 30), to its compact mask.
struct RankCand {
    int v, rv;
    const int *var;     // [c] candidate position -> variable index (ascending)
    const int *card;    // [c]
};

struct RankSets {
    RankSpace rs;
    RankCand rc;
    int by_mask;
    __host__ __device__ __forceinline__ int rv() const { return rc.rv; }
    __device__ __forceinline__ void build_cols(const BicData &d, uint32_t idx, SetCols &sc) const {
        const int l = rs_layer_of(rs, idx);
        uint8_t e[kMaxRankLayers];
        rs_unrank(rs.binom, rs.bstride, rs.c, l, idx - rs.layer_base[l], e);   // one thread: straight from global
        sc.col[0] = d.codes + (int64_t)rc.v * d.n_stride;
        sc.stride[0] = 1;
        uint32_t base = (uint32_t)rc.rv;
        float pen = (float)(rc.rv - 1);
        uint64_t mask = 0;
        for (int i = 0; i < l; i++) {
            const int cd = __ldg(rc.card + e[i]);
            sc.col[i + 1] = d.codes + (int64_t)__ldg(rc.var + e[i]) * d.n_stride;
            sc.stride[i + 1] = base;
            base *= (uint32_t)cd;
            pen = __fmul_rn(pen, (float)cd);
            mask |= (uint64_t)1 << e[i];
        }
        sc.ncols = l + 1;
        sc.cells = base;
        sc.tval = pen;
        sc.out = by_mask ? mask : idx;
    }
};

// cells of every set of [first, first + count) -> tier lists (0: <= t0 cells, 1: <= t1, 2: global, with its cell count;
// 3: too large, only counted)
__global__ void __launch_bounds__(256) bic_classify_kernel(RankSets fam, uint32_t first, uint32_t count, uint32_t t0, uint32_t t1, uint64_t cell_limit,
                                                           uint32_t *list0, uint32_t *list1, GlobalSet *list2, unsigned long long *counters) {
    extern __shared__ uint32_t s_binom[];
    const RankSpace &rs = fam.rs;
    rs_load_binom(rs, s_binom);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    int tier = -1;
    uint32_t idx = 0;
    uint64_t cells = 0;
    if (i < count) {
        idx = first + i;
        const int l = rs_layer_of(rs, idx);
        uint8_t e[kMaxRankLayers];
        rs_unrank(s_binom, rs.bstride, rs.c, l, idx - rs.layer_base[l], e);
        cells = (uint64_t)fam.rc.rv;
        for (int j = 0; j < l; j++) { cells *= (uint64_t)__ldg(fam.rc.card + e[j]); if (cells > cell_limit) cells = cell_limit + 1; }
        tier = cells <= t0 ? 0 : cells <= t1 ? 1 : cells <= cell_limit ? 2 : 3;
    }
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int t = 0; t < 4; t++) {
        const unsigned b = __ballot_sync(0xffffffffu, tier == t);
        if (b == 0) continue;
        unsigned long long basepos = 0;
        const int leader = __ffs(b) - 1;
        if (lane == leader) basepos = atomicAdd(&counters[t], (unsigned long long)__popc(b));
        basepos = __shfl_sync(0xffffffffu, basepos, leader);
        const unsigned long long pos = basepos + __popc(b & ((1u << lane) - 1));
        if (tier == t && t < 2) (t == 0 ? list0 : list1)[pos] = idx;
        if (tier == t && t == 2) list2[pos] = GlobalSet{idx, (uint32_t)cells, 0};
    }
}


// ------------------------------------------------------------------------------------------------ K4, literal form
// find_best_subset_score AS WRITTEN (BIC_OLS.cpp:125-172; SURVEY.md Q5) under Armadillo >= 10.5, where arma::uvec(n) is
// zero-filled: the vector of remaining parents handed to each recursive call is only partly filled, its tail names
// variable 0, and VARSET_CLEAR is an XOR (typedefs.h:657), so a zero entry TOGGLES variable 0: subsets that are not
// subsets get looked up and half-explored sets are marked `checked`.  This kernel emulates that recursion, one thread per
// parent set, with an explicit stack and a private `checked` bitset, so that `score --accept=literal-zero` reproduces the
// cache of the reference as compiled today (the default "clean" DP restates the evident intent of the same lines).
// Sets live in a LOCAL universe: bit i < k = the i-th member of S (ascending), bit k = variable 0 when it is not a member.
// Dependencies: a look-up can reach a set of S's own layer only by replacing a member with variable 0; such a set contains
// variable 0 (the lowest candidate), so a layer is processed in two launches: sets containing candidate 0, then the rest.
constexpr int kLiteralMaxK = 12;

struct LiteralFrame {
    uint16_t parents, thin;
    uint8_t np, idx, i, j, inner, var;
    float best;
    uint8_t pv[kLiteralMaxK], nv[kLiteralMaxK];
};

__global__ void __launch_bounds__(128) accept_literal_kernel(RankSpace enumr /*rank space used to enumerate the layer*/, RankSpace lay /*layout of `table`*/, int layer,
                                                             int zero_cand /*compact position of variable 0 among the candidates, -1: not a candidate*/,
                                                             int phase /*0: only sets with candidate 0, 1: only sets without, 2: all*/, float *__restrict__ table,
                                                             LiteralFrame *__restrict__ frames /*[threads][kLiteralMaxK + 1]*/, uint32_t *__restrict__ checked /*[threads][256]*/) {
    const uint32_t n_layer = enumr.layer_base[layer + 1] - enumr.layer_base[layer];
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_layer) return;
    uint8_t e[kMaxRankLayers];
    rs_unrank(enumr.binom, enumr.bstride, enumr.c, layer, r, e);
    uint64_t S = 0;
    for (int i = 0; i < layer; i++) S |= (uint64_t)1 << e[i];
    const bool has0 = zero_cand >= 0 && ((S >> zero_cand) & 1);
    if (phase == 0 && !has0) return;
    if (phase == 1 && has0) return;
    const uint64_t idx = out_index(lay, S);
    const float ts = table[idx];
    if (is_sentinel(ts)) return;
    const int k = layer;
    if (k == 0) { table[idx] = -ts; return; }
    if (ts > 0.0f) { table[idx] = -ts; return; }                    // BIC_OLS.cpp:213-224: "bad" set, stored by the caller
    if (ts == 0.0f) { table[idx] = sentinel(); return; }            // returned as -0.0: neither side stores it
    // ---- best = find_best_subset_score(parents, cache, parent_vec, num_parents, checked) ----
    LiteralFrame *st = frames + (size_t)r * (kLiteralMaxK + 1);
    uint32_t *chk = checked + (size_t)r * 256;                       // 2^(k+1) <= 8192 bits
    for (int w = 0; w < ((1 << (k + 1)) + 31) / 32; w++) chk[w] = 0;
    chk[0] = 1u;                                                     // checked.insert(empty set) (:231)
    const int zpos = has0 ? 0 : k;                                   // local position of variable 0 (a member is local bit 0: it is the lowest index)
    auto lookup = [&](uint32_t local, float &val) -> bool {          // cache.find(local set)
        uint64_t m = 0;
        for (int i = 0; i < k; i++) if ((local >> i) & 1) m |= (uint64_t)1 << e[i];
        if ((local >> k) & 1) { if (zero_cand < 0) return false; m |= (uint64_t)1 << zero_cand; }
        if (__popcll(m) > lay.K && lay.binom) return false;
        const float x = table[out_index(lay, m)];
        if (is_sentinel(x)) return false;
        val = x;
        return true;
    };
    int sp = 0;
    st[0].parents = (uint16_t)((1u << k) - 1); st[0].np = (uint8_t)k; st[0].idx = 0; st[0].inner = 0; st[0].best = 0.0f;
    for (int i = 0; i < k; i++) st[0].pv[i] = (uint8_t)i;
    float result = 0.0f;
    while (true) {
        LiteralFrame &F = st[sp];
        if (!F.inner) {
            if (F.idx == F.np) {                                     // return best_score
                const float ret = F.best;
                if (sp == 0) { result = ret; break; }
                sp--;
                LiteralFrame &G = st[sp];
                chk[G.thin >> 5] |= 1u << (G.thin & 31);             // checked.insert(thin_parents) (:166)
                if (ret > G.best) G.best = ret;
                G.i++;
                continue;
            }
            F.var = F.pv[F.idx];
            const uint16_t thin = F.parents ^ (uint16_t)(1u << F.var);   // VARSET_CLEAR is XOR
            if ((chk[thin >> 5] >> (thin & 31)) & 1u) { F.idx++; continue; }
            float val;
            if (lookup(thin, val)) { if (val > F.best) F.best = val; F.idx++; continue; }
            F.thin = thin; F.inner = 1; F.i = 0; F.j = 0;
            for (int q = 0; q < kLiteralMaxK; q++) F.nv[q] = (uint8_t)zpos;   // arma::uvec(num_parents - 1), zero-filled: variable 0
        }
        bool called = false;
        while (F.i < F.np) {
            if (F.var == F.pv[F.i]) { F.i++; continue; }
            F.nv[F.j++] = F.pv[F.i];
            LiteralFrame &N = st[sp + 1];                            // find_best_subset_score(thin_parents, cache, new_parent_vec, num_parents - 1, ...)
            N.parents = F.thin; N.np = (uint8_t)(F.np - 1); N.idx = 0; N.inner = 0; N.best = 0.0f;
            for (int q = 0; q < kLiteralMaxK; q++) N.pv[q] = F.nv[q];
            sp++;
            called = true;
            break;
        }
        if (called) continue;
        F.inner = 0;
        F.idx++;
    }
    // :233-249 with bic_threshold = 0
    const float nv = -ts;
    table[idx] = result >= nv ? sentinel() : nv;
}

} // namespace urlgpu
