// order_kernels.cuh — exact structure search over the order graph of one skeleton component, layer by layer (sm_100a).
//
// The search space of run_astar_on_one_scc (astar/astar_main.cpp:216-546, host/search_host.hpp:367-432): the nodes are the
// subsets S of a component C (k = |C| <= 36 variables), S is reached from S\{v} by adding the leaf v with its best cached
// parent set inside S\{v}, and the goal is C.  A* keeps a hash map and a heap over the nodes it generates (~70-80 bytes
// each); here the graph is swept once, one launch per layer, so every node is final when the next layer reads it.  A sweep
// of layer l reads only layer l-1 and the backtrack reads only leaves, so costs are kept for two adjacent layers, indexed by
// colex rank inside the layer, and a leaf byte for every node at base_l + rank (base_l = sum_{m<l} C(k, m)):
// 2^k + 8 C(k, k/2) bytes in all.  With S = {e_0 < ... < e_{l-1}}, rank(S) = sum_i C(e_i, i+1) and
// rank(S \ e_j) = sum_{i<j} C(e_i, i+1) + sum_{i>j} C(e_i, i).
//
//   best(v, U)  the first entry of v's cache, in (score, |S|, mask) order, whose parent set is inside U.  Each variable gets a
//               dense uint32 table T_v over the lattice of its candidates cand_v (the union of its entries inside C, c_v < k
//               bits): T_v[U] = the SORTED POSITION of best(v, U), kOrderNone if there is none.  Built by scattering every
//               entry's position to its compact mask (atomicMin: duplicates keep the first) and a subset-min transform,
//               T[U] = min(T[U], T[U\b]) for every bit b: the low kOrderSegBits bits per 2048-entry segment in shared memory
//               (order_table_low_kernel), each higher bit in one coalesced global pass (order_table_high_kernel).  Positions
//               order like the sparse parent list, so the list's tie rule comes for free and a look-up is one gather.
//   layer l     order_layer_kernel: one thread takes kOrderRun consecutive colex nodes of the layer (unrank the first with the
//               shared-memory binomial table, Gosper successor for the rest).  A first pass over S's bits sums C(e_i, i); then
//               for every v in S, ascending, keeping both prefixes of rank(S \ v): the skeleton test (astar_main.cpp:300-307:
//               the leaf must touch S\{v} unless S\{v} is empty), cost[S\v] from the previous layer, the compaction of S\v
//               into cand_v's bits through five byte look-up tables in shared memory, T_v, the score, and g = cost + score
//               rounded once (__fadd_rn).  cost[S] = min g, leaf[S] = the smallest v attaining it; a node with no admissible
//               predecessor gets cost +inf and leaf kOrderUnreached.
//   backtrack   order_backtrack_kernel, one thread: walks leaf[] back from C and writes the cost, the k leaves and the k
//               sorted positions of their parent sets into one small buffer.
//
// Bound: a layer reads 4 + 4 bytes (cost, table) per (S, v) pair, k 2^(k-1) pairs in all, at addresses that differ from
// node to node: HBM and L2 sector traffic, not arithmetic, sets the time.
#pragma once
#include "common.cuh"

namespace urlgpu {

constexpr int kOrderMaxVars = 36;            // 2^36 + 8 C(36, 18) = 141 GB of nodes; 37 would need 279 GB
constexpr int kOrderSegBits = 11;            // 2048-entry segments of the subset-min transform (8 KB of shared memory)
constexpr int kOrderRun = 4;                 // consecutive colex nodes per thread and grid-stride step
constexpr int kOrderBinom = kOrderMaxVars + 1;
constexpr int kOrderLut = 5;                 // byte look-up tables per variable: bits 0..39 of a compact mask
constexpr uint32_t kOrderNone = 0xFFFFFFFFu; // T_v: no cached subset (best = FLT_MAX)
constexpr uint8_t kOrderUnreached = 0xFF;    // leaf[]: no admissible predecessor

struct OrderVar {            // variable at position j of C
    unsigned long long table; // offset of T_j in the table buffer (uint32 elements)
    unsigned long long adj;   // skeleton neighbours as a compact mask over C; all of C without a skeleton
    unsigned long long cand;  // cand_j as a compact mask over C
    uint32_t score;           // offset of j's sorted scores
    uint8_t shift[kOrderLut]; // popcount of cand_j below byte b: where byte b's compacted bits go
};

__host__ __device__ __forceinline__ size_t order_smem_bytes(int k) {
    return (size_t)kOrderBinom * kOrderBinom * sizeof(unsigned long long) + (size_t)k * sizeof(OrderVar) + (size_t)k * kOrderLut * 256;
}

// ------------------------------------------------------------------------------------------------ best-parent tables
// T[where[i]] = min(T[where[i]], pos[i])
__global__ void __launch_bounds__(256) order_scatter_kernel(const unsigned long long *__restrict__ where, const uint32_t *__restrict__ pos, uint64_t n,
                                                            uint32_t *__restrict__ T) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicMin(T + __ldg(where + i), __ldg(pos + i));
}

// the low `bits` bits of the subset-min transform of one table, one 2^bits segment per CTA
__global__ void __launch_bounds__(1024) order_table_low_kernel(uint32_t *__restrict__ T, int bits) {
    __shared__ uint32_t s[1 << kOrderSegBits];
    const uint32_t n = 1u << bits;
    uint32_t *seg = T + ((size_t)blockIdx.x << bits);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s[i] = seg[i];
    __syncthreads();
    for (int b = 0; b < bits; b++) {
        for (uint32_t i = threadIdx.x; i < n / 2; i += blockDim.x) {
            const uint32_t u = ((i >> b) << (b + 1)) | (i & ((1u << b) - 1));   // bit b clear
            s[u | (1u << b)] = min(s[u | (1u << b)], s[u]);
        }
        __syncthreads();
    }
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) seg[i] = s[i];
}

// one bit b >= kOrderSegBits of the transform: T[U | b] = min(T[U | b], T[U]) for the 2^(c-1) masks U without b
__global__ void __launch_bounds__(256) order_table_high_kernel(uint32_t *__restrict__ T, int b, uint64_t half) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half) return;
    const uint64_t u = ((i >> b) << (b + 1)) | (i & ((1ull << b) - 1));
    const uint64_t w = u | (1ull << b);
    T[w] = min(T[w], T[u]);
}

// ------------------------------------------------------------------------------------------------ layer sweep
// rank r of layer l -> the k-bit mask with that colex rank (B[b * kOrderBinom + i] = C(b, i))
__device__ __forceinline__ unsigned long long order_unrank(const unsigned long long *B, int k, int l, unsigned long long r) {
    unsigned long long S = 0;
    int hi = k - 1;
    for (int i = l; i >= 1; i--) {
        int lo = i - 1, h = hi;                   // largest b in [i-1, hi] with C(b, i) <= r
        while (lo < h) {
            const int mid = (lo + h + 1) >> 1;
            if (B[mid * kOrderBinom + i] <= r) lo = mid; else h = mid - 1;
        }
        S |= 1ull << lo;
        r -= B[lo * kOrderBinom + i];
        hi = lo - 1;
    }
    return S;
}
// Gosper successor; k <= 36, so x + low never overflows
__device__ __forceinline__ unsigned long long order_next(unsigned long long x) {
    const unsigned long long low = x & (~x + 1), r = x + low;
    return r | (((x ^ r) >> 2) >> (__ffsll((long long)x) - 1));
}
// colex rank of S inside its layer
__device__ __forceinline__ unsigned long long order_rank(const unsigned long long *B, unsigned long long S) {
    unsigned long long r = 0;
    int i = 1;
    for (; S; S &= S - 1, i++) r += B[(__ffsll((long long)S) - 1) * kOrderBinom + i];
    return r;
}

// layer `layer` from layer - 1: cost_prev / cost_cur are indexed by colex rank, leaf by `base` + rank
__global__ void __launch_bounds__(256) order_layer_kernel(const OrderVar *__restrict__ vars, const uint8_t *__restrict__ lut,
                                                          const unsigned long long *__restrict__ binom, const uint32_t *__restrict__ T,
                                                          const float *__restrict__ scores, int k, int layer, unsigned long long count,
                                                          unsigned long long base, const float *__restrict__ cost_prev,
                                                          float *__restrict__ cost_cur, uint8_t *__restrict__ leaf) {
    extern __shared__ __align__(16) unsigned char order_smem[];
    unsigned long long *s_binom = reinterpret_cast<unsigned long long *>(order_smem);
    OrderVar *s_var = reinterpret_cast<OrderVar *>(s_binom + kOrderBinom * kOrderBinom);
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(s_var + k);
    for (int i = threadIdx.x; i < kOrderBinom * kOrderBinom; i += blockDim.x) s_binom[i] = __ldg(binom + i);
    for (int i = threadIdx.x; i < k; i += blockDim.x) s_var[i] = vars[i];
    for (int i = threadIdx.x; i < k * kOrderLut * 64; i += blockDim.x)
        reinterpret_cast<uint32_t *>(s_lut)[i] = __ldg(reinterpret_cast<const uint32_t *>(lut) + i);
    __syncthreads();
    const unsigned long long runs = (count + kOrderRun - 1) / kOrderRun;
    for (unsigned long long run = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; run < runs; run += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long first = run * kOrderRun;
        const uint32_t nrun = (uint32_t)min((unsigned long long)kOrderRun, count - first);
        unsigned long long S = order_unrank(s_binom, k, layer, first);
        for (uint32_t u = 0; u < nrun; u++) {
            unsigned long long above = 0;                              // sum_i C(e_i, i)
            {
                int i = 0;
                for (unsigned long long m = S; m; m &= m - 1, i++) above += s_binom[(__ffsll((long long)m) - 1) * kOrderBinom + i];
            }
            unsigned long long below = 0;                              // sum_{i<j} C(e_i, i+1)
            float best = __int_as_float(0x7f800000);
            uint32_t best_leaf = kOrderUnreached;
            int j = 0;
            for (unsigned long long m = S; m; m &= m - 1, j++) {
                const int v = __ffsll((long long)m) - 1;
                above -= s_binom[v * kOrderBinom + j];
                const unsigned long long rprev = below + above;
                below += s_binom[v * kOrderBinom + j + 1];
                const unsigned long long prev = S ^ (1ull << v);
                const OrderVar &V = s_var[v];
                if (prev && !(prev & V.adj)) continue;                 // the leaf must touch the sub-network
                const float c = __ldg(cost_prev + rprev);
                if (c == __int_as_float(0x7f800000)) continue;        // S\v unreached
                const uint8_t *L = s_lut + v * (kOrderLut * 256);
                const unsigned long long idx = (unsigned long long)L[prev & 255] | ((unsigned long long)L[256 + ((prev >> 8) & 255)] << V.shift[1]) |
                                               ((unsigned long long)L[512 + ((prev >> 16) & 255)] << V.shift[2]) |
                                               ((unsigned long long)L[768 + ((prev >> 24) & 255)] << V.shift[3]) |
                                               ((unsigned long long)L[1024 + ((prev >> 32) & 255)] << V.shift[4]);
                const uint32_t pos = __ldg(T + V.table + idx);
                const float s = pos == kOrderNone ? 3.402823466e+38f : __ldg(scores + V.score + pos);
                const float g = __fadd_rn(c, s);
                if (g == __int_as_float(0x7f800000)) continue;
                if (g < best) { best = g; best_leaf = (uint32_t)v; }   // strict: the smallest v among equal costs
            }
            const unsigned long long r = first + u;
            cost_cur[r] = best;
            leaf[base + r] = (uint8_t)best_leaf;
            if (u + 1 < nrun) S = order_next(S);
        }
    }
}

// out[0] = cost(C) bits, out[1] = 1 iff C was reached, out[2 + i] = leaf at step i of the order, out[2 + k + i] = its position;
// cost_full is the one cost of layer k, leaf[base_l + rank] as in the layer kernel
__global__ void order_backtrack_kernel(const OrderVar *__restrict__ vars, const unsigned long long *__restrict__ binom,
                                       const uint32_t *__restrict__ T, const float *__restrict__ cost_full,
                                       const uint8_t *__restrict__ leaf, int k, uint32_t *__restrict__ out) {
    if (blockIdx.x | threadIdx.x) return;
    unsigned long long S = (1ull << k) - 1, base = ((1ull << k) - 1);   // base_k = 2^k - C(k, k)
    out[0] = __float_as_uint(cost_full[0]);
    out[1] = 0;
    for (int i = k - 1; i >= 0; i--) {
        const uint32_t v = leaf[base + order_rank(binom, S)];
        if (v == kOrderUnreached) return;
        const unsigned long long prev = S ^ (1ull << v);
        unsigned long long idx = 0;
        int j = 0;
        for (unsigned long long m = vars[v].cand; m; m &= m - 1, j++)
            if ((prev >> (__ffsll((long long)m) - 1)) & 1) idx |= 1ull << j;
        out[2 + i] = v;
        out[2 + k + i] = T[vars[v].table + idx];
        base -= binom[k * kOrderBinom + i];                    // base_i = base_{i+1} - C(k, i)
        S = prev;
    }
    out[1] = 1;
}

// ------------------------------------------------------------------------------------------------ local search
// urlgpu_order_local_search: insertion hill climbing over the admissible orders of a component of up to 256 variables, with the
// exact search's objective (the float32 left-to-right path sum of best(pi_m, {pi_0..pi_{m-1}})) and its best-parent tables.
// One CTA per restart (resident CTAs stride over the restarts); the whole state of a restart lives in shared memory.
//
//   state       ord[m] (the variable at position m, as a position in C), at[v] (its inverse), b[m] = best(ord[m], pred_m),
//               g[m] = the float32 sum of b[0..m) (g[0] = +0, one rounding per step), pre[m] = the set {ord[0..m)} (4 words).
//   look-up     a policy.  ClimbTable (urlgpu_order_local_search): compact U onto cand_v's <= 32 bits by testing at[] of
//               cand_v's variables, then one gather from T_v, as in the exact search.  ClimbList (urlgpu_order_local_search_sparse):
//               the first entry of v's sorted list whose parent set, W = ceil(k/64) words over C's positions, lies inside U's
//               words (pre[lim] with `out` cleared and `in` set); no limit on c_v.  Both lists and tie orders are the ones the
//               tables are built from, so both policies return the same sorted position.  One gather from v's sorted scores.
//               The move look-ups of ClimbList are warp-cooperative (32 consecutive entries a step, a ballot, the lowest lane),
//               targets in descending order, so the U of pi_i's own look-ups only shrinks and each of them starts at the last hit.
//   iteration   one warp per source i.  For j > i the variables at i+1..j lose pi_i (X[m] = best(pi_m, pred_m \ pi_i)) and pi_i
//               lands at j (Y[j] = best(pi_i, {pi_0..pi_j} \ pi_i)); for j < i the variables at j..i-1 gain pi_i (X[m]) and pi_i
//               lands at j (Y[j] = best(pi_i, {pi_0..pi_{j-1}})): 2(k-1) look-ups per source, O(k^2) per iteration.  Each lane
//               then sums its targets' paths left to right and re-adds the unchanged suffix until its running sum has the bits
//               of the old g at the same position (from there on both sums are the same).  The argmin is a block reduction of
//               a 64-bit key: order-preserving float bits (-0 folded to +0), then i, then j.
//   output      per restart: the final cost, the number of moves, the order and the sorted position of each family.
constexpr int kClimbMaxVars = 256;
constexpr int kClimbMaxCand = 32;
constexpr int kClimbWords = kClimbMaxVars / 64;
constexpr int kClimbThreads = 256;
constexpr int kClimbWarps = kClimbThreads / 32;

struct OrderClimbVar {       // variable at position j of C
    union {
        unsigned long long table;           // ClimbTable: offset of T_j in the table buffer (uint32 elements)
        unsigned long long nent;            // ClimbList: the number of j's entries
    };
    unsigned long long adj[kClimbWords];    // skeleton neighbours over C's positions; all of C without a skeleton
    uint32_t score;                         // offset of j's sorted scores (and, for ClimbList, of its entries' words)
    uint32_t ncand;                         // c_j
    uint8_t cand[kClimbMaxCand];            // ClimbTable: cand_j as positions in C, ascending
};

__host__ __device__ __forceinline__ size_t order_climb_smem_bytes(int k) {
    return (size_t)k * sizeof(OrderClimbVar) + (size_t)(k + 1) * kClimbWords * 8 + kClimbWarps * 8 + (size_t)(2 * k + 1) * 4 +
           (size_t)kClimbWarps * k * 2 * 4 + (size_t)k * 2 + (size_t)kClimbWarps * k * 2;
}

__device__ __forceinline__ uint64_t climb_draw(uint64_t &x) {   // splitmix64
    uint64_t z = (x += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// the sorted position of best(v, U), U = {u : at[u] < lim, u != out} + {in}, pre[lim] = {u : at[u] < lim} (kClimbWords words);
// kOrderNone if v has no entry inside U
struct ClimbTable {
    static constexpr bool kWarp = false;
    const uint32_t *__restrict__ T;         // every T_v
    __device__ __forceinline__ uint32_t pos(const OrderClimbVar &V, const uint8_t *at, const unsigned long long *, int lim, int out, int in) const {
        uint32_t idx = 0;
        for (uint32_t t = 0; t < V.ncand; t++) {
            const int u = V.cand[t];
            if (((int)at[u] < lim && u != out) || u == in) idx |= 1u << t;
        }
        return __ldg(T + V.table + idx);
    }
};
struct ClimbList {
    static constexpr bool kWarp = true;         // the move look-ups by warp_pos
    const unsigned long long *__restrict__ E;   // word w of sorted entry e at E[w * stride + e]
    uint32_t stride;                            // the number of entries
    int words;                                  // W = ceil(k / 64)
    // the complement of U's words
    __device__ __forceinline__ void outside(unsigned long long (&notU)[kClimbWords], const unsigned long long *pre, int lim, int out, int in) const {
#pragma unroll
        for (int w = 0; w < kClimbWords; w++)
            notU[w] = ~((pre[lim * kClimbWords + w] & ~(w == (out >> 6) ? 1ull << (out & 63) : 0ull)) | (w == (in >> 6) ? 1ull << (in & 63) : 0ull));
    }
    // does sorted entry e (from the start of the entries) lie inside U?
    __device__ __forceinline__ bool inside(const unsigned long long (&notU)[kClimbWords], uint32_t e) const {
        unsigned long long miss = __ldg(E + e) & notU[0];
#pragma unroll
        for (int w = 1; w < kClimbWords; w++) if (w < words) miss |= __ldg(E + (size_t)w * stride + e) & notU[w];
        return miss == 0;
    }
    __device__ __forceinline__ uint32_t pos(const OrderClimbVar &V, const uint8_t *, const unsigned long long *pre, int lim, int out, int in) const {
        unsigned long long notU[kClimbWords];
        outside(notU, pre, lim, out, in);
        const uint32_t n = (uint32_t)V.nent;
        for (uint32_t e = 0; e < n; e++) if (inside(notU, V.score + e)) return e;
        return kOrderNone;
    }
    // the same look-up by the whole warp, 32 consecutive entries a step from `start` (every lane gets the answer)
    __device__ __forceinline__ uint32_t warp_pos(const OrderClimbVar &V, const unsigned long long *pre, int lim, int out, int in, uint32_t start, int lane) const {
        unsigned long long notU[kClimbWords];
        outside(notU, pre, lim, out, in);
        const uint32_t n = (uint32_t)V.nent;
        for (uint32_t b = start; b < n; b += 32) {
            const uint32_t hits = __ballot_sync(0xFFFFFFFFu, b + lane < n && inside(notU, V.score + b + lane));
            if (hits) return b + __ffs(hits) - 1;
        }
        return kOrderNone;
    }
};
template <class Look>
__device__ __forceinline__ float climb_best(const Look &look, const OrderClimbVar &V, const uint8_t *at, const unsigned long long *pre, int lim, int out,
                                            int in, const float *__restrict__ scores) {
    const uint32_t pos = look.pos(V, at, pre, lim, out, in);
    return pos == kOrderNone ? 3.402823466e+38f : __ldg(scores + V.score + pos);
}
// does v have a skeleton neighbour in the set P, leaving out position `out`?
__device__ __forceinline__ bool climb_touches(const OrderClimbVar &V, const unsigned long long *P, int out) {
    unsigned long long any = 0;
#pragma unroll
    for (int w = 0; w < kClimbWords; w++) any |= V.adj[w] & P[w] & ~(w == (out >> 6) ? 1ull << (out & 63) : 0ull);
    return any != 0;
}
// order-preserving key of a float32 cost, -0 folded to +0
__device__ __forceinline__ uint32_t climb_key(float g) {
    const uint32_t u = g == 0.0f ? 0u : __float_as_uint(g);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

template <class Look>
__global__ void __launch_bounds__(kClimbThreads) order_climb_kernel(const OrderClimbVar *__restrict__ vars, const Look look,
                                                                    const float *__restrict__ scores, int k, uint32_t restarts, unsigned long long seed,
                                                                    float *__restrict__ r_cost, uint32_t *__restrict__ r_moves,
                                                                    uint8_t *__restrict__ r_order, uint32_t *__restrict__ r_pos) {
    extern __shared__ __align__(16) unsigned char climb_smem[];
    OrderClimbVar *s_var = reinterpret_cast<OrderClimbVar *>(climb_smem);
    unsigned long long *s_pre = reinterpret_cast<unsigned long long *>(s_var + k);         // [k + 1][kClimbWords]
    unsigned long long *s_key = s_pre + (k + 1) * kClimbWords;                              // [kClimbWarps]
    float *s_b = reinterpret_cast<float *>(s_key + kClimbWarps);                             // [k]
    float *s_g = s_b + k;                                                                   // [k + 1]
    float *s_x = s_g + k + 1;                                                               // [kClimbWarps][k]
    float *s_y = s_x + kClimbWarps * k;                                                     // [kClimbWarps][k]
    uint8_t *s_ord = reinterpret_cast<uint8_t *>(s_y + kClimbWarps * k);                    // [k]
    uint8_t *s_at = s_ord + k;                                                              // [k]
    uint8_t *s_okx = s_at + k;                                                              // [kClimbWarps][k]
    uint8_t *s_oky = s_okx + kClimbWarps * k;                                               // [kClimbWarps][k]
    __shared__ int s_flag;
    __shared__ uint32_t s_moves;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < k; i += blockDim.x) s_var[i] = vars[i];
    __syncthreads();

    for (uint32_t r = blockIdx.x; r < restarts; r += gridDim.x) {
        // start: a random admissible order (one thread; k draws)
        if (threadIdx.x == 0) {
            uint64_t x = seed + 0xD1B54A32D192ED03ull * ((uint64_t)r + 1);
            unsigned long long *placed = s_pre, *front = s_pre + kClimbWords;   // scratch: pre[] is rebuilt from the order
            for (int w = 0; w < kClimbWords; w++) placed[w] = front[w] = 0;
            int ok = 1;
            for (int m = 0; m < k; m++) {
                const uint64_t z = climb_draw(x);
                int v;
                if (m == 0) {
                    v = (int)(z % (uint64_t)k);
                } else {
                    int nf = 0;
                    for (int w = 0; w < kClimbWords; w++) nf += __popcll(front[w]);
                    if (nf == 0) { ok = 0; break; }
                    int want = (int)(z % (uint64_t)nf), w = 0;
                    while (want >= __popcll(front[w])) want -= __popcll(front[w++]);
                    unsigned long long f = front[w];
                    for (; want; want--) f &= f - 1;
                    v = 64 * w + __ffsll((long long)f) - 1;
                }
                s_ord[m] = (uint8_t)v;
                placed[v >> 6] |= 1ull << (v & 63);
                for (int w = 0; w < kClimbWords; w++) front[w] = (front[w] | s_var[v].adj[w]) & ~placed[w];
            }
            s_flag = ok;
            s_moves = 0;
        }
        __syncthreads();
        if (!s_flag) {                                            // the component has no admissible order
            if (threadIdx.x == 0) { r_cost[r] = __int_as_float(0x7f800000); r_moves[r] = 0; }
            for (int m = threadIdx.x; m < k; m += blockDim.x) { r_order[(size_t)r * k + m] = 0; r_pos[(size_t)r * k + m] = kOrderNone; }
            __syncthreads();
            continue;
        }
        for (;;) {
            // the state of the current order: at[], pre[], b[], g[]
            for (int m = threadIdx.x; m < k; m += blockDim.x) s_at[s_ord[m]] = (uint8_t)m;
            if (threadIdx.x < kClimbWords) {
                unsigned long long acc = 0;
                s_pre[threadIdx.x] = 0;
                for (int m = 0; m < k; m++) {
                    const int v = s_ord[m];
                    if ((v >> 6) == (int)threadIdx.x) acc |= 1ull << (v & 63);
                    s_pre[(m + 1) * kClimbWords + threadIdx.x] = acc;
                }
            }
            __syncthreads();
            for (int m = threadIdx.x; m < k; m += blockDim.x) s_b[m] = climb_best(look, s_var[s_ord[m]], s_at, s_pre, m, -1, -1, scores);
            __syncthreads();
            if (threadIdx.x == 0) {
                float g = 0.0f;
                s_g[0] = g;
                for (int m = 0; m < k; m++) s_g[m + 1] = g = __fadd_rn(g, s_b[m]);
            }
            __syncthreads();

            // every move (i, j): one warp per source i
            float *X = s_x + warp * k, *Y = s_y + warp * k;
            uint8_t *okX = s_okx + warp * k, *okY = s_oky + warp * k;
            unsigned long long best = ~0ull;
            for (int i = warp; i < k; i += kClimbWarps) {
                const int vi = s_ord[i];
                const OrderClimbVar &Vi = s_var[vi];
                if constexpr (Look::kWarp) {
                    // targets in descending order: U of the Y look-ups only shrinks, so each scan starts at the last hit
                    uint32_t ystart = 0;
                    for (int t = k - 1; t >= 0; t--) {
                        if (t == i) continue;
                        const OrderClimbVar &Vt = s_var[s_ord[t]];
                        const uint32_t px = t > i ? look.warp_pos(Vt, s_pre, t, vi, -1, 0, lane) : look.warp_pos(Vt, s_pre, t, -1, vi, 0, lane);
                        const uint32_t py = t > i ? look.warp_pos(Vi, s_pre, t + 1, vi, -1, ystart, lane) : look.warp_pos(Vi, s_pre, t, -1, -1, ystart, lane);
                        ystart = py == kOrderNone ? (uint32_t)Vi.nent : py;
                        if (lane == 0) {
                            X[t] = px == kOrderNone ? 3.402823466e+38f : __ldg(scores + Vt.score + px);
                            Y[t] = py == kOrderNone ? 3.402823466e+38f : __ldg(scores + Vi.score + py);
                        }
                    }
                }
                for (int t = lane; t < k; t += 32) {
                    if (t == i) continue;
                    const OrderClimbVar &Vt = s_var[s_ord[t]];
                    if (t > i) {
                        if constexpr (!Look::kWarp) {
                            X[t] = climb_best(look, Vt, s_at, s_pre, t, vi, -1, scores);
                            Y[t] = climb_best(look, Vi, s_at, s_pre, t + 1, vi, -1, scores);
                        }
                        okX[t] = t == 1 || climb_touches(Vt, s_pre + t * kClimbWords, vi);
                        okY[t] = climb_touches(Vi, s_pre + (t + 1) * kClimbWords, vi);
                    } else {
                        if constexpr (!Look::kWarp) {
                            X[t] = climb_best(look, Vt, s_at, s_pre, t, -1, vi, scores);
                            Y[t] = climb_best(look, Vi, s_at, s_pre, t, -1, -1, scores);
                        }
                        okX[t] = t > 0 || ((Vt.adj[vi >> 6] >> (vi & 63)) & 1);
                        okY[t] = t == 0 || climb_touches(Vi, s_pre + t * kClimbWords, -1);
                    }
                }
                __syncwarp();
                for (int j = lane; j < k; j += 32) {
                    if (j == i || !okY[j]) continue;
                    bool ok = true;
                    float g;
                    int m0;
                    if (j > i) {
                        g = s_g[i];
                        for (int m = i + 1; m <= j && ok; m++) { ok = okX[m]; g = __fadd_rn(g, X[m]); }
                        g = __fadd_rn(g, Y[j]);
                        m0 = j + 1;
                    } else {
                        g = __fadd_rn(s_g[j], Y[j]);
                        for (int m = j; m < i && ok; m++) { ok = okX[m]; g = __fadd_rn(g, X[m]); }
                        m0 = i + 1;
                    }
                    if (!ok) continue;
                    for (int m = m0; m < k; m++) {
                        if (__float_as_uint(g) == __float_as_uint(s_g[m])) { g = s_g[k]; break; }
                        g = __fadd_rn(g, s_b[m]);
                    }
                    const unsigned long long key = ((unsigned long long)climb_key(g) << 32) | ((unsigned long long)i << 8) | (unsigned long long)j;
                    best = min(best, key);
                }
                __syncwarp();
            }
            for (int o = 16; o; o >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
            if (lane == 0) s_key[warp] = best;
            __syncthreads();

            // the move, if it strictly lowers the cost
            if (threadIdx.x == 0) {
                unsigned long long key = s_key[0];
                for (int w = 1; w < kClimbWarps; w++) key = min(key, s_key[w]);
                int take = 0;
                if (key != ~0ull) {
                    const uint32_t kc = (uint32_t)(key >> 32);
                    const float c = __uint_as_float((kc & 0x80000000u) ? (kc & 0x7FFFFFFFu) : ~kc);
                    take = c < s_g[k];
                }
                if (take) {
                    const int i = (int)((key >> 8) & 255), j = (int)(key & 255);
                    const uint8_t v = s_ord[i];
                    if (j > i) for (int m = i; m < j; m++) s_ord[m] = s_ord[m + 1];
                    else for (int m = i; m > j; m--) s_ord[m] = s_ord[m - 1];
                    s_ord[j] = v;
                    s_moves++;
                }
                s_flag = take;
            }
            __syncthreads();
            if (!s_flag) break;
        }

        // the local optimum of restart r
        for (int m = threadIdx.x; m < k; m += blockDim.x) {
            r_order[(size_t)r * k + m] = s_ord[m];
            r_pos[(size_t)r * k + m] = look.pos(s_var[s_ord[m]], s_at, s_pre, m, -1, -1);
        }
        if (threadIdx.x == 0) { r_cost[r] = s_g[k]; r_moves[r] = s_moves; }
        __syncthreads();
    }
}

} // namespace urlgpu
