// bic_kernels.cuh — K1: discrete BIC counting + log-likelihood (sm_100a).
//
// Replaces ADTree::makeContab (ad_tree/ad_tree.cpp:95-164), LogLikelihoodCalculator::calculate
// (scoring_function/log_likelihood_calculator.cpp:22-77) and BICScoringFunction::calculateScore
// (scoring_function/bic_scoring_function.cpp:32-76) of the reference.
//
// Data layout: codes column-major uint8 [p][n_stride], n_stride = n rounded up to 16 so every column starts
// 16-byte aligned and rows are read with 128-bit loads.  A contingency table of (v, S) is a dense int32 array
// indexed  x_v + r_v * paIdx,  paIdx = mixed radix over the parents in ascending variable index, lowest
// index least significant (log_likelihood_calculator.cpp:61-73).
//
// Arithmetic contract (SURVEY.md Q4): qlog[c] = (int64) ilogi[c] * 2^23 where ilogi[c] = (float)(c*ln c) is the
// reference's own float table (log_likelihood_calculator.h:30-38) built on the host with glibc log.  The
// log-likelihood  sum_cells ilogi[n_ijk] - sum_j ilogi[n_ij]  is accumulated as an exact int64 (every float
// table entry is a multiple of 2^-23), so the result is independent of summation order, thread count and
// GPU count.  It is rounded ONCE to float32, then  score -= tVal * base  in float32 without contraction
// (bic_scoring_function.cpp:73).
#pragma once
#include "common.cuh"
#include <type_traits>

namespace urlgpu {

struct BicData {
    const uint8_t *codes;   // [p][n_stride]
    int64_t n, n_stride;
    const long long *qlog;  // [n+2]
    const long long *qcfg;  // [n+2] per-configuration term: qlog itself (BIC), qlog + the log-regret of the child's arity (fNML)
    int cfg_min;            // configurations with at most this many records contribute nothing (BIC: 1, fNML: 0)
    float base;             // (float)(ln(N)/2); 0 for fNML and BDeu (no penalty term)
    float ess;              // > 0: BDeu with this equivalent sample size (direct-counting kernels only); 0: table look-ups
    double acc_scale;       // the accumulator's unit: 2^-23 (BIC, fNML), 2^-30 (BDeu)
};

// Per-variable candidate description (kernel argument, by value).
struct CandInfo {
    int c;                          // number of candidates (v excluded)
    int v;                          // the child variable
    int rv;                         // its cardinality
    int max_parents;
    int var[kMaxDenseCand];         // candidate -> variable index (ascending)
    int card[kMaxDenseCand];
};

// Where a set's score goes.  DENSE layout: a table of 2^c floats indexed by the compact mask.  RANK layout
// (rank_kernels.cuh): a table of sum_{l<=K} C(c,l) floats indexed by layer base + colex rank of the set, which is the
// reference's enumeration order (score_calculator.cpp:76-120); binom == nullptr selects the dense layout.
constexpr int kMaxRankCand = 255;
constexpr int kMaxRankLayers = 32;
struct RankSpace {                       // kernel argument, by value
    int c, K;                            // candidates, largest set size
    int bstride;                         // columns of the binomial table (K + 2)
    const uint32_t *binom;               // device: [256][bstride], binom[b * bstride + i] = C(b, i) saturating at 2^32 - 1
    uint32_t layer_base[kMaxRankLayers + 2];   // first index of layer l; [K + 1] = T
};
// compact mask (c <= 64) -> table index
__device__ __forceinline__ uint64_t out_index(const RankSpace &rs, uint64_t mask) {
    if (rs.binom == nullptr) return mask;
    uint32_t r = 0;
    int i = 0;
    for (uint64_t m = mask; m; m &= m - 1) { i++; r += __ldg(rs.binom + (__ffsll((long long)m) - 1) * rs.bstride + i); }
    return (uint64_t)rs.layer_base[i] + r;
}

// column list of one set, built by one thread into shared memory
struct SetCols {
    const uint8_t *col[kMaxCols];
    uint32_t stride[kMaxCols];
    int ncols;
    uint32_t cells;
    float tval;
    uint64_t out;   // where the set's score goes
};

// ---------------------------------------------------------------------------------------------------------
// How the direct-counting kernels below name a set (its 32-bit `key`).  A policy fills the set's SetCols: columns,
// cell count, penalty and output index.  MaskSets: key = compact mask over the candidates of a CandInfo (the cube
// path's root tables, in cube order; they never write scores).  RankSets (rank_kernels.cuh): key = colex index.
// ListSets: key = position in a caller's list of (child, parent set) entries (urlgpu_score_sets).
// ---------------------------------------------------------------------------------------------------------
struct MaskSets {
    CandInfo ci;
    __host__ __device__ __forceinline__ int rv() const { return ci.rv; }
    __device__ __forceinline__ void build_cols(const BicData &d, uint32_t mask, SetCols &sc) const {
        // child first with stride 1, then the parents in ascending variable index
        sc.col[0] = d.codes + (int64_t)ci.v * d.n_stride;
        sc.stride[0] = 1;
        uint32_t base = (uint32_t)ci.rv;
        int nc = 1;
        float pen = (float)(ci.rv - 1); // bic_scoring_function.cpp:21
        for (int i = 0; i < ci.c; i++)
            if ((mask >> i) & 1) {
                sc.col[nc] = d.codes + (int64_t)ci.var[i] * d.n_stride;
                sc.stride[nc] = base;
                base *= (uint32_t)ci.card[i];
                pen = __fmul_rn(pen, (float)ci.card[i]); // :25, float product, ascending variable order
                nc++;
            }
        sc.ncols = nc;
        sc.cells = base;
        sc.tval = pen;
        sc.out = mask;
    }
};

// The entries of one launch share the child arity `child_rv` (bic_score_tables_kernel and the fNML table take one per launch).
// Columns, cell count and penalty are built exactly as MaskSets builds them; the score goes to the entry's position.
struct ListSets {
    const ListEntry *ent;
    const int *par;     // parents of all entries, ascending per entry
    const int *card;    // [p]
    int child_rv;
    __host__ __device__ __forceinline__ int rv() const { return child_rv; }
    __device__ __forceinline__ void build_cols(const BicData &d, uint32_t key, SetCols &sc) const {
        const ListEntry e = ent[key];
        sc.col[0] = d.codes + (int64_t)e.v * d.n_stride;
        sc.stride[0] = 1;
        uint32_t base = (uint32_t)child_rv;
        float pen = (float)(child_rv - 1);
        for (int i = 0; i < e.k; i++) {
            const int q = __ldg(par + e.off + i), cd = __ldg(card + q);
            sc.col[i + 1] = d.codes + (int64_t)q * d.n_stride;
            sc.stride[i + 1] = base;
            base *= (uint32_t)cd;
            pen = __fmul_rn(pen, (float)cd);
        }
        sc.ncols = e.k + 1;
        sc.cells = base;
        sc.tval = pen;
        sc.out = key;
    }
};

// accumulate the mixed-radix index of 16 consecutive rows
__device__ __forceinline__ void accum16(uint4 w, uint32_t s, uint32_t (&idx)[16]) {
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int q = 0; q < 4; q++) {
        idx[4 * q + 0] += (ws[q] & 0xffu) * s;
        idx[4 * q + 1] += ((ws[q] >> 8) & 0xffu) * s;
        idx[4 * q + 2] += ((ws[q] >> 16) & 0xffu) * s;
        idx[4 * q + 3] += (ws[q] >> 24) * s;
    }
}

// stream rows [row0,row1) (row0 multiple of 16) of one set into `hist` (shared or global int32 table)
template <typename HistPtr>
__device__ __forceinline__ void count_rows(const SetCols &sc, int64_t row0, int64_t row1, HistPtr hist, int tid, int nthreads) {
    const int64_t full_end = row0 + ((row1 - row0) / 16) * 16;
    const int ncols = sc.ncols;
    for (int64_t r = row0 + (int64_t)tid * 16; r < full_end; r += (int64_t)nthreads * 16) {
        uint32_t idx[16];
#pragma unroll
        for (int i = 0; i < 16; i++) idx[i] = 0;
        int c = 0;
        for (; c + 1 < ncols; c += 2) { // two loads in flight
            const uint4 w0 = ld_stream_u4(reinterpret_cast<const uint4 *>(sc.col[c] + r));
            const uint4 w1 = ld_stream_u4(reinterpret_cast<const uint4 *>(sc.col[c + 1] + r));
            accum16(w0, sc.stride[c], idx);
            accum16(w1, sc.stride[c + 1], idx);
        }
        if (c < ncols) accum16(ld_stream_u4(reinterpret_cast<const uint4 *>(sc.col[c] + r)), sc.stride[c], idx);
#pragma unroll
        for (int i = 0; i < 16; i++) atomicAdd(&hist[idx[i]], 1);
    }
    // ragged tail (< 16 rows)
    for (int64_t r = full_end + tid; r < row1; r += nthreads) {
        uint32_t idx = 0;
        for (int c = 0; c < ncols; c++) idx += (uint32_t)sc.col[c][r] * sc.stride[c];
        atomicAdd(&hist[idx], 1);
    }
}

// sum_cells q[n_ijk] - sum_j q[n_ij] over parent configurations [j0,j1)
template <typename HistPtr>
__device__ __forceinline__ long long score_configs(HistPtr hist, int rv, int64_t j0, int64_t j1, const long long *__restrict__ qlog,
                                                   const long long *__restrict__ qcfg, int cfg_min, int tid, int nthreads) {
    long long acc = 0;
    for (int64_t j = j0 + tid; j < j1; j += nthreads) {
        const int64_t b = j * rv;
        int nij = 0;
        for (int k = 0; k < rv; k++) {
            const int cnt = hist[b + k];
            nij += cnt;
            if (cnt > 1) acc += __ldg(&qlog[cnt]); // q[0] = q[1] = 0
        }
        if (nij > cfg_min) acc -= __ldg(&qcfg[nij]);
    }
    return acc;
}

__device__ __forceinline__ float bic_finalize(long long acc, float tval, float base, double acc_scale = 1.0 / 8388608.0) {
    // one rounding of acc * acc_scale to float32, then the float32 penalty.  acc reaches FP64 rounded to odd (truncated, the
    // lowest bit set when that dropped anything): a second rounding to 24 bits of a 53-bit round-to-odd value is the one
    // correct rounding, also at |acc| >= 2^53 (BIC from 2^30 nats, BDeu near 1e8 records), where round-to-nearest twice is not
    double d = __ll2double_rz(acc);
    if (__double2ll_rz(d) != acc) d = __longlong_as_double(__double_as_longlong(d) | 1);
    const float ll = __double2float_rn(d * acc_scale);
    return __fsub_rn(ll, __fmul_rn(tval, base)); // bic_scoring_function.cpp:73, no FMA contraction
}

// BDeu (bdeu_scoring_function.cpp:25-123, enableDeCamposPruning off) over parent configurations [j0,j1) of a set with
// `nconf` configurations in all:
//   sum_{cells, n_ijk > 0} [ (float)lgamma(a_ijk (+) n_ijk) - (float)lgamma(a_ijk) ]  +  sum_{j, n_ij > 0} [ (float)lgamma(a_ij) - lgamma(a_ij (+) n_ij) ]
// with a_ij = ess / r, a_ijk = ess / (r * r_v) in float32 and (+) the float32 addition the reference performs before
// calling lgamma (:108, :117).  Contract: every bracket is evaluated in FP64, rounded to the 2^-30 grid and the grid values
// are summed as exact integers — independent of summation order like the BIC contract; the reference itself keeps a
// float32 running sum in contingency-tree / hash-map order.
template <typename HistPtr>
__device__ __forceinline__ long long score_configs_bdeu(HistPtr hist, int rv, int64_t nconf, int64_t j0, int64_t j1, float ess, int tid, int nthreads) {
    const float a_ij = __fdiv_rn(ess, (float)(int)nconf);                 // :32 (float / int)
    const float a_ijk = __fdiv_rn(ess, (float)(int)(nconf * rv));         // :35-36
    const double lg_ij = (double)__double2float_rn(lgamma((double)a_ij));   // float members of `scratch`
    const double lg_ijk = (double)__double2float_rn(lgamma((double)a_ijk));
    long long acc = 0;
    for (int64_t j = j0 + tid; j < j1; j += nthreads) {
        const int64_t b = j * rv;
        int nij = 0;
        for (int k = 0; k < rv; k++) {
            const int cnt = hist[b + k];
            nij += cnt;
            if (cnt > 0) {
                const double temp = (double)__double2float_rn(lgamma((double)__fadd_rn(a_ijk, (float)cnt)));   // :105-108
                acc += __double2ll_rn((temp - lg_ijk) * 1073741824.0);
            }
        }
        if (nij > 0) acc += __double2ll_rn((lg_ij - lgamma((double)__fadd_rn(a_ij, (float)nij))) * 1073741824.0);   // :116-118
    }
    return acc;
}

// the per-set score sum of the direct-counting kernels: table look-ups (BIC, fNML) or BDeu's lgamma terms
template <typename HistPtr>
__device__ __forceinline__ long long score_configs_of(const BicData &d, HistPtr hist, int rv, int64_t nconf, int64_t j0, int64_t j1, int tid, int nthreads) {
    if (d.ess > 0.f) return score_configs_bdeu(hist, rv, nconf, j0, j1, d.ess, tid, nthreads);
    return score_configs(hist, rv, j0, j1, d.qlog, d.qcfg, d.cfg_min, tid, nthreads);
}

// ---------------------------------------------------------------------------------------------------------
// K1 (shared-memory tiers): one CTA per listed set; whole table in shared memory.  Outputs, each optional: the score at
// SetCols::out, the table at table_offs[item] of tables_out, the exact accumulator at acc_out[item].
// ---------------------------------------------------------------------------------------------------------
template <class Sets>
__global__ void bic_count_smem_kernel(BicData d, Sets fam, const uint32_t *__restrict__ work, float *__restrict__ scores,
                                      const uint64_t *__restrict__ table_offs, int *__restrict__ tables_out, long long *__restrict__ acc_out) {
    extern __shared__ __align__(16) int hist[];
    __shared__ SetCols sc;
    __shared__ long long red[32];
    if (threadIdx.x == 0) fam.build_cols(d, work[blockIdx.x], sc);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < sc.cells; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    count_rows(sc, 0, d.n, hist, threadIdx.x, blockDim.x);
    __syncthreads();
    if (table_offs) { // cube roots: the table is the parent of marginalised children
        int *dst = tables_out + table_offs[blockIdx.x];
        for (uint32_t i = threadIdx.x; i < sc.cells; i += blockDim.x) dst[i] = hist[i];
    }
    if (!scores && !acc_out) return;
    const int rv = fam.rv();
    long long acc = score_configs_of(d, hist, rv, sc.cells / rv, 0, sc.cells / rv, threadIdx.x, blockDim.x);
    acc = block_sum_ll(acc, red);
    if (threadIdx.x == 0) {
        if (scores) scores[sc.out] = bic_finalize(acc, sc.tval, d.base, d.acc_scale);
        if (acc_out) acc_out[blockIdx.x] = acc;
    }
}

// ---------------------------------------------------------------------------------------------------------
// K1 (global tier): tables live in an L2-resident scratch buffer; grid = (set in batch, row slice).
// ---------------------------------------------------------------------------------------------------------
struct GlobalSet {
    uint32_t key;
    uint32_t cells;
    uint64_t table_off; // in int32 elements
};

template <class Sets>
__global__ void bic_count_global_kernel(BicData d, Sets fam, const GlobalSet *__restrict__ sets, int *__restrict__ tables, int64_t rows_per_slice) {
    __shared__ SetCols sc;
    const GlobalSet gs = sets[blockIdx.x];
    if (threadIdx.x == 0) fam.build_cols(d, gs.key, sc);
    __syncthreads();
    const int64_t row0 = (int64_t)blockIdx.y * rows_per_slice;
    int64_t row1 = row0 + rows_per_slice;
    if (row1 > d.n) row1 = d.n;
    if (row0 >= row1) return;
    count_rows(sc, row0, row1, tables + gs.table_off, threadIdx.x, blockDim.x);
}

__global__ void bic_score_tables_kernel(BicData d, int rv, const GlobalSet *__restrict__ sets, const int *__restrict__ tables,
                                        long long *__restrict__ acc_out /*[batch]*/, int64_t configs_per_chunk) {
    __shared__ long long red[32];
    const GlobalSet gs = sets[blockIdx.x];
    const int64_t nconf = gs.cells / rv;
    const int64_t j0 = (int64_t)blockIdx.y * configs_per_chunk;
    if (j0 >= nconf) return;
    int64_t j1 = j0 + configs_per_chunk;
    if (j1 > nconf) j1 = nconf;
    long long acc = score_configs_of(d, tables + gs.table_off, rv, nconf, j0, j1, threadIdx.x, blockDim.x);
    acc = block_sum_ll(acc, red);
    if (threadIdx.x == 0 && acc != 0) atomicAdd(reinterpret_cast<unsigned long long *>(&acc_out[blockIdx.x]), (unsigned long long)acc);
}

// scores (and, optionally, the exact fixed-point log-likelihood) of the global tier at SetCols::out
template <class Sets>
__global__ void bic_finalize_kernel(BicData d, Sets fam, const GlobalSet *__restrict__ sets, const long long *__restrict__ acc, int nsets,
                                    float *__restrict__ scores, long long *__restrict__ ll_fixed) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsets) return;
    SetCols sc;
    fam.build_cols(d, sets[i].key, sc);
    scores[sc.out] = bic_finalize(acc[i], sc.tval, d.base, d.acc_scale);
    if (ll_fixed) ll_fixed[sc.out] = acc[i];
}

// store rule of the caller: empty set stored iff score < 1, others iff score < 0 (score_calculator.cpp:59,111)
__global__ void bic_store_rule_kernel(float *__restrict__ scores, uint64_t n_masks, int max_parents) {
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_masks) return;
    if (__popcll(m) > max_parents) return; // already sentinel
    const float s = scores[m];
    if (is_sentinel(s)) return;
    const bool stored = (m == 0) ? (s < 1.0f) : (s < 0.0f);
    if (!stored) scores[m] = sentinel();
}


// ---------------------------------------------------------------------------------------------------------
// K1 "cube": derive a child table by summing one parent digit out, and score it in the same pass.
//
// The candidate family of a variable is closed under taking subsets, so only the ROOT tables (the largest
// sets) are counted from the rows; every other table is the marginal of a table one variable larger:
//   child[x_v + rv*(lo + hi*Bc)] = sum_{a<r} parent[x_v + rv*(lo + (hi*r + a)*Bc)]
// where the dropped digit has stride Bc (in parent-configuration units) and arity r.  Each parent cell is read
// exactly once, each child cell written once: a pure streaming pass (HBM/L2 bound), no atomics on the tables.
// The log-likelihood terms of the child are accumulated on the fly (exact int64, see the file header).
// ---------------------------------------------------------------------------------------------------------
struct CubePair {
    uint64_t parent_off, child_off;   // int32 elements
    uint32_t groups;                  // child configurations / (g0 * g1)
    uint32_t Bc;                      // stride of the dropped digit, in configurations
    uint32_t r;                       // arity of the dropped digit
    uint32_t chunk0;                  // first block of this pair
    uint32_t acc[4];                  // accumulators of the child T, T \ {0}, T \ {1} and T \ {0,1} (see "GROUPS")
    uint32_t g0, g1;                  // a group is g0 * g1 configurations: the arities of cube bits 0 and 1 that T holds, else 1
    uint32_t flags;                   // kCubeStore | kCubeScore*
    uint32_t fmt;                     // bit 0: the parent table holds uint16 cells, bit 1: the child table does (see "16-bit tables")
    uint32_t magic;                   // floor((2^32 - 1) / Bc): fast_div instead of a hardware division per group
};
constexpr uint32_t kCubeStore = 1;        // a later pass reads T's table: it is written
constexpr uint32_t kCubeScoreChild = 2;   // score T (a set of the family: layer <= K); acc[s] is scored iff flags & (2 << s)
constexpr uint32_t kCubeScoreLeaf = 4;    // score T \ {0} from the group's sums over digit 0
constexpr uint32_t kCubeScoreDrop1 = 8;   // score T \ {1} from the sums over digit 1
constexpr uint32_t kCubeScoreDrop01 = 16; // score T \ {0,1} from the sums over both

// GROUPS.  A set T derived in a pass has children T \ {b} for the b below run(T), the number of trailing cube bits T holds.
// Digits 0 and 1 are the two lowest digits of a configuration index, so the g0 * g1 consecutive configurations
// a0 + g0 * (a1 + g1 * h) of T (g0, g1 = arities of bits 0 and 1) sum over a0 to configuration a1 + g1 * h of T \ {0}, over a1
// to configuration a0 + g0 * h of T \ {1}, and over both to configuration h of T \ {0,1}.  A thread that derives T in such
// groups holds the counts of all four sets in registers and scores them there.  So T \ {1} (run 1: its only child is
// T \ {0,1}) needs no pass of its own, and only tables of sets with run >= 3 are written.  The dropped digit z >= 2 of such a
// T has a stride Bc that is a multiple of g0 * g1, so a group is contiguous in the parent as well.  Where the parent's pass
// built no two-digit groups, pairs keep the shape (card[0], 1) for a T without bit 1 (scoring T and T \ {0}) and (1, 1) for a
// T without bit 0: the children root \ {1} and root \ {0} of a root table written by a kernel that builds no groups, and
// the children T \ {1} of a fused root's children T (bic_root_kernel scores T and T \ {0} in groups of card[0]).

constexpr int kCubeThreads = 256;
#ifndef URLGPU_CUBE_UNROLL
#define URLGPU_CUBE_UNROLL 2
#endif
constexpr int kCubeUnroll = URLGPU_CUBE_UNROLL;
// configurations per block: a block ends with four block-wide sums (T and its three marginals), so a block does enough
// groups to amortise them.  On one B200 (1000 W) the derive kernel took 88.8 ms per configs[3] step at 16384, 95.1 at
// 4096, 91.3 at 32768 (DESIGN §5)
constexpr uint32_t kCubeConfigsPerBlock = 16384;

// N consecutive cells.  p is aligned to N cells as far as the table allows (tables start 16-byte aligned and a run of N cells
// starts at a multiple of N): the widest vector access that divides N.
template <int N>
__device__ __forceinline__ void load_cfg(const int *__restrict__ p, int (&v)[N]) {
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N / 4; i++) { const int4 t = reinterpret_cast<const int4 *>(p)[i]; v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w; }
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int i = 0; i < N / 2; i++) { const int2 t = reinterpret_cast<const int2 *>(p)[i]; v[2 * i] = t.x; v[2 * i + 1] = t.y; }
    } else {
#pragma unroll
        for (int k = 0; k < N; k++) v[k] = p[k];
    }
}
template <int N>
__device__ __forceinline__ void store_cfg(int *__restrict__ p, const int (&v)[N]) {
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N / 4; i++) reinterpret_cast<int4 *>(p)[i] = make_int4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int i = 0; i < N / 2; i++) reinterpret_cast<int2 *>(p)[i] = make_int2(v[2 * i], v[2 * i + 1]);
    } else {
#pragma unroll
        for (int k = 0; k < N; k++) p[k] = v[k];
    }
}

// 16-bit tables.  At the layers that carry almost all of the cube path's traffic (|S| >= 8 at n = 1e6) a table has far more
// cells than any cell has records — the largest count in such tables of configs[3] is ~2e4 — so they are written with
// uint16 cells: half the bytes through HBM for the kernel that is bound by them.  This is SPECULATIVE: a store that
// would not fit saturates and raises a per-call flag; the caller then discards the variable's scores and recomputes them
// with 32-bit tables (urlgpu.cu: table16 fallback), so results stay exact for any data.
__device__ __forceinline__ uint32_t pack16(int a, int b) { return (uint32_t)min(a, 65535) | ((uint32_t)min(b, 65535) << 16); }
template <int N>
__device__ __forceinline__ void load_cfg16(const uint16_t *__restrict__ p, int (&v)[N]) {
    if constexpr (N % 8 == 0) {
#pragma unroll
        for (int i = 0; i < N / 8; i++) {
            const uint4 t = reinterpret_cast<const uint4 *>(p)[i];
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int q = 0; q < 4; q++) { v[8 * i + 2 * q] = w[q] & 0xffff; v[8 * i + 2 * q + 1] = w[q] >> 16; }
        }
    } else if constexpr (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N / 4; i++) { const uint2 t = reinterpret_cast<const uint2 *>(p)[i]; v[4 * i] = t.x & 0xffff; v[4 * i + 1] = t.x >> 16; v[4 * i + 2] = t.y & 0xffff; v[4 * i + 3] = t.y >> 16; }
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int i = 0; i < N / 2; i++) { const uint32_t t = reinterpret_cast<const uint32_t *>(p)[i]; v[2 * i] = t & 0xffff; v[2 * i + 1] = t >> 16; }
    } else {
#pragma unroll
        for (int k = 0; k < N; k++) v[k] = p[k];
    }
}
template <int N>
__device__ __forceinline__ bool store_cfg16(uint16_t *__restrict__ p, const int (&v)[N]) { // true: a count did not fit
    int mx = v[0];
#pragma unroll
    for (int k = 1; k < N; k++) mx = max(mx, v[k]);
    if constexpr (N % 8 == 0) {
#pragma unroll
        for (int i = 0; i < N / 8; i++)
            reinterpret_cast<uint4 *>(p)[i] = make_uint4(pack16(v[8 * i], v[8 * i + 1]), pack16(v[8 * i + 2], v[8 * i + 3]), pack16(v[8 * i + 4], v[8 * i + 5]), pack16(v[8 * i + 6], v[8 * i + 7]));
    } else if constexpr (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N / 4; i++) reinterpret_cast<uint2 *>(p)[i] = make_uint2(pack16(v[4 * i], v[4 * i + 1]), pack16(v[4 * i + 2], v[4 * i + 3]));
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int i = 0; i < N / 2; i++) reinterpret_cast<uint32_t *>(p)[i] = pack16(v[2 * i], v[2 * i + 1]);
    } else {
#pragma unroll
        for (int k = 0; k < N; k++) p[k] = (uint16_t)min(v[k], 65535);
    }
    return mx > 65535;
}

// sum_k q[cnt_k] - q[n_j] of the RV counts cnt[off .. off + RV) of one configuration (q[0] = q[1] = 0)
template <int RV, int N>
__device__ __forceinline__ void score_cfg(long long &acc, const int (&cnt)[N], int off, const long long *__restrict__ qlog, const long long *__restrict__ qcfg, int cfg_min) {
    int nij = 0;
#pragma unroll
    for (int k = 0; k < RV; k++) nij += cnt[off + k];
    if (nij > cfg_min) {
#pragma unroll
        for (int k = 0; k < RV; k++)
            if (cnt[off + k] > 1) acc += __ldg(&qlog[cnt[off + k]]);
        acc -= __ldg(&qcfg[nij]);
    }
}
// scores of a compile-time group of G0 * G1 configurations of T held in registers (see "GROUPS"): T, T \ {0}, T \ {1}, T \ {0,1}
// add(q, v) adds v to the sum of set q (0: T, 1: T \ {0}, 2: T \ {1}, 3: T \ {0,1})
template <int RV, int G0, int G1, typename AddFn>
__device__ __forceinline__ void score_group(const int (&cnt)[G0 * G1 * RV], uint32_t flags, AddFn add, const long long *__restrict__ qlog,
                                            const long long *__restrict__ qcfg, int cfg_min) {
    // a dimension of 1 (a unary cube digit) sums one configuration: the marginal is T itself, as the flags may still ask
    if (flags & kCubeScoreChild) {
        long long v = 0;
#pragma unroll
        for (int m = 0; m < G0 * G1; m++) score_cfg<RV>(v, cnt, m * RV, qlog, qcfg, cfg_min);
        add(0, v);
    }
    if (flags & kCubeScoreLeaf) {
        long long v = 0;
#pragma unroll
        for (int a1 = 0; a1 < G1; a1++) {
            int s[RV];
#pragma unroll
            for (int k = 0; k < RV; k++) {
                s[k] = cnt[G0 * a1 * RV + k];
#pragma unroll
                for (int a0 = 1; a0 < G0; a0++) s[k] += cnt[(a0 + G0 * a1) * RV + k];
            }
            score_cfg<RV>(v, s, 0, qlog, qcfg, cfg_min);
        }
        add(1, v);
    }
    if (flags & kCubeScoreDrop1) {
        long long v = 0;
#pragma unroll
        for (int a0 = 0; a0 < G0; a0++) {
            int s[RV];
#pragma unroll
            for (int k = 0; k < RV; k++) {
                s[k] = cnt[a0 * RV + k];
#pragma unroll
                for (int a1 = 1; a1 < G1; a1++) s[k] += cnt[(a0 + G0 * a1) * RV + k];
            }
            score_cfg<RV>(v, s, 0, qlog, qcfg, cfg_min);
        }
        add(2, v);
    }
    if (flags & kCubeScoreDrop01) {
        int s[RV];
#pragma unroll
        for (int k = 0; k < RV; k++) {
            s[k] = cnt[k];
#pragma unroll
            for (int m = 1; m < G0 * G1; m++) s[k] += cnt[m * RV + k];
        }
        long long v = 0;
        score_cfg<RV>(v, s, 0, qlog, qcfg, cfg_min);
        add(3, v);
    }
}

// a group of run-time shape g0 x g1, configuration by configuration: cfg(m, cnt) gives the counts of T's configuration m of
// the group, put(m, cnt) stores them if T is written.  T \ {0} is summed in registers on the way; T \ {1} and T \ {0,1} sum
// across the a1 rows, so they read the group's cells again (from L1 or shared memory).
template <int RV, typename CfgFn, typename PutFn, typename AddFn>
__device__ __forceinline__ void score_group_any(uint32_t g0, uint32_t g1, CfgFn cfg, PutFn put, uint32_t flags, AddFn add,
                                                const long long *__restrict__ qlog, const long long *__restrict__ qcfg, int cfg_min) {
#pragma unroll 1
    for (uint32_t a1 = 0; a1 < g1; a1++) {
        int l0[RV] = {};
#pragma unroll 1
        for (uint32_t a0 = 0; a0 < g0; a0++) {
            const uint32_t m = a0 + g0 * a1;
            int cnt[RV];
            cfg(m, cnt);
            put(m, cnt);
            if (flags & kCubeScoreChild) { long long v = 0; score_cfg<RV>(v, cnt, 0, qlog, qcfg, cfg_min); add(0, v); }
#pragma unroll
            for (int k = 0; k < RV; k++) l0[k] += cnt[k];
        }
        if (flags & kCubeScoreLeaf) { long long v = 0; score_cfg<RV>(v, l0, 0, qlog, qcfg, cfg_min); add(1, v); }
    }
    if (flags & (kCubeScoreDrop1 | kCubeScoreDrop01)) {
        int l01[RV] = {};
#pragma unroll 1
        for (uint32_t a0 = 0; a0 < g0; a0++) {
            int l1[RV] = {};
#pragma unroll 1
            for (uint32_t a1 = 0; a1 < g1; a1++) {
                int t[RV];
                cfg(a0 + g0 * a1, t);
#pragma unroll
                for (int k = 0; k < RV; k++) l1[k] += t[k];
            }
            if (flags & kCubeScoreDrop1) { long long v = 0; score_cfg<RV>(v, l1, 0, qlog, qcfg, cfg_min); add(2, v); }
#pragma unroll
            for (int k = 0; k < RV; k++) l01[k] += l1[k];
        }
        if (flags & kCubeScoreDrop01) { long long v = 0; score_cfg<RV>(v, l01, 0, qlog, qcfg, cfg_min); add(3, v); }
    }
}

// child arity known at run time only: no counts are kept in registers.  Sum over `cell(m, k)` (cell k of T's configuration m
// of the group) of the no configurations o of a marginal, each the sum of ni configurations o * so + i * si of T, and score them.
template <typename CellFn>
__device__ __forceinline__ long long score_marginal(CellFn cell, int rv, uint32_t no, uint32_t so, uint32_t ni, uint32_t si,
                                                    const long long *__restrict__ qlog, const long long *__restrict__ qcfg, int cfg_min) {
    long long acc = 0;
    for (uint32_t o = 0; o < no; o++) {
        int nij = 0;
        for (int k = 0; k < rv; k++) {
            int cnt = 0;
            for (uint32_t i = 0; i < ni; i++) cnt += cell(o * so + i * si, k);
            nij += cnt;
            if (cnt > 1) acc += __ldg(&qlog[cnt]);
        }
        if (nij > cfg_min) acc -= __ldg(&qcfg[nij]);
    }
    return acc;
}
// the three marginals of a run-time group that the flags ask for
template <typename CellFn, typename AddFn>
__device__ __forceinline__ void score_marginals(CellFn cell, int rv, uint32_t g0, uint32_t g1, uint32_t flags, AddFn add,
                                                const long long *__restrict__ qlog, const long long *__restrict__ qcfg, int cfg_min) {
    if (flags & kCubeScoreLeaf) add(1, score_marginal(cell, rv, g1, g0, g0, 1, qlog, qcfg, cfg_min));
    if (flags & kCubeScoreDrop1) add(2, score_marginal(cell, rv, g0, 1, g1, g0, qlog, qcfg, cfg_min));
    if (flags & kCubeScoreDrop01) add(3, score_marginal(cell, rv, 1, 0, g0 * g1, 1, qlog, qcfg, cfg_min));
}

// block -> pair map (one load per block instead of a dependent binary search by thread 0 while 255 threads wait)
__global__ void cube_map_kernel(const CubePair *__restrict__ pairs, int npairs, uint32_t total, uint32_t *__restrict__ block_pair) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int lo = 0, hi = npairs - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (pairs[mid].chunk0 <= i) lo = mid; else hi = mid - 1;
    }
    block_pair[i] = (uint32_t)lo;
}

// RV > 0: compile-time child arity (2,3,4); RV == 0: generic arity rv_dyn.  A block derives kCubeConfigsPerBlock / (g0 * g1) groups.
template <int RV>
__global__ void __launch_bounds__(kCubeThreads, RV == 4 ? 5 : 6) cube_derive_kernel(const CubePair *__restrict__ pairs, const uint32_t *__restrict__ block_pair, const int *__restrict__ parent_tab,
                                                                   int *__restrict__ child_tab, int rv_dyn, const long long *__restrict__ qlog,
                                                                   const long long *__restrict__ qcfg, int cfg_min, long long *__restrict__ acc_all,
                                                                   int *__restrict__ ovf_flag /*16-bit tables: a count did not fit*/,
                                                                   int qn /*entries of qlog*/) {
    __shared__ long long red[4][32];
    __shared__ uint32_t s_acc[4];   // the accumulators, parked until thread 0 needs them (registers are tight for RV = 4)
    __shared__ long long s_sum[3][kCubeThreads];   // this thread's sums of T \ {0}, T \ {1}, T \ {0,1}: registers hold T's alone
    (void)qn;
    const CubePair pr = pairs[__ldg(&block_pair[blockIdx.x])];
    if (threadIdx.x < 4) s_acc[threadIdx.x] = pr.acc[threadIdx.x];
    const int rv = RV > 0 ? RV : rv_dyn;
    const uint32_t G = pr.g0 * pr.g1, gpb = max(1u, kCubeConfigsPerBlock / G);
    const uint32_t g0 = (blockIdx.x - pr.chunk0) * gpb;
    const uint32_t g1 = min(g0 + gpb, pr.groups);
    const uint32_t flags = pr.flags;
    const bool store = flags & kCubeStore;
    const int *__restrict__ P = parent_tab + pr.parent_off;
    int *__restrict__ Cc = child_tab + pr.child_off;
    long long acc = 0;   // T
#pragma unroll
    for (int q = 0; q < 3; q++) s_sum[q][threadIdx.x] = 0;
    auto add = [&](int q, long long v) { if (q == 0) acc += v; else s_sum[q - 1][threadIdx.x] += v; };
    if constexpr (RV > 0) {
        // configuration indices fit 32 bits (a table has at most 2^30 cells): one IMAD + one IMAD.WIDE per address.  Arity 4 keeps
        // 64-bit indices: ptxas allocates 44 registers for that form and 58 (or spills) for the 32-bit one
        using idx_t = std::conditional_t<RV == 4, uint64_t, uint32_t>;
        // G0 x G1 (compile time) configurations per group, U groups per thread and iteration: r * G0 * G1 * U configurations' loads
        // in flight.  P16 / C16 (compile time per instantiation, uniform per block): parent / child table in uint16 cells
        auto run = [&](auto G0c, auto G1c, auto P16c, auto C16c) {
            constexpr int G0 = decltype(G0c)::value, G1 = decltype(G1c)::value, N = G0 * G1 * RV, U = G0 * G1 == 1 ? kCubeUnroll : 1;
            constexpr int UA = G0 * G1 == 1 ? 2 : 1;   // loads of the dropped digit in flight: one group of N cells for a group > 1
            constexpr bool P16 = decltype(P16c)::value, C16 = decltype(C16c)::value;
            const uint16_t *__restrict__ Ph = reinterpret_cast<const uint16_t *>(P);
            uint16_t *__restrict__ Ch = reinterpret_cast<uint16_t *>(Cc);
            auto load = [&](idx_t pc, int (&v)[N]) { if constexpr (P16) load_cfg16<N>(Ph + pc * (idx_t)RV, v); else load_cfg<N>(P + pc * (idx_t)RV, v); };
            bool ovf = false;
            for (uint32_t g = g0 + threadIdx.x; g < g1; g += U * kCubeThreads) {
                uint32_t gg[U];
                idx_t pc[U];
                bool on[U];
                int cnt[U][N];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    gg[u] = g + u * kCubeThreads;
                    on[u] = gg[u] < g1;
                    const uint32_t ju = (on[u] ? gg[u] : g) * (G0 * G1);
                    const uint32_t hi = fast_div(ju, pr.Bc, pr.magic), lo = ju - hi * pr.Bc;
                    pc[u] = (idx_t)lo + (idx_t)hi * pr.r * pr.Bc;
                }
#pragma unroll
                for (int u = 0; u < U; u++) load(pc[u], cnt[u]);
#pragma unroll UA
                for (uint32_t a = 1; a < pr.r; a++) {
                    int t[U][N];
#pragma unroll
                    for (int u = 0; u < U; u++) load(pc[u] + (idx_t)a * pr.Bc, t[u]);
#pragma unroll
                    for (int u = 0; u < U; u++)
#pragma unroll
                        for (int k = 0; k < N; k++) cnt[u][k] += t[u][k];
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    if (!on[u]) continue;
                    if (store) {
                        if constexpr (C16) ovf |= store_cfg16<N>(Ch + (idx_t)gg[u] * (idx_t)N, cnt[u]); else store_cfg<N>(Cc + (idx_t)gg[u] * (idx_t)N, cnt[u]);
                    }
                    score_group<RV, G0, G1>(cnt[u], flags, add, qlog, qcfg, cfg_min);
                }
            }
            if (ovf) *ovf_flag = 1;
        };
        // any other shape: the group's configurations one after another
        auto run_any = [&](auto P16c, auto C16c) {
            constexpr bool P16 = decltype(P16c)::value, C16 = decltype(C16c)::value;
            const uint16_t *__restrict__ Ph = reinterpret_cast<const uint16_t *>(P);
            uint16_t *__restrict__ Ch = reinterpret_cast<uint16_t *>(Cc);
            auto load = [&](idx_t pc, int (&v)[RV]) { if constexpr (P16) load_cfg16<RV>(Ph + pc * (idx_t)RV, v); else load_cfg<RV>(P + pc * (idx_t)RV, v); };
            bool ovf = false;
            for (uint32_t g = g0 + threadIdx.x; g < g1; g += kCubeThreads) {
                const uint32_t jg = g * G, hi = fast_div(jg, pr.Bc, pr.magic), lo = jg - hi * pr.Bc;
                const idx_t pg = (idx_t)lo + (idx_t)hi * pr.r * pr.Bc;
                auto cfg = [&](uint32_t m, int (&cnt)[RV]) {
                    load(pg + m, cnt);
#pragma unroll 1
                    for (uint32_t a = 1; a < pr.r; a++) {
                        int t[RV];
                        load(pg + m + (idx_t)a * pr.Bc, t);
#pragma unroll
                        for (int k = 0; k < RV; k++) cnt[k] += t[k];
                    }
                };
                auto put = [&](uint32_t m, const int (&cnt)[RV]) {
                    if (!store) return;
                    if constexpr (C16) ovf |= store_cfg16<RV>(Ch + ((idx_t)jg + m) * (idx_t)RV, cnt); else store_cfg<RV>(Cc + ((idx_t)jg + m) * (idx_t)RV, cnt);
                };
                score_group_any<RV>(pr.g0, pr.g1, cfg, put, flags, add, qlog, qcfg, cfg_min);
            }
            if (ovf) *ovf_flag = 1;
        };
        auto by_group = [&](auto P16c, auto C16c) {
            using I1 = std::integral_constant<int, 1>;
            using I2 = std::integral_constant<int, 2>;
            if (pr.g0 == 2 && pr.g1 == 2) run(I2{}, I2{}, P16c, C16c);
            else if (pr.g0 == 2 && pr.g1 == 1) run(I2{}, I1{}, P16c, C16c);
            else if (G == 1) run(I1{}, I1{}, P16c, C16c);
            else run_any(P16c, C16c);
        };
        switch (pr.fmt & 3u) {
        case 0: by_group(std::false_type{}, std::false_type{}); break;
        case 1: by_group(std::true_type{}, std::false_type{}); break;
        case 2: by_group(std::false_type{}, std::true_type{}); break;
        default: by_group(std::true_type{}, std::true_type{}); break;
        }
    } else {
        const uint16_t *Ph = reinterpret_cast<const uint16_t *>(P);
        uint16_t *Ch = reinterpret_cast<uint16_t *>(Cc);
        auto at = [&](uint64_t i) { return (pr.fmt & 1u) ? (int)Ph[i] : P[i]; };
        for (uint32_t g = g0 + threadIdx.x; g < g1; g += kCubeThreads) {
            const uint32_t jg = g * G, hi = jg / pr.Bc, lo = jg - hi * pr.Bc;
            const uint64_t pg = (uint64_t)lo + (uint64_t)hi * pr.r * pr.Bc;
            auto cell = [&](uint32_t m, int k) {   // an arity this wide keeps no counts in registers: marginals read the cells again (L1)
                int cnt = 0;
                for (uint32_t a = 0; a < pr.r; a++) cnt += at((pg + m + (uint64_t)a * pr.Bc) * rv + k);
                return cnt;
            };
            for (uint32_t m = 0; m < G; m++) {
                const uint64_t j = (uint64_t)jg + m;
                int nij = 0;
                for (int k = 0; k < rv; k++) {
                    const int cnt = cell(m, k);
                    if (store) {
                        if (pr.fmt & 2u) { Ch[j * rv + k] = (uint16_t)min(cnt, 65535); if (cnt > 65535) *ovf_flag = 1; }
                        else Cc[j * rv + k] = cnt;
                    }
                    nij += cnt;
                    if ((flags & kCubeScoreChild) && cnt > 1) acc += __ldg(&qlog[cnt]);
                }
                if ((flags & kCubeScoreChild) && nij > cfg_min) acc -= __ldg(&qcfg[nij]);
            }
            score_marginals(cell, rv, pr.g0, pr.g1, flags, add, qlog, qcfg, cfg_min);
        }
    }
#pragma unroll
    for (int q = 0; q < 4; q++)
        if (flags & (kCubeScoreChild << q)) {
            const long long v = block_sum_ll(q == 0 ? acc : s_sum[q - 1][threadIdx.x], red[q]);
            if (threadIdx.x == 0 && v != 0) atomicAdd(reinterpret_cast<unsigned long long *>(&acc_all[s_acc[q]]), (unsigned long long)v);
        }
}

// scores[res_mask] from the exact accumulators; tVal multiplied in ascending variable order (result-order CandInfo)
__global__ void cube_finalize_kernel(BicData d, CandInfo ci_res, const uint32_t *__restrict__ res_masks, const long long *__restrict__ acc, int nsets,
                                     float *__restrict__ scores, RankSpace om) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsets) return;
    const uint32_t mask = res_masks[i];
    if (mask == 0xffffffffu) return; // a set outside this call's part of the family (urlgpu_score_part)
    float pen = (float)(ci_res.rv - 1);
    for (int b = 0; b < ci_res.c; b++)
        if ((mask >> b) & 1) pen = __fmul_rn(pen, (float)ci_res.card[b]);
    scores[out_index(om, mask)] = bic_finalize(acc[i], pen, d.base, d.acc_scale);
}

} // namespace urlgpu
