// tree_kernels.cuh — the cube path's root kernel (bic_kernels.cuh, urlgpu.cu bic_score_family_cube): the large root
// tables of a family are counted in shared-memory slices of bucketed, bit-packed rows.
//
// Replaces ADTree::makeContab (ad_tree/ad_tree.cpp:95-164) + LogLikelihoodCalculator::calculate
// (scoring_function/log_likelihood_calculator.cpp:22-77) for the root tables of a candidate family.
//
// Per variable:
//   1. rows are packed to one 64-bit word (w = 2, 4 or 8 bits per column by the largest arity; field 0 = child,
//      field 1+i = cube bit i) and bucketed by the joint value of the top `dmax` cube digits (tree_key /
//      tree_scatter kernels + a device scan): rows with a given prefix of top digits are contiguous; one coalesced
//      8-byte load fetches a whole row, and its cell index is the sum of one look-up per BYTE of the word in
//      per-slice tables built in shared memory (byte value -> sum of field value * stride over the byte's fields).
//   2. bic_root_kernel: one CTA per (root, slice).  A slice fixes the root's present top digits (the rows it needs
//      are `nseg` contiguous segments, one per joint value of the ABSENT top digits) and histograms the remaining
//      digits with shared-memory atomics; the slice is then written to the root's table, or, for a fused root, its
//      children are marginalised out of it and scored on chip (see CubeRoot below).
#pragma once
#include "bic_kernels.cuh"
#include <type_traits>

namespace urlgpu {

constexpr int kPreMax = 16;             // prefix products of the lowest digits kept in TreeVar (run of the cube path's fused roots)
constexpr int kTreeMaxZone = 20;        // bucketed top digits
constexpr uint32_t kTreeMaxBuckets = 1u << 20;

struct TreeVar {                        // per-variable constants (kernel argument, by value)
    int c, rv, dmax;
    int w;                              // bits per packed field (2, 4 or 8); field f sits at bit f*w
    uint32_t P_dmax;                    // number of buckets = joint arity of the top dmax digits
    uint16_t card[kMaxDenseCand];       // cube order
    uint32_t pre[kPreMax + 1];          // pre[b] = prod_{i<b} card[i] (saturating at 2^31)
    uint32_t magic[kPreMax + 1];        // floor((2^32-1) / pre[b]) for fast_div
    uint32_t cmagic[kPreMax];           // floor((2^32-1) / card[b]) of the lowest digits
    const unsigned long long *rows;     // [n] packed rows, bucketed
    const uint32_t *prefix_off;         // [P_dmax + 1] first row of every bucket
};

struct TreeRoot {                       // built on the host: how one root table is cut into slices
    uint32_t mask;                      // cube mask of the root
    uint32_t chunk0;                    // first CTA of this root
    uint32_t nslices;
    uint32_t H;                         // units per slice
    uint32_t nseg;                      // row segments per slice
    uint32_t q_stride;                  // buckets per joint value of the zone digits (P_dmax / P_zone)
    uint8_t z, npres, nabs, gmask, ng, pad[3]; // gmask: bytes of the packed row that hold an in-slice field (ng of them)
    uint8_t glist[8];                   // those bytes, ascending
    uint16_t fstride[32];               // stride of packed field f in the slice table (0: not an in-slice column)
    uint16_t pres_card[kTreeMaxZone];   // present zone digits, lowest first (slice index is mixed radix over them)
    uint32_t pres_weight[kTreeMaxZone]; //   weight of the digit inside the zone prefix index
    uint16_t abs_card[kTreeMaxZone];    // absent zone digits, lowest first (segment index is mixed radix over them)
    uint32_t abs_weight[kTreeMaxZone];
    uint32_t pres_magic[kTreeMaxZone];  // floor((2^32-1)/card) of the zone digits: fast_div instead of a hardware division
    uint32_t abs_magic[kTreeMaxZone];
};

// ---- bucketing ---------------------------------------------------------------------------------------------
__global__ void tree_key_kernel(BicData d, CandInfo ci_cube, int dmax, uint32_t *__restrict__ keys, uint32_t *__restrict__ hist) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.n) return;
    uint32_t key = 0;
    for (int b = ci_cube.c - 1; b >= ci_cube.c - dmax; b--) key = key * (uint32_t)ci_cube.card[b] + d.codes[(int64_t)ci_cube.var[b] * d.n_stride + r];
    keys[r] = key;
    atomicAdd(&hist[key], 1u);
}

// exclusive prefix sum of the bucket histogram (<= 2^20 + 1 entries) in three small kernels: per-tile sums (4096 entries per CTA),
// a one-CTA scan of the tile sums, per-tile rescan.  (cub::DeviceScan did this in round 1; the hot path carries no library kernel.)
constexpr int kScanTile = 4096, kScanThreads = 256, kScanPer = kScanTile / kScanThreads;
__global__ void __launch_bounds__(kScanThreads) bucket_scan_sums_kernel(const uint32_t *__restrict__ hist, uint32_t n, uint32_t *__restrict__ tile_sum) {
    __shared__ uint32_t red[kScanThreads / 32];
    const uint32_t base = blockIdx.x * kScanTile;
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < kScanPer; k++) { const uint32_t i = base + k * kScanThreads + threadIdx.x; if (i < n) s += hist[i]; }
    s = __reduce_add_sync(0xffffffffu, s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < kScanThreads / 32; w++) t += red[w]; tile_sum[blockIdx.x] = t; }
}
__global__ void __launch_bounds__(1024) bucket_scan_tiles_kernel(uint32_t *__restrict__ tile_sum, uint32_t ntiles) { // in place, exclusive; ntiles <= 1024
    __shared__ uint32_t part[1024];
    const uint32_t v = threadIdx.x < ntiles ? tile_sum[threadIdx.x] : 0;
    part[threadIdx.x] = v;
    __syncthreads();
    for (uint32_t o = 1; o < 1024; o <<= 1) {
        const uint32_t x = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
        __syncthreads();
        part[threadIdx.x] += x;
        __syncthreads();
    }
    if (threadIdx.x < ntiles) tile_sum[threadIdx.x] = part[threadIdx.x] - v;
}
__global__ void __launch_bounds__(kScanThreads) bucket_scan_final_kernel(const uint32_t *__restrict__ hist, uint32_t n, const uint32_t *__restrict__ tile_off,
                                                                         uint32_t *__restrict__ off) {
    __shared__ uint32_t wsum[kScanThreads / 32];
    const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanPer;   // every thread a contiguous run of 16 entries (64 bytes)
    uint32_t v[kScanPer], s = 0;
#pragma unroll
    for (int k = 0; k < kScanPer; k++) { v[k] = base + k < n ? hist[base + k] : 0; s += v[k]; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    uint32_t run = tile_off[blockIdx.x] + x - s;
    for (int w = 0; w < warp; w++) run += wsum[w];
#pragma unroll
    for (int k = 0; k < kScanPer; k++) { if (base + k < n) off[base + k] = run; run += v[k]; }
}

__global__ void tree_scatter_kernel(BicData d, CandInfo ci_cube, TreeVar tv, const uint32_t *__restrict__ keys, uint32_t *__restrict__ cursor,
                                    unsigned long long *__restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.n) return;
    unsigned long long w = (unsigned long long)d.codes[(int64_t)ci_cube.v * d.n_stride + r];
    for (int i = 0; i < ci_cube.c; i++) w |= (unsigned long long)d.codes[(int64_t)ci_cube.var[i] * d.n_stride + r] << ((i + 1) * tv.w);
    out[atomicAdd(&cursor[keys[r]], 1u)] = w; // order inside a bucket is arbitrary: counts do not depend on it
}

// exact warp sum of any int64 values whose sum fits int64, in three 32-bit REDUX operations: bits 0-23 and 24-47 as
// unsigned parts (32 of them sum below 2^29) and the arithmetic high part v >> 48 (|v >> 48| <= 2^15, 32 of them below 2^20).
// Two parts (24 low bits + v >> 24 in an int) would wrap once a lane or the warp reached 2^55, i.e. 2^32 nats of a BIC
// accumulator: one configuration of a 256-ary child holding 7.75e8 records of a slice is enough.
__device__ __forceinline__ long long warp_sum_ll_redux(long long v) {
    const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(v & 0xFFFFFF));
    const unsigned mid = __reduce_add_sync(0xffffffffu, (unsigned)((v >> 24) & 0xFFFFFF));
    const int hi = __reduce_add_sync(0xffffffffu, (int)(v >> 48));
    return (long long)(((unsigned long long)(long long)hi << 48) + ((unsigned long long)mid << 24) + lo);   // modulo 2^64
}

// ---- count the slice's rows.  The rows are `nseg` contiguous segments of the bucketed rows; they are walked as ONE
// concatenated range (segbeg/segoff in shared memory): a warp takes 128 consecutive positions per step, lane l the
// positions l, l+32, l+64, l+96, so every load is coalesced inside a segment and four loads are in flight per lane.
// NG = number of bytes of the packed word that hold an in-slice field (compile time: the look-ups unroll).
template <int NG, int NW>
__device__ __forceinline__ void tree_count(const unsigned long long *__restrict__ rows, const uint32_t *segbeg, const uint32_t *segoff, uint32_t nseg,
                                           uint32_t total, int *tab, const uint16_t *lut, const uint8_t *glist, int warp, int lane) {
    uint32_t gsh[NG];
#pragma unroll
    for (int i = 0; i < NG; i++) gsh[i] = 8u * glist[i];
    for (uint32_t base = (uint32_t)warp * 128u; base < total; base += NW * 128u) {
        const uint32_t p0 = base + lane;
        uint32_t seg = 0;
        if (nseg > 1 && p0 < total) { // last segment with segoff[seg] <= p0
            uint32_t lo = 0, hi = nseg - 1;
            while (lo < hi) {
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (segoff[mid] <= p0) lo = mid; else hi = mid - 1;
            }
            seg = lo;
        }
        unsigned long long w[4];
        bool ok[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const uint32_t p = p0 + 32u * u;
            ok[u] = p < total;
            if (ok[u]) {
                while (segoff[seg + 1] <= p) seg++; // also skips empty segments
                w[u] = __ldg(rows + segbeg[seg] + (p - segoff[seg]));
            }
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (ok[u]) {
                uint32_t idx = 0;
#pragma unroll
                for (int i = 0; i < NG; i++) idx += lut[(gsh[i] << 5) + ((uint32_t)(w[u] >> gsh[i]) & 255u)];
                atomicAdd(&tab[idx], 1);
            }
    }
}

// slices with more segments than the shared-memory segment tables hold (a root whose present digits all sit below many
// absent ones): warp `warp` owns segments warp, warp + W, ... and fetches the bounds of 32 of them at once
template <int NG, typename BoundsFn, int NW>
__device__ __forceinline__ void tree_count_fragmented(const unsigned long long *__restrict__ rows, BoundsFn seg_bounds, uint32_t nseg, int *tab,
                                                      const uint16_t *lut, const uint8_t *glist, int warp, int lane) {
    uint32_t gsh[NG];
#pragma unroll
    for (int i = 0; i < NG; i++) gsh[i] = 8u * glist[i];
    for (uint32_t j0 = 0; warp + NW * j0 < nseg; j0 += 32) {
        const uint32_t seg = warp + NW * (j0 + lane);
        uint32_t r0 = 0, r1 = 0;
        if (seg < nseg) seg_bounds(seg, r0, r1);
        const uint32_t left = (nseg - warp - NW * j0 + NW - 1) / NW;
        const int cnt = (int)min(32u, left);
        for (int k = 0; k < cnt; k++) {
            const uint32_t b0 = __shfl_sync(0xffffffffu, r0, k), b1 = __shfl_sync(0xffffffffu, r1, k);
            for (uint32_t g = b0 + lane; g < b1; g += 32) {
                const unsigned long long w = __ldg(rows + g);
                uint32_t idx = 0;
#pragma unroll
                for (int i = 0; i < NG; i++) idx += lut[(gsh[i] << 5) + ((uint32_t)(w >> gsh[i]) & 255u)];
                atomicAdd(&tab[idx], 1);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// bic_root_kernel: one CTA per (root, slice) histograms the slice in shared memory from the bucketed packed rows, then
//   * plain root (nchild == 0): the slice is written to its place in the root's dense global table;
//   * fused root (nchild == z > 0): the root is only an ancestor (layer K+1), so its table is never written.  The
//     CTA sums each run digit b < z out of the slice (a block-wide pass: the slice holds the whole run), scores
//     child b = root \ {b} on the fly and writes the child's slice to ITS global table unless b == 0 (nothing is
//     derived from a set that lacks bit 0).  This removes the write and the z reads of the largest layer of tables.
//     For b >= 1 a thread sums whole groups of card[0] consecutive child configurations (pre[b] is a multiple of card[0]),
//     so it also holds the counts of the child's leaf root \ {b, 0} and scores it (bic_kernels.cuh, "LEAF").
// ---------------------------------------------------------------------------------------------------------
constexpr int kRootMaxChild = 16;

struct CubeRoot {
    TreeRoot t;                              // slicing description; t.z = fused run (0 for a plain root)
    unsigned long long table_off;            // plain: the root's table in `tables` (int32 elements)
    unsigned long long child_off[kRootMaxChild];   // fused: child b's table in `child_tables`
    uint32_t child_acc[kRootMaxChild];       // and its accumulator
    uint32_t leaf_acc[kRootMaxChild];        // accumulator of the leaf root \ {b, 0} of child b >= 1
    uint32_t nchild;                         // fused: children drop bit b, bfirst <= b < nchild (== run length)
    uint16_t bfirst, score;                  // layers above K only hold sets with their lowest bits forced: the first droppable bit;
                                             // score bit 0: score the children, bit 1: score the leaves of children b >= 1
    uint32_t child16;                        // bit b: child b's table holds uint16 cells (bic_kernels.cuh, "16-bit tables")
    uint32_t pad16;
};

__global__ void root_map_kernel(const CubeRoot *__restrict__ roots, int nroots, uint32_t total, uint32_t *__restrict__ cta_root) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int lo = 0, hi = nroots - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (roots[mid].t.chunk0 <= i) lo = mid; else hi = mid - 1;
    }
    cta_root[i] = (uint32_t)lo;
}

template <int RV, int NW>
__global__ void __launch_bounds__(NW * 32, 2) bic_root_kernel(TreeVar tv, const CubeRoot *__restrict__ roots, const uint32_t *__restrict__ cta_root,
                                                                const long long *__restrict__ qlog, const long long *__restrict__ qcfg, int cfg_min,
                                                                int *__restrict__ tables, int *__restrict__ child_tables,
                                                                long long *__restrict__ acc_out, uint32_t table_budget /*cells*/, uint32_t seg_cap,
                                                                int *__restrict__ ovf_flag, int qn /*entries of qlog*/) {
    extern __shared__ __align__(16) int s_dyn[];              // [table_budget] slice table, then segbeg[seg_cap], segoff[seg_cap + 1]
    __shared__ CubeRoot cr;
    __shared__ uint16_t s_lut[8 * 256];
    __shared__ unsigned long long s_cacc[2][kRootMaxChild]; // per-child exact sums of this CTA: [0] the child b, [1] its leaf
    constexpr int kRootThreads = NW * 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rv = RV > 0 ? RV : tv.rv;
    {
        const uint32_t ri = cta_root[blockIdx.x];
        const uint32_t *src = reinterpret_cast<const uint32_t *>(roots + ri);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&cr);
        for (int i = tid; i < (int)(sizeof(CubeRoot) / 4); i += kRootThreads) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    const TreeRoot &rt = cr.t;
    const int z = rt.z;
    (void)qn;
    if (tid < 2 * kRootMaxChild) s_cacc[tid / kRootMaxChild][tid % kRootMaxChild] = 0;
    const uint32_t S0 = rt.H * (uint32_t)rv * tv.pre[z];
    const uint32_t si = blockIdx.x - rt.chunk0;
    {
        int4 *t4 = reinterpret_cast<int4 *>(s_dyn);
        for (uint32_t i = tid; i < (S0 + 3) / 4; i += kRootThreads) t4[i] = make_int4(0, 0, 0, 0);
        const int w = tv.w, fpb = 8 / w;
        const uint32_t fm = (1u << w) - 1u;
        for (int e = tid; e < 8 * 256; e += kRootThreads) {
            const int g = e >> 8;
            if (!((rt.gmask >> g) & 1)) continue;
            const uint32_t val = e & 255;
            uint32_t sum = 0;
            for (int k = 0; k < fpb; k++) sum += ((val >> (k * w)) & fm) * rt.fstride[g * fpb + k];
            s_lut[e] = (uint16_t)sum;
        }
    }
    // ---- count ----
    {
        uint32_t *s_segbeg = reinterpret_cast<uint32_t *>(s_dyn + table_budget);
        uint32_t *s_segoff = s_segbeg + seg_cap;
        const uint32_t nseg = rt.nseg;
        uint32_t qb = 0;
        {
            uint32_t rem = si;
            for (int a = 0; a < rt.npres; a++) {
                const uint32_t cb = rt.pres_card[a], qq = fast_div(rem, cb, rt.pres_magic[a]);
                qb += (rem - qq * cb) * rt.pres_weight[a];
                rem = qq;
            }
        }
        auto seg_bounds = [&](uint32_t seg, uint32_t &r0, uint32_t &r1) {
            uint32_t q = qb, rs = seg;
            for (int a = 0; a < rt.nabs; a++) {
                const uint32_t cb = rt.abs_card[a], qq = fast_div(rs, cb, rt.abs_magic[a]);
                q += (rs - qq * cb) * rt.abs_weight[a];
                rs = qq;
            }
            r0 = __ldg(&tv.prefix_off[(size_t)q * rt.q_stride]);
            r1 = __ldg(&tv.prefix_off[(size_t)(q + 1) * rt.q_stride]);
        };
        if (nseg <= seg_cap) {
            for (uint32_t seg = tid; seg < nseg; seg += kRootThreads) {
                uint32_t r0, r1;
                seg_bounds(seg, r0, r1);
                s_segbeg[seg] = r0;
                s_segoff[seg] = r1 - r0;
            }
            __syncthreads();
            if (warp == 0) {
                uint32_t carry = 0;
                for (uint32_t b0 = 0; b0 < nseg; b0 += 32) {
                    const uint32_t i = b0 + lane;
                    const uint32_t len = i < nseg ? s_segoff[i] : 0;
                    uint32_t x = len;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
                    if (i < nseg) s_segoff[i] = carry + x - len;
                    carry += __shfl_sync(0xffffffffu, x, 31);
                }
                if (lane == 0) s_segoff[nseg] = carry;
            }
            __syncthreads();
            const uint32_t total = s_segoff[nseg];
            switch (rt.ng) {
#define URLGPU_ROOT_COUNT(NG) case NG: tree_count<NG, NW>(tv.rows, s_segbeg, s_segoff, nseg, total, s_dyn, s_lut, rt.glist, warp, lane); break;
                URLGPU_ROOT_COUNT(1) URLGPU_ROOT_COUNT(2) URLGPU_ROOT_COUNT(3) URLGPU_ROOT_COUNT(4)
                URLGPU_ROOT_COUNT(5) URLGPU_ROOT_COUNT(6) URLGPU_ROOT_COUNT(7) URLGPU_ROOT_COUNT(8)
#undef URLGPU_ROOT_COUNT
            default: break;
            }
        } else {
            __syncthreads(); // the look-up tables
            switch (rt.ng) {
#define URLGPU_ROOT_COUNT(NG) case NG: tree_count_fragmented<NG, decltype(seg_bounds), NW>(tv.rows, seg_bounds, nseg, s_dyn, s_lut, rt.glist, warp, lane); break;
                URLGPU_ROOT_COUNT(1) URLGPU_ROOT_COUNT(2) URLGPU_ROOT_COUNT(3) URLGPU_ROOT_COUNT(4)
                URLGPU_ROOT_COUNT(5) URLGPU_ROOT_COUNT(6) URLGPU_ROOT_COUNT(7) URLGPU_ROOT_COUNT(8)
#undef URLGPU_ROOT_COUNT
            default: break;
            }
        }
    }
    __syncthreads();
    if (cr.nchild == 0) { // plain root: the slice goes to its place in the dense table (slicing digits are the most significant)
        const unsigned long long off = cr.table_off + (unsigned long long)si * S0;
        if ((S0 & 3u) == 0 && (off & 3ull) == 0) {
            int4 *dst = reinterpret_cast<int4 *>(tables + off);
            const int4 *src4 = reinterpret_cast<const int4 *>(s_dyn);
            for (uint32_t i = tid; i < S0 / 4; i += kRootThreads) dst[i] = src4[i];
        } else {
            int *dst = tables + off;
            for (uint32_t i = tid; i < S0; i += kRootThreads) dst[i] = s_dyn[i];
        }
        return;
    }
    // fused root: children b = bfirst .. z-1
    const uint32_t cfg_src = S0 / (uint32_t)rv;
    const bool score = cr.score & 1u;
    for (int b = cr.bfirst; b < z; b++) {
        const uint32_t r = tv.card[b], pre = tv.pre[b], magic = tv.magic[b];
        const uint32_t cfg_dst = fast_div(cfg_src, r, tv.cmagic[b]); // r divides the run product: exact
        const bool c16 = (cr.child16 >> b) & 1u;
        int *dst = child_tables + cr.child_off[b] + (c16 ? 0ull : (unsigned long long)si * ((unsigned long long)cfg_dst * rv));
        uint16_t *dst16 = reinterpret_cast<uint16_t *>(child_tables + cr.child_off[b]) + (unsigned long long)si * ((unsigned long long)cfg_dst * rv);
        const bool store = b > 0;
        const bool sleaf = b > 0 && (cr.score & 2u);
        const uint32_t r0 = b > 0 ? tv.card[0] : 1u;   // configurations per group
        bool ovf = false;
        long long acc = 0, lacc = 0;
        if constexpr (RV > 0) {
            // R = compile-time arity of the digit summed out (2, 3, 4), 0 = run-time loop; G = compile-time group size
            auto pass = [&](auto RC, auto GC) {
                constexpr int R = decltype(RC)::value, G = decltype(GC)::value, N = G * RV;
                for (uint32_t g = tid; g < cfg_dst / G; g += kRootThreads) {
                    const uint32_t j = g * G, hi = fast_div(j, pre, magic), lo = j - hi * pre;
                    const uint32_t p0 = lo + hi * r * pre;
                    int cnt[N];
                    load_cfg<N>(s_dyn + (size_t)p0 * RV, cnt);
                    if constexpr (R > 0) {
#pragma unroll
                        for (int a = 1; a < R; a++) {
                            int t[N];
                            load_cfg<N>(s_dyn + (size_t)(p0 + a * pre) * RV, t);
#pragma unroll
                            for (int k = 0; k < N; k++) cnt[k] += t[k];
                        }
                    } else {
#pragma unroll 2
                        for (uint32_t a = 1; a < r; a++) {
                            int t[N];
                            load_cfg<N>(s_dyn + (size_t)(p0 + a * pre) * RV, t);
#pragma unroll
                            for (int k = 0; k < N; k++) cnt[k] += t[k];
                        }
                    }
                    if (store) {
                        if (c16) ovf |= store_cfg16<N>(dst16 + (size_t)j * RV, cnt);
                        else store_cfg<N>(dst + (size_t)j * RV, cnt);
                    }
                    if (score)
#pragma unroll
                        for (int m = 0; m < G; m++) score_cfg<RV>(acc, cnt, m * RV, qlog, qcfg, cfg_min);
                    if (sleaf) {
                        int leaf[RV];
                        sum_group<RV, G>(cnt, leaf);
                        score_cfg<RV>(lacc, leaf, 0, qlog, qcfg, cfg_min);
                    }
                }
            };
            // r0 >= 3: the group's configurations one after another, each added into the leaf's counts in registers
            auto pass_any = [&]() {
                for (uint32_t g = tid; g < cfg_dst / r0; g += kRootThreads) {
                    const uint32_t jg = g * r0, hi = fast_div(jg, pre, magic), lo = jg - hi * pre;
                    const uint32_t pg = lo + hi * r * pre;
                    int leaf[RV] = {};
#pragma unroll 1
                    for (uint32_t m = 0; m < r0; m++) {
                        int cnt[RV];
                        load_cfg<RV>(s_dyn + (size_t)(pg + m) * RV, cnt);
#pragma unroll 2
                        for (uint32_t a = 1; a < r; a++) {
                            int t[RV];
                            load_cfg<RV>(s_dyn + (size_t)(pg + m + a * pre) * RV, t);
#pragma unroll
                            for (int k = 0; k < RV; k++) cnt[k] += t[k];
                        }
                        if (store) {
                            if (c16) ovf |= store_cfg16<RV>(dst16 + (size_t)(jg + m) * RV, cnt);
                            else store_cfg<RV>(dst + (size_t)(jg + m) * RV, cnt);
                        }
                        if (score) score_cfg<RV>(acc, cnt, 0, qlog, qcfg, cfg_min);
#pragma unroll
                        for (int k = 0; k < RV; k++) leaf[k] += cnt[k];
                    }
                    if (sleaf) score_cfg<RV>(lacc, leaf, 0, qlog, qcfg, cfg_min);
                }
            };
            auto by_arity = [&](auto GC) {
                switch (r) {
                case 2: pass(std::integral_constant<int, 2>{}, GC); break;
                case 3: pass(std::integral_constant<int, 3>{}, GC); break;
                case 4: pass(std::integral_constant<int, 4>{}, GC); break;
                default: pass(std::integral_constant<int, 0>{}, GC); break;
                }
            };
            if (r0 == 1) by_arity(std::integral_constant<int, 1>{});
            else if (r0 == 2) by_arity(std::integral_constant<int, 2>{});
            else pass_any();
        } else {
            for (uint32_t g = tid; g < cfg_dst / r0; g += kRootThreads) {
                const uint32_t jg = g * r0, hi = fast_div(jg, pre, magic), lo = jg - hi * pre;
                const uint32_t pg = lo + hi * r * pre;
                for (uint32_t m = 0; m < r0; m++) {
                    const uint32_t j = jg + m, p0 = pg + m;
                    int nij = 0;
                    for (int k = 0; k < rv; k++) {
                        int cnt = 0;
                        for (uint32_t a = 0; a < r; a++) cnt += s_dyn[(size_t)(p0 + a * pre) * rv + k];
                        if (store) {
                            if (c16) { dst16[(size_t)j * rv + k] = (uint16_t)min(cnt, 65535); ovf |= cnt > 65535; }
                            else dst[(size_t)j * rv + k] = cnt;
                        }
                        nij += cnt;
                        if (score && cnt > 1) acc += __ldg(&qlog[cnt]);
                    }
                    if (score && nij > cfg_min) acc -= __ldg(&qcfg[nij]);
                }
                if (sleaf) { // the leaf's counts: the group's cells summed again from shared memory
                    int nl = 0;
                    for (int k = 0; k < rv; k++) {
                        int cnt = 0;
                        for (uint32_t m = 0; m < r0; m++)
                            for (uint32_t a = 0; a < r; a++) cnt += s_dyn[(size_t)(pg + m + a * pre) * rv + k];
                        nl += cnt;
                        if (cnt > 1) lacc += __ldg(&qlog[cnt]);
                    }
                    if (nl > cfg_min) lacc -= __ldg(&qcfg[nl]);
                }
            }
        }
        if (ovf) *ovf_flag = 1;
        // no barrier between children: every warp adds its exact partial sums to the child's shared accumulators
        if (score) {
            acc = warp_sum_ll_redux(acc);
            if (lane == 0 && acc != 0) atomicAdd(&s_cacc[0][b], (unsigned long long)acc);
        }
        if (sleaf) {
            lacc = warp_sum_ll_redux(lacc);
            if (lane == 0 && lacc != 0) atomicAdd(&s_cacc[1][b], (unsigned long long)lacc);
        }
    }
    if (cr.score) {
        __syncthreads();
        if (tid >= (int)cr.bfirst && tid < z) {
            const unsigned long long a = s_cacc[0][tid], la = s_cacc[1][tid];
            if (score && a != 0) atomicAdd(reinterpret_cast<unsigned long long *>(&acc_out[cr.child_acc[tid]]), a);
            if (la != 0) atomicAdd(reinterpret_cast<unsigned long long *>(&acc_out[cr.leaf_acc[tid]]), la);
        }
    }
}

} // namespace urlgpu
