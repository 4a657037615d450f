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
//   * fused root (nchild == z > 0): the root is only an ancestor (layer K+1 or K+2), so its table is never written.  The
//     CTA sums each run digit b < z out of the slice (a block-wide pass: the slice holds the whole run) and scores child
//     T = root \ {b} on the fly.  This removes the write and the z reads of the largest layer of tables.  For b >= 1 a thread
//     sums whole groups of card[0] consecutive child configurations (pre[b] is a multiple of card[0]), so it also holds the
//     counts of T \ {0} and scores it (bic_kernels.cuh, "GROUPS").  T is written iff b >= 2: the derive kernel reads it for
//     T \ {1} (and T \ {0,1}), which stay out of the root kernel, whose two CTAs per SM score less efficiently than the
//     derive kernel's six; T = root \ {1} has no child left to derive and is not written.  The host sets which sets a pass
//     scores (CubeRoot::flags): above layer K only sets whose lowest bits are forced belong to the family.
// ---------------------------------------------------------------------------------------------------------
constexpr int kRootMaxChild = 16;

struct CubeRoot {
    TreeRoot t;                              // slicing description; t.z = fused run (0 for a plain root)
    unsigned long long table_off;            // plain: the root's table in `tables` (int32 elements)
    unsigned long long child_off[kRootMaxChild];   // fused: table of pass b's child root \ {b} in `child_tables` (b >= 2)
    uint32_t acc[kRootMaxChild][2];          // accumulators of pass b's sets T = root \ {b} and T \ {0}
    uint32_t nchild;                         // fused: passes b < nchild (== run length)
    uint32_t child16;                        // bit b: child b's table holds uint16 cells (bic_kernels.cuh, "16-bit tables")
    uint8_t flags[kRootMaxChild];            // pass b: kCubeStore | kCubeScore* (bic_kernels.cuh); 0: no pass b
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
    __shared__ unsigned long long s_cacc[kRootMaxChild][2]; // exact sums of this CTA: pass b's T and T \ {0}
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
    if (tid < 2 * kRootMaxChild) s_cacc[tid >> 1][tid & 1] = 0;
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
    // fused root: passes b < z (see the kernel's header)
    const uint32_t cfg_src = S0 / (uint32_t)rv;
    for (int b = 0; b < z; b++) {
        const uint32_t flags = cr.flags[b];
        if (!flags) continue;
        const uint32_t r = tv.card[b], pre = tv.pre[b], magic = tv.magic[b];
        const uint32_t cfg_dst = fast_div(cfg_src, r, tv.cmagic[b]); // r divides the run product: exact
        const uint32_t G = b == 0 ? 1u : tv.card[0];   // configurations per group
        const bool c16 = (cr.child16 >> b) & 1u;
        int *dst = child_tables + cr.child_off[b] + (c16 ? 0ull : (unsigned long long)si * ((unsigned long long)cfg_dst * rv));
        uint16_t *dst16 = reinterpret_cast<uint16_t *>(child_tables + cr.child_off[b]) + (unsigned long long)si * ((unsigned long long)cfg_dst * rv);
        const bool store = flags & kCubeStore;
        bool ovf = false;
        long long acc[2] = {0, 0};
        auto add = [&](int q, long long v) { if (q < 2) acc[q] += v; };   // passes score T and T \ {0} only
        if constexpr (RV > 0) {
            // R = compile-time arity of the digit summed out (2, 3, 4), 0 = run-time loop; G0 = compile-time group size
            auto pass = [&](auto RC, auto G0c) {
                constexpr int R = decltype(RC)::value, G0 = decltype(G0c)::value, N = G0 * RV;
                for (uint32_t g = tid; g < cfg_dst / G0; g += kRootThreads) {
                    const uint32_t j = g * G0, hi = fast_div(j, pre, magic), lo = j - hi * pre;
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
                    score_group<RV, G0, 1>(cnt, flags, add, qlog, qcfg, cfg_min);
                }
            };
            // any other group shape: the group's configurations one after another
            auto pass_any = [&]() {
                for (uint32_t g = tid; g < cfg_dst / G; g += kRootThreads) {
                    const uint32_t jg = g * G, hi = fast_div(jg, pre, magic), lo = jg - hi * pre;
                    const uint32_t pg = lo + hi * r * pre;
                    auto cfg = [&](uint32_t m, int (&cnt)[RV]) {
                        load_cfg<RV>(s_dyn + (size_t)(pg + m) * RV, cnt);
#pragma unroll 2
                        for (uint32_t a = 1; a < r; a++) {
                            int t[RV];
                            load_cfg<RV>(s_dyn + (size_t)(pg + m + a * pre) * RV, t);
#pragma unroll
                            for (int k = 0; k < RV; k++) cnt[k] += t[k];
                        }
                    };
                    auto put = [&](uint32_t m, const int (&cnt)[RV]) {
                        if (!store) return;
                        if (c16) ovf |= store_cfg16<RV>(dst16 + (size_t)(jg + m) * RV, cnt);
                        else store_cfg<RV>(dst + (size_t)(jg + m) * RV, cnt);
                    };
                    score_group_any<RV>(G, 1u, cfg, put, flags, add, qlog, qcfg, cfg_min);
                }
            };
            auto by_arity = [&](auto G0c) {
                switch (r) {
                case 2: pass(std::integral_constant<int, 2>{}, G0c); break;
                case 3: pass(std::integral_constant<int, 3>{}, G0c); break;
                case 4: pass(std::integral_constant<int, 4>{}, G0c); break;
                default: pass(std::integral_constant<int, 0>{}, G0c); break;
                }
            };
            if (G == 1) by_arity(std::integral_constant<int, 1>{});
            else if (G == 2) by_arity(std::integral_constant<int, 2>{});
            else pass_any();
        } else {
            for (uint32_t g = tid; g < cfg_dst / G; g += kRootThreads) {
                const uint32_t jg = g * G, hi = fast_div(jg, pre, magic), lo = jg - hi * pre;
                const uint32_t pg = lo + hi * r * pre;
                auto cell = [&](uint32_t m, int k) {   // marginals sum the group's cells again from shared memory
                    int cnt = 0;
                    for (uint32_t a = 0; a < r; a++) cnt += s_dyn[(size_t)(pg + m + a * pre) * rv + k];
                    return cnt;
                };
                for (uint32_t m = 0; m < G; m++) {
                    const uint32_t j = jg + m;
                    int nij = 0;
                    for (int k = 0; k < rv; k++) {
                        const int cnt = cell(m, k);
                        if (store) {
                            if (c16) { dst16[(size_t)j * rv + k] = (uint16_t)min(cnt, 65535); ovf |= cnt > 65535; }
                            else dst[(size_t)j * rv + k] = cnt;
                        }
                        nij += cnt;
                        if ((flags & kCubeScoreChild) && cnt > 1) acc[0] += __ldg(&qlog[cnt]);
                    }
                    if ((flags & kCubeScoreChild) && nij > cfg_min) acc[0] -= __ldg(&qcfg[nij]);
                }
                score_marginals(cell, rv, G, 1u, flags, add, qlog, qcfg, cfg_min);
            }
        }
        if (ovf) *ovf_flag = 1;
        // no barrier between passes: every warp adds its exact partial sums to the pass's shared accumulators
#pragma unroll
        for (int q = 0; q < 2; q++)
            if (flags & (kCubeScoreChild << q)) {
                const long long v = warp_sum_ll_redux(acc[q]);
                if (lane == 0 && v != 0) atomicAdd(&s_cacc[b][q], (unsigned long long)v);
            }
    }
    __syncthreads();
    if (tid < 2 * z) {
        const int b = tid >> 1, q = tid & 1;
        const unsigned long long a = s_cacc[b][q];
        if ((cr.flags[b] & (kCubeScoreChild << q)) && a != 0) atomicAdd(reinterpret_cast<unsigned long long *>(&acc_out[cr.acc[b][q]]), a);
    }
}

} // namespace urlgpu
