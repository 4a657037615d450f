// common.cuh — shared device helpers for the urlgpu kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace urlgpu {

// "not stored / not scored" marker inside dense score tables: a quiet NaN with a payload no arithmetic produces.
__host__ __device__ constexpr uint32_t kSentinelBits = 0x7fc0beefu;
__device__ __forceinline__ float sentinel() { return __uint_as_float(kSentinelBits); }
__device__ __forceinline__ bool is_sentinel(float x) { return __float_as_uint(x) == kSentinelBits; }

constexpr int kMaxDenseCand = 30;   // dense-by-compact-mask tables: 2^c floats
constexpr int kMaxCols = 32;        // columns of one contingency table (|S|+1)

// One entry of a caller's list of parent sets (urlgpu_score_sets): the child, its parent count and the first of its parents
// in a separate array of variable indices (ascending per entry).  Shared by K1 (ListSets) and K3 (cbic_sets_kernel).
struct ListEntry {
    int v;
    int k;
    uint32_t off;
};

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum of int64 (integer: order independent, so any tree is deterministic)
__device__ __forceinline__ long long block_sum_ll(long long v, long long *smem32) {
    v = warp_sum_ll(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) smem32[warp] = v;
    __syncthreads();
    const int nw = (blockDim.x + 31) >> 5;
    v = (threadIdx.x < nw) ? smem32[threadIdx.x] : 0;
    if (warp == 0) v = warp_sum_ll(v);
    return v; // valid in thread 0
}

// 128-bit read-only streaming load (rows are read once per set; keep them out of L1)
__device__ __forceinline__ uint4 ld_stream_u4(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// floor(j / d) by multiplication: m = floor((2^32-1) / d) (d >= 2), at most one correction step
__device__ __forceinline__ uint32_t fast_div(uint32_t j, uint32_t d, uint32_t m) {
    if (d == 1) return j;
    uint32_t q = __umulhi(j, m);
    if (j - q * d >= d) q++;
    return q;
}

__global__ void fill_u32_kernel(uint32_t *__restrict__ t, uint64_t n, uint32_t v) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) t[i] = v;
}

} // namespace urlgpu
