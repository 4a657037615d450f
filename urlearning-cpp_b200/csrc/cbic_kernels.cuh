// cbic_kernels.cuh — K2 (standardise + FP64 Gram), K3 (per-set residual variance + score), K4 (acceptance DP)
// for the continuous "cBIC" score (sm_100a).
//
// Replaces BIC_OLS_Function's constructor (scoring_function/BIC_OLS.cpp:30-123), calculateScoreAndBeta
// (:277-389, incl. the mlpack LinearRegression Train/ComputeError it calls) and calculateScore +
// find_best_subset_score (:125-276) of the reference.
//
// The reference refits an OLS on n rows for every parent set (O(k^2 n) per set).  Here the data is reduced ONCE
// to the Gram matrix G = Z^T Z of the standardised columns; the residual sum of squares of regressing z_v on
// z_S is the Schur complement  RSS = G_vv - g_Sv^T G_SS^-1 g_Sv.  Candidate sets are walked as a binary
// decision tree over the compact candidate bits (highest bit first); including a candidate is one symmetric
// rank-1 "sweep" of the Schur complement restricted to the still-undecided candidates, so a set whose lowest
// member is bit j costs j(j+1)/2 FMAs and on average ~4 FMAs per set, instead of a k^3/3 factorisation.
#pragma once
#include "common.cuh"
#include "log_table.cuh"

namespace urlgpu {

// ------------------------------------------------------------------------------------------------ K2
// Fixed-order reductions: every partial is produced by a fixed (block, thread) -> row mapping and the partials
// are combined sequentially, so the result does not depend on scheduling.

constexpr int kRedBlocks = 256;
constexpr int kRedThreads = 256;

// out[col*kRedBlocks + b] = sum over this block's rows of f(x - shift[col])   (mode 0: x-shift, mode 1: (x-shift)^2)
__global__ void col_partial_kernel(const double *__restrict__ x, int64_t n, int64_t stride, const double *__restrict__ shift, int mode,
                                   double *__restrict__ out) {
    __shared__ double sh[kRedThreads];
    const int col = blockIdx.y;
    const double s = shift ? shift[col] : 0.0;
    const double *xc = x + (int64_t)col * stride;
    double acc = 0;
    for (int64_t r = (int64_t)blockIdx.x * kRedThreads + threadIdx.x; r < n; r += (int64_t)kRedBlocks * kRedThreads) {
        const double t = xc[r] - s;
        acc += mode ? t * t : t;
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = kRedThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[col * kRedBlocks + blockIdx.x] = sh[0];
}

// sequential combine of the kRedBlocks partials of each column
__global__ void col_combine_kernel(const double *__restrict__ partial, int p, double *__restrict__ out) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= p) return;
    double acc = 0;
    for (int b = 0; b < kRedBlocks; b++) acc += partial[col * kRedBlocks + b];
    out[col] = acc;
}

// mean = sum/n ; after centring: m2 = mean of centred column, var = (acc2 - acc3^2/n)/(n-1) (Armadillo op_var), dev = sqrt(var)
__global__ void mean_kernel(const double *__restrict__ sum, int p, double n, double *__restrict__ mean) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col < p) mean[col] = sum[col] / n;
}
__global__ void dev_kernel(const double *__restrict__ acc2, const double *__restrict__ acc3, int p, double n, double *__restrict__ dev) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col < p) dev[col] = sqrt((acc2[col] - acc3[col] * acc3[col] / n) / (n - 1.0));
}
// z = (x - mean) / dev   (BIC_OLS.cpp:76-77)
// x has row pitch x_stride; z has row pitch z_stride >= n and is zero beyond n (the Gram kernel streams whole chunks)
__global__ void standardise_kernel(const double *__restrict__ x, int64_t n, int64_t x_stride, const double *__restrict__ mean,
                                   const double *__restrict__ dev, double *__restrict__ z, int64_t z_stride) {
    const int col = blockIdx.y;
    const double m = mean[col], d = dev[col];
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < z_stride; r += (int64_t)gridDim.x * blockDim.x)
        z[(int64_t)col * z_stride + r] = r < n ? __ddiv_rn(x[(int64_t)col * x_stride + r] - m, d) : 0.0;
}

// Gram partials on the FP64 tensor pipe (DMMA): G = Z^T Z is the only dense contraction of the path.
// tcgen05/wgmma have no f64 kind, so the math is mma.sync.m8n8k4.f64 (SASS DMMA); the operand stream is TMA:
//   * Z is variable-major ([p][n_stride], records contiguous, n_stride a multiple of kGramKC with zeros beyond n).
//   * A CTA owns one 64x64 tile pair (ta <= tb) of G for one row slice.  A producer warp streams the slice in chunks of
//     kGramKC records: per chunk one bulk copy (cp.async.bulk, 256 B) per variable row of the A and B tiles into a
//     kGramStages-deep ring of padded shared-memory tiles, completion on an mbarrier (expect_tx); four consumer warps
//     (one 32x32 sub-tile each: 4x4 MMA tiles, 32 FP64 accumulators per lane) wait on the stage's full barrier, read
//     their fragments from shared memory (row pitch 36 doubles: the 8 rows x 4 records of a fragment fall into 32 distinct
//     8-byte bank pairs) and hand the stage back through an empty barrier.
//   * lane l holds Z[a0 + l/4][r + l%4] for A (row major, 8 variables x 4 records) and Z[b0 + l/4][r + l%4] for B (column
//     major): both operands are the same layout, which is why no transposition is ever needed.
// Every (tile pair, slice) partial is produced by one warp in ascending record order and the slices are combined in fixed
// order: the Gram is bit-identical for any scheduling.  Grid = (tile pair, row slice) with the tile pair fastest, so the
// CTAs running together stream the same rows and Z comes from HBM once (L2 serves the p/64-fold reuse).
constexpr int kGramTile = 64;
constexpr int kGramKC = 32;                       // records per chunk: 256-byte bulk copies
constexpr int kGramPitch = kGramKC + 4;           // doubles per shared-memory row
constexpr int kGramStages = 3;
constexpr int kGramConsumers = 4;                 // warps
constexpr int kGramThreads = (kGramConsumers + 1) * 32;
constexpr size_t kGramStageDoubles = (size_t)2 * kGramTile * kGramPitch;
constexpr size_t kGramSmemBytes = kGramStages * kGramStageDoubles * sizeof(double) + 2 * kGramStages * sizeof(unsigned long long);

__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS UBLKCP); 16-byte aligned, size % 16 == 0
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__global__ void __launch_bounds__(kGramThreads) gram_partial_kernel(const double *__restrict__ z, int64_t n_stride, int p, int64_t rows_per_slice, int tiles,
                                                                   double *__restrict__ partial /*[slices][p][p]*/) {
    extern __shared__ __align__(128) unsigned char gram_smem[];
    double *tilebuf = reinterpret_cast<double *>(gram_smem);
    unsigned long long *full = reinterpret_cast<unsigned long long *>(gram_smem + kGramStages * kGramStageDoubles * sizeof(double));
    unsigned long long *empty = full + kGramStages;
    // blockIdx.x enumerates the upper-triangular tile pairs (ta <= tb)
    int ta = 0, rem = blockIdx.x;
    while (rem >= tiles - ta) { rem -= tiles - ta; ta++; }
    const int tb = ta + rem;
    const bool diag = ta == tb;
    const int slice = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t s0 = (int64_t)slice * rows_per_slice;           // multiples of kGramKC
    const int64_t s1 = min(s0 + rows_per_slice, n_stride);
    const int nchunks = (int)((s1 - s0) / kGramKC);
    const int rows_a = min(kGramTile, p - ta * kGramTile), rows_b = diag ? 0 : min(kGramTile, p - tb * kGramTile);
    // rows of the tiles beyond p are never copied: zero them once in every stage
    for (int st = 0; st < kGramStages; st++) {
        double *A = tilebuf + st * kGramStageDoubles, *B = A + kGramTile * kGramPitch;
        for (int i = threadIdx.x; i < (kGramTile - rows_a) * kGramPitch; i += kGramThreads) A[rows_a * kGramPitch + i] = 0.0;
        if (!diag) for (int i = threadIdx.x; i < (kGramTile - rows_b) * kGramPitch; i += kGramThreads) B[rows_b * kGramPitch + i] = 0.0;
    }
    if (threadIdx.x == 0) {
        for (int st = 0; st < kGramStages; st++) { mbar_init(&full[st], 1); mbar_init(&empty[st], kGramConsumers); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (warp == kGramConsumers) { // ---- producer warp: lane l copies rows l, l + 32 of A and of B
        const uint32_t chunk_bytes = (uint32_t)((rows_a + rows_b) * kGramKC * sizeof(double));
        for (int c = 0; c < nchunks; c++) {
            const int st = c % kGramStages;
            if (c >= kGramStages) mbar_wait(&empty[st], ((c / kGramStages) - 1) & 1);
            double *A = tilebuf + st * kGramStageDoubles, *B = A + kGramTile * kGramPitch;
            if (lane == 0) mbar_arrive_expect_tx(&full[st], chunk_bytes);
            __syncwarp();
            const int64_t r = s0 + (int64_t)c * kGramKC;
            for (int row = lane; row < rows_a; row += 32)
                bulk_g2s(A + row * kGramPitch, z + (int64_t)(ta * kGramTile + row) * n_stride + r, kGramKC * sizeof(double), &full[st]);
            for (int row = lane; row < rows_b; row += 32)
                bulk_g2s(B + row * kGramPitch, z + (int64_t)(tb * kGramTile + row) * n_stride + r, kGramKC * sizeof(double), &full[st]);
        }
        return;
    }
    // ---- consumer warps: warp w owns rows [32 (w/2), +32) of the A tile and columns [32 (w%2), +32) of the B tile
    const int wa = (warp >> 1) * 32, wb = (warp & 1) * 32;
    const int vrow = lane >> 2, kk = lane & 3;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int c = 0; c < nchunks; c++) {
        const int st = c % kGramStages;
        mbar_wait(&full[st], (c / kGramStages) & 1);
        const double *A = tilebuf + st * kGramStageDoubles;
        const double *B = diag ? A : A + kGramTile * kGramPitch;
        const double *pa = A + (wa + vrow) * kGramPitch + kk, *pb = B + (wb + vrow) * kGramPitch + kk;
#pragma unroll
        for (int k = 0; k < kGramKC; k += 4) {
            double fa[4], fb[4];
#pragma unroll
            for (int t = 0; t < 4; t++) { fa[t] = pa[t * 8 * kGramPitch + k]; fb[t] = pb[t * 8 * kGramPitch + k]; }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) dmma_8x8x4(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);
    }
    // C fragment: lane holds C[row = lane/4][col = (lane%4)*2 + {0,1}] of each 8x8 tile
    double *out = partial + (int64_t)slice * p * p;
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int a = ta * kGramTile + wa + i * 8 + vrow, b = tb * kGramTile + wb + j * 8 + kk * 2;
            if (a < p && b < p) out[(int64_t)a * p + b] = acc[i][j][0];
            if (a < p && b + 1 < p) out[(int64_t)a * p + b + 1] = acc[i][j][1];
        }
}
// G[a][b] = sum over slices in slice order (fixed order); mirror to the lower triangle
__global__ void gram_combine_kernel(const double *__restrict__ partial, int p, int slices, double *__restrict__ g) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p * p) return;
    const int a = idx / p, b = idx % p;
    if (b < a) return;
    if ((a / kGramTile) > (b / kGramTile)) return;
    double acc = 0;
    for (int s = 0; s < slices; s++) acc += partial[(int64_t)s * p * p + a * p + b];
    g[a * p + b] = acc;
    g[b * p + a] = acc;
}

// FP64 peak probes (urlgpu_probe_fp64): the denominators of the K2/K3 roofline fractions are MEASURED on the device the
// bench runs on, not taken from a data sheet.  dfma: 8 independent FMA chains per thread; dmma: 8 independent
// m8n8k4 accumulator tiles per warp.  Operands stay in registers, so the result is the issue rate of the FP64 pipes.
__global__ void __launch_bounds__(256) probe_dfma_kernel(double *out, int iters, double a, double b) {
    double x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = (double)(threadIdx.x + i);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) x[i] = fma(x[i], a, b);
    }
    double sum = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) sum += x[i];
    if (sum == 123.456) out[0] = sum; // never true for the arguments used: keeps the chains alive
}
__global__ void __launch_bounds__(256) probe_dmma_kernel(double *out, int iters, double a, double b) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; i++) { c[i][0] = (double)threadIdx.x; c[i][1] = (double)i; }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) dmma_8x8x4(c[i][0], c[i][1], a, b);
    }
    double sum = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) sum += c[i][0] + c[i][1];
    if (sum == 123.456) out[0] = sum;
}

// ------------------------------------------------------------------------------------------------ K3

struct CbicParams {
    int max_parents;
    double n;         // row count (num_err, BIC_OLS.cpp:348)
    double lam_logn;  // lambda*log(n)  (:366, evaluated left to right)
    double log_n;     // log(n)
    // Pivot guard (SURVEY Q13): a candidate whose Schur pivot has dropped to <= piv_tol (1e-10 * the largest diagonal entry of
    // the candidate Gram) is a linear combination of the candidates already swept.  Its sweep is skipped (inv = 0 turns every
    // FMA of the sweep into the identity), so RSS equals the least-squares RSS without that column — what arma::solve's
    // rank-deficient fallback gives the reference (BIC_OLS.cpp:313-315) — instead of Inf/NaN; the penalty still counts it.
    double piv_tol;
};
// 1/d for a positive, normal pivot: hardware seed (MUFU.RCP64H) + two Newton steps = full double precision (<= 1 ulp), without
// the special-case slow path of the IEEE division.  Every cBIC kernel divides through this function, so all of them
// (dense DFS / tree, rank space, per-set) see the same bits.
__device__ __forceinline__ double pivot_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(fma(-d, r, 1.0), r, r);
    r = fma(fma(-d, r, 1.0), r, r);
    return r;
}
__device__ __forceinline__ double guarded_inv(double d, double tol) { return d > tol ? pivot_rcp(d) : 0.0; }

// ln(x) in FP64 for the score n*ln(RSS/n): x = 2^e * m, m in [1, 2) falls into one of 128 intervals with centre c_i;
// ln(m) = -ln(1/c_i) + ln1p(r), r = m * (1/c_i) - 1 (one FMA, |r| <= 2^-8), ln1p by a degree-5 polynomial (truncation
// 6e-16 absolute).  Accuracy ~2e-16 relative to |ln x| >= 1 (measured against libm over 1e-300..1e300), at a third of the
// instructions of the library routine, which K3 — instruction-issue bound at one logarithm per parent set — is made of.
// Zero, negative, subnormal, infinite and NaN arguments go to the library routine (same results as before for those).
__device__ __forceinline__ double cbic_log(double x) {
    const long long ix = __double_as_longlong(x);
    const int hi = (int)(ix >> 32);
    if (hi < 0x00100000 || hi >= 0x7ff00000) return log(x);
    const int e = (hi >> 20) - 1023;
    const double2 t = __ldg(&kLogTable[(hi >> 13) & 0x7f]);
    const double m = __longlong_as_double((ix & 0x000fffffffffffffLL) | 0x3ff0000000000000LL);
    const double r = fma(m, t.x, -1.0);
    double q = fma(r, 0.2, -0.25);
    q = fma(q, r, 0.33333333333333331);
    q = fma(q, r, -0.5);
    return fma((double)e, 0.69314718055994529, t.y + fma(r * r, q, r));
}

// packed lower-triangular index, element order (v, cand0, cand1, ...)
__host__ __device__ __forceinline__ int tri(int a, int b) { return a * (a + 1) / 2 + b; }

// One warp sweeps candidate `piv` out of the packed matrix A over (v, cand_0 .. cand_{piv-1}, ...) in shared memory:
// the rows above the pivot are updated in place, the lanes striding over each row.
__device__ __forceinline__ void cbic_warp_sweep(double *A, int piv, double piv_tol, int lane) {
    const double inv = guarded_inv(A[tri(piv, piv)], piv_tol);
    for (int a = 0; a < piv; a++) {
        const double f = -A[tri(piv, a)] * inv;
        for (int b = lane; b <= a; b += 32) A[tri(a, b)] = fma(f, A[tri(piv, b)], A[tri(a, b)]);
    }
    __syncwarp();
}

// Level A: one warp per prefix (the high candidate bits).  Starting from a matrix over (v, cand_0 .. cand_{c_in-1}), walk
// the `bits` highest candidates from the top: an included one is swept out (Schur complement), either way it is then
// dropped.  The prefix index p = (q << bits) | local: q selects the input matrix (in_stride = 0: one shared matrix),
// bit (bits-1) of `local` is candidate c_in-1.  Run in two stages (host: 9 + 9 bits at c = 29) so the sweeps of the top
// bits are shared by the 2^bits prefixes below them; every element still sees the same sequence of FMAs.
// Output: the remaining matrix over (v, cand_0 .. cand_{c_in-bits-1}), either contiguous per prefix (transposed == 0:
// out[p * outsz + e], the next stage's input) or entry-major (transposed == 1: out[e * n_out + p], what the DFS reads).
__global__ void cbic_roots_kernel(const double *__restrict__ in, size_t in_stride, int c_in, int bits, int max_parents, uint32_t n_out,
                                  double *__restrict__ out, int transposed, double piv_tol) {
    extern __shared__ double smat[]; // [warps][tri size]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t P = blockIdx.x * (blockDim.x >> 5) + warp;
    const int tsz = (c_in + 1) * (c_in + 2) / 2;
    double *A = smat + warp * tsz;
    if (P >= n_out) return;
    if (__popc(P) > max_parents) return; // whole subtree unscored
    const double *src = in + (size_t)(P >> bits) * in_stride;
    for (int e = lane; e < tsz; e += 32) A[e] = src[e];
    __syncwarp();
    for (int t = bits - 1; t >= 0; t--)
        if ((P >> t) & 1) cbic_warp_sweep(A, c_in - bits + t + 1 /*position of the candidate in (v, c0, c1, ...)*/, piv_tol, lane);
    const int c_out = c_in - bits;
    const int outsz = (c_out + 1) * (c_out + 2) / 2;
    if (transposed) { for (int e = lane; e < outsz; e += 32) out[(size_t)e * n_out + P] = A[e]; }
    else { for (int e = lane; e < outsz; e += 32) out[(size_t)P * outsz + e] = A[e]; }
}

// the_score of one set from its RSS (BIC_OLS.cpp:302-305,366): k == 0 -> 0.0.
// n*log(RSS/n) is evaluated as n*(log(RSS) - log(n)) with log(n) hoisted: one FP64 division less per set.
__device__ __forceinline__ double cbic_the_score64(double rss, int k, const CbicParams &prm) {
    if (k == 0) return 0.0;
    return prm.n * (cbic_log(rss) - prm.log_n) + prm.lam_logn * (double)k;
}

// Listed parent sets (urlgpu_score_sets; urlgpu_score_one is a list of one): one warp per set gathers the packed sub-Gram over
// (v, parents ascending) from the p x p Gram into its slice of shared memory — the order of cbic_sub_gram — and sweeps every
// parent out, highest first: the sequence of FMAs the family kernels apply to this set.  O(k^3) work, no 2^k tables.  One
// launch covers the sets of one size k; `work` lists their keys (positions in the caller's list), the outputs go to the key:
// the_score in FP64 and the float score -the_score.
__global__ void cbic_sets_kernel(const double *__restrict__ gram, int p, const ListEntry *__restrict__ ent, const int *__restrict__ par,
                                 const uint32_t *__restrict__ work, uint32_t count, int k, CbicParams prm, float *__restrict__ scores,
                                 double *__restrict__ the_score) {
    extern __shared__ double smat[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t i = blockIdx.x * (blockDim.x >> 5) + warp;
    if (i >= count) return;
    const uint32_t key = work[i];
    const ListEntry e = ent[key];
    double *A = smat + (size_t)warp * ((k + 1) * (k + 2) / 2);
    for (int a = 0; a <= k; a++) {
        const double *row = gram + (size_t)(a == 0 ? e.v : par[e.off + a - 1]) * p;
        for (int b = lane; b <= a; b += 32) A[tri(a, b)] = row[b == 0 ? e.v : par[e.off + b - 1]];
    }
    __syncwarp();
    for (int piv = k; piv >= 1; piv--) cbic_warp_sweep(A, piv, prm.piv_tol, lane);
    if (lane == 0) {
        const double ts = cbic_the_score64(A[0], k, prm);
        the_score[key] = ts;
        scores[key] = -__double2float_rn(ts); // BIC_OLS.cpp:223,245,275
    }
}

// Level B: template-recursive DFS over the J low candidate bits.  A has (j+1)(j+2)/2 packed entries over
// (v, cand0..cand_{j-1}).  Low masks are emitted in ascending order (exclude branch first).  Every level is inlined, so
// all matrices live in registers; the scores of the 16 sets below a level-4 node are collected in registers and written
// together.
template <int j>
__device__ __forceinline__ void cbic_sweep(const double *A, double *B, double piv_tol) {
    const double inv = guarded_inv(A[tri(j, j)], piv_tol);
#pragma unroll
    for (int a = 0; a < j; a++) {
        const double f = -A[tri(j, a)] * inv;
#pragma unroll
        for (int b = 0; b <= a; b++) B[tri(a, b)] = fma(f, A[tri(j, b)], A[tri(a, b)]);
    }
}

// bottom three levels: LOCAL = the low mask bits decided so far (compile time -> buf[] stays in registers)
constexpr int kBufLevel = 4;             // the scores of the 2^kBufLevel sets below such a node are written together: 64 contiguous bytes
constexpr int kBufSets = 1 << kBufLevel; // (32-byte sector writes reached DRAM as read-modify-writes: 2.7x the table size written, 0.9x read)

template <int j, uint32_t LOCAL>
__device__ __forceinline__ void cbic_dfs_buf(const double *A, int k, const CbicParams &prm, float (&buf)[kBufSets]) {
    if constexpr (j == 0) {
        buf[LOCAL] = (float)cbic_the_score64(A[0], k, prm);
    } else {
        cbic_dfs_buf<j - 1, LOCAL>(A, k, prm, buf);
        if (k < prm.max_parents) {
            double B[j * (j + 1) / 2];
            cbic_sweep<j>(A, B, prm.piv_tol);
            cbic_dfs_buf<j - 1, (LOCAL | (1u << (j - 1)))>(B, k + 1, prm, buf);
        } else {
#pragma unroll
            for (uint32_t m = 0; m < (1u << (j - 1)); m++) buf[LOCAL | (1u << (j - 1)) | m] = sentinel();
        }
    }
}

template <int j>
__device__ __forceinline__ void cbic_dfs_inl(const double *A, uint32_t low, int k, const CbicParams &prm, float *__restrict__ out) {
    if constexpr (j == kBufLevel) {
        float buf[kBufSets];
        cbic_dfs_buf<kBufLevel, 0u>(A, k, prm, buf);
        // streaming stores (st.global.cs) for the 2^c scores: measured 8.8 -> 8.3 ms per variable at config 3 against the
        // default store policy
        float4 *o4 = reinterpret_cast<float4 *>(out + low); // low is a multiple of kBufSets here
#pragma unroll
        for (int q = 0; q < kBufSets / 4; q++) __stcs(o4 + q, make_float4(buf[4 * q], buf[4 * q + 1], buf[4 * q + 2], buf[4 * q + 3]));
    } else if constexpr (j == 0) {
        out[low] = (float)cbic_the_score64(A[0], k, prm);
    } else {
        cbic_dfs_inl<j - 1>(A, low, k, prm, out); // candidate j-1 excluded: leading principal submatrix
        if (k < prm.max_parents) {
            double B[j * (j + 1) / 2];
            cbic_sweep<j>(A, B, prm.piv_tol);
            cbic_dfs_inl<j - 1>(B, low | (1u << (j - 1)), k + 1, prm, out);
        } else {
            for (uint32_t m = 0; m < (1u << (j - 1)); m++) out[low | (1u << (j - 1)) | m] = sentinel();
        }
    }
}

// one thread per prefix, J = 0..4: kBufLevel is the widest DFS whose matrices all fit the registers the launch bound
// leaves (J = 5 and 6 spill); wider level-B widths go to cbic_tree_kernel below
constexpr int kDfsMinBlocks = 5;
template <int J>
__global__ void __launch_bounds__(128, kDfsMinBlocks) cbic_dfs_kernel(const double *__restrict__ roots, CbicParams prm, uint32_t n_prefix, float *__restrict__ ts_out) {
    static_assert(J <= kBufLevel, "wider level-B widths use cbic_tree_kernel");
    const uint32_t P = blockIdx.x * blockDim.x + threadIdx.x;
    if (P >= n_prefix) return;
    float *out = ts_out + ((size_t)P << J);
    const int k0 = __popc(P);
    if (k0 > prm.max_parents) {
        for (uint32_t m = 0; m < (1u << J); m++) out[m] = sentinel();
        return;
    }
    double A[(J + 1) * (J + 2) / 2];
#pragma unroll
    for (int e = 0; e < (J + 1) * (J + 2) / 2; e++) A[e] = roots[(size_t)e * n_prefix + P];
    cbic_dfs_inl<J>(A, 0u, k0, prm, out);
}

// Level B, CTA form (J >= 7): a per-thread DFS this wide keeps the matrices of its upper levels on the thread's stack —
// 2.9 KB per thread at J = 11, 270 MB over the resident threads, which spills out of L2 and tripled the DRAM traffic of
// K3 (ncu, round 1).  Here one CTA of 2^(J-4) threads owns one prefix: the levels J .. 5 are expanded BREADTH FIRST in shared
// memory, all threads sharing each level's element-wise sweeps, and every thread then walks its own 4-bit subtree
// (16 sets) with all matrices in registers.  An "exclude" child is the leading principal submatrix of its parent, i.e. a
// PREFIX of the parent's packed array: it is never copied, only "include" children get storage (2802 doubles = 22 KB at
// J = 11).  Every element sees exactly the FMA sequence of the DFS, so scores are bit-identical.  No local memory.
constexpr int kTreeJB = 4;
__host__ __device__ constexpr int tri_size(int j) { return (j + 1) * (j + 2) / 2; }   // packed entries of a matrix over (v, cand_0 .. cand_{j-1})
template <int J> __host__ __device__ constexpr int cbic_tree_base(int level) {          // first double of the include-children of `level` (level < J)
    int off = tri_size(J);
    for (int l = J - 1; l > level; l--) off += (1 << (J - 1 - l)) * tri_size(l);
    return off;
}
template <int J> __host__ __device__ constexpr int cbic_tree_doubles() { return cbic_tree_base<J>(kTreeJB - 1); }

// storage of matrix m of `level`: trailing exclude decisions make it a view (prefix) of an ancestor's storage
__device__ __forceinline__ int cbic_tree_offset(const int *s_base, int level, uint32_t m) {
    if (m == 0) return 0;
    const int t = __ffs(m) - 1;
    const int l = level + t;
    return s_base[l] + (int)((m >> t) >> 1) * ((l + 1) * (l + 2) / 2);
}

// one level of the breadth-first expansion: the 2^(J-j) parents of level j share the CTA's threads evenly (a power of two
// of threads per parent), so everything that depends on the parent is computed once per thread and level
template <int J, int LEVEL>
__device__ __forceinline__ void cbic_tree_expand(double *S, double *inv /*[2][2^(J-kTreeJB)]*/, const unsigned char *tri_row, const int *s_base, int k0,
                                                 const CbicParams &prm, int tid) {
    if constexpr (LEVEL > kTreeJB) {
        constexpr int j = LEVEL;                        // parents: matrices over (v, cand_0 .. cand_{j-1}); pivot = row j
        constexpr int P = 1 << (J - j), E = tri_size(j - 1), NT = 1 << (J - kTreeJB), TPP = NT / P;
        const int m = tid / TPP, part = tid % TPP;
        const double *A = S + cbic_tree_offset(s_base, j, (uint32_t)m);
        const double inv_m = inv[(j & 1) * NT + m];
        double *inv_out = inv + ((j - 1) & 1) * NT;
        double *out = S + cbic_tree_base<J>(j - 1) + m * E;
        const bool include = k0 + __popc(m) < prm.max_parents;
        const double *prow = A + tri(j, 0);
        for (int e = part; e < E; e += TPP) {
            const int a = tri_row[e], b = e - a * (a + 1) / 2;
            const bool last = e == E - 1;               // element (j-1, j-1): the next pivot of both children
            if (last) inv_out[2 * m] = guarded_inv(A[e], prm.piv_tol);
            if (include) {
                const double f = -prow[a] * inv_m;
                const double x = fma(f, prow[b], A[e]);
                out[e] = x;
                if (last) inv_out[2 * m + 1] = guarded_inv(x, prm.piv_tol);
            }
        }
        __syncthreads();
        cbic_tree_expand<J, LEVEL - 1>(S, inv, tri_row, s_base, k0, prm, tid);
    }
}

// 72 registers hold every matrix (7 CTAs of 128 threads per SM at J = 11); left to itself, ptxas picks 64 at J = 10, 11
// and spills
template <int J>
__global__ void __maxnreg__(72) cbic_tree_kernel(const double *__restrict__ roots /*[n_prefix][tri_size(J)]*/, CbicParams prm, uint32_t n_prefix,
                                                 float *__restrict__ ts_out) {
    constexpr int NT = 1 << (J - kTreeJB);
    __shared__ double S[cbic_tree_doubles<J>()];
    __shared__ double inv[2 * NT];
    __shared__ unsigned char tri_row[tri_size(J - 1)];
    __shared__ int s_base[J + 1];
    const uint32_t P = blockIdx.x;
    const int tid = threadIdx.x;
    float *out = ts_out + ((size_t)P << J);
    const int k0 = __popc(P);
    if (k0 > prm.max_parents) { // whole subtree unscored
        for (uint32_t m = tid; m < (1u << J); m += NT) out[m] = sentinel();
        return;
    }
    for (int e = tid; e < tri_size(J); e += NT) S[e] = roots[(size_t)P * tri_size(J) + e];
    for (int e = tid; e < tri_size(J - 1); e += NT) {
        int a = 0;
        while ((a + 1) * (a + 2) / 2 <= e) a++;
        tri_row[e] = (unsigned char)a;
    }
    if (tid <= J) { // first double of the include-children of each level
        int off = tri_size(J);
        for (int l = J - 1; l > tid; l--) off += (1 << (J - 1 - l)) * tri_size(l);
        s_base[tid] = tid == J ? 0 : off;
    }
    __syncthreads();
    if (tid == 0) inv[(J & 1) * NT] = guarded_inv(S[tri(J, J)], prm.piv_tol);
    __syncthreads();
    cbic_tree_expand<J, J>(S, inv, tri_row, s_base, k0, prm, tid);
    // every thread: its level-4 matrix into registers, 16 sets, 64 contiguous bytes of scores
    const int k = k0 + __popc(tid);
    const uint32_t low = (uint32_t)tid << kTreeJB;
    if (k > prm.max_parents) {
#pragma unroll
        for (int q = 0; q < (1 << kTreeJB); q++) out[low + q] = sentinel();
        return;
    }
    double A[tri_size(kTreeJB)];
    const double *src = S + cbic_tree_offset(s_base, kTreeJB, (uint32_t)tid);
#pragma unroll
    for (int e = 0; e < tri_size(kTreeJB); e++) A[e] = src[e];
    cbic_dfs_inl<kTreeJB>(A, low, k, prm, out);
}

// ------------------------------------------------------------------------------------------------ K4 / K5 rules
// K4 — acceptance DP of the shipped `score` for cBIC ("clean" recursion, SURVEY.md Q5), layers ascending:
//   ts >  0            -> stored by the caller, val = -ts           (BIC_OLS.cpp:213-224, score_calculator.cpp:111-113)
//   ts == 0            -> not stored
//   ts <  0 (or NaN)   -> stored iff F(S) < -ts                     (BIC_OLS.cpp:233-249)
//   F(S) = max(0, max_{i in S, S\i != {}} g(S\i)),  g(T) = stored(T) ? val(T) : F(T)   (BIC_OLS.cpp:125-172)
//   In: table[mask] = the_score (float) or sentinel (not scored).  Out: table[mask] = stored value or sentinel.
// K5 — subset-dominance prune (ScoreCalculator::prune, score_calculator.cpp:150-197) as a DP on the dense table:
//   M(S) = max(val'(S), max_i M(S\i)),  keep S iff stored and val(S) > max_i M(S\i)  (ties: the subset, having
//   the smaller mask, sorts first and wins — compareSecond :137-148).  The empty set is always kept.
// URLGPU_CBIC_NO_ACCEPT: store -the_score for every scored set (dense table or rank-space scores alike)
__global__ void cbic_negate_kernel(float *__restrict__ table, uint64_t n) {
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    const float ts = table[m];
    if (!is_sentinel(ts)) table[m] = -ts;
}

// ------------------------------------------------------------------------------------------------ K4/K5, segment form
// The layer-by-layer kernels above scan all 2^c masks once per layer.  The segment form walks the table ONCE:
// a mask is split into (H, low) with `lb` low bits; one CTA owns the 2^lb-entry segment of a high part H.
// A set depends only on sets one element smaller: (H, low\b) — same segment, lower popcount — and (H\hb, low) —
// the same offset in the segments of H's sub-masks.  Launching the high parts in order of popcount(H) makes
// every dependency segment final, so a CTA (1) folds the popcount(H) dependency segments into one max array with
// coalesced reads, (2) runs the within-segment DP over popcount sub-layers in shared memory, (3) writes the
// segment back.  Traffic: (3 + popcount(H)) * 2^lb * 4 B per segment instead of ~c full-table scans.
constexpr int kSegMaxLb = 11;

struct SegLists {
    const uint32_t *high_sorted;  // all 2^hb high masks sorted by (popcount, value)
    const uint16_t *low_sorted;   // all 2^lb low masks sorted by (popcount, value)
    int low_off[kSegMaxLb + 2];   // start of each popcount class in low_sorted
};

// MODE 0: cBIC acceptance (see cbic_accept_layer_kernel), aux = gtab.  MODE 1: subset-dominance prune, aux = mtab.
template <int MODE>
__global__ void __launch_bounds__(256) segment_dp_kernel(float *__restrict__ table, float *__restrict__ aux, SegLists sl, int high_begin, int lb, int a /*popcount of the high parts of this launch*/,
                                                         int max_parents) {
    __shared__ __align__(16) float s_val[1 << kSegMaxLb];
    __shared__ __align__(16) float s_aux[1 << kSegMaxLb];
    __shared__ __align__(16) float s_dep[1 << kSegMaxLb];
    const uint32_t H = sl.high_sorted[high_begin + blockIdx.x];
    const uint32_t seg = 1u << lb;
    const size_t base = (size_t)H << lb;
    const float neutral = MODE == 0 ? 0.0f : -INFINITY;
    if ((seg & 3u) == 0) {
        // 128-bit loads, the dependency segments taken four at a time: up to 4 independent loads in flight per thread and
        // vector (the loop over the set bits of H has an unknown trip count, one load per iteration left the memory
        // system at ~2.5 TB/s)
        auto fold = [&](float4 d, const float4 g) {
            if (MODE == 0) { d.x = g.x > d.x ? g.x : d.x; d.y = g.y > d.y ? g.y : d.y; d.z = g.z > d.z ? g.z : d.z; d.w = g.w > d.w ? g.w : d.w; }
            else { d.x = fmaxf(d.x, g.x); d.y = fmaxf(d.y, g.y); d.z = fmaxf(d.z, g.z); d.w = fmaxf(d.w, g.w); }
            return d;
        };
        const float4 n4 = make_float4(neutral, neutral, neutral, neutral);
        for (uint32_t i = threadIdx.x * 4u; i < seg; i += blockDim.x * 4u) {
            const float4 v = *reinterpret_cast<const float4 *>(table + base + i);
            float4 d = n4;
            uint32_t rem = H;
            while (rem) {
                uint32_t b[4];
#pragma unroll
                for (int q = 0; q < 4; q++) { b[q] = rem & (~rem + 1); rem ^= b[q]; }
                float4 g[4];
#pragma unroll
                for (int q = 0; q < 4; q++) g[q] = b[q] ? *reinterpret_cast<const float4 *>(aux + ((size_t)(H ^ b[q]) << lb) + i) : n4;
#pragma unroll
                for (int q = 0; q < 4; q++) d = fold(d, g[q]);
            }
            *reinterpret_cast<float4 *>(s_val + i) = v;
            *reinterpret_cast<float4 *>(s_aux + i) = n4;
            *reinterpret_cast<float4 *>(s_dep + i) = d;
        }
    } else {
        for (uint32_t i = threadIdx.x; i < seg; i += blockDim.x) {
            s_val[i] = table[base + i];
            s_aux[i] = neutral;
            float d = neutral;
            for (uint32_t hb = H; hb; hb &= hb - 1) {
                const float g = aux[((size_t)(H ^ (hb & (~hb + 1))) << lb) + i];
                d = MODE == 0 ? (g > d ? g : d) : fmaxf(d, g);
            }
            s_dep[i] = d;
        }
    }
    __syncthreads();
    for (int j = 0; j <= lb; j++) {
        const int layer = a + j;
        if (layer <= max_parents) {
            for (int idx = sl.low_off[j] + threadIdx.x; idx < sl.low_off[j + 1]; idx += blockDim.x) {
                const uint32_t low = sl.low_sorted[idx];
                const float v = s_val[low];
                if (MODE == 0) {
                    if (is_sentinel(v)) continue;
                    if (layer == 0) { s_val[low] = -v; s_aux[low] = 0.0f; continue; }
                    if (v > 0.0f) { s_val[low] = -v; s_aux[low] = -v; continue; }
                    float F = 0.0f;
                    if (layer > 1) {
                        F = s_dep[low] > F ? s_dep[low] : F;
                        for (uint32_t b = low; b; b &= b - 1) {
                            const float g = s_aux[low ^ (b & (~b + 1))];
                            if (g > F) F = g;
                        }
                    }
                    if (v == 0.0f) { s_val[low] = sentinel(); s_aux[low] = F; continue; }
                    const float val = -v;
                    if (F >= val) { s_val[low] = sentinel(); s_aux[low] = F; }
                    else { s_val[low] = val; s_aux[low] = val; }
                } else {
                    float best = s_dep[low];
                    for (uint32_t b = low; b; b &= b - 1) best = fmaxf(best, s_aux[low ^ (b & (~b + 1))]);
                    const bool stored = !is_sentinel(v);
                    if (stored && layer > 0 && !(v > best)) s_val[low] = sentinel();
                    s_aux[low] = stored ? fmaxf(best, v) : best;
                }
            }
        }
        __syncthreads();
    }
    if ((seg & 3u) == 0) {
        for (uint32_t i = threadIdx.x * 4u; i < seg; i += blockDim.x * 4u) {
            *reinterpret_cast<float4 *>(table + base + i) = *reinterpret_cast<const float4 *>(s_val + i);
            *reinterpret_cast<float4 *>(aux + base + i) = *reinterpret_cast<const float4 *>(s_aux + i);
        }
    } else {
        for (uint32_t i = threadIdx.x; i < seg; i += blockDim.x) {
            table[base + i] = s_val[i];
            aux[base + i] = s_aux[i];
        }
    }
}

} // namespace urlgpu
