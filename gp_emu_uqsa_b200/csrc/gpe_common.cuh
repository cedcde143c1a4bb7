// gp_emu_uqsa_b200 -- shared device/host helpers (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <type_traits>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "gp_emu_uqsa_b200 kernels are written for sm_100a (B200) only"
#endif

namespace gpe {

constexpr int NB = 128;        // leaf block / padding granule of every n x n matrix
constexpr int NUM_SMS = 148;   // B200

// ---- opt-in to more than 48 KB of dynamic shared memory: a per-device function attribute, set the first time a
// kernel needs a given size on the current device (one static instance per launch site)
struct SmemOptIn {
    size_t have[16] = {};
    template <class Kern>
    cudaError_t ensure(Kern kernel, size_t bytes) {
        if (bytes <= 48 * 1024) return cudaSuccess;
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 15;
        if (bytes <= have[dev]) return cudaSuccess;
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e == cudaSuccess) have[dev] = bytes;
        return e;
    }
};

// ---- cp.async (LDGSTS) 16-byte copies, the staging path for FP64 DMMA tiles -------------
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ---- FP64 tensor-pipe MMA: D(8x8) += A(8x4) * B(4x8); SASS: DMMA.8x8x4 ------------------
// lane l: a = A[l>>2][l&3], b = B[l&3][l>>2], c0,c1 = C[l>>2][2*(l&3)+{0,1}]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---- mbarrier (shared::cta) helpers for the warp-specialised producer/consumer pipeline ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(a), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(a) : "memory");
}
// arrive on `bar` once every cp.async previously issued by this thread has landed
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
    unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(a) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    unsigned done;
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- exp() for the Gaussian kernel entries ------------------------------------------------------------------
// CUDA's exp(double) materialises every polynomial coefficient with a pair of UMOV/IMAD.MOV (a DFMA immediate holds
// only the high 32 bits of a double): 22 UMOV + 15 IMAD per call, which made the covariance and gradient kernels
// issue-bound (ncu: FP64 pipe 53-57 % busy, 134 issue slots per entry for 50 FP64 instructions).  Here the
// constants sit in the constant bank and are DFMA operands directly.  Same method and accuracy class as the library
// routine: k = rint(x log2 e) by the 1.5*2^52 trick, r = x - k ln2 in two parts (fdlibm split), exp(r) on
// |r| <= ln2/2 as 1 + r(1 + r q(r)) with the Taylor coefficients to r^13 (truncation 6e-18), scaled by 2^k through the
// exponent field; arguments outside (-708, 708) (denormal, zero or infinite results) are scaled by two multiplications.
// tools/ub_exp.cu measures it against exp(): max 1 ulp apart on 2^26 arguments of the kernel's range.
static __constant__ double GPE_EXP_K[16] = {
    1.4426950408889634074,       // log2(e)
    -6.93147180369123816490e-01, // -ln2 hi (low 21 bits zero: k * hi is exact)
    -1.90821492927058770002e-10, // -ln2 lo
    1.0 / 6227020800.0, 1.0 / 479001600.0, 1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 362880.0, 1.0 / 40320.0,
    1.0 / 5040.0, 1.0 / 720.0, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5, 0.0};
__device__ __forceinline__ double gpe_exp(double x) {
    const double magic = 6755399441055744.0;           // 1.5 * 2^52 (low word zero: a DFMA immediate)
    const double t = fma(x, GPE_EXP_K[0], magic);
    const int k = __double2loint(t);
    const double kd = t - magic;
    double r = fma(kd, GPE_EXP_K[1], x);
    r = fma(kd, GPE_EXP_K[2], r);
    double q = GPE_EXP_K[3];
#pragma unroll
    for (int i = 4; i <= 14; i++) q = fma(q, r, GPE_EXP_K[i]);
    q = fma(q, r, 1.0);
    q = fma(q, r, 1.0);
    if (fabs(x) < 708.0) return __hiloint2double(__double2hiint(q) + (k << 20), __double2loint(q));
    // rare: results that are denormal, zero, infinite or NaN -- scale in two steps so the last product rounds once
    if (x != x) return x;
    if (x > 710.0) return __longlong_as_double(0x7ff0000000000000ll);
    if (x < -746.0) return 0.0;
    const int k1 = k >> 1, k2 = k - k1;
    return q * __hiloint2double((k1 + 1023) << 20, 0) * __hiloint2double((k2 + 1023) << 20, 0);
}

// ---- Matérn 5/2 from the scaled squared distance D = sum_k ((x_ik - x_jk) / delta_k)^2, r = sqrt(D) ----------------------
// R = (1 + sqrt5 r + 5D/3) exp(-sqrt5 r) is the correlation; G = (5/6)(1 + sqrt5 r) exp(-sqrt5 r) is its derivative factor,
// dR/dtheta_k = G Delta_k^2 for delta_k = exp(theta_k / 2).  One exponential serves both; sqrt is the IEEE one.
constexpr int FAMILY_GAUSSIAN = 0, FAMILY_MATERN52 = 1;
__device__ __forceinline__ double gpe_matern52(double D, double& G) {
    const double s5r = 2.23606797749978969641 * __dsqrt_rn(D);
    const double e = gpe_exp(-s5r);
    const double p = 1.0 + s5r;
    G = (5.0 / 6.0) * p * e;
    return fma(D, 5.0 / 3.0, p) * e;
}
__device__ __forceinline__ double gpe_matern52(double D) {
    double G;
    return gpe_matern52(D, G);   // (G is dead code here)
}
// kappa = -2 R'(0) of the family (R as a function of D): the prior variance of a scaled derivative of the process
template <int FAM>
constexpr double FAMILY_KAPPA = FAM == FAMILY_MATERN52 ? 5.0 / 3.0 : 2.0;

// f(std::integral_constant<int, FAMILY_...>{}) for the run-time family: the one place where a family picks the kernel
// instantiations a launch site runs.  A static inside the generic lambda f is one per family instantiation.
template <class F>
decltype(auto) with_family(int family, F&& f) {
    if (family == FAMILY_MATERN52) return f(std::integral_constant<int, FAMILY_MATERN52>{});
    return f(std::integral_constant<int, FAMILY_GAUSSIAN>{});
}
// Prior covariance c·k(D) of two distinct points at scaled squared distance D
template <int FAM>
__device__ __forceinline__ double cov_prior(double cscale, double D) {
    return cscale * (FAM == FAMILY_MATERN52 ? gpe_matern52(D) : gpe_exp(-D));
}

// ---- squared-distance tiles: the D of every covariance tile c k(D) ---------------------------------------------------------------
// The inputs, scaled by 1/delta, are held k-major in shared memory: the row tile Xi [d][RA RS] and the column tile Xj [d][2 CH + 2].
// A thread owns RA x 4 entries, rows ty + RS a and columns 2tx + {0, 1}, CH + 2tx + {0, 1}: the row operand is a broadcast, the
// column operand a conflict-free double2.  Two shapes are in use: 4 x 4 (RS 16, CH 32: 64 x 64 entries, strides 64 / 66) and
// 8 x 4 (RS 8, CH 64: 64 rows x 128 points, strides 64 / 130).  Direct differences (no |x|^2+|y|^2-2xy GEMM trick: it would lose
// cond(A) digits and break the 1e-10 parity target).

// the operands of input k: xi[a] = Xi[k][ty + RS a], xj = Xj[k][2tx, 2tx + 1, CH + 2tx, CH + 2tx + 1]
template <int RA, int RS, int CH>
__device__ __forceinline__ void tile_operands(const double* Xi, const double* Xj, int k, int ty, int tx, double (&xi)[RA],
                                              double (&xj)[4]) {
#pragma unroll
    for (int a = 0; a < RA; a++) xi[a] = Xi[k * (RA * RS) + ty + RS * a];
    const double2 v0 = *reinterpret_cast<const double2*>(&Xj[k * (2 * CH + 2) + 2 * tx]);
    const double2 v1 = *reinterpret_cast<const double2*>(&Xj[k * (2 * CH + 2) + CH + 2 * tx]);
    xj[0] = v0.x; xj[1] = v0.y; xj[2] = v1.x; xj[3] = v1.y;
}

// D[a][c] = sum_k (xi[a] - xj[c])^2, accumulated in input order
template <int RA, int RS, int CH>
__device__ __forceinline__ void sqdist_tile(const double* Xi, const double* Xj, int d, int ty, int tx, double (&D)[RA][4]) {
#pragma unroll
    for (int a = 0; a < RA; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) D[a][c] = 0.0;
    for (int k = 0; k < d; k++) {
        double xi[RA], xj[4];
        tile_operands<RA, RS, CH>(Xi, Xj, k, ty, tx, xi, xj);
#pragma unroll
        for (int a = 0; a < RA; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const double df = xi[a] - xj[c];
                D[a][c] = fma(df, df, D[a][c]);
            }
    }
}

// The two tiles of the 4 x 4 shape from the rows i0 + r and j0 + r (r < 64) of X [n][d], scaled by w [d], zero for rows >= n.
// 256 threads; no integer division: thread -> (row, k mod 4), 4 lanes read 32 contiguous bytes of a row.
__device__ __forceinline__ void fill_scaled_tiles(const double* __restrict__ X, const double* __restrict__ w, int n, int d, int i0,
                                                  int j0, double* Xi, double* Xj, int tid) {
    const int row = tid >> 2, gi = i0 + row, gj = j0 + row;
    for (int k = tid & 3; k < d; k += 4) {
        Xi[k * 64 + row] = (gi < n) ? X[(size_t)gi * d + k] * w[k] : 0.0;
        Xj[k * 66 + row] = (gj < n) ? X[(size_t)gj * d + k] * w[k] : 0.0;
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum; result valid in thread 0. `red` must hold >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = 0.0;
    if (w == 0) {
        s = (l < nw) ? red[l] : 0.0;
        s = warp_sum(s);
    }
    return s;
}

}  // namespace gpe
