// gp_emu_uqsa_b200 -- shared device/host helpers (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

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
