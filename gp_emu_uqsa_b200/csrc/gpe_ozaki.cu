// FP64 GEMM on the INT8 tensor cores by integer modular arithmetic (see gpe_ozaki.cuh for the scheme).
#include "gpe_ozaki.cuh"

#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

namespace gpe {

// pairwise coprime moduli <= 256, largest first (255 = 3.5.17, 253 = 11.23, 247 = 13.19, 217 = 7.31, the rest prime)
static const uint32_t OZ_MODULI[OZ_MAXMOD] = {256, 255, 253, 251, 247, 241, 239, 233, 229, 227,
                                              223, 217, 211, 199, 197, 193, 191, 181, 179, 173};

// ---------------------------------------------------------------------------------------------- host constants
struct OzConst {
    uint32_t p[OZ_MAXMOD];      // modulus
    uint32_t m32[OZ_MAXMOD];    // ceil(2^32 / p): floor(t / p) = umulhi(t, m32) for t < 2^20
    uint32_t m39[OZ_MAXMOD];    // ceil(2^39 / p): floor(t / p) = (t * m39) >> 39 for t < 2^31
    uint32_t clo[OZ_MAXMOD];    // bytes 256^0..256^3 mod p
    uint32_t chi[OZ_MAXMOD];    // bytes 256^4..256^7 mod p
    uint32_t c0[OZ_MAXMOD];     // (-2^63) mod p
    uint32_t np[OZ_MAXMOD];     // -p mod 2^32 (a table entry, so that the compiler cannot turn q * np + t back into a negation and a multiply)
};
struct OzCrt {
    uint32_t f2[OZ_MAXMOD], f1[OZ_MAXMOD], f0[OZ_MAXMOD];   // floor(2^96 y_i / p_i), most significant limb first
    double P;                                               // product of the moduli, correctly rounded
    int plen;                                               // bit length of the product
};

static OzConst make_const() {
    OzConst c;
    for (int a = 0; a < OZ_MAXMOD; a++) {
        const uint32_t p = OZ_MODULI[a];
        c.p[a] = p;
        c.m32[a] = (uint32_t)(((1ull << 32) + p - 1) / p);
        c.m39[a] = (uint32_t)(((1ull << 39) + p - 1) / p);
        uint32_t pw = 1 % p, lo = 0, hi = 0;
        for (int j = 0; j < 8; j++) {
            if (j < 4) lo |= pw << (8 * j);
            else hi |= pw << (8 * (j - 4));
            pw = (pw * 256u) % p;
        }
        c.clo[a] = lo;
        c.chi[a] = hi;
        uint32_t t = 1 % p;                 // 2^63 mod p
        for (int j = 0; j < 63; j++) t = (t * 2u) % p;
        c.c0[a] = (p - t) % p;
        c.np[a] = 0u - p;
    }
    return c;
}

static OzCrt make_crt(int nmod) {
    OzCrt c;
    memset(&c, 0, sizeof c);
    // product in 32-bit limbs (little endian), exact
    uint32_t L[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < nmod; a++) {
        uint64_t carry = 0;
        for (int j = 0; j < 8; j++) {
            const uint64_t v = (uint64_t)L[j] * OZ_MODULI[a] + carry;
            L[j] = (uint32_t)v;
            carry = v >> 32;
        }
    }
    int top = 255;
    while (top > 0 && !((L[top >> 5] >> (top & 31)) & 1u)) top--;
    c.plen = top + 1;
    // round to nearest even at 53 bits
    auto bit = [&](int i) -> uint64_t { return i < 0 ? 0 : ((L[i >> 5] >> (i & 31)) & 1u); };
    uint64_t mant = 0;
    for (int i = 0; i < 53; i++) mant = (mant << 1) | bit(top - i);
    const uint64_t half = bit(top - 53);
    bool sticky = false;
    for (int i = top - 54; i >= 0; i--) sticky |= bit(i) != 0;
    if (half && (sticky || (mant & 1))) mant++;
    c.P = std::ldexp((double)mant, top - 52);
    for (int a = 0; a < nmod; a++) {
        const uint32_t p = OZ_MODULI[a];
        uint32_t Mi = 1 % p;
        for (int b = 0; b < nmod; b++)
            if (b != a) Mi = (Mi * (OZ_MODULI[b] % p)) % p;
        uint32_t y = 0;
        for (uint32_t t = 0; t < p; t++)
            if ((Mi * t) % p == 1 % p) { y = t; break; }
        const unsigned __int128 f = (((unsigned __int128)y) << 96) / p;
        c.f2[a] = (uint32_t)(f >> 64);
        c.f1[a] = (uint32_t)(f >> 32);
        c.f0[a] = (uint32_t)f;
    }
    return c;
}

int oz_operand_bits(int nmod, int K) {
    static int plen[OZ_MAXMOD + 1] = {0};
    if (!plen[nmod]) plen[nmod] = make_crt(nmod).plen;
    int lk = 0;
    while ((1 << lk) < K) lk++;
    int b = (plen[nmod] - 2 - lk) / 2;
    return b > 63 ? 63 : b;
}

static __constant__ OzConst OZC;

static cudaError_t upload_const() {
    static std::mutex mu;
    static bool done[16] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    if (done[dev & 15]) return cudaSuccess;
    const OzConst c = make_const();
    cudaError_t e = cudaMemcpyToSymbol(OZC, &c, sizeof c);
    if (e == cudaSuccess) done[dev & 15] = true;
    return e;
}

// ---------------------------------------------------------------------------------------------- step 1: residues
// Element (r, k) of the operand is src[r * ld + k] (KC) or src[k * ld + r] (!KC).  Planes: [item][modulus][R][K] bytes.
// One pass for the row maxima (scale exponent s = bits - 1 - floor(log2 max)), a second over the same data (L2 / L1
// hits) for the residues: v = trunc(x 2^s) as a 64-bit integer in offset binary, its eight bytes weighted by
// 256^j mod p with two DP4A, the 20-bit sum reduced by one multiply-high.
__device__ __forceinline__ int oz_scale_exp(double mx, int bits) {
    if (!(mx > 0.0)) return 0;
    const int e = (int)((__double2hiint(mx) >> 20) & 0x7ff) - 1023;     // floor(log2 mx) for normal numbers
    int s = bits - 1 - e;
    return max(-1000, min(1000, s));
}
__device__ __forceinline__ double oz_pow2(int e) { return __hiloint2double((1023 + e) << 20, 0); }

__device__ __forceinline__ void oz_to_u64(double x, double p1, double p2, uint32_t& lo, uint32_t& hi) {
    const long long v = __double2ll_rz(x * p1 * p2);
    const unsigned long long u = (unsigned long long)v ^ 0x8000000000000000ull;
    lo = (uint32_t)u;
    hi = (uint32_t)(u >> 32);
}
__device__ __forceinline__ uint32_t oz_residue(uint32_t lo, uint32_t hi, uint32_t clo, uint32_t chi, uint32_t c0,
                                               uint32_t m32, uint32_t np) {
    uint32_t t = __dp4a(lo, clo, c0);
    t = __dp4a(hi, chi, t);
    return __umulhi(t, m32) * np + t;       // np = -p (mod 2^32): one multiply-add, no separate negation on the FMA-heavy pipe
}

#ifndef OZ_COMB_MINB
#define OZ_COMB_MINB 3
#endif
#ifndef OZ_CONV_MINB
#define OZ_CONV_MINB 4
#endif
constexpr int OZ_CV = 8;      // consecutive k per thread in the conversion
// k range of row r that the residue GEMM can read: tri 0 all, > 0 "k <= r" (up to the end of r's granule of `tri` rows),
// < 0 "k >= r" (from the start of r's granule of `-tri` rows).  The granule is the row count of the GEMM's work unit for this
// operand (128 x cluster size for the A role, 256 for the B role).  Nothing outside the range is written or read.
__device__ __forceinline__ void oz_row_range(int tri, int r, int K, int& klo, int& khi) {
    klo = 0;
    khi = K;
    if (tri > 0) khi = min(K, (r / tri + 1) * tri);
    else if (tri < 0) klo = min(K, (r / -tri) * -tri);
}
__device__ __forceinline__ uint32_t oz_pack4(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
    return __byte_perm(__byte_perm(r0, r1, 0x0040), __byte_perm(r2, r3, 0x0040), 0x5410);   // PRMT: the ALU pipe is idle here
}
// residues of eight values for modulus a, packed
__device__ __forceinline__ uint2 oz_residues8(const uint32_t (&lo)[OZ_CV], const uint32_t (&hi)[OZ_CV], int a) {
    // modulus 0 is 256 (and 2^63 = 0 mod 256): the residue is the low byte, no arithmetic (a is uniform across the warp)
    if (a == 0) return make_uint2(oz_pack4(lo[0], lo[1], lo[2], lo[3]), oz_pack4(lo[4], lo[5], lo[6], lo[7]));
    const uint32_t clo = OZC.clo[a], chi = OZC.chi[a], c0 = OZC.c0[a], m32 = OZC.m32[a], np = OZC.np[a];
    uint32_t r[OZ_CV];
#pragma unroll
    for (int j = 0; j < OZ_CV; j++) r[j] = oz_residue(lo[j], hi[j], clo, chi, c0, m32, np);
    return make_uint2(oz_pack4(r[0], r[1], r[2], r[3]), oz_pack4(r[4], r[5], r[6], r[7]));
}

// K-contiguous operand: one warp per row.
__global__ void __launch_bounds__(256, OZ_CONV_MINB) oz_convert_kc_kernel(const double* __restrict__ src, int ld, long long sS, int R, int K,
                                                            int nmod, int bits, int tri, uint8_t* __restrict__ planes,
                                                            int* __restrict__ sexp, double fixed_max) {
    const int b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + warp;
    if (r >= R) return;
    const double* row = src + (size_t)b * sS + (size_t)r * ld;
    uint8_t* Pb = planes + (size_t)b * nmod * R * K;
    int klo, khi;
    oz_row_range(tri, r, K, klo, khi);
    double mx = fixed_max;          // > 0: the caller's bound on |x| replaces the pass over the row (one scale for all rows)
    if (!(fixed_max > 0.0)) {
        for (int k = klo + lane * 2; k < khi; k += 64) {
            const double2 v = *reinterpret_cast<const double2*>(row + k);
            mx = fmax(mx, fmax(fabs(v.x), fabs(v.y)));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    const int s = oz_scale_exp(mx, bits);
    if (lane == 0) sexp[(size_t)b * R + r] = s;
    const double p1 = oz_pow2(s / 2), p2 = oz_pow2(s - s / 2);
    const size_t plane = (size_t)R * K;
    for (int k0 = klo + lane * OZ_CV; k0 < khi; k0 += 32 * OZ_CV) {
        uint32_t lo[OZ_CV], hi[OZ_CV];
#pragma unroll
        for (int j = 0; j < OZ_CV; j += 2) {
            const double2 v = *reinterpret_cast<const double2*>(row + k0 + j);
            oz_to_u64(v.x, p1, p2, lo[j], hi[j]);
            oz_to_u64(v.y, p1, p2, lo[j + 1], hi[j + 1]);
        }
        uint8_t* dst = Pb + (size_t)r * K + k0;
#pragma unroll 2
        for (int a = 0; a < nmod; a++) *reinterpret_cast<uint2*>(dst + (size_t)a * plane) = oz_residues8(lo, hi, a);
    }
}

// Operand stored [k][r]: a CTA takes 32 rows r (adjacent in memory); thread (tx, ty) reads eight k of row tx per 64-wide
// slab (each load 256 contiguous bytes across the warp), the residues of all moduli are transposed through shared memory
// and leave as 64-byte row segments.
constexpr int OZ_THALF = 10;  // moduli staged at a time
constexpr int OZ_TS = 72;     // bytes per staged row (64 + 8: conflict-free 8-byte stores of a half-warp)
__global__ void __launch_bounds__(256) oz_convert_t_kernel(const double* __restrict__ src, int ld, long long sS, int R, int K,
                                                           int nmod, int bits, int tri, uint8_t* __restrict__ planes,
                                                           int* __restrict__ sexp, double fixed_max) {
    __shared__ double red[8][33];
    __shared__ int s_sh[32];
    __shared__ __align__(16) uint8_t stage[OZ_THALF * 32 * OZ_TS];
    const int b = blockIdx.y;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int r0 = blockIdx.x * 32, r = r0 + tx;           // R is a multiple of 32; the 32 rows share one granule
    const double* col = src + (size_t)b * sS + r;
    uint8_t* Pb = planes + (size_t)b * nmod * R * K;
    int klo, khi;
    oz_row_range(tri, r0, K, klo, khi);
    if (fixed_max > 0.0) {          // the caller's bound on |x| replaces the pass over the data (one scale for all rows)
        if (ty == 0) {
            const int s = oz_scale_exp(fixed_max, bits);
            s_sh[tx] = s;
            sexp[(size_t)b * R + r] = s;
        }
    } else {
        double mx = 0.0;
        for (int k = klo + ty; k < khi; k += 8) mx = fmax(mx, fabs(col[(size_t)k * ld]));
        red[ty][tx] = mx;
        __syncthreads();
        if (ty == 0) {
#pragma unroll
            for (int j = 1; j < 8; j++) mx = fmax(mx, red[j][tx]);
            const int s = oz_scale_exp(mx, bits);
            s_sh[tx] = s;
            sexp[(size_t)b * R + r] = s;
        }
    }
    __syncthreads();
    const int s = s_sh[tx];
    const double p1 = oz_pow2(s / 2), p2 = oz_pow2(s - s / 2);
    const size_t plane = (size_t)R * K;
    const int orow = threadIdx.x >> 3, och = threadIdx.x & 7;      // write-out: row, 8-byte chunk
    for (int k0 = klo; k0 < khi; k0 += 64) {
        uint32_t lo[OZ_CV], hi[OZ_CV];
        const double* cp = col + (size_t)(k0 + ty * OZ_CV) * ld;
#pragma unroll
        for (int j = 0; j < OZ_CV; j++) oz_to_u64(cp[(size_t)j * ld], p1, p2, lo[j], hi[j]);
        uint8_t* dst = Pb + (size_t)(r0 + orow) * K + k0 + och * 8;
        // the moduli in groups of OZ_THALF: 23 KB of staging, so that the kernel fits on an SM beside a CTA of the residue GEMM
        for (int a0 = 0; a0 < nmod; a0 += OZ_THALF) {
            const int na = min(OZ_THALF, nmod - a0);
#pragma unroll 2
            for (int a = 0; a < na; a++)
                *reinterpret_cast<uint2*>(stage + (a * 32 + tx) * OZ_TS + ty * 8) = oz_residues8(lo, hi, a0 + a);
            __syncthreads();
            for (int a = 0; a < na; a++)
                *reinterpret_cast<uint2*>(dst + (size_t)(a0 + a) * plane) =
                    *reinterpret_cast<const uint2*>(stage + (a * 32 + orow) * OZ_TS + och * 8);
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------------- step 2: residue GEMM
struct OzGemmArgs {
    int M, N, K, nmod, nbp;      // nbp = items * nmod plane products
    int kmode, lower;
    int nmajor;                  // one operand much larger than L2 (prediction): units that share a tile of it are consecutive (oz_unit)
    int tiles_m, tiles_n, T;     // tiles per plane product
    uint8_t* D;                  // [nbp][M][N]
    uint32_t p[OZ_MAXMOD], m39[OZ_MAXMOD], np[OZ_MAXMOD];
};

constexpr int OZ_STAGES = 4;
constexpr int OZ_A_BYTES = OZ_BM * OZ_BK, OZ_B_BYTES = OZ_BN * OZ_BK;
constexpr int OZ_STAGE_BYTES = OZ_A_BYTES + OZ_B_BYTES;
constexpr int OZ_THREADS = 192;   // warp 0: TMA producer, warp 1: MMA issuer, warps 2..5: epilogue (TMEM lane quarters 2,3,0,1)
constexpr size_t OZ_SMEM = (size_t)OZ_STAGES * OZ_STAGE_BYTES + 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor, K-major operand in the 128-byte-swizzled layout TMA writes (rows of 128 bytes,
// 8-row groups 1024 bytes apart): start address >> 4 in [0,14), leading byte offset (unused for swizzled K-major) in
// [16,30), stride byte offset 1024 >> 4 in [32,46), version 1 in [46,48), layout type 2 = SWIZZLE_128B in [61,64)
__device__ __forceinline__ uint64_t oz_desc(uint32_t saddr) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor: D format S32 = 2 at [4,6), A / B format U8 = 0 at [7,10) / [10,13), both K-major, N >> 3 at
// [17,23), M >> 4 at [24,29)
constexpr uint32_t OZ_IDESC = (2u << 4) | ((uint32_t)(OZ_BN >> 3) << 17) | ((uint32_t)(OZ_BM >> 4) << 24);

__device__ __forceinline__ void oz_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void oz_tma_load(void* smem, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(
            smem_u32(smem)),
        "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}
#ifndef OZ_PREFETCH
#define OZ_PREFETCH 0
#endif
__device__ __forceinline__ void oz_tma_prefetch(const CUtensorMap* tm, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];\n" ::"l"(tm), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void oz_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}

// Work unit t of a plane product -> (um, tn), heaviest first.  A unit is CL vertically adjacent 128x256 tiles (rows
// um*CL .. um*CL+CL-1 of the tile grid) computed by the CL CTAs of a cluster, which share the tile of B.
template <int CL>
__device__ __forceinline__ void oz_unit(const OzGemmArgs& g, int t, int& um, int& tn) {
    const int units_m = g.tiles_m / CL;
    if (g.lower) {              // rows ascending (k >= i: heaviest first), tn up to the diagonal of the unit's last row
        int row = 0, before = 0;
        while (true) {
            const int cnt = min(g.tiles_n, (row * CL + CL - 1) / 2 + 1);
            if (t < before + cnt) break;
            before += cnt;
            row++;
        }
        um = row;
        tn = t - before;
        return;
    }
    switch (g.kmode) {
        case KM_LE_J:
            if (g.nmajor) {       // the mirror image: a tall A (the prediction product with its roles swapped), tn fastest, rotated
                um = t / g.tiles_n;
                tn = g.tiles_n - 1 - (t % g.tiles_n + um) % g.tiles_n;
            } else {
                tn = g.tiles_n - 1 - t / units_m;
                um = t % units_m;
            }
            break;
        case KM_GE_J: tn = t / units_m; um = t % units_m; break;
        case KM_LE_I:
            if (g.nmajor) {
                // a wide B (the prediction's 65 536 points: 134 MB per plane, more than L2): the units_m units of one column
                // tile are consecutive, so the clusters that run side by side read that tile of B from L2 and DRAM sees it
                // once; the row unit is rotated by tn so that a cluster's static sequence (stride = number of clusters) walks
                // through all k ranges whatever the two counts' common divisor
                tn = t / units_m;
                um = units_m - 1 - (t % units_m + tn) % units_m;
            } else {
                um = units_m - 1 - t / g.tiles_n;
                tn = t % g.tiles_n;
            }
            break;
        default: um = t / g.tiles_n; tn = t % g.tiles_n; break;
    }
}
// k blocks of a unit (the same for all CTAs of the cluster: they run their pipelines in lock step)
template <int CL>
__device__ __forceinline__ void oz_krange(const OzGemmArgs& g, int um, int tn, int& kb0, int& kb1) {
    const int nkb = g.K / OZ_BK;
    kb0 = 0;
    kb1 = nkb;
    switch (g.kmode) {
        case KM_LE_J: kb1 = min(nkb, (tn + 1) * (OZ_BN / OZ_BK)); break;
        case KM_GE_J: kb0 = min(nkb - 1, tn * (OZ_BN / OZ_BK)); break;
        case KM_LE_I: kb1 = min(nkb, (um + 1) * CL * (OZ_BM / OZ_BK)); break;
        case KM_GE_I: kb0 = min(nkb - 1, um * CL * (OZ_BM / OZ_BK)); break;
        default: break;
    }
}

__device__ __forceinline__ uint32_t oz_cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void oz_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void oz_tma_load_mc(void* smem, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar,
                                               uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3, "
        "%4}], [%5], %6;\n" ::"r"(smem_u32(smem)),
        "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void oz_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
                     smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}

// CL = 1: every CTA loads its own 128 x 128 tile of A and 256 x 128 tile of B per k block (48 KB per 4 MMAs: the kernel is
// bound by the L2 -> SM bandwidth, 90 B/clk/SM at the INT8 peak).  CL = 2: the two CTAs of a cluster work on vertically
// adjacent tiles; each loads its own tile of A and one half of the shared tile of B, multicast into both CTAs' shared
// memory (32 KB from L2 per CTA and k block).  A stage is released when the MMAs of both CTAs have read it (their
// tcgen05.commit arrives on both CTAs' empty barriers); a CTA's full barrier counts the bytes of all three copies.
template <int CL>
__global__ void __launch_bounds__(OZ_THREADS, 1) oz_gemm_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB,
                                                                 const __grid_constant__ OzGemmArgs g) {
    extern __shared__ uint8_t oz_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)oz_smem_raw + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t full_bar[OZ_STAGES], empty_bar[OZ_STAGES], tfull_bar[2], tempty_bar[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rank = CL > 1 ? (int)oz_cluster_rank() : 0;
    const long long cid = blockIdx.x / CL, ncl = gridDim.x / CL;
    constexpr uint16_t MASK = (uint16_t)((1u << CL) - 1u);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < OZ_STAGES; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], CL);
        }
#pragma unroll
        for (int s = 0; s < 2; s++) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmB) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_s)), "n"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (CL > 1) oz_cluster_sync();            // the peer's barriers exist before anything is multicast to them
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem = tmem_base_s;
    const long long total = (long long)g.nbp * g.T;

    if (warp == 0) {
        if (lane == 0) {                      // ---- TMA producer
            int stage = 0;
            uint32_t phase = 0;
            for (long long w = cid; w < total; w += ncl) {
                const int bp = (int)(w / g.T), t = (int)(w - (long long)bp * g.T);
                int um, tn, kb0, kb1;
                oz_unit<CL>(g, t, um, tn);
                oz_krange<CL>(g, um, tn, kb0, kb1);
                const int tm = um * CL + rank;
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    oz_mbar_expect_tx(&full_bar[stage], OZ_STAGE_BYTES);
                    uint8_t* sa = smem + stage * OZ_STAGE_BYTES;
                    oz_tma_load(sa, &tmA, kb * OZ_BK, tm * OZ_BM, bp, &full_bar[stage]);
                    if (CL == 1) {
                        oz_tma_load(sa + OZ_A_BYTES, &tmB, kb * OZ_BK, tn * OZ_BN, bp, &full_bar[stage]);
                    } else {
                        constexpr int HB = OZ_BN / CL;          // rows of B this CTA fetches for the cluster
                        oz_tma_load_mc(sa + OZ_A_BYTES + rank * HB * OZ_BK, &tmB, kb * OZ_BK, tn * OZ_BN + rank * HB, bp,
                                       &full_bar[stage], MASK);
                    }
                    if (OZ_PREFETCH > 0 && kb + OZ_PREFETCH < kb1) {      // pull the k block OZ_PREFETCH ahead into L2
                        oz_tma_prefetch(&tmA, (kb + OZ_PREFETCH) * OZ_BK, tm * OZ_BM, bp);
                        oz_tma_prefetch(&tmB, (kb + OZ_PREFETCH) * OZ_BK, tn * OZ_BN + (CL > 1 ? rank * (OZ_BN / CL) : 0), bp);
                    }
                    if (++stage == OZ_STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                      // ---- MMA issuer
            int stage = 0, as = 0;
            uint32_t phase = 0, aphase = 0;
            for (long long w = cid; w < total; w += ncl) {
                const int bp = (int)(w / g.T), t = (int)(w - (long long)bp * g.T);
                int um, tn, kb0, kb1;
                oz_unit<CL>(g, t, um, tn);
                oz_krange<CL>(g, um, tn, kb0, kb1);
                mbar_wait(&tempty_bar[as], aphase ^ 1u);
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t dcol = tmem + (uint32_t)(as * OZ_BN);
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&full_bar[stage], phase);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint32_t sa = smem_u32(smem + stage * OZ_STAGE_BYTES);
                    const uint64_t da = oz_desc(sa), db = oz_desc(sa + OZ_A_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < OZ_BK / 32; k4++) {
                        const uint32_t accum = (kb > kb0 || k4 > 0) ? 1u : 0u;
                        asm volatile(
                            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                            "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}\n" ::"r"(dcol),
                            "l"(da + (uint64_t)(k4 * 2)), "l"(db + (uint64_t)(k4 * 2)), "r"(OZ_IDESC), "r"(accum), "r"(0u), "r"(0u),
                            "r"(0u), "r"(0u)
                            : "memory");
                    }
                    if (CL == 1) oz_commit(&empty_bar[stage]);
                    else oz_commit_mc(&empty_bar[stage], MASK);
                    if (++stage == OZ_STAGES) { stage = 0; phase ^= 1u; }
                }
                oz_commit(&tfull_bar[as]);
                as ^= 1;
                if (as == 0) aphase ^= 1u;
            }
        }
    } else {                                  // ---- epilogue: accumulator -> residues mod p -> 8-bit planes
        const int quad = warp & 3;
        int as = 0;
        uint32_t aphase = 0;
        for (long long w = cid; w < total; w += ncl) {
            const int bp = (int)(w / g.T), t = (int)(w - (long long)bp * g.T);
            int um, tn;
            oz_unit<CL>(g, t, um, tn);
            const int tm = um * CL + rank;
            const int a = bp % g.nmod;
            const uint32_t np = g.np[a], m39 = g.m39[a];
            mbar_wait(&tfull_bar[as], aphase);
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            const int row = tm * OZ_BM + quad * 32 + lane;
            uint8_t* drow = g.D + ((size_t)bp * g.M + row) * g.N + (size_t)tn * OZ_BN;
            const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * OZ_BN);
#pragma unroll 1
            for (int c = 0; c < OZ_BN / 32; c++) {
                uint32_t v[32];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                      "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
                      "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
                      "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                    : "r"(tbase + (uint32_t)(c * 32)));
                asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
                uint32_t wv[8];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    uint32_t r[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        const uint32_t x = v[4 * j + e];
                        const uint32_t q = (uint32_t)(((unsigned long long)x * m39) >> 39);
                        r[e] = q * np + x;
                    }
                    wv[j] = oz_pack4(r[0], r[1], r[2], r[3]);
                }
                uint4* d4 = reinterpret_cast<uint4*>(drow + c * 32);
                d4[0] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                d4[1] = make_uint4(wv[4], wv[5], wv[6], wv[7]);
            }
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            mbar_arrive(&tempty_bar[as]);
            as ^= 1;
            if (as == 0) aphase ^= 1u;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (CL > 1) oz_cluster_sync();            // no CTA leaves while its peer can still multicast into it
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "n"(512));
}

// ---------------------------------------------------------------------------------------------- step 3: CRT
struct OzCombArgs {
    int M, N, nmod, lower, accumulate;
    double alpha, P;
    uint32_t f2[OZ_MAXMOD], f1[OZ_MAXMOD], f0[OZ_MAXMOD];
};

// thread: one row, eight consecutive columns (a warp reads 256 contiguous bytes of each residue plane).  V / P =
// frac(sum_i r_i f_i) in 96-bit fixed point: three 64-bit accumulators of 8-bit x 32-bit products, carries resolved once;
// the top 64 bits read as a signed number centre the result in (-P/2, P/2).  NMOD > 0: the loop over the moduli is
// unrolled so that all plane loads are in flight together.
template <int NMOD>
__global__ void __launch_bounds__(256, OZ_COMB_MINB) oz_combine_kernel(const uint8_t* __restrict__ D, const int* __restrict__ sA,
                                                         const int* __restrict__ sB, double* __restrict__ C, int ldc,
                                                         long long sC, const __grid_constant__ OzCombArgs g) {
    const int b = blockIdx.z;
    const int row = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int col = blockIdx.x * 256 + (threadIdx.x & 31) * 8;
    if (g.lower && (col >> 7) > (row >> 7)) return;
    const int nmod = NMOD > 0 ? NMOD : g.nmod;
    const uint8_t* d = D + ((size_t)b * nmod * g.M + row) * g.N + col;
    const size_t plane = (size_t)g.M * g.N;
    unsigned long long a1[8], a0[8];
    uint32_t a2[8];                           // only its low 32 bits reach the result: the sum is taken modulo 1
#pragma unroll
    for (int j = 0; j < 8; j++) { a2[j] = 0u; a1[j] = a0[j] = 0ull; }
    if (NMOD > 0) {
        uint2 w[NMOD > 0 ? NMOD : 1];
#pragma unroll
        for (int a = 0; a < NMOD; a++) w[a] = __ldg(reinterpret_cast<const uint2*>(d + a * plane));
#pragma unroll
        for (int a = 0; a < NMOD; a++) {
            const uint32_t f2 = g.f2[a], f1 = g.f1[a], f0 = g.f0[a];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t r = __byte_perm(j < 4 ? w[a].x : w[a].y, 0u, 0x4440 | (j & 3));
                a2[j] += r * f2;
                a1[j] += (unsigned long long)r * f1;
                a0[j] += (unsigned long long)r * f0;
            }
        }
    } else {
        for (int a = 0; a < nmod; a++) {
            const uint2 w = __ldg(reinterpret_cast<const uint2*>(d + a * plane));
            const uint32_t f2 = g.f2[a], f1 = g.f1[a], f0 = g.f0[a];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t r = __byte_perm(j < 4 ? w.x : w.y, 0u, 0x4440 | (j & 3));
                a2[j] += r * f2;
                a1[j] += (unsigned long long)r * f1;
                a0[j] += (unsigned long long)r * f0;
            }
        }
    }
    const double ra = oz_pow2(-sA[(size_t)b * g.M + row]) * g.P;      // both exact powers of two times P: one rounding below
    const int4 sb0 = *reinterpret_cast<const int4*>(sB + (size_t)b * g.N + col);
    const int4 sb1 = *reinterpret_cast<const int4*>(sB + (size_t)b * g.N + col + 4);
    const int sbv[8] = {sb0.x, sb0.y, sb0.z, sb0.w, sb1.x, sb1.y, sb1.z, sb1.w};
    double out[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const unsigned long long mid = a1[j] + (a0[j] >> 32);
        const uint32_t top = (uint32_t)(a2[j] + (mid >> 32));
        const long long hi64 = (long long)(((unsigned long long)top << 32) | (mid & 0xffffffffull));
        const double frac = fma((double)(uint32_t)a0[j], 0x1p-96, (double)hi64 * 0x1p-64);
        out[j] = frac * ra * oz_pow2(-sbv[j]);
    }
    double* c = C + (size_t)b * sC + (size_t)row * ldc + col;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        double4 v;
        if (g.accumulate) {
            const double4 o = *reinterpret_cast<const double4*>(c + 4 * h);
            v = make_double4(fma(g.alpha, out[4 * h], o.x), fma(g.alpha, out[4 * h + 1], o.y), fma(g.alpha, out[4 * h + 2], o.z),
                             fma(g.alpha, out[4 * h + 3], o.w));
        } else {
            v = make_double4(g.alpha * out[4 * h], g.alpha * out[4 * h + 1], g.alpha * out[4 * h + 2], g.alpha * out[4 * h + 3]);
        }
        *reinterpret_cast<double4*>(c + 4 * h) = v;
    }
}

// The same recombination for the prediction product Z = L^-1 C, of which only the column norms are wanted
// (EPI_SUMSQ of the DMMA kernels): part[ti][col] = sum over the 128 rows of row tile ti of Z^2.  A CTA takes one row tile
// and 256 columns; warp w walks rows 16 w .. 16 w + 15, thread = eight columns; the eight warps' sums meet in shared memory.
template <int NMOD>
__global__ void __launch_bounds__(256, 2) oz_combine_sumsq_kernel(const uint8_t* __restrict__ D, const int* __restrict__ sA,
                                                                              const int* __restrict__ sB, double* __restrict__ part,
                                                                              int ldp, const __grid_constant__ OzCombArgs g) {
    __shared__ double red[8][256 + 8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ti = blockIdx.y;
    const int col = blockIdx.x * 256 + lane * 8;
    const int nmod = NMOD > 0 ? NMOD : g.nmod;
    const size_t plane = (size_t)g.M * g.N;
    const int4 sb0 = *reinterpret_cast<const int4*>(sB + col);
    const int4 sb1 = *reinterpret_cast<const int4*>(sB + col + 4);
    const int sbv[8] = {sb0.x, sb0.y, sb0.z, sb0.w, sb1.x, sb1.y, sb1.z, sb1.w};
    double cs[8], acc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { cs[j] = oz_pow2(-sbv[j]); acc[j] = 0.0; }
    for (int rr = 0; rr < 16; rr++) {
        const int row = ti * 128 + warp * 16 + rr;
        const uint8_t* d = D + (size_t)row * g.N + col;
        unsigned long long a1[8], a0[8];
        uint32_t a2[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { a2[j] = 0u; a1[j] = a0[j] = 0ull; }
        if (NMOD > 0) {
            uint2 w[NMOD > 0 ? NMOD : 1];
#pragma unroll
            for (int a = 0; a < NMOD; a++) w[a] = __ldg(reinterpret_cast<const uint2*>(d + a * plane));
#pragma unroll
            for (int a = 0; a < NMOD; a++) {
                const uint32_t f2 = g.f2[a], f1 = g.f1[a], f0 = g.f0[a];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint32_t r = __byte_perm(j < 4 ? w[a].x : w[a].y, 0u, 0x4440 | (j & 3));
                    a2[j] += r * f2;
                    a1[j] += (unsigned long long)r * f1;
                    a0[j] += (unsigned long long)r * f0;
                }
            }
        } else {
            for (int a = 0; a < nmod; a++) {
                const uint2 w = __ldg(reinterpret_cast<const uint2*>(d + a * plane));
                const uint32_t f2 = g.f2[a], f1 = g.f1[a], f0 = g.f0[a];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint32_t r = __byte_perm(j < 4 ? w.x : w.y, 0u, 0x4440 | (j & 3));
                    a2[j] += r * f2;
                    a1[j] += (unsigned long long)r * f1;
                    a0[j] += (unsigned long long)r * f0;
                }
            }
        }
        const double ra = oz_pow2(-sA[row]) * g.P;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const unsigned long long mid = a1[j] + (a0[j] >> 32);
            const uint32_t top = (uint32_t)(a2[j] + (mid >> 32));
            const long long hi64 = (long long)(((unsigned long long)top << 32) | (mid & 0xffffffffull));
            const double frac = fma((double)(uint32_t)a0[j], 0x1p-96, (double)hi64 * 0x1p-64);
            const double z = frac * ra * cs[j];
            acc[j] = fma(z, z, acc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < 8; j++) red[warp][lane * 8 + j] = acc[j];
    __syncthreads();
    {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; w++) s += red[w][threadIdx.x];
        part[(size_t)ti * ldp + blockIdx.x * 256 + threadIdx.x] = s;
    }
}

// Row norms: the prediction product with its roles swapped, Z^T = C^T L^-T (rows = points, columns = training points), so
// that the triangular factor sits on the column side, where the k range of a unit is exact to 256 whatever the cluster size.
// out[row] = sum over all N columns of (Z^T)^2.  A warp takes one row at a time (ROWS_PER_CTA / 8 rows per warp), a lane eight
// consecutive columns of each 256-column segment; the lanes' sums meet by shuffles.
constexpr int OZ_RS_ROWS = 32;
template <int NMOD>
__global__ void __launch_bounds__(256, 2) oz_combine_rowsumsq_kernel(const uint8_t* __restrict__ D, const int* __restrict__ sA,
                                                                     const int* __restrict__ sB, double* __restrict__ out,
                                                                     const __grid_constant__ OzCombArgs g) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nmod = NMOD > 0 ? NMOD : g.nmod;
    const size_t plane = (size_t)g.M * g.N;
    for (int rr = 0; rr < OZ_RS_ROWS / 8; rr++) {
        const int row = blockIdx.x * OZ_RS_ROWS + rr * 8 + warp;
        double acc = 0.0;
        for (int c0 = 0; c0 < g.N; c0 += 256) {
            const int col = c0 + lane * 8;
            const uint8_t* d = D + (size_t)row * g.N + col;
            unsigned long long a1[8], a0[8];
            uint32_t a2[8];
#pragma unroll
            for (int j = 0; j < 8; j++) { a2[j] = 0u; a1[j] = a0[j] = 0ull; }
            if (NMOD > 0) {
                uint2 w[NMOD > 0 ? NMOD : 1];
#pragma unroll
                for (int a = 0; a < NMOD; a++) w[a] = __ldg(reinterpret_cast<const uint2*>(d + a * plane));
#pragma unroll
                for (int a = 0; a < NMOD; a++) {
                    const uint32_t f2 = g.f2[a], f1 = g.f1[a], f0 = g.f0[a];
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const uint32_t r = __byte_perm(j < 4 ? w[a].x : w[a].y, 0u, 0x4440 | (j & 3));
                        a2[j] += r * f2;
                        a1[j] += (unsigned long long)r * f1;
                        a0[j] += (unsigned long long)r * f0;
                    }
                }
            } else {
                for (int a = 0; a < nmod; a++) {
                    const uint2 w = __ldg(reinterpret_cast<const uint2*>(d + a * plane));
                    const uint32_t f2 = g.f2[a], f1 = g.f1[a], f0 = g.f0[a];
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const uint32_t r = __byte_perm(j < 4 ? w.x : w.y, 0u, 0x4440 | (j & 3));
                        a2[j] += r * f2;
                        a1[j] += (unsigned long long)r * f1;
                        a0[j] += (unsigned long long)r * f0;
                    }
                }
            }
            const int4 sb0 = *reinterpret_cast<const int4*>(sB + col);
            const int4 sb1 = *reinterpret_cast<const int4*>(sB + col + 4);
            const int sbv[8] = {sb0.x, sb0.y, sb0.z, sb0.w, sb1.x, sb1.y, sb1.z, sb1.w};
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const unsigned long long mid = a1[j] + (a0[j] >> 32);
                const uint32_t top = (uint32_t)(a2[j] + (mid >> 32));
                const long long hi64 = (long long)(((unsigned long long)top << 32) | (mid & 0xffffffffull));
                const double frac = fma((double)(uint32_t)a0[j], 0x1p-96, (double)hi64 * 0x1p-64);
                const double z = frac * g.P * oz_pow2(-sbv[j]);      // the row's own scale is applied once, to the sum
                acc = fma(z, z, acc);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            const double ra = oz_pow2(-sA[row]);
            out[row] = acc * ra * ra;
        }
    }
}

// ---------------------------------------------------------------------------------------------- host side
void OzWs::release() {
    cudaFree(PA); cudaFree(PB); cudaFree(PD); cudaFree(sA); cudaFree(sB);
    PA = PB = PD = nullptr; sA = sB = nullptr;
    capA = capB = capD = capS = 0;
}

bool oz_supported(const GemmP& p, int epi) {
    if (epi == EPI_SUMSQ) {     // column norms of a single product (prediction): partials [M / 128][N]
        if (p.batch != 1 || p.lower || p.accumulate) return false;
    } else if (epi != EPI_STORE) {
        return false;
    }
    if (p.M % OZ_BM || p.N % OZ_BN || p.K % OZ_BK || p.K > 32768) return false;
    if ((p.kmode == KM_LE_J || p.kmode == KM_GE_J) && p.K != p.N) return false;
    if ((p.kmode == KM_LE_I || p.kmode == KM_GE_I) && p.K != p.M) return false;
    if (p.lower && p.M != p.N) return false;
    if (epi == EPI_STORE && (p.ldc % 4 || ((uintptr_t)p.C & 31) || (p.sC % 4))) return false;
    if (p.lda % 2 || p.ldb % 2 || ((uintptr_t)p.A & 15) || ((uintptr_t)p.B & 15) || (p.sA % 2) || (p.sB % 2)) return false;
    return true;
}

bool oz_sumsq_swapped(const GemmP& p, int epi) {
    return epi == EPI_SUMSQ && p.kmode == KM_LE_I && p.M % OZ_BN == 0 && p.N % OZ_BM == 0 && p.N % OZ_RS_ROWS == 0;
}

static bool same_operand(const GemmP& p, int layout) {
    return p.A == p.B && p.lda == p.ldb && p.sA == p.sB && p.M == p.N && layout != GEMM_NN;
}

cudaError_t oz_reserve(OzWs& ws, const GemmP& p, int layout, int nmod) {
    const bool same = same_operand(p, layout);
    const size_t needA = (size_t)p.batch * nmod * p.M * p.K, needB = same ? 0 : (size_t)p.batch * nmod * p.N * p.K;
    const size_t needD = (size_t)p.batch * nmod * p.M * p.N, needS = (size_t)p.batch * (size_t)(p.M > p.N ? p.M : p.N);
    auto grown = [&]() { ws.have_a = false; ws.grew = true; };
    auto grow = [&](uint8_t*& ptr, size_t& cap, size_t need) -> cudaError_t {
        if (need <= cap) return cudaSuccess;
        grown();
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&ptr, need);
        if (e == cudaSuccess) cap = need;
        return e;
    };
    cudaError_t e;
    if ((e = grow(ws.PA, ws.capA, needA)) != cudaSuccess) return e;
    if ((e = grow(ws.PB, ws.capB, needB)) != cudaSuccess) return e;
    if ((e = grow(ws.PD, ws.capD, needD)) != cudaSuccess) return e;
    if (needS > ws.capS) {
        grown();
        cudaFree(ws.sA); cudaFree(ws.sB);
        ws.sA = ws.sB = nullptr;
        ws.capS = 0;
        if ((e = cudaMalloc(&ws.sA, needS * sizeof(int))) != cudaSuccess) return e;
        if ((e = cudaMalloc(&ws.sB, needS * sizeof(int))) != cudaSuccess) return e;
        ws.capS = needS;
    }
    return cudaSuccess;
}

typedef CUresult (*OzEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static OzEncodeFn encode_fn() {
    static OzEncodeFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* f = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<OzEncodeFn>(f);
    }
    return fn;
}

// 3-D map over residue planes [nbp][R][K] bytes: box = 128 bytes of k x `rows` rows x 1 plane, 128-byte swizzle
static cudaError_t make_map(CUtensorMap* out, const uint8_t* base, int K, int R, int nbp, int rows) {
    OzEncodeFn fn = encode_fn();
    if (!fn) return cudaErrorNotSupported;
    const cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)R, (cuuint64_t)nbp};
    const cuuint64_t gstr[2] = {(cuuint64_t)K, (cuuint64_t)K * (cuuint64_t)R};
    const cuuint32_t box[3] = {(cuuint32_t)OZ_BK, (cuuint32_t)rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

static cudaError_t launch_convert(bool kc, const double* src, int ld, long long sS, int R, int K, int nmod, int bits, int tri,
                                  uint8_t* planes, int* sexp, int batch, cudaStream_t st, double fixed_max = 0.0) {
    if (kc) {
        dim3 grid((R + 7) / 8, batch);
        oz_convert_kc_kernel<<<grid, 256, 0, st>>>(src, ld, sS, R, K, nmod, bits, tri, planes, sexp, fixed_max);
    } else {
        dim3 grid(R / 32, batch);
        oz_convert_t_kernel<<<grid, 256, 0, st>>>(src, ld, sS, R, K, nmod, bits, tri, planes, sexp, fixed_max);
    }
    return cudaGetLastError();
}

cudaError_t oz_gemm(const GemmP& p, int layout, int epi, int nmod, OzWs& ws, cudaStream_t st, const OzHint& hint, const OzHook& hook) {
    if (nmod < 2 || nmod > OZ_MAXMOD || !oz_supported(p, epi)) return cudaErrorInvalidValue;
    cudaError_t e;
    if ((e = upload_const()) != cudaSuccess) return e;
    static OzCrt crt[OZ_MAXMOD + 1];
    static bool have_crt[OZ_MAXMOD + 1] = {false};
    static OzConst hc = make_const();
    {   // (two handles may be driven from two host threads)
        static std::mutex crt_mu;
        std::lock_guard<std::mutex> lk(crt_mu);
        if (!have_crt[nmod]) { crt[nmod] = make_crt(nmod); have_crt[nmod] = true; }
    }
    const bool same = same_operand(p, layout);
    if ((e = oz_reserve(ws, p, layout, nmod)) != cudaSuccess) return e;
    const int bits = oz_operand_bits(nmod, p.K);
    const bool a_kc = layout != GEMM_TN, b_kc = layout == GEMM_NT;
    // column norms of Z = A B with A lower triangular (prediction): run as Z^T = B^T A^T, the triangular factor on the column side
    const bool swap = oz_sumsq_swapped(p, epi);
    // cluster size of the residue GEMM: pairs wherever the row tiles pair up.  Quadruples cut the L2 -> SM traffic further (24
    // instead of 32 KB per k block) but only 33 of them are resident at once (132 of the 148 SMs: the GPCs' SM counts are not
    // multiples of four) and row-triangular operands are then converted and read in 512-row granules; same-box A/B at n = 4096,
    // 32 items: 44.4-44.9 (pairs) against 45.4-45.9 ms per step; the prediction product (one item, 65 536 columns, k <= i)
    // 13.6 Mpred/s with pairs against 13.35 with quadruples
    const int tiles_m = (swap ? p.N : p.M) / OZ_BM;
    const int CL = tiles_m % 2 == 0 ? 2 : 1;
    // k ranges of triangular operands (zero blocks are neither converted nor read): granule = rows of the GEMM's work unit
    const int gA = swap ? OZ_BN : std::max(OZ_BM * CL, same ? OZ_BN : 0);
    const int triA = p.kmode == KM_LE_I ? gA : (p.kmode == KM_GE_I ? -gA : 0);
    const int triB = p.kmode == KM_LE_J ? OZ_BN : (p.kmode == KM_GE_J ? -OZ_BN : 0);
    hook(0, true, st);
    const OzWs::Key keyA{p.A, p.lda, p.sA, p.M, p.K, p.batch, nmod, bits, triA, a_kc ? 1 : 0};
    if (!(hint.reuse_a && ws.have_a && ws.key_a == keyA && ws.tag_a == hint.a_tag)) {
        if ((e = launch_convert(a_kc, p.A, p.lda, p.sA, p.M, p.K, nmod, bits, triA, ws.PA, ws.sA, p.batch, st)) != cudaSuccess) return e;
    }
    ws.key_a = keyA;
    ws.tag_a = hint.a_tag;
    ws.have_a = true;
    const uint8_t* PBp = ws.PA;
    const int* sBp = ws.sA;
    if (!same) {
        if ((e = launch_convert(b_kc, p.B, p.ldb, p.sB, p.N, p.K, nmod, bits, triB, ws.PB, ws.sB, p.batch, st, hint.b_bound)) != cudaSuccess)
            return e;
        PBp = ws.PB;
        sBp = ws.sB;
    }
    hook(0, false, st);
    // residue GEMM
    hook(1, true, st);
    CUtensorMap tmA, tmB;
    const int nbp = p.batch * nmod;
    OzGemmArgs g;
    if (swap) {
        if ((e = make_map(&tmA, PBp, p.K, p.N, nbp, OZ_BM)) != cudaSuccess) return e;
        g.M = p.N; g.N = p.M; g.kmode = KM_LE_J;
        g.tiles_m = p.N / OZ_BM; g.tiles_n = p.M / OZ_BN;
        if ((e = make_map(&tmB, ws.PA, p.K, p.M, nbp, OZ_BN / CL)) != cudaSuccess) return e;
    } else {
        if ((e = make_map(&tmA, ws.PA, p.K, p.M, nbp, OZ_BM)) != cudaSuccess) return e;
        g.M = p.M; g.N = p.N; g.kmode = p.kmode;
        g.tiles_m = p.M / OZ_BM; g.tiles_n = p.N / OZ_BN;
        if ((e = make_map(&tmB, PBp, p.K, p.N, nbp, OZ_BN / CL)) != cudaSuccess) return e;
    }
    g.K = p.K; g.nmod = nmod; g.nbp = nbp; g.lower = p.lower;
    g.nmajor = (!p.lower && (swap || (p.kmode == KM_LE_I && g.tiles_n > 2 * (g.tiles_m / CL)))) ? 1 : 0;
    const int units_m = g.tiles_m / CL;
    if (p.lower) {
        int T = 0;
        for (int r = 0; r < units_m; r++) T += std::min(g.tiles_n, (r * CL + CL - 1) / 2 + 1);
        g.T = T;
    } else {
        g.T = units_m * g.tiles_n;
    }
    g.D = ws.PD;
    for (int a = 0; a < OZ_MAXMOD; a++) { g.p[a] = hc.p[a]; g.m39[a] = hc.m39[a]; g.np[a] = hc.np[a]; }
    const long long total = (long long)nbp * g.T;
    if (CL == 1) {
        static SmemOptIn optin;
        if ((e = optin.ensure(oz_gemm_kernel<1>, OZ_SMEM)) != cudaSuccess) return e;
        const int grid = (int)std::min<long long>(NUM_SMS, total);
        oz_gemm_kernel<1><<<grid, OZ_THREADS, OZ_SMEM, st>>>(tmA, tmB, g);
    } else {
        static SmemOptIn optin2;
        if ((e = optin2.ensure(oz_gemm_kernel<2>, OZ_SMEM)) != cudaSuccess) return e;
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.blockDim = dim3(OZ_THREADS); cfg.dynamicSmemBytes = OZ_SMEM; cfg.stream = st; cfg.attrs = attr; cfg.numAttrs = 1;
        static int max_clusters[16] = {0};
        int dev = 0;
        cudaGetDevice(&dev);
        int& mc = max_clusters[dev & 15];
        if (!mc) {       // clusters that are resident at once: a persistent grid must not exceed them
            cfg.gridDim = dim3(NUM_SMS / CL * CL);
            int n = 0;
            cudaError_t qe = cudaOccupancyMaxActiveClusters(&n, oz_gemm_kernel<2>, &cfg);
            if (qe != cudaSuccess || n < 1) n = NUM_SMS / CL - 4;
            mc = std::min(n, NUM_SMS / CL);
            if (getenv("GPE_OZAKI_VERBOSE")) fprintf(stderr, "oz_gemm: cluster %d, %d clusters resident\n", CL, mc);
        }
        const int ncl = (int)std::min<long long>(mc, total);
        cfg.gridDim = dim3(CL * ncl);
        if ((e = cudaLaunchKernelEx(&cfg, oz_gemm_kernel<2>, tmA, tmB, g)) != cudaSuccess) return e;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    hook(1, false, st);
    // CRT + scale + store
    hook(2, true, st);
    OzCombArgs c;
    c.M = p.M; c.N = p.N; c.nmod = nmod; c.lower = p.lower; c.accumulate = p.accumulate; c.alpha = p.alpha; c.P = crt[nmod].P;
    for (int a = 0; a < OZ_MAXMOD; a++) { c.f2[a] = crt[nmod].f2[a]; c.f1[a] = crt[nmod].f1[a]; c.f0[a] = crt[nmod].f0[a]; }
    if (swap) {
        c.M = p.N; c.N = p.M;
        const unsigned rgrid = (unsigned)(p.N / OZ_RS_ROWS);
        switch (nmod) {
            case 14: oz_combine_rowsumsq_kernel<14><<<rgrid, 256, 0, st>>>(ws.PD, sBp, ws.sA, p.C, c); break;
            case 15: oz_combine_rowsumsq_kernel<15><<<rgrid, 256, 0, st>>>(ws.PD, sBp, ws.sA, p.C, c); break;
            case 16: oz_combine_rowsumsq_kernel<16><<<rgrid, 256, 0, st>>>(ws.PD, sBp, ws.sA, p.C, c); break;
            case 17: oz_combine_rowsumsq_kernel<17><<<rgrid, 256, 0, st>>>(ws.PD, sBp, ws.sA, p.C, c); break;
            case 18: oz_combine_rowsumsq_kernel<18><<<rgrid, 256, 0, st>>>(ws.PD, sBp, ws.sA, p.C, c); break;
            default: oz_combine_rowsumsq_kernel<0><<<rgrid, 256, 0, st>>>(ws.PD, sBp, ws.sA, p.C, c); break;
        }
        hook(2, false, st);
        return cudaGetLastError();
    }
    if (epi == EPI_SUMSQ) {
        dim3 sgrid(p.N / 256, p.M / 128);
        switch (nmod) {
            case 14: oz_combine_sumsq_kernel<14><<<sgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, c); break;
            case 15: oz_combine_sumsq_kernel<15><<<sgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, c); break;
            case 16: oz_combine_sumsq_kernel<16><<<sgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, c); break;
            case 17: oz_combine_sumsq_kernel<17><<<sgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, c); break;
            case 18: oz_combine_sumsq_kernel<18><<<sgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, c); break;
            default: oz_combine_sumsq_kernel<0><<<sgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, c); break;
        }
        hook(2, false, st);
        return cudaGetLastError();
    }
    dim3 cgrid(p.N / 256, p.M / 8, p.batch);
    switch (nmod) {
        case 14: oz_combine_kernel<14><<<cgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, p.sC, c); break;
        case 15: oz_combine_kernel<15><<<cgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, p.sC, c); break;
        case 16: oz_combine_kernel<16><<<cgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, p.sC, c); break;
        case 17: oz_combine_kernel<17><<<cgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, p.sC, c); break;
        case 18: oz_combine_kernel<18><<<cgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, p.sC, c); break;
        default: oz_combine_kernel<0><<<cgrid, 256, 0, st>>>(ws.PD, ws.sA, sBp, p.C, p.ldc, p.sC, c); break;
    }
    hook(2, false, st);
    return cudaGetLastError();
}

}  // namespace gpe
