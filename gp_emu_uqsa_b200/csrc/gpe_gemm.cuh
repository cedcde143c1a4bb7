// Batched FP64 GEMM family on the FP64 tensor pipe (DMMA.8x8x4 via mma.sync.m8n8k4.f64).
//
// One kernel template serves every dense contraction on the hot path -- the SYRK/TRMM
// updates of the recursive Cholesky+inverse, LAUUM (A^-1 = L^-T L^-1), the skinny
// triangular products for the GLS mean, and the prediction product Z = L^-1 C -- by
//   * choosing how each operand is stored (K-contiguous or M/N-contiguous), which only
//     changes the shared-memory indexing of the fragment loads (no transposes are made),
//   * restricting the K range per output tile (triangular operands: zero tiles skipped),
//   * optionally computing only tiles that touch the lower triangle of C.
// tcgen05/UMMA has no FP64 kind, so FP64 tiles are fed Ampere-style: cp.async (LDGSTS) 16-byte
// copies into padded shared memory (row stride == 4 mod 16 doubles => the 8-byte fragment
// loads of a half-warp hit 16 distinct bank pairs), 4-stage pipeline, one barrier per k-tile.
// Measured roof (tools/ub_fp64.cu on B200): 37.2 TFLOP/s, DMMA == DFMA peak.
#pragma once
#include "gpe_common.cuh"
#include <cstdlib>

namespace gpe {

enum KMode : int {
    KM_FULL = 0,
    KM_LE_J = 1,  // k <  (tj+1)*BN   (B lower-triangular, stored [n][k])
    KM_GE_J = 2,  // k >= tj*BN       (B lower-triangular, stored [k][n])
    KM_LE_I = 3,  // k <  (ti+1)*BM   (A lower-triangular, stored [m][k])
    KM_GE_I = 4,  // k >= ti*BM       (A lower-triangular, stored [k][m])
};

enum Epi : int {
    EPI_STORE = 0,  // C = alpha*acc (+ C)
    EPI_SUMSQ = 1,  // part[b][ti][col] = sum_rows acc^2   (column norms of Z = L^-1 C)
};

// How the operands of launch_gemm are stored: A [M][K] or, transposed, [K][M]; B [N][K] or, not transposed, [K][N].
enum Layout : int {
    GEMM_NT = 0,  // C = A B^T   (A [M][K], B [N][K]: both K-contiguous)
    GEMM_NN = 1,  // C = A B     (A [M][K], B [K][N])
    GEMM_TN = 2,  // C = A^T B   (A [K][M], B [K][N])
};

struct GemmP {
    const double* A;
    const double* B;
    double* C;          // EPI_SUMSQ: partial buffer [batch][tiles_m][N]
    int lda, ldb, ldc;  // leading dimensions (elements)
    long long sA = 0, sB = 0, sC = 0;  // batch strides (elements)
    int M, N, K;
    double alpha = 1.0;
    int accumulate = 0;  // 1: C += alpha*acc
    int kmode = KM_FULL;
    int lower = 0;  // 1: skip tiles strictly above the diagonal (square C)
    int batch = 1;
};

constexpr int GEMM_BK = 16;
constexpr int GEMM_STAGES = 4;

template <int ROWS, bool KC>
struct TileShape {
    static constexpr int LD = KC ? (GEMM_BK + 4) : (ROWS + 4);
    static constexpr int ELEMS = KC ? ROWS * LD : GEMM_BK * LD;
};

// Issue the cp.async copies of one operand tile.  KC: g -> element (row0, k0), row stride ld.
// !KC: g -> element (k0, row0), k stride ld.
template <int ROWS, bool KC, int NT>
__device__ __forceinline__ void load_tile(double* s, const double* __restrict__ g, int ld, int tid) {
    constexpr int LD = TileShape<ROWS, KC>::LD;
    if (KC) {
        constexpr int CH = ROWS * (GEMM_BK / 2);
#pragma unroll
        for (int c = tid; c < CH; c += NT) {
            int row = c >> 3, c2 = c & 7;
            cp_async16(s + row * LD + c2 * 2, g + (size_t)row * ld + c2 * 2);
        }
    } else {
        constexpr int CPR = ROWS / 2;
        constexpr int CH = GEMM_BK * CPR;
#pragma unroll
        for (int c = tid; c < CH; c += NT) {
            int kr = c / CPR, c2 = c % CPR;
            cp_async16(s + kr * LD + c2 * 2, g + (size_t)kr * ld + c2 * 2);
        }
    }
}

// Producer-warp flavour: one warp copies the whole tile; modest unrolling keeps its register
// footprint below the consumers' so the kernel-wide allocation is set by the math warps.
template <int ROWS, bool KC>
__device__ __forceinline__ void load_tile_warp(double* s, const double* __restrict__ g, int ld, int lane) {
    constexpr int LD = TileShape<ROWS, KC>::LD;
    if (KC) {
        const int c2 = lane & 7, r0 = lane >> 3;           // 4 rows x 8 chunks per pass
        const double* gp = g + (size_t)r0 * ld + c2 * 2;
        double* sp = s + r0 * LD + c2 * 2;
#pragma unroll 8
        for (int it = 0; it < ROWS / 4; it++) {
            cp_async16(sp, gp);
            gp += (size_t)4 * ld;
            sp += 4 * LD;
        }
    } else {
        constexpr int CPR = ROWS / 2;                       // chunks per k-row
        constexpr int PASSES = CPR / 32;
#pragma unroll 4
        for (int kr = 0; kr < GEMM_BK; kr++) {
#pragma unroll
            for (int ps = 0; ps < PASSES; ps++) {
                int c2 = lane + 32 * ps;
                cp_async16(s + kr * LD + c2 * 2, g + (size_t)kr * ld + c2 * 2);
            }
        }
    }
}

template <int BM, int BN, int WMW, int WNW, bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(WMW* WNW * 32, 1) gemm_dmma_kernel(GemmP p) {
    constexpr int NT = WMW * WNW * 32;
    constexpr int WTM = BM / WMW, WTN = BN / WNW;
    constexpr int FM = WTM / 8, FN = WTN / 8;
    constexpr int A_EL = TileShape<BM, A_KC>::ELEMS, B_EL = TileShape<BN, B_KC>::ELEMS;
    constexpr int A_LD = TileShape<BM, A_KC>::LD, B_LD = TileShape<BN, B_KC>::LD;
    extern __shared__ __align__(16) double smem[];

    // Heaviest tiles first: with a triangular operand the k-range grows with tj (KM_LE_J) or ti (KM_LE_I);
    // walking those indices downwards leaves the short tiles for the tail of the launch
    // (B200: TRMM 8.80 -> 8.68 ms at n = 2048 x 32 items, prediction 6.86 -> 6.98 Mpred/s).
    const int tj = (p.kmode == KM_LE_J) ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
    const int ti = (p.kmode == KM_LE_I) ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y;
    const int b = blockIdx.z;
    if (p.lower && (ti + 1) * BM <= tj * BN) return;
    const int m0 = ti * BM, n0 = tj * BN;

    int kbeg = 0, kend = p.K;
    switch (p.kmode) {
        case KM_LE_J: kend = min(p.K, (tj + 1) * BN); break;
        case KM_GE_J: kbeg = min(p.K, tj * BN); break;
        case KM_LE_I: kend = min(p.K, (ti + 1) * BM); break;
        case KM_GE_I: kbeg = min(p.K, ti * BM); break;
        default: break;
    }
    const int KT = (kend - kbeg + GEMM_BK - 1) / GEMM_BK;

    const double* Ag = p.A + (size_t)b * p.sA + (A_KC ? ((size_t)m0 * p.lda + kbeg) : ((size_t)kbeg * p.lda + m0));
    const double* Bg = p.B + (size_t)b * p.sB + (B_KC ? ((size_t)n0 * p.ldb + kbeg) : ((size_t)kbeg * p.ldb + n0));
    const size_t a_kstep = A_KC ? (size_t)GEMM_BK : (size_t)GEMM_BK * p.lda;
    const size_t b_kstep = B_KC ? (size_t)GEMM_BK : (size_t)GEMM_BK * p.ldb;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm0 = (warp / WNW) * WTM, wn0 = (warp % WNW) * WTN;
    const int fr = lane >> 2, fc = lane & 3;

    double acc[FM][FN][2];
#pragma unroll
    for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    double* As = smem;
    double* Bs = smem + GEMM_STAGES * A_EL;

#pragma unroll
    for (int s = 0; s < GEMM_STAGES - 1; s++) {
        if (s < KT) {
            load_tile<BM, A_KC, NT>(As + s * A_EL, Ag + s * a_kstep, p.lda, tid);
            load_tile<BN, B_KC, NT>(Bs + s * B_EL, Bg + s * b_kstep, p.ldb, tid);
        }
        cp_async_commit();
    }

    // fragment base offsets inside a stage
    const int a_off = A_KC ? ((wm0 + fr) * A_LD + fc) : (fc * A_LD + wm0 + fr);
    const int b_off = B_KC ? ((wn0 + fr) * B_LD + fc) : (fc * B_LD + wn0 + fr);
    constexpr int a_fstep = A_KC ? 8 * A_LD : 8;      // next 8-row fragment
    constexpr int b_fstep = B_KC ? 8 * B_LD : 8;
    constexpr int a_kk = A_KC ? 4 : 4 * A_LD;         // next k4 step
    constexpr int b_kk = B_KC ? 4 : 4 * B_LD;

    for (int kt = 0; kt < KT; kt++) {
        cp_async_wait<GEMM_STAGES - 2>();
        __syncthreads();
        {
            int nk = kt + GEMM_STAGES - 1;
            if (nk < KT) {
                int s = nk % GEMM_STAGES;
                load_tile<BM, A_KC, NT>(As + s * A_EL, Ag + nk * a_kstep, p.lda, tid);
                load_tile<BN, B_KC, NT>(Bs + s * B_EL, Bg + nk * b_kstep, p.ldb, tid);
            }
            cp_async_commit();
        }
        const double* at = As + (kt % GEMM_STAGES) * A_EL + a_off;
        const double* bt = Bs + (kt % GEMM_STAGES) * B_EL + b_off;
#pragma unroll
        for (int kk = 0; kk < GEMM_BK / 4; kk++) {
            double af[FM], bf[FN];
#pragma unroll
            for (int i = 0; i < FM; i++) af[i] = at[kk * a_kk + i * a_fstep];
#pragma unroll
            for (int j = 0; j < FN; j++) bf[j] = bt[kk * b_kk + j * b_fstep];
#pragma unroll
            for (int i = 0; i < FM; i++)
#pragma unroll
                for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
    }
    cp_async_wait<0>();

    if (EPI == EPI_STORE) {
        double* Cg = p.C + (size_t)b * p.sC + (size_t)(m0 + wm0 + fr) * p.ldc + n0 + wn0 + 2 * fc;
#pragma unroll
        for (int i = 0; i < FM; i++)
#pragma unroll
            for (int j = 0; j < FN; j++) {
                double2* dst = reinterpret_cast<double2*>(Cg + (size_t)(8 * i) * p.ldc + 8 * j);
                double2 v;
                v.x = p.alpha * acc[i][j][0];
                v.y = p.alpha * acc[i][j][1];
                if (p.accumulate) {
                    double2 o = *dst;
                    v.x += o.x;
                    v.y += o.y;
                }
                *dst = v;
            }
    } else {
        // column sums of squares over this tile's BM rows -> part[b][ti][n0 + col]
        __syncthreads();                 // all warps are done with the operand stages
        double* red = smem;              // [WMW][BN]
#pragma unroll
        for (int j = 0; j < FN; j++) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int i = 0; i < FM; i++) {
                s0 = fma(acc[i][j][0], acc[i][j][0], s0);
                s1 = fma(acc[i][j][1], acc[i][j][1], s1);
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (fr == 0) {
                red[(warp / WNW) * BN + wn0 + 8 * j + 2 * fc] = s0;
                red[(warp / WNW) * BN + wn0 + 8 * j + 2 * fc + 1] = s1;
            }
        }
        __syncthreads();
        for (int c = tid; c < BN; c += NT) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < WMW; w++) s += red[w * BN + c];
            p.C[(size_t)b * p.sC + (size_t)ti * p.ldc + n0 + c] = s;
        }
    }
}

template <int BM, int BN, bool A_KC, bool B_KC>
constexpr size_t gemm_smem_bytes() {
    return (size_t)GEMM_STAGES * (TileShape<BM, A_KC>::ELEMS + TileShape<BN, B_KC>::ELEMS) * sizeof(double);
}

template <int BM, int BN, int WMW, int WNW, bool A_KC, bool B_KC, int EPI>
inline cudaError_t launch_gemm_cfg(const GemmP& p, cudaStream_t st) {
    auto kern = gemm_dmma_kernel<BM, BN, WMW, WNW, A_KC, B_KC, EPI>;
    constexpr size_t smem = gemm_smem_bytes<BM, BN, A_KC, B_KC>();
    static SmemOptIn optin;
    if (cudaError_t e = optin.ensure(kern, smem); e != cudaSuccess) return e;
    if (p.M % BM || p.N % BN || p.K % GEMM_BK) return cudaErrorInvalidValue;
    dim3 grid(p.N / BN, p.M / BM, p.batch);
    kern<<<grid, WMW * WNW * 32, smem, st>>>(p);
    return cudaGetLastError();
}


// ------------------------------------------------------------------------------------------------
// Warp-specialised 128x128 variant (the hot configuration): 8 consumer warps (2x4, warp tile 64x32,
// 32 DMMA per k4 step) + 1 producer warp that issues every cp.async of the tile.  Stages are handed
// over with mbarriers (full: cp.async.mbarrier.arrive.noinc by the 32 producer lanes; empty: one
// arrive per consumer warp), so there is no block-wide barrier in the main loop: consumer warps
// drift apart and keep the FP64 tensor pipe fed while others wait, and the LSU back-pressure /
// address arithmetic of the copies never stalls a math warp (ncu r01: barrier 5.8 % + long-scoreboard
// 5.2 % of samples in the single-role kernel).
constexpr int WS_CONSUMERS = 8;
constexpr int WS_COLGROUP = 16;      // column blocks per L2-resident group of a row-triangular launch
constexpr int WS_THREADS = (WS_CONSUMERS + 1) * 32;

// WMW = warp rows of the 8 math warps: 2 -> 2x4 warps of 64x32 (column-triangular and dense launches),
// 4 -> 4x2 warps of 32x64 (row-triangular launches: four row levels for the per-warp k range below).
template <bool A_KC, bool B_KC, int EPI, int WMW = 2>
__global__ void __launch_bounds__(WS_THREADS, 1) gemm_dmma_ws_kernel(GemmP p) {
    constexpr int BM = 128, BN = 128, WNW = WS_CONSUMERS / WMW;
    constexpr int WTM = BM / WMW, WTN = BN / WNW, FM = WTM / 8, FN = WTN / 8;
    constexpr int A_EL = TileShape<BM, A_KC>::ELEMS, B_EL = TileShape<BN, B_KC>::ELEMS;
    constexpr int A_LD = TileShape<BM, A_KC>::LD, B_LD = TileShape<BN, B_KC>::LD;
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) uint64_t full_bar[GEMM_STAGES], empty_bar[GEMM_STAGES];

    // Heaviest tiles first: with a triangular operand the k-range grows with tj (KM_LE_J) or ti (KM_LE_I);
    // walking those indices downwards leaves the short tiles for the tail of the launch
    // (B200: TRMM 8.80 -> 8.68 ms at n = 2048 x 32 items, prediction 6.86 -> 6.98 Mpred/s).
    // Tile order.  Column-triangular / dense launches: column index fastest, heaviest columns first.
    // Row-triangular launches (k <= i, k >= i; 1-D grid): column blocks are taken in groups of WS_COLGROUP;
    // inside a group the row index runs from the heaviest to the lightest tile and the column index fastest,
    // so (a) the group's slice of B (<= 32 MB at 2048 rows) is read from HBM once and then served from L2 to all row tiles --
    // with the plain column-fastest order every row tile streamed B from HBM again: ncu on the prediction
    // product Z = L^-1 C showed 9.18 GB of DRAM reads per 65 536-point chunk for a 1.07 GB operand, L2 hit rate
    // 47 % -- and (b) the launch still ends on its shortest tiles.
    const bool rowtri = (p.kmode == KM_LE_I || p.kmode == KM_GE_I);
    int tj, ti;
    if (rowtri) {
        const int ntx = p.N / BN, nty = (p.M + BM - 1) / BM, id = (int)blockIdx.x;
        const int full = (ntx / WS_COLGROUP) * WS_COLGROUP * nty;      // CTAs in complete groups
        int g0, gsz, r;
        if (id < full) { g0 = (id / (WS_COLGROUP * nty)) * WS_COLGROUP; gsz = WS_COLGROUP; r = id % (WS_COLGROUP * nty); }
        else { g0 = (ntx / WS_COLGROUP) * WS_COLGROUP; gsz = ntx - g0; r = id - full; }
        const int y = r / gsz;
        tj = g0 + (r - y * gsz);
        ti = (p.kmode == KM_LE_I) ? nty - 1 - y : y;
    } else {
        tj = (p.kmode == KM_LE_J) ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
        ti = (int)blockIdx.y;
    }
    const int b = blockIdx.z;
    if (p.lower && (ti + 1) * BM <= tj * BN) return;
    const int m0 = ti * BM, n0 = tj * BN;
    int kbeg = 0, kend = p.K;
    switch (p.kmode) {
        case KM_LE_J: kend = min(p.K, (tj + 1) * BN); break;
        case KM_GE_J: kbeg = min(p.K, tj * BN); break;
        case KM_LE_I: kend = min(p.K, (ti + 1) * BM); break;
        case KM_GE_I: kbeg = min(p.K, ti * BM); break;
        default: break;
    }
    const int KT = (kend - kbeg + GEMM_BK - 1) / GEMM_BK;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < GEMM_STAGES; s++) {
            mbar_init(&full_bar[s], 32);
            mbar_init(&empty_bar[s], WS_CONSUMERS);
        }
    }
    __syncthreads();

    double* As = smem;
    double* Bs = smem + GEMM_STAGES * A_EL;

    if (warp == WS_CONSUMERS) {
        // ===== producer warp =====
        const double* Ag = p.A + (size_t)b * p.sA + (A_KC ? ((size_t)m0 * p.lda + kbeg) : ((size_t)kbeg * p.lda + m0));
        const double* Bg = p.B + (size_t)b * p.sB + (B_KC ? ((size_t)n0 * p.ldb + kbeg) : ((size_t)kbeg * p.ldb + n0));
        const size_t a_kstep = A_KC ? (size_t)GEMM_BK : (size_t)GEMM_BK * p.lda;
        const size_t b_kstep = B_KC ? (size_t)GEMM_BK : (size_t)GEMM_BK * p.ldb;
        for (int kt = 0; kt < KT; kt++) {
            const int s = kt % GEMM_STAGES;
            if (kt >= GEMM_STAGES) mbar_wait(&empty_bar[s], ((kt / GEMM_STAGES) - 1) & 1);
            load_tile_warp<BM, A_KC>(As + s * A_EL, Ag + kt * a_kstep, p.lda, lane);
            load_tile_warp<BN, B_KC>(Bs + s * B_EL, Bg + kt * b_kstep, p.ldb, lane);
            cp_async_mbar_arrive_noinc(&full_bar[s]);
        }
        cp_async_wait<0>();
        if (EPI != EPI_STORE) named_bar_sync(1, WS_THREADS);
        return;
    }

    // ===== consumer warps =====
    // Warp w runs on SM sub-partition w % 4.  Column ownership is mirrored for the second warp row
    // (warps 4..7 take columns 3,2,1,0), so each sub-partition hosts one warp from the light and one from
    // the heavy end of a triangular operand (see the per-warp k range below).
    // (4x2 grid: warps 0..3 take rows 0..3 of column 0, warps 4..7 rows 3..0 of column 1.)
    const int wrow = (WMW == 2) ? warp / 4 : (warp < 4 ? warp : 7 - warp);
    const int wcol = (WMW == 2) ? (warp < 4 ? warp : 7 - warp) : warp / 4;
    const int wm0 = wrow * WTM, wn0 = wcol * WTN;
    const int fr = lane >> 2, fc = lane & 3;
    // Per-warp k range.  The CTA-level range [kbeg, kend) already drops the k-tiles that are zero for the
    // whole 128x128 tile; inside the 128-wide diagonal block of the triangular operand a 64x32 warp tile
    // still meets only zeros for part of it (B lower: columns n see k <= n, or k >= n when stored [k][n];
    // A lower: rows likewise).  Those k-tiles are waited for and released but not multiplied:
    // 37.5 % (column modes) / 25 % (row modes) of the diagonal block's DMMAs, with no change to the
    // inner loop.
    int wk_lo = 0, wk_hi = KT;
    switch (p.kmode) {
        case KM_LE_J: wk_hi = min(KT, (n0 + wn0 + WTN - kbeg + GEMM_BK - 1) / GEMM_BK); break;
        case KM_GE_J: wk_lo = max(0, (n0 + wn0 - kbeg) / GEMM_BK); break;
        case KM_LE_I: wk_hi = min(KT, (m0 + wm0 + WTM - kbeg + GEMM_BK - 1) / GEMM_BK); break;
        case KM_GE_I: wk_lo = max(0, (m0 + wm0 - kbeg) / GEMM_BK); break;
        default: break;
    }
    double acc[FM][FN][2];
#pragma unroll
    for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int a_off = A_KC ? ((wm0 + fr) * A_LD + fc) : (fc * A_LD + wm0 + fr);
    const int b_off = B_KC ? ((wn0 + fr) * B_LD + fc) : (fc * B_LD + wn0 + fr);
    constexpr int a_fstep = A_KC ? 8 * A_LD : 8;
    constexpr int b_fstep = B_KC ? 8 * B_LD : 8;
    constexpr int a_kk = A_KC ? 4 : 4 * A_LD;
    constexpr int b_kk = B_KC ? 4 : 4 * B_LD;

    // Ragged last row tile (column-norm launches only: the prediction product Z = L^-1 C with M = K = n rounded up to 16
    // instead of the 128-padded size -- n = 2000: 80 live rows in the last, heaviest tile).  Rows >= M of the operand are
    // the identity padding of L^-1, whose entries at k < K are zero, so they contribute nothing either way; warps whose
    // rows are all (or in their upper half) beyond M skip those fragment rows.  Warp-uniform, decided outside the k loop.
    int fm_n = FM;
    if (EPI == EPI_SUMSQ && m0 + wm0 + WTM > p.M) {
        const int live = p.M - m0 - wm0;
        fm_n = live <= 0 ? 0 : (live <= WTM / 2 ? FM / 2 : FM);
    }
    for (int kt = 0; kt < KT; kt++) {
        const int s = kt % GEMM_STAGES;
        mbar_wait(&full_bar[s], (kt / GEMM_STAGES) & 1);
        const double* at = As + s * A_EL + a_off;
        const double* bt = Bs + s * B_EL + b_off;
        if (kt >= wk_lo && kt < wk_hi) {
            if (EPI != EPI_SUMSQ || fm_n == FM) {
#pragma unroll
                for (int kk = 0; kk < GEMM_BK / 4; kk++) {
                    double af[FM], bf[FN];
#pragma unroll
                    for (int i = 0; i < FM; i++) af[i] = at[kk * a_kk + i * a_fstep];
#pragma unroll
                    for (int j = 0; j < FN; j++) bf[j] = bt[kk * b_kk + j * b_fstep];
#pragma unroll
                    for (int i = 0; i < FM; i++)
#pragma unroll
                        for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
                }
            } else if (fm_n == FM / 2) {
#pragma unroll
                for (int kk = 0; kk < GEMM_BK / 4; kk++) {
                    double af[FM / 2], bf[FN];
#pragma unroll
                    for (int i = 0; i < FM / 2; i++) af[i] = at[kk * a_kk + i * a_fstep];
#pragma unroll
                    for (int j = 0; j < FN; j++) bf[j] = bt[kk * b_kk + j * b_fstep];
#pragma unroll
                    for (int i = 0; i < FM / 2; i++)
#pragma unroll
                        for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
    }

    if (EPI == EPI_STORE) {
        double* Cg = p.C + (size_t)b * p.sC + (size_t)(m0 + wm0 + fr) * p.ldc + n0 + wn0 + 2 * fc;
#pragma unroll
        for (int i = 0; i < FM; i++)
#pragma unroll
            for (int j = 0; j < FN; j++) {
                double2* dst = reinterpret_cast<double2*>(Cg + (size_t)(8 * i) * p.ldc + 8 * j);
                double2 v;
                v.x = p.alpha * acc[i][j][0];
                v.y = p.alpha * acc[i][j][1];
                if (p.accumulate) {
                    double2 o = *dst;
                    v.x += o.x;
                    v.y += o.y;
                }
                *dst = v;
            }
    } else {
        named_bar_sync(1, WS_THREADS);      // every stage consumed, producer drained: smem is free
        double* red = smem;                 // [WMW][BN]
#pragma unroll
        for (int j = 0; j < FN; j++) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int i = 0; i < FM; i++) {
                s0 = fma(acc[i][j][0], acc[i][j][0], s0);
                s1 = fma(acc[i][j][1], acc[i][j][1], s1);
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (fr == 0) {
                red[wrow * BN + wn0 + 8 * j + 2 * fc] = s0;
                red[wrow * BN + wn0 + 8 * j + 2 * fc + 1] = s1;
            }
        }
        named_bar_sync(2, WS_CONSUMERS * 32);
        for (int c = tid; c < BN; c += WS_CONSUMERS * 32) {
            double tot = 0.0;
#pragma unroll
            for (int w = 0; w < WMW; w++) tot += red[w * BN + c];
            p.C[(size_t)b * p.sC + (size_t)ti * p.ldc + n0 + c] = tot;
        }
    }
}

template <bool A_KC, bool B_KC, int EPI, int WMW>
inline cudaError_t launch_gemm_ws_shape(const GemmP& p, cudaStream_t st) {
    auto kern = gemm_dmma_ws_kernel<A_KC, B_KC, EPI, WMW>;
    constexpr size_t smem = gemm_smem_bytes<128, 128, A_KC, B_KC>();
    static SmemOptIn optin;
    if (cudaError_t e = optin.ensure(kern, smem); e != cudaSuccess) return e;
    const bool rowtri = (p.kmode == KM_LE_I || p.kmode == KM_GE_I);
    const bool ragged_ok = (EPI == EPI_SUMSQ) && p.kmode == KM_LE_I && p.M % GEMM_BK == 0;      // see the kernel's fm_n
    if ((p.M % 128 && !ragged_ok) || p.N % 128 || p.K % GEMM_BK) return cudaErrorInvalidValue;
    dim3 grid = rowtri ? dim3(((p.M + 127) / 128) * (p.N / 128), 1, p.batch) : dim3(p.N / 128, p.M / 128, p.batch);
    kern<<<grid, WS_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

// row-triangular launches (k <= i, k >= i) get the 4x2 warp grid, everything else the 2x4 grid
template <bool A_KC, bool B_KC, int EPI>
inline cudaError_t launch_gemm_ws(const GemmP& p, cudaStream_t st) {
    if (p.kmode == KM_LE_I || p.kmode == KM_GE_I) return launch_gemm_ws_shape<A_KC, B_KC, EPI, 4>(p, st);
    return launch_gemm_ws_shape<A_KC, B_KC, EPI, 2>(p, st);
}


// ------------------------------------------------------------------------------------------------
// Two-CTAs-per-SM flavour of the warp-specialised kernel: 128x64 tile, 4 consumer warps + 1 producer warp (160 threads),
// 3 stages (<= 92 KB), so that two CTAs are resident on an SM.  With one CTA per SM the tensor pipe idles while a new
// CTA fills its pipeline (barrier init, first loads from L2/HBM) and while the old one stores its tile: a few
// microseconds per CTA, 2-3 % of a 190 us LAUUM tile but 8-15 % of the 30-70 us tiles of the h = 512 recursion level
// (round 1: 86.5 / 77 / 56 % of the algorithmic roof at h = 2048 / 1024 / 512).  Two independent CTAs hide each other's
// ramps; the warp tiles (64x32 / 32x64), fragment loads and the k loop are those of the one-CTA kernel, 8 math warps
// per SM as before.
constexpr int WS2_CONSUMERS = 4;
constexpr int WS2_THREADS = (WS2_CONSUMERS + 1) * 32;
constexpr int WS2_STAGES = 3;
constexpr int WS2_COLGROUP = 32;     // 64-column blocks per L2-resident group of a row-triangular launch (2048 columns, as WS_COLGROUP)

template <bool A_KC, bool B_KC, int EPI, int WMW>
__global__ void __launch_bounds__(WS2_THREADS, 2) gemm_dmma_ws2_kernel(GemmP p) {
    constexpr int BM = 128, BN = 64, WNW = WS2_CONSUMERS / WMW;
    constexpr int WTM = BM / WMW, WTN = BN / WNW, FM = WTM / 8, FN = WTN / 8;      // 2x2 warps of 64x32, or 4x1 of 32x64
    constexpr int A_EL = TileShape<BM, A_KC>::ELEMS, B_EL = TileShape<BN, B_KC>::ELEMS;
    constexpr int A_LD = TileShape<BM, A_KC>::LD, B_LD = TileShape<BN, B_KC>::LD;
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) uint64_t full_bar[WS2_STAGES], empty_bar[WS2_STAGES];

    const bool rowtri = (p.kmode == KM_LE_I || p.kmode == KM_GE_I);
    int tj, ti;
    if (rowtri) {
        const int ntx = p.N / BN, nty = p.M / BM, id = (int)blockIdx.x;
        const int full = (ntx / WS2_COLGROUP) * WS2_COLGROUP * nty;
        int g0, gsz, r;
        if (id < full) { g0 = (id / (WS2_COLGROUP * nty)) * WS2_COLGROUP; gsz = WS2_COLGROUP; r = id % (WS2_COLGROUP * nty); }
        else { g0 = (ntx / WS2_COLGROUP) * WS2_COLGROUP; gsz = ntx - g0; r = id - full; }
        const int y = r / gsz;
        tj = g0 + (r - y * gsz);
        ti = (p.kmode == KM_LE_I) ? nty - 1 - y : y;
    } else {
        tj = (p.kmode == KM_LE_J) ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
        ti = (int)blockIdx.y;
    }
    const int b = blockIdx.z;
    if (p.lower && (ti + 1) * BM <= tj * BN) return;
    const int m0 = ti * BM, n0 = tj * BN;
    int kbeg = 0, kend = p.K;
    switch (p.kmode) {
        case KM_LE_J: kend = min(p.K, (tj + 1) * BN); break;
        case KM_GE_J: kbeg = min(p.K, (tj * BN / GEMM_BK) * GEMM_BK); break;
        case KM_LE_I: kend = min(p.K, (ti + 1) * BM); break;
        case KM_GE_I: kbeg = min(p.K, ti * BM); break;
        default: break;
    }
    const int KT = (kend - kbeg + GEMM_BK - 1) / GEMM_BK;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < WS2_STAGES; s++) {
            mbar_init(&full_bar[s], 32);
            mbar_init(&empty_bar[s], WS2_CONSUMERS);
        }
    }
    __syncthreads();

    double* As = smem;
    double* Bs = smem + WS2_STAGES * A_EL;

    if (warp == WS2_CONSUMERS) {
        const double* Ag = p.A + (size_t)b * p.sA + (A_KC ? ((size_t)m0 * p.lda + kbeg) : ((size_t)kbeg * p.lda + m0));
        const double* Bg = p.B + (size_t)b * p.sB + (B_KC ? ((size_t)n0 * p.ldb + kbeg) : ((size_t)kbeg * p.ldb + n0));
        const size_t a_kstep = A_KC ? (size_t)GEMM_BK : (size_t)GEMM_BK * p.lda;
        const size_t b_kstep = B_KC ? (size_t)GEMM_BK : (size_t)GEMM_BK * p.ldb;
        for (int kt = 0; kt < KT; kt++) {
            const int s = kt % WS2_STAGES;
            if (kt >= WS2_STAGES) mbar_wait(&empty_bar[s], ((kt / WS2_STAGES) - 1) & 1);
            load_tile_warp<BM, A_KC>(As + s * A_EL, Ag + kt * a_kstep, p.lda, lane);
            load_tile_warp<BN, B_KC>(Bs + s * B_EL, Bg + kt * b_kstep, p.ldb, lane);
            cp_async_mbar_arrive_noinc(&full_bar[s]);
        }
        cp_async_wait<0>();
        if (EPI != EPI_STORE) named_bar_sync(1, WS2_THREADS);
        return;
    }

    // consumer warps.  2x2 grid: warps 0, 1 take columns 0, 1 of row 0, warps 2, 3 columns 1, 0 of row 1 (mirrored, so the light
    // and the heavy end of a column-triangular operand share an SM sub-partition pair); 4x1 grid: warp w takes row w.
    const int wrow = (WMW == 2) ? warp / 2 : warp;
    const int wcol = (WMW == 2) ? (warp < 2 ? warp : 3 - warp) : 0;
    const int wm0 = wrow * WTM, wn0 = wcol * WTN;
    const int fr = lane >> 2, fc = lane & 3;
    int wk_lo = 0, wk_hi = KT;
    switch (p.kmode) {
        case KM_LE_J: wk_hi = min(KT, (n0 + wn0 + WTN - kbeg + GEMM_BK - 1) / GEMM_BK); break;
        case KM_GE_J: wk_lo = max(0, (n0 + wn0 - kbeg) / GEMM_BK); break;
        case KM_LE_I: wk_hi = min(KT, (m0 + wm0 + WTM - kbeg + GEMM_BK - 1) / GEMM_BK); break;
        case KM_GE_I: wk_lo = max(0, (m0 + wm0 - kbeg) / GEMM_BK); break;
        default: break;
    }
    double acc[FM][FN][2];
#pragma unroll
    for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int a_off = A_KC ? ((wm0 + fr) * A_LD + fc) : (fc * A_LD + wm0 + fr);
    const int b_off = B_KC ? ((wn0 + fr) * B_LD + fc) : (fc * B_LD + wn0 + fr);
    constexpr int a_fstep = A_KC ? 8 * A_LD : 8;
    constexpr int b_fstep = B_KC ? 8 * B_LD : 8;
    constexpr int a_kk = A_KC ? 4 : 4 * A_LD;
    constexpr int b_kk = B_KC ? 4 : 4 * B_LD;

    for (int kt = 0; kt < KT; kt++) {
        const int s = kt % WS2_STAGES;
        mbar_wait(&full_bar[s], (kt / WS2_STAGES) & 1);
        const double* at = As + s * A_EL + a_off;
        const double* bt = Bs + s * B_EL + b_off;
        if (kt >= wk_lo && kt < wk_hi) {
#pragma unroll
            for (int kk = 0; kk < GEMM_BK / 4; kk++) {
                double af[FM], bf[FN];
#pragma unroll
                for (int i = 0; i < FM; i++) af[i] = at[kk * a_kk + i * a_fstep];
#pragma unroll
                for (int j = 0; j < FN; j++) bf[j] = bt[kk * b_kk + j * b_fstep];
#pragma unroll
                for (int i = 0; i < FM; i++)
#pragma unroll
                    for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
    }

    if (EPI == EPI_STORE) {
        double* Cg = p.C + (size_t)b * p.sC + (size_t)(m0 + wm0 + fr) * p.ldc + n0 + wn0 + 2 * fc;
#pragma unroll
        for (int i = 0; i < FM; i++)
#pragma unroll
            for (int j = 0; j < FN; j++) {
                double2* dst = reinterpret_cast<double2*>(Cg + (size_t)(8 * i) * p.ldc + 8 * j);
                double2 v;
                v.x = p.alpha * acc[i][j][0];
                v.y = p.alpha * acc[i][j][1];
                if (p.accumulate) {
                    double2 o = *dst;
                    v.x += o.x;
                    v.y += o.y;
                }
                *dst = v;
            }
    } else {
        named_bar_sync(1, WS2_THREADS);     // every stage consumed, producer drained: smem is free
        double* red = smem;                 // [WMW][BN]
#pragma unroll
        for (int j = 0; j < FN; j++) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int i = 0; i < FM; i++) {
                s0 = fma(acc[i][j][0], acc[i][j][0], s0);
                s1 = fma(acc[i][j][1], acc[i][j][1], s1);
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (fr == 0) {
                red[wrow * BN + wn0 + 8 * j + 2 * fc] = s0;
                red[wrow * BN + wn0 + 8 * j + 2 * fc + 1] = s1;
            }
        }
        named_bar_sync(2, WS2_CONSUMERS * 32);
        for (int c = tid; c < BN; c += WS2_CONSUMERS * 32) {
            double tot = 0.0;
#pragma unroll
            for (int w = 0; w < WMW; w++) tot += red[w * BN + c];
            p.C[(size_t)b * p.sC + (size_t)ti * p.ldc + n0 + c] = tot;
        }
    }
}

template <bool A_KC, bool B_KC>
constexpr size_t gemm_ws2_smem_bytes() {
    return (size_t)WS2_STAGES * (TileShape<128, A_KC>::ELEMS + TileShape<64, B_KC>::ELEMS) * sizeof(double);
}

template <bool A_KC, bool B_KC, int EPI, int WMW>
inline cudaError_t launch_gemm_ws2_shape(const GemmP& p, cudaStream_t st) {
    auto kern = gemm_dmma_ws2_kernel<A_KC, B_KC, EPI, WMW>;
    constexpr size_t smem = gemm_ws2_smem_bytes<A_KC, B_KC>();
    static SmemOptIn optin;
    if (cudaError_t e = optin.ensure(kern, smem); e != cudaSuccess) return e;
    static bool carve = false;
    if (!carve) {       // two CTAs of ~90 KB each must both find shared memory: ask for the largest carve-out
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carve = true;
    }
    if (p.M % 128 || p.N % 64 || p.K % GEMM_BK) return cudaErrorInvalidValue;
    const bool rowtri = (p.kmode == KM_LE_I || p.kmode == KM_GE_I);
    dim3 grid = rowtri ? dim3((p.M / 128) * (p.N / 64), 1, p.batch) : dim3(p.N / 64, p.M / 128, p.batch);
    kern<<<grid, WS2_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

template <bool A_KC, bool B_KC, int EPI>
inline cudaError_t launch_gemm_ws2(const GemmP& p, cudaStream_t st) {
    if (p.kmode == KM_LE_I || p.kmode == KM_GE_I) return launch_gemm_ws2_shape<A_KC, B_KC, EPI, 4>(p, st);
    return launch_gemm_ws2_shape<A_KC, B_KC, EPI, 2>(p, st);
}

// Layouts: GEMM_NT = (A_KC,B_KC), GEMM_NN = (A_KC,!B_KC), GEMM_TN = (!A_KC,!B_KC).
// Tile choice: 128x64 tiles, two CTAs per SM, when 128x128 tiles still fill the machine, else 64x64 (or 32x32);
// N == 32 panels use 128x32.  Column norms (EPI_SUMSQ) take the 128x64 kernel, or the 128x128 one for a ragged M.
cudaError_t launch_gemm(const GemmP& p, int layout, int epi, cudaStream_t st);
// does an EPI_STORE product take the two-CTAs-per-SM kernel, i.e. do 128x128 tiles fill the machine?
bool gemm_fills_machine(const GemmP& p);

}  // namespace gpe
