// LAUUM with the gradient reduction in its epilogue (K3 + K1g fused).
//
// Reference arithmetic replaced: the per-hyper-parameter solve / trace expressions of
// _emulatoroptimise.py:345-372 and :450-487, which collapse (SURVEY A.2) to
//     grad_k = 1/2 sum_ij T^k_ij W_ij,   W = A^-1 - U U^T,   U = [A^-1 H K^-T | sqrt(f) A^-1 (y - H beta)],
// with T^k built from E_ij = exp(-sum_k ((x_ik - x_jk)/delta_k)^2)  (_emulatorkernels.py:53-71, :126-144).
//
// Round 1 formed A^-1 = L^-T L^-1 with the generic DMMA GEMM, stored its lower tiles (8 n^2 / 2 bytes per item) and
// read them back in a separate reduction kernel that also recomputed E and the U.U^T dot products on the FP64 ALU
// (3.15 ms per 32-item step, 0.32 of the FP64 roof, long-scoreboard bound on the A^-1 loads).  Here a 128x128 tile of
// W never leaves the registers of the CTA that computed it:
//   * the k loop runs over L^-1 (k >= i, as LAUUM) and then over the NR columns of U, whose tiles come from a
//     pre-negated k-major copy (-U^T as the A operand, U^T as the B operand), so W = A^-1 - U U^T falls out of the
//     tensor pipe and the 2 x 18 FMA per entry of the old dot products disappear;
//   * the epilogue stages the scaled input tiles X_i / delta, X_j / delta in the (now free) pipeline stages, reads
//     E_ij = exp(-D_ij) for the 64 entries a lane holds from the copy the covariance build kept (the FP64 pipe is the
//     bottleneck of this path and HBM is idle: 8 bytes per entry are cheaper than 2d + 22 FP64 instructions), and
//     reduces sum W E Delta_k^2 (k < d), sum W E, sum_diag W, sum_diag W r into one partial row per tile, which
//     grad_finalize_kernel adds up in a fixed order.
// A^-1 is not written at all on this path (the sensitivity code builds it on demand with the generic kernel).
#include "gpe_gemm.cuh"
#include "gpe_kernels.cuh"

#include <algorithm>
#include <cstdlib>

namespace gpe {

struct LauumGradP {
    const double* Li;      // [B][np][np]  L^-1 (lower; upper blocks zero)
    long long sL;
    int np, n, d;
    int ku;                // k-tiles of the U part (ceil(nu / 16))
    const double* Ut;      // [B][NR][np]   U^T
    const double* nUt;     // [B][NR][np]  -U^T
    long long sU;
    const double* X;       // [n][d]
    const double* r;       // [n] or null
    const double* winv;    // [B][d]  1 / delta
    const double* E;       // [B][np][np]  exp(-D) as written by the covariance build (lower 64x64 tiles)
    long long sE;
    double* part;          // [B][ntile][d + 3]
    int ntile;
};

constexpr int LG_LDX = 128 + 4;     // row stride of the k-major X tiles in the epilogue

__device__ __forceinline__ void tri_decode_lg(int t, int& ti, int& tj) {
    int r = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((r + 1) * (r + 2) / 2 <= t) r++;
    while (r * (r + 1) / 2 > t) r--;
    ti = r;
    tj = t - r * (r + 1) / 2;
}

__global__ void __launch_bounds__(WS_THREADS, 1) lauum_grad_kernel(LauumGradP p) {
    constexpr int BM = 128, BN = 128, WMW = 4, WNW = WS_CONSUMERS / WMW;
    constexpr int WTM = BM / WMW, WTN = BN / WNW, FM = WTM / 8, FN = WTN / 8;       // warp tile 32 x 64: FM = 4, FN = 8
    constexpr int A_EL = TileShape<BM, false>::ELEMS, B_EL = TileShape<BN, false>::ELEMS;
    constexpr int A_LD = TileShape<BM, false>::LD, B_LD = TileShape<BN, false>::LD;
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) uint64_t full_bar[GEMM_STAGES], empty_bar[GEMM_STAGES];

    // lower-triangle tiles, row by row: tile t = ti (ti + 1) / 2 + tj.  Row ti has the k range [ti * 128, np):
    // the launch starts on its longest tiles and ends on its shortest
    int ti, tj;
    tri_decode_lg((int)blockIdx.x, ti, tj);
    const int tile_id = (int)blockIdx.x;
    const int b = blockIdx.z;
    const int m0 = ti * BM, n0 = tj * BN;
    const int kbeg = m0;
    const int KT0 = (p.np - kbeg) / GEMM_BK, KT = KT0 + p.ku;
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
        // ===== producer warp: L^-1 tiles (both operands: rows k, columns m0.. / n0..), then the U tiles =====
        const double* Lb = p.Li + (size_t)b * p.sL;
        const double* Ag = Lb + (size_t)kbeg * p.np + m0;
        const double* Bg = Lb + (size_t)kbeg * p.np + n0;
        const double* Au = p.nUt + (size_t)b * p.sU + m0;
        const double* Bu = p.Ut + (size_t)b * p.sU + n0;
        const size_t kstep = (size_t)GEMM_BK * p.np;
        for (int kt = 0; kt < KT; kt++) {
            const int s = kt % GEMM_STAGES;
            if (kt >= GEMM_STAGES) mbar_wait(&empty_bar[s], ((kt / GEMM_STAGES) - 1) & 1);
            if (kt < KT0) {
                load_tile_warp<BM, false>(As + s * A_EL, Ag + kt * kstep, p.np, lane);
                load_tile_warp<BN, false>(Bs + s * B_EL, Bg + kt * kstep, p.np, lane);
            } else {
                load_tile_warp<BM, false>(As + s * A_EL, Au + (kt - KT0) * kstep, p.np, lane);
                load_tile_warp<BN, false>(Bs + s * B_EL, Bu + (kt - KT0) * kstep, p.np, lane);
            }
            cp_async_mbar_arrive_noinc(&full_bar[s]);
            // the epilogue reads this tile's 128 x 128 block of E (written by the covariance build a whole factorisation
            // ago: it comes from HBM).  Ask L2 for it while the consumers still have a few k-tiles to go.
            if (kt == KT - GEMM_STAGES - 4 || (KT < GEMM_STAGES + 5 && kt == 0)) {
                const double* Eg = p.E + (size_t)b * p.sE + (size_t)m0 * p.np + n0;
#pragma unroll 4
                for (int q = 0; q < 32; q++) {                 // 128 rows x 8 lines of 128 bytes
                    const int li = q * 32 + lane;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(Eg + (size_t)(li >> 3) * p.np + (li & 7) * 16));
                }
            }
        }
        cp_async_wait<0>();
        return;
    }

    // ===== consumer warps: 4 x 2 grid, warps 0..3 rows 0..3 of column 0, warps 4..7 rows 3..0 of column 1 =====
    const int wrow = (warp < 4 ? warp : 7 - warp), wcol = warp / 4;
    const int wm0 = wrow * WTM, wn0 = wcol * WTN;
    const int fr = lane >> 2, fc = lane & 3;
    // inside the diagonal block of L^-1 (k in [m0, m0 + 128)) rows k < m see only zeros of the A operand
    const int wk_lo = wm0 / GEMM_BK;
    double acc[FM][FN][2];
#pragma unroll
    for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int a_off = fc * A_LD + wm0 + fr;
    const int b_off = fc * B_LD + wn0 + fr;
    constexpr int a_kk = 4 * A_LD, b_kk = 4 * B_LD;

    // Diagonal tiles (ti == tj): only entries on or below the diagonal are used.  With the 4 x 2 warp grid the warps of
    // rows 0, 1 in column 1 have nothing to do and the warps (row 0, column 0), (row 2, column 1) need only their left four
    // fragment columns: per SM sub-partition that is 48 / 48 / 32 / 32 DMMAs per k4 step instead of 64 -- the tile costs
    // 3/4 (diagonal tiles are 8.8 % of a LAUUM launch at n = 4096).  Warp-uniform, decided outside the k loop.
    int jn = FN;
    if (ti == tj) jn = (wcol == 0) ? (wrow == 0 ? FN / 2 : FN) : (wrow == 3 ? FN : (wrow == 2 ? FN / 2 : 0));
    for (int kt = 0; kt < KT; kt++) {
        const int s = kt % GEMM_STAGES;
        mbar_wait(&full_bar[s], (kt / GEMM_STAGES) & 1);
        const double* at = As + s * A_EL + a_off;
        const double* bt = Bs + s * B_EL + b_off;
        if (kt >= wk_lo) {
            if (jn == FN) {
#pragma unroll
                for (int kk = 0; kk < GEMM_BK / 4; kk++) {
                    double af[FM], bf[FN];
#pragma unroll
                    for (int i = 0; i < FM; i++) af[i] = at[kk * a_kk + i * 8];
#pragma unroll
                    for (int j = 0; j < FN; j++) bf[j] = bt[kk * b_kk + j * 8];
#pragma unroll
                    for (int i = 0; i < FM; i++)
#pragma unroll
                        for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
                }
            } else if (jn == FN / 2) {
#pragma unroll
                for (int kk = 0; kk < GEMM_BK / 4; kk++) {
                    double af[FM], bf[FN / 2];
#pragma unroll
                    for (int i = 0; i < FM; i++) af[i] = at[kk * a_kk + i * 8];
#pragma unroll
                    for (int j = 0; j < FN / 2; j++) bf[j] = bt[kk * b_kk + j * 8];
#pragma unroll
                    for (int i = 0; i < FM; i++)
#pragma unroll
                        for (int j = 0; j < FN / 2; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
    }

    // ===== epilogue: acc = W tile.  The pipeline stages are free: stage the E tile and the scaled input tiles there. =====
    const int d = p.d, n = p.n;
    named_bar_sync(2, WS_CONSUMERS * 32);           // every consumer is past its last stage read
    double* Es = smem;                              // [128][LG_LDX]  exp(-D) of this tile (from the covariance build's copy);
                                                    //                later the per-lane partial sums [d][256]
    double* Xi = Es + 128 * LG_LDX;                 // [d][LG_LDX]  rows m0 .. m0 + 127, k-major, scaled by 1 / delta
    double* Xj = Xi + (size_t)d * LG_LDX;           // [d][LG_LDX]  rows n0 ..
    double* red = Xj + (size_t)d * LG_LDX;          // [8][3]
    {
        // thread -> 16-byte chunk (tid & 63) of rows (tid >> 6) + 4 it
        const double* src = p.E + (size_t)b * p.sE + (size_t)(m0 + (tid >> 6)) * p.np + n0 + 2 * (tid & 63);
        double* dst = Es + (tid >> 6) * LG_LDX + 2 * (tid & 63);
        const size_t sstep = (size_t)4 * p.np;
#pragma unroll 4
        for (int it = 0; it < 32; it++) {
            cp_async16(dst, src);
            src += sstep;
            dst += 4 * LG_LDX;
        }
        cp_async_commit();
        const double* __restrict__ w = p.winv + (size_t)b * d;
        const double* __restrict__ Xg = p.X;
        const int row = tid >> 1, gi = m0 + row, gj = n0 + row;
        for (int k = tid & 1; k < d; k += 2) {
            const double wk = __ldg(w + k);
            const double vi = (gi < n) ? __ldg(Xg + (size_t)gi * d + k) : 0.0;
            const double vj = (gj < n) ? __ldg(Xg + (size_t)gj * d + k) : 0.0;
            Xi[k * LG_LDX + row] = vi * wk;
            Xj[k * LG_LDX + row] = vj * wk;
        }
        cp_async_wait<0>();
    }
    named_bar_sync(2, WS_CONSUMERS * 32);

    const int row0 = wm0 + fr, col0 = wn0 + 2 * fc;          // lane's entries: rows row0 + 8 i, columns col0 + 8 j + {0, 1}
    double sE = 0.0, sD = 0.0, sDr = 0.0;
    // pass 1: acc <- t = 2 W E for the pairs below the diagonal inside the n x n matrix, 0 elsewhere; the diagonal sums
    // on the way.  Tiles strictly below the diagonal and inside the matrix -- all but a few -- need no case analysis.
    if (ti > tj && m0 + BM <= n) {
#pragma unroll
        for (int j = 0; j < FN; j++)
#pragma unroll
            for (int i = 0; i < FM; i++) {
                const double2 ev = *reinterpret_cast<const double2*>(Es + (row0 + 8 * i) * LG_LDX + col0 + 8 * j);
                const double t0 = 2.0 * acc[i][j][0] * ev.x, t1 = 2.0 * acc[i][j][1] * ev.y;
                acc[i][j][0] = t0;
                acc[i][j][1] = t1;
                sE += t0 + t1;
            }
    } else {
        const bool diag_tile = (ti == tj);
#pragma unroll
        for (int j = 0; j < FN; j++)
#pragma unroll
            for (int i = 0; i < FM; i++) {
                const int gi = m0 + row0 + 8 * i;
                const double2 ev = *reinterpret_cast<const double2*>(Es + (row0 + 8 * i) * LG_LDX + col0 + 8 * j);
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int gj = n0 + col0 + 8 * j + e;
                    const double wv = acc[i][j][e];
                    double tv = 2.0 * wv * (e ? ev.y : ev.x);
                    bool below = gi < n;                        // gj < gi < n off the diagonal tiles
                    if (diag_tile) {
                        below = below && gj < gi;               // each pair once, from below; selected, not multiplied by 0:
                        if (gi == gj && gi < n) {               // the copy of E holds the lower 64x64 tiles only
                            sD += wv;
                            if (p.r != nullptr) sDr = fma(wv, p.r[gi], sDr);
                        }
                    }
                    tv = below ? tv : 0.0;
                    acc[i][j][e] = tv;
                    sE += tv;
                }
            }
    }
    sE = warp_sum(sE); sD = warp_sum(sD); sDr = warp_sum(sDr);
    if (lane == 0) { red[warp * 3] = sE; red[warp * 3 + 1] = sD; red[warp * 3 + 2] = sDr; }
    // pass 2: per dimension, sum t * Delta_k^2 over the lane's 64 entries.  With all 64 t's in registers (128 of the 168
    // a thread of a 9-warp CTA can have) the compiler has no room to overlap the sub -> mul -> fma triples and every
    // instruction waits for the one before (ncu: stall_wait on each of them, 44 % of the FP64 issue rate).  So the
    // right half of the warp tile (fragment columns 4..7) is parked in shared memory -- each lane overwrites the E
    // entries it has just consumed, no other lane touches them -- and the two halves are reduced one after the other
    // with eight triples in flight.  The lane's partial sums go to shared memory; cross-lane sums happen once at the end.
#pragma unroll
    for (int j = FN / 2; j < FN; j++)
#pragma unroll
        for (int i = 0; i < FM; i++)
            *reinterpret_cast<double2*>(Es + (row0 + 8 * i) * LG_LDX + col0 + 8 * j) = make_double2(acc[i][j][0], acc[i][j][1]);
    double* gpart = Xj + (size_t)d * LG_LDX + 8 * 3;      // [d][256], behind the reduction rows
    auto half_pass = [&](const double (&t)[FM][FN / 2][2], int jbase, bool add) {
        for (int k = 0; k < d; k++) {
            double xi[FM];
#pragma unroll
            for (int i = 0; i < FM; i++) xi[i] = Xi[k * LG_LDX + row0 + 8 * i];
            double g[FM][2];
#pragma unroll
            for (int i = 0; i < FM; i++) g[i][0] = g[i][1] = 0.0;
#pragma unroll
            for (int j = 0; j < FN / 2; j++) {
                const double2 xj = *reinterpret_cast<const double2*>(Xj + k * LG_LDX + col0 + 8 * (jbase + j));
                double d0[FM], d1[FM], m0[FM], m1[FM];
#pragma unroll
                for (int i = 0; i < FM; i++) { d0[i] = xi[i] - xj.x; d1[i] = xi[i] - xj.y; }
#pragma unroll
                for (int i = 0; i < FM; i++) { m0[i] = t[i][j][0] * d0[i]; m1[i] = t[i][j][1] * d1[i]; }
#pragma unroll
                for (int i = 0; i < FM; i++) { g[i][0] = fma(m0[i], d0[i], g[i][0]); g[i][1] = fma(m1[i], d1[i], g[i][1]); }
            }
            const double gs = ((g[0][0] + g[0][1]) + (g[1][0] + g[1][1])) + ((g[2][0] + g[2][1]) + (g[3][0] + g[3][1]));
            if (add) gpart[k * 256 + tid] += gs;
            else gpart[k * 256 + tid] = gs;
        }
    };
    {
        double t[FM][FN / 2][2];
#pragma unroll
        for (int i = 0; i < FM; i++)
#pragma unroll
            for (int j = 0; j < FN / 2; j++) { t[i][j][0] = acc[i][j][0]; t[i][j][1] = acc[i][j][1]; }
        half_pass(t, 0, false);
#pragma unroll
        for (int i = 0; i < FM; i++)
#pragma unroll
            for (int j = 0; j < FN / 2; j++) {
                const double2 v = *reinterpret_cast<const double2*>(Es + (row0 + 8 * i) * LG_LDX + col0 + 8 * (j + FN / 2));
                t[i][j][0] = v.x;
                t[i][j][1] = v.y;
            }
        half_pass(t, FN / 2, true);
    }
    named_bar_sync(2, WS_CONSUMERS * 32);
    const int nv = d + 3;
    double* pout = p.part + ((size_t)b * p.ntile + tile_id) * nv;
    // dimension k: 16 threads add 16 lane partials each, then a 16-lane butterfly -- a fixed order
    for (int k0 = 0; k0 < d; k0 += 16) {
        const int k = k0 + (tid >> 4), part = tid & 15;
        double sacc = 0.0;
        if (k < d) {
#pragma unroll
            for (int q = 0; q < 16; q++) sacc += gpart[k * 256 + part * 16 + q];
        }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (k < d && part == 0) pout[k] = sacc;
    }
    if (tid < 3) {
        double sacc = 0.0;
#pragma unroll
        for (int w = 0; w < WS_CONSUMERS; w++) sacc += red[w * 3 + tid];
        pout[d + tid] = sacc;
    }
}


// -U^T and U^T, k-major: Ut[b][c][i] = U[b][i][c]
__global__ void __launch_bounds__(256) ut_kernel(const double* __restrict__ U, int np, double* __restrict__ Ut, double* __restrict__ nUt) {
    __shared__ double T[32][NR + 1];
    const int b = blockIdx.y, i0 = blockIdx.x * 32;
    const double* Ub = U + ((size_t)b * np + i0) * NR;
    for (int e = threadIdx.x; e < 32 * NR; e += 256) T[e / NR][e % NR] = Ub[e];
    __syncthreads();
    for (int e = threadIdx.x; e < 32 * NR; e += 256) {
        const int c = e / 32, i = e % 32;
        const double v = T[i][c];
        const size_t o = ((size_t)b * NR + c) * np + i0 + i;
        Ut[o] = v;
        nUt[o] = -v;
    }
}

static size_t lauum_grad_smem(int d) {
    // the epilogue's E tile, two k-major input tiles and the reduction rows reuse the pipeline stages
    const size_t epi = ((size_t)128 * LG_LDX + (size_t)2 * d * LG_LDX + 8 * 3 + (size_t)256 * d) * sizeof(double);
    return std::max(epi, gemm_smem_bytes<128, 128, false, false>());
}

bool lauum_grad_supported(int d) { return lauum_grad_smem(d) <= 227 * 1024; }

cudaError_t launch_lauum_grad(const double* Li, long long sL, int np, int n, int d, int nu, const double* U, double* Ut, double* nUt,
                              const double* X, const double* r, const double* winv, const double* E, long long sE, double* part,
                              int B, cudaStream_t st) {
    if (np % 128 || !lauum_grad_supported(d)) return cudaErrorInvalidValue;
    ut_kernel<<<dim3(np / 32, B), 256, 0, st>>>(U, np, Ut, nUt);
    LauumGradP p;
    p.Li = Li; p.sL = sL; p.np = np; p.n = n; p.d = d;
    p.ku = (nu + GEMM_BK - 1) / GEMM_BK;
    p.Ut = Ut; p.nUt = nUt; p.sU = (long long)NR * np;
    p.X = X; p.r = r; p.winv = winv; p.E = E; p.sE = sE; p.part = part;
    const int T = np / 128;
    p.ntile = T * (T + 1) / 2;
    const size_t smem = lauum_grad_smem(d);
    static SmemOptIn optin;
    if (cudaError_t e = optin.ensure(lauum_grad_kernel, smem); e != cudaSuccess) return e;
    lauum_grad_kernel<<<dim3(p.ntile, 1, B), WS_THREADS, smem, st>>>(p);
    return cudaGetLastError();
}

int lauum_grad_ntiles(int npad) {
    const int T = npad / 128;
    return T * (T + 1) / 2;       // partial rows per item: one per 128x128 lower tile
}

}  // namespace gpe
