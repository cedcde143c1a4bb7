// Non-GEMM kernels of the likelihood path.  Reference arithmetic being replaced:
//   _emulatorkernels.py:39-71 / :112-144 (var, grad_delta_A, grad_nugget_A),
//   _emulatoroptimise.py:305-378 / :412-493 (loglikelihood_mucm / _gp4ml).
#include "gpe_kernels.cuh"
#include "gpe_b200.h"

#include <algorithm>
#include <cstdlib>

namespace gpe {

// =========================================================================== prep
__global__ void prep_theta_kernel(const double* __restrict__ theta, int B, int p, int d, int mode,
                                  double fixed_nugget, ItemPar* par, double* winv) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* t = theta + (size_t)b * p;
    for (int k = 0; k < d; k++) winv[(size_t)b * d + k] = 1.0 / exp(t[k] / 2.0);
    int idx = d;
    double nug = fixed_nugget;
    if (mode & GPE_MODE_NUGGET_FREE) nug = exp(t[idx++] / 2.0);
    double sigma = 1.0, s2 = 1.0;
    if (!(mode & GPE_MODE_MUCM)) {
        sigma = exp(t[idx] / 2.0);
        s2 = sigma * sigma;
    }
    ItemPar ip;
    bool alt = mode & GPE_MODE_ALT_NUGGET;
    ip.c = alt ? 1.0 : (1.0 - nug);
    ip.offs = s2 * ip.c;
    ip.diagv = alt ? s2 * (1.0 + nug * nug) : s2;
    ip.radd = alt ? 1.0 : 0.0;
    ip.s2A = s2;
    ip.nugget = nug;
    ip.sigma = sigma;
    ip.pad_ = 0.0;
    par[b] = ip;
}

void launch_prep_theta(const double* theta, int B, int p, int d, int mode, double fixed_nugget,
                       ItemPar* par, double* winv, cudaStream_t st) {
    prep_theta_kernel<<<(B + 127) / 128, 128, 0, st>>>(theta, B, p, d, mode, fixed_nugget, par, winv);
}

// =========================================================================== K1 covariance build
// 64x64 tile per CTA, 256 threads, 4x4 entries per thread (the 4 x 4 shape of sqdist_tile, gpe_common.cuh).
constexpr int CT = 64;

// lower-triangle tile index t = ti (ti + 1) / 2 + tj  ->  (ti, tj): 1-D grids launch no empty CTAs for the upper half
__device__ __forceinline__ void tri_decode(int t, int& ti, int& tj) {
    int r = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((r + 1) * (r + 2) / 2 <= t) r++;
    while (r * (r + 1) / 2 > t) r--;
    ti = r;
    tj = t - r * (r + 1) / 2;
}

// GMODE 0: covariance (the hot path: no G registers, no spills under the 80-register cap of 3 CTAs/SM);
// 1: d(s2 A)/d theta_delta[gdim] (grad_delta_A); 2: kernel grad_nugget_A (off-diagonal only; the alt-nugget form
// is a pure diagonal and is assembled by the caller).
// FAM: FAMILY_GAUSSIAN (E = exp(-D) is both the entry and the derivative factor) or FAMILY_MATERN52 (entry R(D); GMODE 1
// uses the derivative factor G(D) in its place; no E copy)
template <int GMODE, int FAM>
__global__ void __launch_bounds__(256, 3) cov_build_kernel(const double* __restrict__ X, const double* __restrict__ r,
                                                        int n, int d, int npad, const ItemPar* __restrict__ par,
                                                        const double* __restrict__ winv, double* __restrict__ A,
                                                        long long sA, int full, int gdim, double* __restrict__ Eout) {
    constexpr int gmode = GMODE;
    int tj = blockIdx.x, ti = blockIdx.y;
    const int b = blockIdx.z;
    if (!full) tri_decode(blockIdx.x, ti, tj);
    extern __shared__ __align__(16) double sm[];
    double* Xi = sm;                   // [d][CT]
    double* Xj = sm + (size_t)d * CT;  // [d][CT+2]
    const int tid = threadIdx.x;
    fill_scaled_tiles(X, winv + (size_t)b * d, n, d, ti * CT, tj * CT, Xi, Xj, tid);
    __syncthreads();
    const ItemPar ip = par[b];
    const int ty = tid >> 4, tx = tid & 15;
    double D[4][4], G[GMODE == 1 ? 4 : 1][4];
    sqdist_tile<4, 16, 32>(Xi, Xj, d, ty, tx, D);
    if constexpr (GMODE == 1) {      // Delta_gdim^2 of each entry (0 <= gdim < d)
        double xi[4], xj[4];
        tile_operands<4, 16, 32>(Xi, Xj, gdim, ty, tx, xi, xj);
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const double df = xi[a] - xj[c];
                G[a][c] = df * df;
            }
    }
    // all 16 exponentials first, outside the padding / diagonal case analysis: straight-line code whose 16 polynomial
    // chains interleave (inside the branches they ran one dependent chain at a time)
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            if constexpr (FAM == FAMILY_GAUSSIAN) D[a][c] = gpe_exp(-D[a][c]);
            else if constexpr (GMODE == 1) gpe_matern52(D[a][c], D[a][c]);
            else D[a][c] = gpe_matern52(D[a][c]);
        }
    double* Ab = A + (size_t)b * sA;
#pragma unroll
    for (int a = 0; a < 4; a++) {
        int gi = ti * CT + ty + 16 * a;
        double ri = (r != nullptr && gi < n) ? r[gi] : 0.0;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            int gj0 = tj * CT + 32 * h + 2 * tx;
            double v[2];
#pragma unroll
            for (int e = 0; e < 2; e++) {
                int gj = gj0 + e;
                double val;
                if (gi >= n || gj >= n) val = (gi == gj && gmode == 0) ? 1.0 : 0.0;     // identity padding
                else if (gi == gj) val = (gmode == 0) ? ip.diagv + ip.radd * ri : 0.0;
                else if constexpr (GMODE == 1) val = ip.offs * G[a][2 * h + e] * D[a][2 * h + e];
                else val = ip.offs * D[a][2 * h + e];
                v[e] = val;
            }
            *reinterpret_cast<double2*>(&Ab[(size_t)gi * npad + gj0]) = make_double2(v[0], v[1]);
            if constexpr (GMODE == 0 && FAM == FAMILY_GAUSSIAN) {
                if (Eout != nullptr)
                    *reinterpret_cast<double2*>(&Eout[(size_t)b * sA + (size_t)gi * npad + gj0]) = make_double2(D[a][2 * h], D[a][2 * h + 1]);
            }
        }
    }
}

cudaError_t launch_cov_build(const double* X, const double* r, int n, int d, int npad, const ItemPar* par,
                             const double* winv, double* A, long long sA, int B, int full, cudaStream_t st, int gmode, int gdim,
                             double* Eout, int family) {
    const int nt = npad / CT;
    dim3 grid = full ? dim3(nt, nt, B) : dim3(nt * (nt + 1) / 2, 1, B);
    size_t smem = (size_t)d * (CT + CT + 2) * sizeof(double);
    return with_family(family, [&](auto fam) {
        static SmemOptIn opt[3];
        auto kern = gmode == 0 ? cov_build_kernel<0, fam> : (gmode == 1 ? cov_build_kernel<1, fam> : cov_build_kernel<2, fam>);
        if (cudaError_t e = opt[gmode].ensure(kern, smem); e != cudaSuccess) return e;
        kern<<<grid, 256, smem, st>>>(X, r, n, d, npad, par, winv, A, sA, full, gdim, Eout);
        return cudaGetLastError();
    });
}

__global__ void unpad_sym_kernel(const double* __restrict__ A, int npad, int n, double* __restrict__ out, int mirror) {
    size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * n) return;
    int i = idx / n, j = idx % n;
    int si = i, sj = j;
    if (mirror && j > i) { si = j; sj = i; }
    out[idx] = A[(size_t)si * npad + sj];
}

void launch_unpad_sym(const double* A, int npad, int n, double* out, int mirror, cudaStream_t st) {
    size_t tot = (size_t)n * n;
    unpad_sym_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(A, npad, n, out, mirror);
}

__global__ void pad_sym_kernel(const double* __restrict__ src, int n, int npad, double* __restrict__ dst) {
    const size_t nn = (size_t)npad * npad;
    const double* sb = src + (size_t)blockIdx.y * n * n;
    double* db = dst + (size_t)blockIdx.y * nn;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < nn; idx += (size_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / npad), j = (int)(idx % npad);
        db[idx] = (i < n && j < n) ? sb[(size_t)i * n + j] : (i == j ? 1.0 : 0.0);
    }
}

void launch_pad_sym(const double* src, int n, int npad, double* dst, int batch, cudaStream_t st) {
    const size_t nn = (size_t)npad * npad;
    const unsigned gx = (unsigned)std::min<size_t>((nn + 255) / 256, 4096);
    pad_sym_kernel<<<dim3(gx, batch), 256, 0, st>>>(src, n, npad, dst);
}

__global__ void unpad_lower_kernel(const double* __restrict__ src, int npad, int n, double* __restrict__ dst) {
    const size_t tot = (size_t)n * n;
    const double* sb = src + (size_t)blockIdx.y * npad * npad;
    double* db = dst + (size_t)blockIdx.y * tot;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < tot; idx += (size_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / n), j = (int)(idx % n);
        db[idx] = (j <= i) ? sb[(size_t)i * npad + j] : 0.0;
    }
}

void launch_unpad_lower(const double* src, int npad, int n, double* dst, int batch, cudaStream_t st) {
    const size_t tot = (size_t)n * n;
    const unsigned gx = (unsigned)std::min<size_t>((tot + 255) / 256, 4096);
    unpad_lower_kernel<<<dim3(gx, batch), 256, 0, st>>>(src, npad, n, dst);
}

// =========================================================================== K2 leaf
// One CTA factors a 128x128 SPD block held in shared memory and inverts its Cholesky factor.
// ---- v3 leaf: blocked, barrier-light, O(n^3) parts on the FP64 tensor pipe -------------------------
// The v1 kernel (left-looking, one column per step) spent one block barrier, one FP64 sqrt and one FP64 divide
// per column on a 1024-thread CTA (238 us per launch of 128x128 blocks, the longest latency chain of an evaluation).
// v3 keeps the block in shared memory and works in 8-wide panels:
//   potrf  (16 panels): (1) the 8x8 diagonal block is factored by ONE warp in registers -- lane i owns
//          row i, pivots and columns travel by shuffles, 1/sqrt(pivot) comes from rsqrt() so there is
//          no divide on the chain; (2) the rows below are solved against it, one thread per row;
//          (3) the trailing block gets its rank-8 update as two DMMA.8x8x4 per lower 8x8 fragment,
//          operands and accumulator read straight from shared memory, two fragments in flight per warp.
//          Look-ahead: in step (3) warp 0 updates only the next diagonal block and factors it at once
//          (step (1) of the next panel) while the warps of the other three scheduler partitions do the
//          rest of the update, so the serial pivot chain and the DMMA work overlap.  2 barriers per panel.
//   trtri: the 8x8 diagonal inverses (one thread per column), then log2(128/8) = 4 doubling levels
//          X21 = -X22 (L21 X11), both products as DMMA fragments with the triangular k ranges; 9 barriers.
// L is kept in the lower triangle (diagonal included), X = L^-1 transposed in the upper triangle, its
// diagonal (1/L_ii) in dinv[]; the log-determinant is summed from the stored pivots afterwards.
// History (tools/perf_leaf.py, 32 blocks per launch): v1 238 us; v2 (same structure, scalar-FMA trailing
// update and inverse levels with register micro-tiles) 107 us, of which 33 us trailing update and 43 us
// inverse levels -- issue-bound, one FMA per instruction; v3 58.7 us; with look-ahead and four DMMA chains per
// warp in the inverse levels 45 us (tools/leaf_phases.cu: 109.6 k -> 82 k cycles).  The row stride is 132 (= 4 mod 16
// doubles, the same rule as the GEMM tiles) so the 8x4 / 4x8 fragment loads are bank-conflict-free; the
// few row-per-thread accesses of the panel solve pay a 4-way conflict instead.
// Phase timing of the leaf for tools/leaf_phases.cu (compiled only there, with -DGPE_LEAF_TIMING): thread 0 adds the
// cycles between barriers to g_leaf_cyc[phase].
#ifdef GPE_LEAF_TIMING
__device__ unsigned long long g_leaf_cyc[16];
#define LEAF_TICK(i) do { if (tid == 0) { long long now_ = clock64(); g_leaf_cyc[i] += (unsigned long long)(now_ - t_last_); t_last_ = now_; } } while (0)
#define LEAF_TICK_INIT long long t_last_ = clock64()
#else
#define LEAF_TICK(i) do { } while (0)
#define LEAF_TICK_INIT do { } while (0)
#endif
constexpr int LT = 512;          // threads of the leaf CTA
constexpr int PW = 8;            // panel width
constexpr int L3 = NB + 4;
constexpr int T3MAX = 64 * 68;

__global__ void __launch_bounds__(LT, 1) leaf_potrf_trtri_v3_kernel(const double* __restrict__ A, double* __restrict__ Linv,
                                                                     int ld, long long sA, long long sL, int off,
                                                                     double* __restrict__ logdet_part, int nleaf,
                                                                     int* __restrict__ status, double* __restrict__ Lfac) {
    extern __shared__ __align__(16) double S[];      // [NB][L3]
    double* Tm = S + NB * L3;                        // [T3MAX] product scratch of the inverse levels
    double* dinv = Tm + T3MAX;                       // [NB] 1 / L_ii
    double* pv = dinv + NB;                          // [NB] pivots
    __shared__ double red[32];
    __shared__ int s_bad;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fc = lane & 3;
    constexpr int NW = LT / 32;
    __shared__ unsigned char tri_rb[128], tri_cb[128];   // lower-triangle enumeration f = rb (rb + 1) / 2 + cb, f < 120
    LEAF_TICK_INIT;
    const double* Ab = A + (size_t)b * sA + (size_t)off * ld + off;
#pragma unroll 8
    for (int e = tid; e < NB * NB; e += LT) {
        int i = e >> 7, j = e & (NB - 1);
        S[i * L3 + j] = (j <= i) ? Ab[(size_t)i * ld + j] : 0.0;
    }
    if (tid < 120) {
        int rb = (int)((sqrtf(8.0f * (float)tid + 1.0f) - 1.0f) * 0.5f);
        while ((rb + 1) * (rb + 2) / 2 <= tid) rb++;
        while (rb * (rb + 1) / 2 > tid) rb--;
        tri_rb[tid] = (unsigned char)rb;
        tri_cb[tid] = (unsigned char)(tid - rb * (rb + 1) / 2);
    }
    if (tid == 0) s_bad = 0;
    __syncthreads();
    LEAF_TICK(0);

    // ------------------------------------------------------------------ potrf, 8-wide panels with look-ahead
    // 8x8 diagonal block in registers of warp 0: lane i owns row i
    auto factor_diag = [&](int j0) {
        double a[PW];
#pragma unroll
        for (int c = 0; c < PW; c++) a[c] = (lane < PW && c <= lane) ? S[(j0 + lane) * L3 + j0 + c] : 0.0;
#pragma unroll
        for (int j = 0; j < PW; j++) {
            double pj = __shfl_sync(0xffffffffu, a[j], j);
            if (!(pj > 0.0)) {           // LAPACK dpotrf: pivot <= 0 or NaN -> info = j + 1
                if (lane == 0 && s_bad == 0) s_bad = off + j0 + j + 1;
                pj = 1.0;
            }
            const double rj = rsqrt(pj);           // (a hand-rolled seed + 2 Newton steps was slower: 2.75 k vs 2.48 k cycles per panel)
            if (lane == j) {
                a[j] = pj * rj;
                pv[j0 + j] = pj;
                dinv[j0 + j] = rj;
            } else {
                a[j] *= rj;
            }
#pragma unroll
            for (int k = j + 1; k < PW; k++) {
                double lk = __shfl_sync(0xffffffffu, a[j], k);
                if (lane >= k) a[k] = fma(-a[j], lk, a[k]);
            }
        }
        if (lane < PW) {
#pragma unroll
            for (int c = 0; c < PW; c++)
                if (c <= lane) S[(j0 + lane) * L3 + j0 + c] = a[c];
        }
    };
    if (warp == 0) factor_diag(0);
    __syncthreads();
    LEAF_TICK(1);
    for (int j0 = 0; j0 < NB - PW; j0 += PW) {
        const int base = j0 + PW, R = NB - base;
        if (tid < R) {                   // panel solve: row r against the diagonal block
            double* row = S + (base + tid) * L3 + j0;
            double x[PW];
#pragma unroll
            for (int c = 0; c < PW; c++) x[c] = row[c];
#pragma unroll
            for (int j = 0; j < PW; j++) {
                double sacc = x[j];
#pragma unroll
                for (int k = 0; k < j; k++) sacc = fma(-x[k], S[(j0 + j) * L3 + j0 + k], sacc);
                x[j] = sacc * dinv[j0 + j];
            }
#pragma unroll
            for (int c = 0; c < PW; c++) row[c] = x[c];
        }
        __syncthreads();
        LEAF_TICK(2);
        // A22 -= L21 L21^T on the lower 8x8 fragments (2 DMMAs each).  Look-ahead: warp 0 updates the next diagonal
        // block (fragment 0) and factors it at once -- the serial pivot chain of panel j + 1 -- while warps 1..15 do the
        // other fragments, two in flight per warp.  (tools/leaf_phases.cu: the chain and the update were 29 % + 24 %
        // of the leaf when they ran one after the other.)
        const int nbk = R >> 3, F = nbk * (nbk + 1) / 2;
        if (warp == 0) {
            const double* ar = S + (base + fr) * L3 + j0 + fc;
            double* cp = S + (base + fr) * L3 + base + 2 * fc;
            double2 c = *reinterpret_cast<double2*>(cp);
            dmma884(c.x, c.y, -ar[0], ar[0]);
            dmma884(c.x, c.y, -ar[4], ar[4]);
            *reinterpret_cast<double2*>(cp) = c;
            __syncwarp();
            factor_diag(base);
        } else if (warp & 3) {
            // warps 4, 8, 12 share warp 0's scheduler and FP64 pipe: they stay out of the update so the pivot chain
            // runs undisturbed (12 workers: chain and update both ~2.1 k cycles per panel instead of 2.75 k)
            constexpr int NWK = NW - NW / 4;
            const int wid = warp - 1 - (warp >> 2);
            for (int f = 1 + wid; f < F; f += 2 * NWK) {
                const int f2 = f + NWK;
                const bool two = f2 < F;
                const int rb = tri_rb[f], cb = tri_cb[f];
                const int rb2 = two ? tri_rb[f2] : rb, cb2 = two ? tri_cb[f2] : cb;
                const double* ar = S + (base + 8 * rb + fr) * L3 + j0 + fc;
                const double* br = S + (base + 8 * cb + fr) * L3 + j0 + fc;
                double* cp = S + (base + 8 * rb + fr) * L3 + base + 8 * cb + 2 * fc;
                const double* ar2 = S + (base + 8 * rb2 + fr) * L3 + j0 + fc;
                const double* br2 = S + (base + 8 * cb2 + fr) * L3 + j0 + fc;
                double* cp2 = S + (base + 8 * rb2 + fr) * L3 + base + 8 * cb2 + 2 * fc;
                const double a0 = ar[0], a4 = ar[4], b0 = br[0], b4 = br[4];
                const double a0b = ar2[0], a4b = ar2[4], b0b = br2[0], b4b = br2[4];
                double2 c = *reinterpret_cast<double2*>(cp);
                double2 c2 = *reinterpret_cast<double2*>(cp2);
                dmma884(c.x, c.y, -a0, b0);
                dmma884(c2.x, c2.y, -a0b, b0b);
                dmma884(c.x, c.y, -a4, b4);
                dmma884(c2.x, c2.y, -a4b, b4b);
                *reinterpret_cast<double2*>(cp) = c;
                if (two) *reinterpret_cast<double2*>(cp2) = c2;
            }
        }
        __syncthreads();
        LEAF_TICK(3);
    }
    {                                    // log-determinant from the pivots: 2 sum log L_ii = sum log pivot_i
        double v = (tid < NB) ? log(pv[tid]) : 0.0;
        double tot = block_sum(v, red);
        if (tid == 0) {
            logdet_part[(size_t)b * nleaf + off / NB] = tot;
            if (s_bad) {
                int bad = s_bad, old = atomicCAS(&status[b], 0, bad);
                while (old != 0 && old > bad) {
                    int prev = atomicCAS(&status[b], old, bad);
                    if (prev == old) break;
                    old = prev;
                }
            }
        }
    }
    LEAF_TICK(4);
    // ------------------------------------------------------------------ trtri
    // X = L^-1 is kept transposed in the upper triangle (X[i][j], i > j, at S[j][i]), its diagonal in dinv.
    if (tid < NB) {                      // inverses of the 8x8 diagonal blocks, one thread per column
        const int o = tid & ~(PW - 1), c = tid & (PW - 1);
        double x[PW];
#pragma unroll
        for (int i = 0; i < PW; i++) {
            double sacc = 0.0;
#pragma unroll
            for (int k = 0; k < i; k++) sacc = fma(S[(o + i) * L3 + o + k], x[k], sacc);
            x[i] = (i == c) ? dinv[o + i] : ((i > c) ? -sacc * dinv[o + i] : 0.0);
        }
#pragma unroll
        for (int i = 0; i < PW; i++)
            if (i > c) S[tid * L3 + o + i] = x[i];
    }
    __syncthreads();
    LEAF_TICK(5);
    int lhb = 0;                         // log2(h / 8)
    for (int h = PW; h < NB; h <<= 1, lhb++) {  // doubling levels: X21 = -X22 (L21 X11) per node of size 2h
        const int hb = h >> 3, F = (NB / (2 * h)) << (2 * lhb), ldT = h + 4;
        // Two fragments per warp in flight, each with two accumulator chains (even / odd k4 steps): four independent
        // DMMA chains per warp.  The k ranges are warp-uniform, so the predicates around the DMMAs are too.
        // T = L21 X11: fragment (rb, cb); X11 is lower triangular: k4 steps from 2 cb on
        for (int f = warp; f < F; f += 2 * NW) {
            const int fB = f + NW;
            const bool two = fB < F;
            const int g = two ? fB : f;
            const int node = f >> (2 * lhb), rem = f & (hb * hb - 1), rb = rem >> lhb, cb = rem & (hb - 1), o = node * 2 * h;
            const int nodeB = g >> (2 * lhb), remB = g & (hb * hb - 1), rbB = remB >> lhb, cbB = remB & (hb - 1), oB = nodeB * 2 * h;
            const double* ar = S + (o + h + 8 * rb + fr) * L3 + o + fc;         // L21[8rb+fr][k]
            const double* arB = S + (oB + h + 8 * rbB + fr) * L3 + oB + fc;
            const int n = 8 * cb + fr, nB = 8 * cbB + fr;                       // this lane's column of X11
            const double* xr = S + (o + n) * L3 + o + fc;                       // X11[k][n] lives at S[o+n][o+k]
            const double* xrB = S + (oB + nB) * L3 + oB + fc;
            const double dn = dinv[o + n], dnB = dinv[oB + nB];
            double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0, p0 = 0.0, p1 = 0.0, q0 = 0.0, q1 = 0.0;
            for (int sidx = 2 * min(cb, cbB); sidx < 2 * hb; sidx += 2) {
                const int k = 4 * sidx + fc, k2 = k + 4;
                if (sidx >= 2 * cb) {
                    const double bv = (k > n) ? xr[4 * sidx] : ((k == n) ? dn : 0.0);
                    const double bv2 = (k2 > n) ? xr[4 * sidx + 4] : ((k2 == n) ? dn : 0.0);
                    dmma884(c0, c1, ar[4 * sidx], bv);
                    dmma884(e0, e1, ar[4 * sidx + 4], bv2);
                }
                if (sidx >= 2 * cbB) {
                    const double bv = (k > nB) ? xrB[4 * sidx] : ((k == nB) ? dnB : 0.0);
                    const double bv2 = (k2 > nB) ? xrB[4 * sidx + 4] : ((k2 == nB) ? dnB : 0.0);
                    dmma884(p0, p1, arB[4 * sidx], bv);
                    dmma884(q0, q1, arB[4 * sidx + 4], bv2);
                }
            }
            double* tp = Tm + node * h * ldT + (8 * rb + fr) * ldT + 8 * cb + 2 * fc;
            tp[0] = c0 + e0;
            tp[1] = c1 + e1;
            if (two) {
                double* tpB = Tm + nodeB * h * ldT + (8 * rbB + fr) * ldT + 8 * cbB + 2 * fc;
                tpB[0] = p0 + q0;
                tpB[1] = p1 + q1;
            }
        }
        __syncthreads();
        LEAF_TICK(6);
        // X21 = -X22 T: X22 lower triangular: k4 steps up to 2 rb + 1 (an even count); result stored transposed
        for (int f = warp; f < F; f += 2 * NW) {
            const int fB = f + NW;
            const bool two = fB < F;
            const int g = two ? fB : f;
            const int node = f >> (2 * lhb), rem = f & (hb * hb - 1), rb = rem >> lhb, cb = rem & (hb - 1), o = node * 2 * h;
            const int nodeB = g >> (2 * lhb), remB = g & (hb * hb - 1), rbB = remB >> lhb, cbB = remB & (hb - 1), oB = nodeB * 2 * h;
            const int r = 8 * rb + fr, rB = 8 * rbB + fr;                       // this lane's row of X22
            const double* xc = S + (o + h + fc) * L3 + o + h + r;               // X22[r][k] lives at S[o+h+k][o+h+r]
            const double* xcB = S + (oB + h + fc) * L3 + oB + h + rB;
            const double* tr = Tm + node * h * ldT + fc * ldT + 8 * cb + fr;    // T[k][8cb+fr]
            const double* trB = Tm + nodeB * h * ldT + fc * ldT + 8 * cbB + fr;
            const double dr = dinv[o + h + r], drB = dinv[oB + h + rB];
            double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0, p0 = 0.0, p1 = 0.0, q0 = 0.0, q1 = 0.0;
            for (int sidx = 0; sidx <= 2 * max(rb, rbB) + 1; sidx += 2) {
                const int k = 4 * sidx + fc, k2 = k + 4;
                if (sidx <= 2 * rb + 1) {
                    const double av = (k < r) ? xc[4 * sidx * L3] : ((k == r) ? dr : 0.0);
                    const double av2 = (k2 < r) ? xc[(4 * sidx + 4) * L3] : ((k2 == r) ? dr : 0.0);
                    dmma884(c0, c1, av, tr[4 * sidx * ldT]);
                    dmma884(e0, e1, av2, tr[(4 * sidx + 4) * ldT]);
                }
                if (sidx <= 2 * rbB + 1) {
                    const double av = (k < rB) ? xcB[4 * sidx * L3] : ((k == rB) ? drB : 0.0);
                    const double av2 = (k2 < rB) ? xcB[(4 * sidx + 4) * L3] : ((k2 == rB) ? drB : 0.0);
                    dmma884(p0, p1, av, trB[4 * sidx * ldT]);
                    dmma884(q0, q1, av2, trB[(4 * sidx + 4) * ldT]);
                }
            }
            double* xo = S + (o + 8 * cb + 2 * fc) * L3 + o + h + r;
            xo[0] = -(c0 + e0);
            xo[L3] = -(c1 + e1);
            if (two) {
                double* xoB = S + (oB + 8 * cbB + 2 * fc) * L3 + oB + h + rB;
                xoB[0] = -(p0 + q0);
                xoB[L3] = -(p1 + q1);
            }
        }
        __syncthreads();
        LEAF_TICK(7);
    }
    // results as 16-byte stores: L^-1 (lower, zeros above the diagonal) and, if asked for, the factor itself
    double* Lb = Linv + (size_t)b * sL + (size_t)off * ld + off;
#pragma unroll 8
    for (int e = tid; e < NB * NB / 2; e += LT) {
        const int i = e >> 6, j = (e & 63) * 2;
        double2 v;
        v.x = (j < i) ? S[j * L3 + i] : ((j == i) ? dinv[i] : 0.0);
        v.y = (j + 1 < i) ? S[(j + 1) * L3 + i] : ((j + 1 == i) ? dinv[i] : 0.0);
        *reinterpret_cast<double2*>(&Lb[(size_t)i * ld + j]) = v;
    }
    if (Lfac != nullptr) {
        double* Fb = Lfac + (size_t)b * sL + (size_t)off * ld + off;
#pragma unroll 8
        for (int e = tid; e < NB * NB / 2; e += LT) {
            const int i = e >> 6, j = (e & 63) * 2;
            double2 v;
            v.x = (j <= i) ? S[i * L3 + j] : 0.0;
            v.y = (j + 1 <= i) ? S[i * L3 + j + 1] : 0.0;
            *reinterpret_cast<double2*>(&Fb[(size_t)i * ld + j]) = v;
        }
    }
    __syncthreads();
    LEAF_TICK(8);
}

void launch_leaf(const double* A, double* Linv, int ld, long long sA, long long sL, int off,
                 double* logdet_part, int nleaf, int* status, int B, cudaStream_t st, double* Lfac) {
    static SmemOptIn opt3;
    const size_t smem3 = (size_t)(NB * L3 + T3MAX + 2 * NB) * sizeof(double);
    opt3.ensure(leaf_potrf_trtri_v3_kernel, smem3);
    leaf_potrf_trtri_v3_kernel<<<B, LT, smem3, st>>>(A, Linv, ld, sA, sL, off, logdet_part, nleaf, status, Lfac);
}

// =========================================================================== K3 pieces
__global__ void build_hy_kernel(const double* __restrict__ H, const double* __restrict__ y, int n, int q, int npad,
                                double* __restrict__ HY) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npad * NR) return;
    int i = idx / NR, c = idx % NR;
    double v = 0.0;
    if (i < n) {
        if (c < q) v = H[(size_t)i * q + c];
        else if (c == q) v = y[i];
    }
    HY[idx] = v;
}

void launch_build_hy(const double* H, const double* y, int n, int q, int npad, double* HY, cudaStream_t st) {
    build_hy_kernel<<<(npad * NR + 255) / 256, 256, 0, st>>>(H, y, n, q, npad, HY);
}

// Gram partials: GP[b][slab][c1][c2] = sum_{i in slab} Wy[i][c1] Wy[i][c2].  One 128-row slab per CTA, loaded in one
// pass (the 512-row slabs in 64-row steps were a chain of dependent global-load latencies: 20-36 us for one item);
// four accumulator chains per entry (rows mod 4), added in a fixed order.
__global__ void __launch_bounds__(1024) gram_kernel(const double* __restrict__ Wy, int npad, double* __restrict__ GP) {
    __shared__ double T[GRAM_SLAB][NR + 1];
    const int slab = blockIdx.x, b = blockIdx.y, nslab = gridDim.x;
    const int c1 = threadIdx.x / NR, c2 = threadIdx.x % NR;
    const double* Wb = Wy + ((size_t)b * npad + (size_t)slab * GRAM_SLAB) * NR;
#pragma unroll
    for (int e = threadIdx.x; e < GRAM_SLAB * NR; e += 1024) T[e / NR][e % NR] = Wb[e];
    __syncthreads();
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll 8
    for (int rr = 0; rr < GRAM_SLAB; rr += 4) {
        a0 = fma(T[rr][c1], T[rr][c2], a0);
        a1 = fma(T[rr + 1][c1], T[rr + 1][c2], a1);
        a2 = fma(T[rr + 2][c1], T[rr + 2][c2], a2);
        a3 = fma(T[rr + 3][c1], T[rr + 3][c2], a3);
    }
    GP[((size_t)b * nslab + slab) * NR * NR + threadIdx.x] = (a0 + a1) + (a2 + a3);
}

void launch_gram(const double* Wy, int npad, int B, double* GP, cudaStream_t st) {
    int nslab = (npad + GRAM_SLAB - 1) / GRAM_SLAB;
    gram_kernel<<<dim3(nslab, B), 1024, 0, st>>>(Wy, npad, GP);
}

// GLS mean + log-likelihood scalars (one CTA per batch item).
//   Wy = L^-1 [H | y] = [w | u];  Q = w^T w = K K^T;  beta = Q^-1 w^T u;  z = u - w beta;
//   quad = |z|^2 = y^T (A^-1 y - A^-1 H beta)      (_emulatoroptimise.py:324-325 / :438)
//   Z = [ w K^-T | sqrt(f) z ]  so that  U = L^-T Z = [ A^-1 H K^-T | sqrt(f) (alpha - Gm beta) ].
__global__ void __launch_bounds__(256) llh_finalize_kernel(const double* __restrict__ Wy, const double* __restrict__ GP,
                                                           const double* __restrict__ logdet_part, int nleaf, int nslab,
                                                           int n, int q, int npad, int mode, ItemPar* par, ItemOut* out,
                                                           double* __restrict__ beta_out, double* __restrict__ Z,
                                                           int* __restrict__ status, const double* __restrict__ beta_override,
                                                           double* __restrict__ Kout) {
    __shared__ double G[NR][NR + 1];
    __shared__ double Kf[NR][NR + 1];
    __shared__ double beta[NR], tv[NR], rK[NR];   // rK[a] = 1 / K_aa
    __shared__ double red[32];
    __shared__ double s_quad, s_sqrtf, s_logdetQ;
    __shared__ int s_badQ;
    const int b = blockIdx.x, tid = threadIdx.x;
    for (int e = tid; e < NR * NR; e += 256) {
        double s = 0.0;
        for (int sl = 0; sl < nslab; sl++) s += GP[((size_t)b * nslab + sl) * NR * NR + e];
        G[e / NR][e % NR] = s;
    }
    if (tid == 0) s_badQ = 0;
    __syncthreads();
    if (tid < 32) {
        // warp-level Cholesky of Q (q <= 31): lane i owns row i
        const int i = tid;
        for (int j = 0; j < q; j++) {
            double s = 0.0, pv = 0.0;
            for (int k = 0; k < j; k++) {
                double kjk = Kf[j][k];
                if (i < q) s = fma(Kf[i][k], kjk, s);
                pv = fma(kjk, kjk, pv);
            }
            double piv = G[j][j] - pv;
            if (!(piv > 0.0)) {
                if (i == 0 && s_badQ == 0) s_badQ = j + 1;
                piv = 1.0;
            }
            const double rk = rsqrt(piv);                // one reciprocal root per column, no divide on the chain
            if (i == j) { Kf[j][j] = piv * rk; rK[j] = rk; }
            else if (i > j && i < q) Kf[i][j] = (G[i][j] - s) * rk;
            else if (i < j) Kf[i][j] = 0.0;
            __syncwarp();
        }
        // log det Q = sum log pivot_j (= 2 sum log K_jj), lanes in parallel
        double lp = (i < q) ? -2.0 * log(rK[i]) : 0.0;
        lp = warp_sum(lp);
        if (i == 0) {
            // K t = w^T u ; K^T beta = t
            for (int a = 0; a < q; a++) {
                double s = G[a][q];
                for (int k = 0; k < a; k++) s -= Kf[a][k] * tv[k];
                tv[a] = s * rK[a];
            }
            for (int a = q - 1; a >= 0; a--) {
                double s = tv[a];
                for (int k = a + 1; k < q; k++) s -= Kf[k][a] * beta[k];
                beta[a] = s * rK[a];
            }
            s_logdetQ = lp;
        }
    }
    __syncthreads();
    const double* Wb = Wy + (size_t)b * npad * NR;
    double* Zb = Z + (size_t)b * npad * NR;
    // pass 1: z_i and quad
    double qp = 0.0;
    for (int i = tid; i < npad; i += 256) {
        const double* wr = Wb + (size_t)i * NR;
        double z = wr[q];
        for (int a = 0; a < q; a++) z = fma(-wr[a], beta[a], z);
        qp = fma(z, z, qp);
        Zb[(size_t)i * NR + q] = z;
    }
    double quad = block_sum(qp, red);
    if (tid == 0) {
        double logdetA = 0.0;
        for (int l = 0; l < nleaf; l++) logdetA += logdet_part[(size_t)b * nleaf + l];
        ItemOut o;
        o.logdetA = logdetA;
        o.logdetQ = s_logdetQ;
        o.quad = quad;
        const double nq = (double)(n - q);
        if (mode & GPE_MODE_MUCM) {
            double sig2 = quad / (nq - 2.0);
            o.sig2 = sig2;
            o.llh = 0.5 * (nq * log(sig2) + logdetA + s_logdetQ);
            o.f = nq / (sig2 * (nq - 2.0));
            o.s2g = sig2;
            par[b].sigma = sqrt(sig2);
        } else {
            o.sig2 = par[b].s2A;
            o.llh = 0.5 * (quad + logdetA + s_logdetQ + nq * log(2.0 * 3.14159265358979323846));
            o.f = 1.0;
            o.s2g = par[b].s2A;
        }
        o.pad_ = 0.0;
        out[b] = o;
        s_quad = quad;
        s_sqrtf = sqrt(o.f);
        for (int a = 0; a < q; a++) beta_out[(size_t)b * NR + a] = beta[a];
        if (Kout != nullptr)
            for (int a = 0; a < q; a++)
                for (int k = 0; k < q; k++) Kout[((size_t)b * NR + a) * NR + k] = (k <= a) ? Kf[a][k] : 0.0;
        if (s_badQ && status[b] == 0) status[b] = npad + s_badQ;
    }
    __syncthreads();
    if (beta_override != nullptr) {   // Posterior with a user-supplied beta (before optimalbeta has run)
        if (tid < q) beta[tid] = beta_override[tid];
        __syncthreads();
        for (int i = tid; i < npad; i += 256) {
            const double* wr = Wb + (size_t)i * NR;
            double z = wr[q];
            for (int a = 0; a < q; a++) z = fma(-wr[a], beta[a], z);
            Zb[(size_t)i * NR + q] = z;
        }
    }
    const double sf = s_sqrtf;
    // pass 2: Z rows: v K^T = w_i  <=>  K v^T = w_i^T  (forward substitution), and scale z
    for (int i = tid; i < npad; i += 256) {
        const double* wr = Wb + (size_t)i * NR;
        double v[NR];
#pragma unroll
        for (int a = 0; a < NR; a++) {
            if (a < q) {
                double s = wr[a];
                for (int k = 0; k < a; k++) s = fma(-Kf[a][k], v[k], s);
                v[a] = s * rK[a];
            } else {
                v[a] = 0.0;
            }
        }
        double* zr = Zb + (size_t)i * NR;
        double zq = zr[q] * sf;
#pragma unroll
        for (int a = 0; a < NR; a++) zr[a] = (a < q) ? v[a] : ((a == q) ? zq : 0.0);
    }
}

void launch_llh_finalize(const double* Wy, const double* GP, const double* logdet_part, int nleaf,
                         int n, int q, int npad, int mode, ItemPar* par, ItemOut* out, double* beta,
                         double* Z, int* status, int B, const double* beta_override, double* Kout, cudaStream_t st) {
    int nslab = (npad + GRAM_SLAB - 1) / GRAM_SLAB;
    llh_finalize_kernel<<<B, 256, 0, st>>>(Wy, GP, logdet_part, nleaf, nslab, n, q, npad, mode, par, out, beta, Z, status,
                                           beta_override, Kout);
}

// =========================================================================== K1g fused gradient reduction
// grad_k = 1/2 sum_ij T^k_ij W_ij,  W = A^-1 - U U^T  (SURVEY A.2; _emulatoroptimise.py:345-372,
// :450-487 collapse to this).  The d gradient matrices T^k are never formed: each 64x64 tile of
// A^-1 is read once, E_ij = exp(-D_ij) is recomputed from X, and d+3 weighted sums are reduced.
constexpr int GD = 16;  // dims accumulated per register pass

// USE_E: E = exp(-D) is read from the copy the covariance build kept (8 B per entry from an idle HBM) instead of being
// recomputed (2d + 22 FP64 instructions per entry on the pipe this kernel is bound by).
// FAM == FAMILY_MATERN52 (recompute path only): t holds 2 W G for the d delta sums and sE collects 2 W R directly.
template <bool USE_E, int FAM>
__global__ void __launch_bounds__(256, 2) grad_partial_kernel(const double* __restrict__ X, const double* __restrict__ r,
                                                           int n, int d, int npad, const double* __restrict__ winv,
                                                           const double* __restrict__ Ainv, long long sAinv,
                                                           const double* __restrict__ U, int nu, double* __restrict__ part,
                                                           const double* __restrict__ E) {
    int ti, tj;
    tri_decode(blockIdx.x, ti, tj);
    const int b = blockIdx.z;
    extern __shared__ __align__(16) double sm[];
    double* Xi = sm;                                // [d][64]
    double* Xj = Xi + (size_t)d * CT;               // [d][66]
    double* Ui = Xj + (size_t)d * (CT + 2);         // [nu][64]
    double* Uj = Ui + (size_t)nu * CT;              // [nu][66]
    double* red = Uj + (size_t)nu * (CT + 2);       // [8][d+3]
    const int tid = threadIdx.x;
    fill_scaled_tiles(X, winv + (size_t)b * d, n, d, ti * CT, tj * CT, Xi, Xj, tid);
    const double* Ub = U + (size_t)b * npad * NR;
    {
        const int row = tid >> 2;
        for (int c = tid & 3; c < nu; c += 4) {
            Ui[c * CT + row] = Ub[(size_t)(ti * CT + row) * NR + c];
            Uj[c * (CT + 2) + row] = Ub[(size_t)(tj * CT + row) * NR + c];
        }
    }
    __syncthreads();
    const int ty = tid >> 4, tx = tid & 15;
    const double* Ab = Ainv + (size_t)b * sAinv;
    double t[4][4];
    double sE = 0.0, sD = 0.0, sDr = 0.0;
    {
        // The A^-1 tile is requested first (ncu: long-scoreboard was the top stall with the loads issued
        // right before their use); its latency hides behind the U.U^T dot products.
        double2 av[4][2];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int h = 0; h < 2; h++)
                av[a][h] = __ldg(reinterpret_cast<const double2*>(&Ab[(size_t)(ti * CT + ty + 16 * a) * npad + tj * CT + 32 * h + 2 * tx]));
        double2 ev[4][2];
        if (USE_E) {
            const double* Eb = E + (size_t)b * sAinv;
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int h = 0; h < 2; h++)
                    ev[a][h] = __ldg(reinterpret_cast<const double2*>(&Eb[(size_t)(ti * CT + ty + 16 * a) * npad + tj * CT + 32 * h + 2 * tx]));
        }
        double D[4][4], dot[4][4];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) dot[a][c] = 0.0;
        for (int k = 0; k < nu; k++) {
            double ui[4], uj[4];
#pragma unroll
            for (int a = 0; a < 4; a++) ui[a] = Ui[k * CT + ty + 16 * a];
            double2 v0 = *reinterpret_cast<const double2*>(&Uj[k * (CT + 2) + 2 * tx]);
            double2 v1 = *reinterpret_cast<const double2*>(&Uj[k * (CT + 2) + 32 + 2 * tx]);
            uj[0] = v0.x; uj[1] = v0.y; uj[2] = v1.x; uj[3] = v1.y;
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int c = 0; c < 4; c++) dot[a][c] = fma(ui[a], uj[c], dot[a][c]);
        }
        // W = A^-1 - U U^T  (dot becomes W)
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                dot[a][2 * h] = av[a][h].x - dot[a][2 * h];
                dot[a][2 * h + 1] = av[a][h].y - dot[a][2 * h + 1];
            }
        if (USE_E) {
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int h = 0; h < 2; h++) { D[a][2 * h] = ev[a][h].x; D[a][2 * h + 1] = ev[a][h].y; }
        } else {
            sqdist_tile<4, 16, 32>(Xi, Xj, d, ty, tx, D);
            if constexpr (FAM == FAMILY_GAUSSIAN) {
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int c = 0; c < 4; c++) D[a][c] = gpe_exp(-D[a][c]);      // 16 interleaved chains, no branches
            }
        }
#pragma unroll
        for (int a = 0; a < 4; a++) {
            int gi = ti * CT + ty + 16 * a;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                int gj0 = tj * CT + 32 * h + 2 * tx;
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    int gj = gj0 + e;
                    double wv = dot[a][2 * h + e];
                    double tv = 0.0;
                    if constexpr (FAM == FAMILY_GAUSSIAN) {
                        // A^-1 is valid on and below the diagonal only (LAUUM computes lower fragments):
                        // every off-diagonal pair is taken once from the lower triangle with weight 2
                        if (gi < n && gj < n) {
                            if (gi == gj) {
                                sD += wv;
                                if (r != nullptr) sDr = fma(wv, r[gi], sDr);
                            } else if (gi > gj) {
                                tv = 2.0 * wv * D[a][2 * h + e];
                            }
                        }
                        sE += tv;
                    } else {
                        double g, sv = 0.0;
                        const double rv = gpe_matern52(D[a][2 * h + e], g);     // unconditional: the chains interleave
                        if (gi < n && gj < n) {
                            if (gi == gj) {
                                sD += wv;
                                if (r != nullptr) sDr = fma(wv, r[gi], sDr);
                            } else if (gi > gj) {
                                tv = 2.0 * wv * g;
                                sv = 2.0 * wv * rv;
                            }
                        }
                        sE += sv;
                    }
                    t[a][2 * h + e] = tv;
                }
            }
        }
    }
    const int nv = d + 3;
    const int warp = tid >> 5, lane = tid & 31;
    double* pout = part + ((size_t)b * gridDim.x + blockIdx.x) * nv;
    sE = warp_sum(sE); sD = warp_sum(sD); sDr = warp_sum(sDr);
    if (lane == 0) { red[warp * nv + d] = sE; red[warp * nv + d + 1] = sD; red[warp * nv + d + 2] = sDr; }
    for (int k0 = 0; k0 < d; k0 += GD) {
        double acc[GD];
#pragma unroll
        for (int kk = 0; kk < GD; kk++) acc[kk] = 0.0;
#pragma unroll
        for (int kk = 0; kk < GD; kk++) {
            int k = k0 + kk;
            if (k < d) {
                double xi[4], xj[4];
                tile_operands<4, 16, 32>(Xi, Xj, k, ty, tx, xi, xj);
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        double df = xi[a] - xj[c];
                        acc[kk] = fma(t[a][c], df * df, acc[kk]);
                    }
            }
        }
#pragma unroll
        for (int kk = 0; kk < GD; kk++) {
            double v = warp_sum(acc[kk]);
            if (lane == 0 && k0 + kk < d) red[warp * nv + k0 + kk] = v;
        }
    }
    __syncthreads();
    for (int v = tid; v < nv; v += 256) {
        double s = 0.0;
#pragma unroll
        for (int wv = 0; wv < 8; wv++) s += red[wv * nv + v];
        pout[v] = s;
    }
}

void launch_grad_partial(const double* X, const double* r, int n, int d, int npad, const double* winv,
                         const double* Ainv, long long sAinv, const double* U, int nu, double* part,
                         int B, cudaStream_t st, const double* E, int family) {
    int nt = npad / CT;
    size_t smem = ((size_t)(d + nu) * (CT + CT + 2) + 8 * (size_t)(d + 3)) * sizeof(double);
    const dim3 grid(nt * (nt + 1) / 2, 1, B);
    with_family(family, [&](auto fam) {
        static SmemOptIn optin, optin_e;
        auto kern = grad_partial_kernel<false, fam>;
        SmemOptIn* opt = &optin;
        if constexpr (fam == FAMILY_GAUSSIAN)      // Matérn: always recomputed, the covariance build keeps no copy of R or G
            if (E != nullptr) { kern = grad_partial_kernel<true, fam>; opt = &optin_e; }      // (same layout and item stride as A^-1)
        opt->ensure(kern, smem);
        kern<<<grid, 256, smem, st>>>(X, r, n, d, npad, winv, Ainv, sAinv, U, nu, part, E);
    });
}

// Sum the tile partials in a fixed order and apply the per-parameter prefactors
// (parameter order [delta.., nugget?, sigma?], _emulatoroptimise.py:94-103).
__global__ void __launch_bounds__(256) grad_finalize_kernel(const double* __restrict__ part, int ntile, int n, int d, int p,
                                                            int mode, const ItemPar* __restrict__ par,
                                                            const ItemOut* __restrict__ out, const int* __restrict__ status,
                                                            double* __restrict__ llh, double* __restrict__ grad,
                                                            double* __restrict__ sigma_hat) {
    extern __shared__ double sums[];  // [d+3]
    __shared__ double red[32];
    const int b = blockIdx.x, tid = threadIdx.x, nv = d + 3;
    const double* pb = part + (size_t)b * ntile * nv;
    for (int v = 0; v < nv; v++) {
        double s = 0.0;
        for (int t = tid; t < ntile; t += 256) s += pb[(size_t)t * nv + v];
        double tot = block_sum(s, red);
        if (tid == 0) sums[v] = tot;
    }
    __syncthreads();
    if (tid == 0) {
        const ItemPar ip = par[b];
        const ItemOut o = out[b];
        const double sE = sums[d], sD = sums[d + 1], sDr = sums[d + 2];
        double* g = grad + (size_t)b * p;
        for (int k = 0; k < d; k++) g[k] = 0.5 * o.s2g * ip.c * sums[k];
        int idx = d;
        if (mode & GPE_MODE_NUGGET_FREE) {
            if (mode & GPE_MODE_ALT_NUGGET) g[idx] = 0.5 * ip.nugget * ip.nugget * o.s2g * sD;
            else g[idx] = 0.5 * (-0.5 * ip.nugget * o.s2g) * sE;
            idx++;
        }
        if (!(mode & GPE_MODE_MUCM)) g[idx] = 0.5 * (ip.offs * sE + ip.diagv * sD + (ip.radd - 1.0) * sDr);
        llh[b] = o.llh;
        sigma_hat[b] = ip.sigma;
        (void)status;
    }
}

void launch_grad_finalize(const double* part, int ntile, int n, int d, int npad, int p, int mode, const ItemPar* par,
                          const ItemOut* out, const int* status, double* llh, double* grad,
                          double* sigma_hat, int B, cudaStream_t st) {
    grad_finalize_kernel<<<B, 256, (d + 3) * sizeof(double), st>>>(part, ntile, n, d, p, mode, par, out, status,
                                                                  llh, grad, sigma_hat);
}

}  // namespace gpe
