// Leave-one-out cross-validation (DESIGN.md section 9c): the per-item statistics, the dense weight pieces and the finalize
// of the LOO objective of a GPE_MODE_LOO batch, and gpe_loo on the fit state.
//
// With A the matrix the likelihood of the same mode factors, P = A^-1 - U_q U_q^T (U_q = A^-1 H K^-T, the first q columns
// of the skinny panel U) and alpha = P y = U[:, q] / sqrt(f), the LOO predictive of y_i with beta re-estimated on the other
// n - 1 points has residual e_i = alpha_i / P_ii and variance s^2 / P_ii.  The objective
//     L = 1/2 sum_i [ log(2 pi s^2 / P_ii) + alpha_i^2 / (s^2 P_ii) ]
// (s^2 = 1 in gp4ml mode; in MUCM mode s^2 is profiled: s^2 = mean_i alpha_i^2 / P_ii) has the gradient
//     dL/dtheta_k = sum_ab W_ab dA_ab/dtheta_k,   W = F F^T - 1/2 [(P c) alpha^T + alpha (P c)^T],   F = P diag(sqrt w),
//     w_i = 1/2 (1/P_ii + alpha_i^2 / (s^2 P_ii^2)),   c_i = alpha_i / (s^2 P_ii).
#include "gpe_handle.h"

#include <climits>
#include <cmath>
#include <vector>

namespace gpe {

// Column layout of the LOO panel V [npad][NR] (the dead Wy panel of the item): the right-hand side of the product P c = F (c / sqrt w)
// must be a column of the B operand, the others ride along.
enum { LOO_CW = 0, LOO_ALPHA = 1, LOO_SQW = 2, LOO_PII = 3 };

// One CTA per item.  Reads diag(A^-1) from the stored lower tiles, U and the item's f; writes V, the objective (out[b].llh),
// sigma_hat (MUCM: s, into par[b].sigma) and, for an item with P_ii <= 0, status = 2 npad + i + 1 (first such i).  An item
// that is flagged here or whose factorisation failed gets an all-zero V, so its products and reduction stay finite and
// leave the other items of the launch alone.
__global__ void __launch_bounds__(256) loo_stats_kernel(const double* __restrict__ Ainv, long long sA, const double* __restrict__ U,
                                                        int n, int q, int npad, int mode, ItemPar* __restrict__ par,
                                                        ItemOut* __restrict__ out, double* __restrict__ V, int* __restrict__ status) {
    __shared__ double red[32];
    __shared__ int s_bad;
    __shared__ double s_s2, s_obj;
    const int b = blockIdx.x, tid = threadIdx.x;
    const double* Ab = Ainv + (size_t)b * sA;
    const double* Ub = U + (size_t)b * npad * NR;
    double* Vb = V + (size_t)b * npad * NR;
    if (tid == 0) s_bad = INT_MAX;
    __syncthreads();
    const double rsf = 1.0 / sqrt(out[b].f);
    double sq = 0.0, slog = 0.0;
    for (int i = tid; i < n; i += 256) {
        const double* ur = Ub + (size_t)i * NR;
        double pii = Ab[(size_t)i * npad + i];
        for (int a = 0; a < q; a++) pii = fma(-ur[a], ur[a], pii);
        const double al = ur[q] * rsf;
        if (!(pii > 0.0) || !isfinite(al)) atomicMin(&s_bad, i);
        Vb[(size_t)i * NR + LOO_ALPHA] = al;
        Vb[(size_t)i * NR + LOO_PII] = pii;
        sq += al * al / pii;
        slog += log(pii);
    }
    sq = block_sum(sq, red);
    __syncthreads();
    slog = block_sum(slog, red);
    const bool mucm = mode & GPE_MODE_MUCM;
    if (tid == 0) {
        const double s2 = mucm ? sq / n : 1.0;
        s_s2 = s2;
        s_obj = 0.5 * ((double)n * log(2.0 * 3.14159265358979323846 * s2) - slog + sq / s2);
    }
    __syncthreads();
    const bool dead = s_bad != INT_MAX || status[b] != 0;
    const double s2 = s_s2;
    for (int i = tid; i < npad; i += 256) {
        double* vr = Vb + (size_t)i * NR;
        double cw = 0.0, al = 0.0, sw = 0.0;
        if (i < n && !dead) {
            const double pii = vr[LOO_PII];
            al = vr[LOO_ALPHA];
            const double c = al / (s2 * pii);
            const double w = 0.5 * (1.0 / pii + al * c / pii);
            sw = sqrt(w);
            cw = c / sw;
        }
        for (int a = 0; a < NR; a++) vr[a] = (a == LOO_CW) ? cw : (a == LOO_ALPHA) ? al : (a == LOO_SQW) ? sw : 0.0;
    }
    if (tid == 0) {
        out[b].llh = dead ? INFINITY : s_obj;
        out[b].sig2 = s2;
        if (mucm) par[b].sigma = sqrt(s2);
        if (s_bad != INT_MAX && status[b] == 0) status[b] = 2 * npad + s_bad + 1;
    }
}

void launch_loo_stats(const double* Ainv, long long sA, const double* U, int n, int q, int npad, int mode, ItemPar* par, ItemOut* out,
                      double* V, int* status, int B, cudaStream_t st) {
    loo_stats_kernel<<<B, 256, 0, st>>>(Ainv, sA, U, n, q, npad, mode, par, out, V, status);
}

// F = P diag(sqrt w) as a dense [npad][npad] matrix per item: the lower-stored A^-1 mirrored, minus U_q U_q^T, columns scaled.
// 64 x 64 tile per CTA; the source tile of A^-1 (always from the lower triangle) goes through shared memory, so reads and
// writes are both row-contiguous.  Rows / columns >= n are zero.
constexpr int LT64 = 64;
__global__ void __launch_bounds__(256) loo_f_kernel(const double* __restrict__ Ainv, long long sA, const double* __restrict__ U,
                                                    const double* __restrict__ V, int n, int q, int npad, double* __restrict__ F) {
    extern __shared__ double sm[];
    double(*T)[LT64 + 1] = reinterpret_cast<double(*)[LT64 + 1]>(sm);                     // [64][65]
    double* Ui = sm + LT64 * (LT64 + 1);                                                    // [q][64]
    double* Uj = Ui + (size_t)q * LT64;                                                     // [q][65]
    double* sw = Uj + (size_t)q * (LT64 + 1);                                               // [64]
    const int tj = blockIdx.x, ti = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
    const double* Ab = Ainv + (size_t)b * sA;
    const double* Ub = U + (size_t)b * npad * NR;
    const double* Vb = V + (size_t)b * npad * NR;
    const int si = ti >= tj ? ti : tj, sj = ti >= tj ? tj : ti;       // source tile in the lower triangle
    for (int e = tid; e < LT64 * LT64; e += 256) {
        const int r = e >> 6, c = e & 63;
        T[r][c] = Ab[(size_t)(si * LT64 + r) * npad + sj * LT64 + c];
    }
    for (int e = tid; e < q * LT64; e += 256) {
        const int r = e / q, a = e % q;
        Ui[a * LT64 + r] = Ub[(size_t)(ti * LT64 + r) * NR + a];
        Uj[a * (LT64 + 1) + r] = Ub[(size_t)(tj * LT64 + r) * NR + a];
    }
    if (tid < LT64) sw[tid] = Vb[(size_t)(tj * LT64 + tid) * NR + LOO_SQW];
    __syncthreads();
    const int ty = tid >> 4, tx = tid & 15;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[a][c] = 0.0;
    for (int k = 0; k < q; k++) {
        double ui[4], uj[4];
#pragma unroll
        for (int a = 0; a < 4; a++) { ui[a] = Ui[k * LT64 + ty + 16 * a]; uj[a] = Uj[k * (LT64 + 1) + tx + 16 * a]; }
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) acc[a][c] = fma(ui[a], uj[c], acc[a][c]);
    }
    double* Fb = F + (size_t)b * sA;
#pragma unroll
    for (int a = 0; a < 4; a++) {
        const int r = ty + 16 * a, gi = ti * LT64 + r;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int cc = tx + 16 * c, gj = tj * LT64 + cc;
            const bool lower_src = ti > tj || (ti == tj && r >= cc);
            const double ainv = lower_src ? T[r][cc] : T[cc][r];
            Fb[(size_t)gi * npad + gj] = (gi < n && gj < n) ? (ainv - acc[a][c]) * sw[cc] : 0.0;
        }
    }
}

void launch_loo_f(const double* Ainv, long long sA, const double* U, const double* V, int n, int q, int npad, double* F, int B,
                  cudaStream_t st) {
    const int nt = npad / LT64;
    const size_t smem = ((size_t)LT64 * (LT64 + 1) + (size_t)q * (2 * LT64 + 1) + LT64) * sizeof(double);
    static SmemOptIn opt;
    opt.ensure(loo_f_kernel, smem);
    loo_f_kernel<<<dim3(nt, nt, B), 256, smem, st>>>(Ainv, sA, U, V, n, q, npad, F);
}

// C (lower triangle, i >= j) = -1/2 [(P c)_i alpha_j + alpha_i (P c)_j]: the rank-2 part of W, written before F F^T is
// accumulated onto it.  Pc [npad][NR] holds P c in column LOO_CW (the product F V).
__global__ void __launch_bounds__(256) loo_rank2_kernel(const double* __restrict__ Pc, const double* __restrict__ V, int npad,
                                                        double* __restrict__ C, long long sC) {
    const int i = blockIdx.x, b = blockIdx.y;
    const double* Pb = Pc + (size_t)b * npad * NR;
    const double* Vb = V + (size_t)b * npad * NR;
    const double pi = Pb[(size_t)i * NR + LOO_CW], ai = Vb[(size_t)i * NR + LOO_ALPHA];
    double* Cr = C + (size_t)b * sC + (size_t)i * npad;
    for (int j = threadIdx.x; j <= i; j += 256)
        Cr[j] = -0.5 * (pi * Vb[(size_t)j * NR + LOO_ALPHA] + ai * Pb[(size_t)j * NR + LOO_CW]);
}

void launch_loo_rank2(const double* Pc, const double* V, int npad, double* C, long long sC, int B, cudaStream_t st) {
    loo_rank2_kernel<<<dim3(npad, B), 256, 0, st>>>(Pc, V, npad, C, sC);
}

// Tile partials of the reduction on W summed in a fixed order, times the exact prefactors of dA/dtheta (the reduction
// returns sum_ij W_ij dA_ij / (prefactor)): delta_k: s2A c; nugget: -1/2 nu s2A (kernel) or s2A nu^2 (alt nugget, diagonal);
// sigma (gp4ml): A - diag(r).
__global__ void __launch_bounds__(256) loo_finalize_kernel(const double* __restrict__ part, int ntile, int d, int p, int mode,
                                                           const ItemPar* __restrict__ par, const ItemOut* __restrict__ out,
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
        const double sE = sums[d], sD = sums[d + 1], sDr = sums[d + 2];
        double* g = grad + (size_t)b * p;
        for (int k = 0; k < d; k++) g[k] = ip.offs * sums[k];
        int idx = d;
        if (mode & GPE_MODE_NUGGET_FREE) {
            if (mode & GPE_MODE_ALT_NUGGET) g[idx] = ip.nugget * ip.nugget * ip.s2A * sD;
            else g[idx] = -0.5 * ip.nugget * ip.s2A * sE;
            idx++;
        }
        if (!(mode & GPE_MODE_MUCM)) g[idx] = ip.offs * sE + ip.diagv * sD + (ip.radd - 1.0) * sDr;
        llh[b] = out[b].llh;
        sigma_hat[b] = ip.sigma;
    }
}

void launch_loo_finalize(const double* part, int ntile, int d, int p, int mode, const ItemPar* par, const ItemOut* out,
                         double* llh, double* grad, double* sigma_hat, int B, cudaStream_t st) {
    loo_finalize_kernel<<<B, 256, (d + 3) * sizeof(double), st>>>(part, ntile, d, p, mode, par, out, llh, grad, sigma_hat);
}

// gpe_loo: one thread per training point i.  diag(A^-1)_i is the squared norm of column i of L^-1 (rows k >= i); P_ii
// subtracts the row norm of U_q; alpha = U[:, q] - U_q t with t = K^T (beta_gls - beta_used) re-centres a state that was
// fitted with a caller's beta on the GLS estimate.  A point with P_ii <= 0 gets NaN for both outputs.
struct LooShift { double t[NR]; };

__global__ void __launch_bounds__(128) loo_fit_kernel(const double* __restrict__ Li, const double* __restrict__ E, const double* __restrict__ y,
                                                      int n, int q, int npad, LooShift sh, double sigma2, double* __restrict__ mean,
                                                      double* __restrict__ var) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;      // four chains, added in a fixed order
    int k = i;
    for (; k + 3 < n; k += 4) {
        const double a0 = Li[(size_t)k * npad + i], a1 = Li[(size_t)(k + 1) * npad + i];
        const double a2 = Li[(size_t)(k + 2) * npad + i], a3 = Li[(size_t)(k + 3) * npad + i];
        d0 = fma(a0, a0, d0); d1 = fma(a1, a1, d1); d2 = fma(a2, a2, d2); d3 = fma(a3, a3, d3);
    }
    for (; k < n; k++) { const double a0 = Li[(size_t)k * npad + i]; d0 = fma(a0, a0, d0); }
    double pii = (d0 + d1) + (d2 + d3);
    const double* er = E + (size_t)i * NR;
    double al = er[q];
    for (int a = 0; a < q; a++) {
        pii = fma(-er[a], er[a], pii);
        al = fma(-er[a], sh.t[a], al);
    }
    if (pii > 0.0) {
        mean[i] = y[i] - al / pii;
        var[i] = sigma2 / pii;
    } else {
        mean[i] = var[i] = NAN;
    }
}

}  // namespace gpe

using namespace gpe;

extern "C" int gpe_loo(gpe_handle* h, double* mean, double* var) {
    if (!h || !mean || !var) return h ? h->fail_msg("bad argument") : -2;
    if (!h->fitted) return h->fail_msg("gpe_fit_state has not succeeded on this handle");
    NvtxRange nvtx("gpe_loo");
    CK(cudaSetDevice(h->device));
    const int n = h->n, q = h->q;
    std::vector<double> K;
    CK(read_small(K, h->fK, (size_t)NR * NR));
    LooShift sh{};
    for (int a = 0; a < q; a++)
        for (int k = a; k < q; k++) sh.t[a] += K[(size_t)k * NR + a] * h->fit_dbeta[k];
    DevOut<double> md(h), vd(h);
    CK(md.stage(mean, (size_t)n));
    CK(vd.stage(var, (size_t)n));
    {
        ProfScope ps(h, gpe_handle::CAT_OTHER, h->st);
        loo_fit_kernel<<<(n + 127) / 128, 128, 0, h->st>>>(h->fLi, h->fE, h->y, n, q, h->npad, sh, h->fit_sigma * h->fit_sigma, md.p, vd.p);
    }
    h->launches++;
    CK(cudaGetLastError());
    CK(md.flush());
    CK(vd.flush());
    CK(cudaStreamSynchronize(h->st));
    return 0;
}
