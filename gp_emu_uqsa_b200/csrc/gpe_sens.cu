// K6 sensitivity / uncertainty integrals and the generic A^-1 B solve on the fitted training matrix.
// Reference arithmetic replaced: sensitivity/_sensitivityclasses.py
//   :40-44   e = A^-1 (f - H beta), G = A^-1 H                      -> gpe_solve
//   :90-102  Rtt, :599-626 P_prod_calc + Pw_calc (n x n product-form matrices) and their
//            contractions tr(A^-1 Pw), G^T Pw G, e^T Pw e (:187-197, :481-495)  -> gpe_sens_contract
//   :628-633 Tw_calc inside the x_w sweep of main_effect (:277-285)            -> gpe_sens_main_effect
//
// With B = diag(1/v), C = diag(1/delta^2) every such matrix has the form
//     P_kl = scale * u_k u_l * exp(-sum_i gamma_i (x_ki - x_li)^2),   u_k = prod_i exp(-a_i (x_ki - m_i)^2)
// (gamma_i = 0 for the integrated-out inputs), i.e. a rank-one-scaled Gaussian kernel: the same
// "build an n x n entry from X, reduce it against A^-1" pattern as the likelihood gradient.  The
// n^2 d tables P_prod / P_b4_prod of the reference (0.5 GB at n=2000, d=16) are never formed.
#include "gpe_handle.h"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace gpe;

#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return h->fail(#call, e__);        \
    } while (0)

namespace {

constexpr int ST = 64;   // tile edge

// rows [n,k] -> zero padded panel [npad, NR]
__global__ void pack_panel_kernel(const double* __restrict__ src, int n, int k, int npad, double* __restrict__ dst) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npad * NR) return;
    int i = idx / NR, c = idx % NR;
    dst[idx] = (i < n && c < k) ? src[(size_t)i * k + c] : 0.0;
}
__global__ void unpack_panel_kernel(const double* __restrict__ src, int n, int k, double* __restrict__ dst) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * k) return;
    int i = idx / k, c = idx % k;
    dst[idx] = src[(size_t)i * NR + c];
}

// One 64x64 tile of P per CTA (full grid: P is needed dense by the panel product); lower tiles
// also reduce sum_kl wgt * Ainv_kl * P_kl into tile partials (fixed-order final sum => deterministic).
__global__ void __launch_bounds__(256) sens_pw_kernel(const double* __restrict__ X, int n, int d, int npad,
                                                      const double* __restrict__ sg /*sqrt(gamma) [d]*/,
                                                      const double* __restrict__ acoef /*[d]*/, const double* __restrict__ mvec /*[d]*/,
                                                      double scale, const double* __restrict__ Ainv, double* __restrict__ P,
                                                      double* __restrict__ tpart) {
    extern __shared__ __align__(16) double sm[];
    double* Xi = sm;                        // [d][64]
    double* Xj = Xi + (size_t)d * ST;       // [d][66]
    double* ui = Xj + (size_t)d * (ST + 2); // [64]
    double* uj = ui + ST;                   // [64]
    __shared__ double red[32];
    const int tj = blockIdx.x, ti = blockIdx.y, tid = threadIdx.x;
    for (int e = tid; e < ST * d; e += 256) {
        int row = e / d, k = e % d;
        int gi = ti * ST + row, gj = tj * ST + row;
        Xi[k * ST + row] = (gi < n) ? X[(size_t)gi * d + k] * sg[k] : 0.0;
        Xj[k * (ST + 2) + row] = (gj < n) ? X[(size_t)gj * d + k] * sg[k] : 0.0;
    }
    if (tid < 2 * ST) {
        int row = tid & (ST - 1);
        int g = (tid < ST ? ti : tj) * ST + row;
        double u = 0.0;
        if (g < n) {
            u = 1.0;
            for (int k = 0; k < d; k++) {      // product of exponentials, dimension order, as the reference forms it
                double dx = X[(size_t)g * d + k] - mvec[k];
                u *= gpe_exp(-acoef[k] * (dx * dx));
            }
        }
        (tid < ST ? ui : uj)[row] = u;
    }
    __syncthreads();
    const int ty = tid >> 4, tx = tid & 15;
    double D[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) D[a][c] = 0.0;
    for (int k = 0; k < d; k++) {
        double xi[4], xj[4];
#pragma unroll
        for (int a = 0; a < 4; a++) xi[a] = Xi[k * ST + ty + 16 * a];
        double2 v0 = *reinterpret_cast<const double2*>(&Xj[k * (ST + 2) + 2 * tx]);
        double2 v1 = *reinterpret_cast<const double2*>(&Xj[k * (ST + 2) + 32 + 2 * tx]);
        xj[0] = v0.x; xj[1] = v0.y; xj[2] = v1.x; xj[3] = v1.y;
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double df = xi[a] - xj[c];
                D[a][c] = fma(df, df, D[a][c]);
            }
    }
    const bool lower = tj <= ti;
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 4; a++) {
        int li = ty + 16 * a, gi = ti * ST + li;
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            int lj0 = 32 * hh + 2 * tx, gj0 = tj * ST + lj0;
            double2 pv;
            pv.x = scale * ui[li] * uj[lj0] * gpe_exp(-D[a][2 * hh]);
            pv.y = scale * ui[li] * uj[lj0 + 1] * gpe_exp(-D[a][2 * hh + 1]);
            *reinterpret_cast<double2*>(&P[(size_t)gi * npad + gj0]) = pv;
            if (lower) {      // A^-1 is valid on and below the diagonal only: off-diagonal pairs weigh 2
                double2 av = *reinterpret_cast<const double2*>(&Ainv[(size_t)gi * npad + gj0]);
                double w0 = (gj0 < gi) ? 2.0 : ((gj0 == gi) ? 1.0 : 0.0);
                double w1 = (gj0 + 1 < gi) ? 2.0 : ((gj0 + 1 == gi) ? 1.0 : 0.0);
                acc = fma(w0 * av.x, pv.x, acc);
                acc = fma(w1 * av.y, pv.y, acc);
            }
        }
    }
    if (lower) {
        double tot = block_sum(acc, red);
        if (tid == 0) tpart[(size_t)ti * (ti + 1) / 2 + tj] = tot;
    }
}

// sums tile partials in a fixed order; also M[c1][c2] = sum_i V[i][c1] Y[i][c2] for the two panels
__global__ void __launch_bounds__(1024) sens_reduce_kernel(const double* __restrict__ tpart, int ntile, const double* __restrict__ V,
                                                           const double* __restrict__ Y, int npad, double* __restrict__ out /*[1 + NR*NR]*/) {
    __shared__ double red[32];
    const int tid = threadIdx.x;
    double s = 0.0;
    for (int t = tid; t < ntile; t += 1024) s += tpart[t];
    double tot = block_sum(s, red);
    if (tid == 0) out[0] = tot;
    const int c1 = tid / NR, c2 = tid % NR;
    double acc = 0.0;
    for (int i = 0; i < npad; i++) acc = fma(V[(size_t)i * NR + c1], Y[(size_t)i * NR + c2], acc);
    out[1 + tid] = acc;
}

// main-effect sweep: one CTA per (x_w value, input P):  sum_k e_k * scale * prod_{i != P} t1_i exp(-t2_i (x_ki-m_i)^2)
//                                                               * exp(-c_P (x_w - x_kP)^2)
__global__ void __launch_bounds__(256) sens_main_effect_kernel(const double* __restrict__ X, int n, int d,
                                                               const double* __restrict__ t1, const double* __restrict__ t2,
                                                               const double* __restrict__ cdiag, const double* __restrict__ mvec,
                                                               const double* __restrict__ evec, double scale,
                                                               const int* __restrict__ which, const double* __restrict__ xw, int points,
                                                               double* __restrict__ out) {
    __shared__ double red[32];
    const int j = blockIdx.x, w = blockIdx.y, P = which[w];
    const double xv = xw[(size_t)w * points + j], cP = cdiag[P];
    double s = 0.0;
    for (int k = threadIdx.x; k < n; k += 256) {
        double val = 1.0;
        for (int i = 0; i < d; i++) {
            if (i == P) continue;
            double dx = X[(size_t)k * d + i] - mvec[i];
            val *= t1[i] * gpe_exp(-t2[i] * (dx * dx));
        }
        double dw = xv - X[(size_t)k * d + P];
        s = fma(scale * val * gpe_exp(-(dw * dw) * cP), evec[k], s);
    }
    double tot = block_sum(s, red);
    if (threadIdx.x == 0) out[(size_t)w * points + j] = tot;
}

// Maximin criterion of the Latin-hypercube design (design_inputs.py:73): argmin over the condensed
// squared-distance vector of one candidate design (+ shared extra points).  The distance is accumulated
// exactly like scipy's pdist('sqeuclidean') kernel -- sequentially over the dimensions, separate multiply
// and add (no FMA contraction) -- so values, and therefore the index of the first minimum, are bit-identical.
constexpr int PD_ROWS = 32;
struct PdBest { double val; long long idx; };

__global__ void __launch_bounds__(256) pdist_argmin_kernel(const double* __restrict__ designs, int n, int dim,
                                                           const double* __restrict__ extra, int ne,
                                                           PdBest* __restrict__ part) {
    __shared__ double rowpt[64];
    __shared__ double rv[8];
    __shared__ long long ri[8];
    const int P = n + ne, blk = blockIdx.x, des = blockIdx.y, tid = threadIdx.x;
    const double* D = designs + (size_t)des * n * dim;
    auto point = [&](int r) -> const double* { return r < n ? D + (size_t)r * dim : extra + (size_t)(r - n) * dim; };
    double best = 1.0e300;
    long long bidx = 0x7fffffffffffffffll;
    const int r0 = blk * PD_ROWS, r1 = min(P - 1, r0 + PD_ROWS);
    for (int i = r0; i < r1; i++) {
        __syncthreads();
        if (tid < dim) rowpt[tid] = point(i)[tid];
        __syncthreads();
        const long long base = (long long)i * P - (long long)i * (i + 1) / 2 - i - 1;      // + j
        for (int j = i + 1 + tid; j < P; j += 256) {
            const double* pj = point(j);
            double acc = 0.0;
            for (int k = 0; k < dim; k++) {
                const double diff = __dsub_rn(rowpt[k], pj[k]);
                acc = __dadd_rn(acc, __dmul_rn(diff, diff));
            }
            if (acc < best) { best = acc; bidx = base + j; }       // indices only grow: first minimum kept
        }
    }
    // block reduce: smallest value, ties -> smallest index
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, best, o);
        long long oi = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (ov < best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
    }
    __syncthreads();
    if ((tid & 31) == 0) { rv[tid >> 5] = best; ri[tid >> 5] = bidx; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 8; w++)
            if (rv[w] < best || (rv[w] == best && ri[w] < bidx)) { best = rv[w]; bidx = ri[w]; }
        part[(size_t)des * gridDim.x + blk].val = best;
        part[(size_t)des * gridDim.x + blk].idx = bidx;
    }
}

int ensure_ainv(gpe_handle* h) {
    if (h->fAinv_valid) return 0;
    const int np = h->npad;
    if (!h->fAinv) CK(cudaMalloc((void**)&h->fAinv, (size_t)np * np * sizeof(double)));
    // LAUUM: A^-1 = Linv^T Linv, lower 128-tiles
    int rc = gpe_run_gemm(h, h->fLi, h->fLi, h->fAinv, np, np, np, 0, 0, 0, np, np, np, 1.0, 0, KM_GE_I, 1, 1, 2, EPI_STORE);
    if (rc) return rc;
    h->fAinv_valid = true;
    return 0;
}

}  // namespace

extern "C" {

int gpe_solve(gpe_handle* h, const double* Bm, int k, double* out) {
    if (!h || !Bm || !out || k < 1) return h ? h->fail_msg("bad argument") : -2;
    if (!h->fitted) return h->fail_msg("gpe_fit_state has not succeeded on this handle");
    NvtxRange nvtx("gpe_solve");
    CK(cudaSetDevice(h->device));
    const int np = h->npad, n = h->n;
    double *src = nullptr, *dst = nullptr, *p0 = nullptr, *p1 = nullptr, *p2 = nullptr;
    const bool in_dev = gpe_is_device_ptr(Bm), out_dev = gpe_is_device_ptr(out);
    TmpDev t_p0(h), t_p1(h), t_p2(h), t_src(h), t_dst(h);
    CK(t_p0.get(&p0, (size_t)np * NR));
    CK(t_p1.get(&p1, (size_t)np * NR));
    CK(t_p2.get(&p2, (size_t)np * NR));
    CK(t_src.get(&src, (size_t)n * NR));
    CK(t_dst.get(&dst, (size_t)n * NR));
    int rc = 0;
    for (int c0 = 0; c0 < k && !rc; c0 += NR) {
        int kc = std::min(NR, k - c0);
        // gather the column block [n, kc] (strided in the source) into a dense staging buffer
        CK(cudaMemcpy2DAsync(src, sizeof(double) * kc, Bm + c0, sizeof(double) * k, sizeof(double) * kc, n,
                             in_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->st));
        pack_panel_kernel<<<(np * NR + 255) / 256, 256, 0, h->st>>>(src, n, kc, np, p0);
        h->launches++;
        // p1 = Linv p0 ; p2 = Linv^T p1   (A^-1 = L^-T L^-1)
        rc = gpe_run_gemm(h, h->fLi, p0, p1, np, NR, NR, 0, 0, 0, np, NR, np, 1.0, 0, KM_LE_I, 0, 1, 1, EPI_STORE);
        if (!rc) rc = gpe_run_gemm(h, h->fLi, p1, p2, np, NR, NR, 0, 0, 0, np, NR, np, 1.0, 0, KM_GE_I, 0, 1, 2, EPI_STORE);
        if (rc) break;
        unpack_panel_kernel<<<(n * kc + 255) / 256, 256, 0, h->st>>>(p2, n, kc, dst);
        h->launches++;
        CK(cudaMemcpy2DAsync(out + c0, sizeof(double) * k, dst, sizeof(double) * kc, sizeof(double) * kc, n,
                             out_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->st));
        CK(cudaStreamSynchronize(h->st));
    }
    cudaStreamSynchronize(h->st);
    if (rc) return rc;
    CK(cudaGetLastError());
    return 0;
}

int gpe_sens_contract(gpe_handle* h, const double* gamma, const double* acoef, const double* mvec, double scale,
                      const double* V, int nv, double* trace_out, double* M_out) {
    if (!h || !gamma || !acoef || !mvec || !V || nv < 1 || nv > NR) return h ? h->fail_msg("bad argument (nv <= 32)") : -2;
    if (h->family != FAMILY_GAUSSIAN) return h->fail_msg("sensitivity integrals need the Gaussian kernel");
    if (!h->fitted) return h->fail_msg("gpe_fit_state has not succeeded on this handle");
    NvtxRange nvtx("gpe_sens_contract");
    CK(cudaSetDevice(h->device));
    const int np = h->npad, n = h->n, d = h->d;
    int rc;
    if ((rc = gpe_ensure_batch_ws(h, 1))) return rc;     // h->S: scratch for P
    if ((rc = ensure_ainv(h))) return rc;
    std::vector<double> g(d), hostbuf(3 * d);
    CK(cudaMemcpy(g.data(), gamma, sizeof(double) * d, cudaMemcpyDefault));
    for (int k = 0; k < d; k++) hostbuf[k] = std::sqrt(g[k]);
    CK(cudaMemcpy(hostbuf.data() + d, acoef, sizeof(double) * d, cudaMemcpyDefault));
    CK(cudaMemcpy(hostbuf.data() + 2 * d, mvec, sizeof(double) * d, cudaMemcpyDefault));
    const int nt = np / ST, ntile = nt * (nt + 1) / 2;
    double *coef = nullptr, *tpart = nullptr, *Vsrc = nullptr, *Vp = nullptr, *Yp = nullptr, *outd = nullptr;
    TmpDev t_coef(h), t_tpart(h), t_Vsrc(h), t_Vp(h), t_Yp(h), t_outd(h);
    CK(t_coef.get(&coef, (size_t)3 * d));
    CK(t_tpart.get(&tpart, (size_t)ntile));
    CK(t_Vsrc.get(&Vsrc, (size_t)n * nv));
    CK(t_Vp.get(&Vp, (size_t)np * NR));
    CK(t_Yp.get(&Yp, (size_t)np * NR));
    CK(t_outd.get(&outd, (size_t)(1 + NR * NR)));
    CK(cudaMemcpyAsync(coef, hostbuf.data(), sizeof(double) * 3 * d, cudaMemcpyHostToDevice, h->st));
    CK(cudaMemcpyAsync(Vsrc, V, sizeof(double) * (size_t)n * nv, cudaMemcpyDefault, h->st));
    pack_panel_kernel<<<(np * NR + 255) / 256, 256, 0, h->st>>>(Vsrc, n, nv, np, Vp);
    size_t smem = ((size_t)d * (ST + ST + 2) + 2 * ST) * sizeof(double);
    static SmemOptIn optin;
    optin.ensure(sens_pw_kernel, smem);
    sens_pw_kernel<<<dim3(nt, nt), 256, smem, h->st>>>(h->X, n, d, np, coef, coef + d, coef + 2 * d, scale, h->fAinv, h->S, tpart);
    h->launches += 2;
    // Y = P Vp   (P dense [np,np] row-major; rows/cols >= n are zero because u = 0 there)
    rc = gpe_run_gemm(h, h->S, Vp, Yp, np, NR, NR, 0, 0, 0, np, NR, np, 1.0, 0, KM_FULL, 0, 1, 1, EPI_STORE);
    if (!rc) {
        sens_reduce_kernel<<<1, 1024, 0, h->st>>>(tpart, ntile, Vp, Yp, np, outd);
        h->launches++;
    }
    std::vector<double> res(1 + NR * NR);
    cudaMemcpyAsync(res.data(), outd, sizeof(double) * res.size(), cudaMemcpyDeviceToHost, h->st);
    cudaStreamSynchronize(h->st);
    if (rc) return rc;
    CK(cudaGetLastError());
    if (trace_out) CK(cudaMemcpy(trace_out, res.data(), sizeof(double), cudaMemcpyDefault));
    if (M_out) {
        std::vector<double> M((size_t)nv * nv);
        for (int a = 0; a < nv; a++)
            for (int b = 0; b < nv; b++) M[(size_t)a * nv + b] = res[1 + a * NR + b];
        CK(cudaMemcpy(M_out, M.data(), sizeof(double) * M.size(), cudaMemcpyDefault));
    }
    return 0;
}

int gpe_sens_main_effect(gpe_handle* h, const double* t1, const double* t2, const double* cdiag, const double* mvec,
                         const double* evec, double scale, const int* which, int nwhich, const double* xw, int points,
                         double* out) {
    if (!h || !h->n || !t1 || !t2 || !cdiag || !mvec || !evec || !which || !xw || !out || nwhich < 1 || points < 1)
        return h ? h->fail_msg("bad argument / no training set") : -2;
    if (h->family != FAMILY_GAUSSIAN) return h->fail_msg("sensitivity integrals need the Gaussian kernel");
    NvtxRange nvtx("gpe_sens_main_effect");
    CK(cudaSetDevice(h->device));
    const int n = h->n, d = h->d;
    std::vector<double> hb(4 * d + n + (size_t)nwhich * points);
    std::vector<int> wh(nwhich);
    CK(cudaMemcpy(hb.data(), t1, sizeof(double) * d, cudaMemcpyDefault));
    CK(cudaMemcpy(hb.data() + d, t2, sizeof(double) * d, cudaMemcpyDefault));
    CK(cudaMemcpy(hb.data() + 2 * d, cdiag, sizeof(double) * d, cudaMemcpyDefault));
    CK(cudaMemcpy(hb.data() + 3 * d, mvec, sizeof(double) * d, cudaMemcpyDefault));
    CK(cudaMemcpy(hb.data() + 4 * d, evec, sizeof(double) * n, cudaMemcpyDefault));
    CK(cudaMemcpy(hb.data() + 4 * d + n, xw, sizeof(double) * (size_t)nwhich * points, cudaMemcpyDefault));
    CK(cudaMemcpy(wh.data(), which, sizeof(int) * nwhich, cudaMemcpyDefault));
    for (int w = 0; w < nwhich; w++)
        if (wh[w] < 0 || wh[w] >= d) return h->fail_msg("input index out of range");
    double *db = nullptr, *od = nullptr;
    int* wd = nullptr;
    TmpDev t_db(h), t_od(h), t_wd(h);
    CK(t_db.get(&db, hb.size()));
    CK(t_od.get(&od, (size_t)nwhich * points));
    CK(t_wd.get(&wd, (size_t)nwhich));
    CK(cudaMemcpyAsync(db, hb.data(), sizeof(double) * hb.size(), cudaMemcpyHostToDevice, h->st));
    CK(cudaMemcpyAsync(wd, wh.data(), sizeof(int) * nwhich, cudaMemcpyHostToDevice, h->st));
    sens_main_effect_kernel<<<dim3(points, nwhich), 256, 0, h->st>>>(h->X, n, d, db, db + d, db + 2 * d, db + 3 * d, db + 4 * d, scale,
                                                                      wd, db + 4 * d + n, points, od);
    h->launches++;
    cudaMemcpyAsync(out, od, sizeof(double) * (size_t)nwhich * points, cudaMemcpyDefault, h->st);
    cudaStreamSynchronize(h->st);
    CK(cudaGetLastError());
    return 0;
}

int gpe_pdist_argmin(gpe_handle* h, const double* designs, int N, int n, int dim, const double* extra, int ne,
                     long long* argmin_out) {
    if (!h || !designs || !argmin_out || N < 1 || n < 1 || dim < 1 || dim > 64 || ne < 0 || (ne > 0 && !extra) || n + ne < 2)
        return h ? h->fail_msg("bad argument (1 <= dim <= 64, at least two points)") : -2;
    NvtxRange nvtx("gpe_pdist_argmin");
    CK(cudaSetDevice(h->device));
    const int P = n + ne, nblk = (P - 1 + PD_ROWS - 1) / PD_ROWS;
    double *dd = nullptr, *de = nullptr;
    PdBest* dp = nullptr;
    TmpDev t_d(h), t_e(h), t_p(h);
    const double* dsrc = designs;
    if (!gpe_is_device_ptr(designs)) {
        CK(t_d.get(&dd, (size_t)N * n * dim));
        CK(cudaMemcpyAsync(dd, designs, sizeof(double) * (size_t)N * n * dim, cudaMemcpyHostToDevice, h->st));
        dsrc = dd;
    }
    const double* esrc = extra;
    if (ne > 0 && !gpe_is_device_ptr(extra)) {
        CK(t_e.get(&de, (size_t)ne * dim));
        CK(cudaMemcpyAsync(de, extra, sizeof(double) * (size_t)ne * dim, cudaMemcpyHostToDevice, h->st));
        esrc = de;
    }
    CK(t_p.get(&dp, (size_t)N * nblk));
    pdist_argmin_kernel<<<dim3(nblk, N), 256, 0, h->st>>>(dsrc, n, dim, esrc, ne, dp);
    h->launches++;
    std::vector<PdBest> part((size_t)N * nblk);
    CK(cudaMemcpyAsync(part.data(), dp, sizeof(PdBest) * part.size(), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    std::vector<long long> res(N);
    for (int k = 0; k < N; k++) {
        PdBest b = part[(size_t)k * nblk];
        for (int t = 1; t < nblk; t++) {
            const PdBest& c = part[(size_t)k * nblk + t];
            if (c.val < b.val || (c.val == b.val && c.idx < b.idx)) b = c;
        }
        res[k] = b.idx;
    }
    CK(cudaMemcpy(argmin_out, res.data(), sizeof(long long) * N, cudaMemcpyDefault));
    return 0;
}

}  // extern "C"
