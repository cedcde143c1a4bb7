// K4 posterior mean / variance over large point sets, K4f full covariance, K5 implausibility.
// Reference arithmetic replaced: Posterior.make_covar/make_mean/make_var
// (_emulatorclasses.py:607-631), kernel.covar (_emulatorkernels.py:75-79, :148-152),
// history_match.py:121-136 / :237-250 / :317-329.
//
// Nothing of size m x m or n x m_total is ever materialised: points are processed in chunks;
// per chunk the cross-covariance tile C [n, mc] is generated on device (optionally straight from
// a flat grid index), Z = L^-1 C runs on the FP64 tensor pipe with the column norms |L^-1 c_j|^2
// reduced in the GEMM epilogue, and a skinny product [A^-1 H K^-T | e]^T C gives the mean and the
// regression-variance term.   v_j = sigma^2 (a*_jj - |L^-1 c_j|^2 + |K^-1 h_j - (Gm K^-T)^T c_j|^2).
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

void gpe_handle::free_fit() {
    auto fr = [](double*& p) { if (p) cudaFree(p); p = nullptr; };
    fr(fLi); fr(fE); fr(fK); fr(fbeta); fr(fwinv); fr(fXs); fr(fAinv);
    fAinv_valid = false;
    for (auto& sl : ps) { fr(sl.C); fr(sl.Part); fr(sl.Aux); fr(sl.X); fr(sl.H); fr(sl.Mean); fr(sl.Var); }
    pchunk = 0;
    fitted = false;
}

namespace {

constexpr int MAXD = 64;
struct GridDesc {
    int d;
    int levels[MAXD];
    double lo[MAXD], step[MAXD];   // coordinate = lo + (digit + 0.5) * step
};
struct BasisDesc {
    int q;
    int idx[NR], pw[NR];
};

// scaled training inputs, k-major, zero padded: Xs[k][i] = X[i][k] / delta_k
__global__ void scale_train_kernel(const double* __restrict__ X, const double* __restrict__ winv, int n, int d, int npad,
                                   double* __restrict__ Xs) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= d * npad) return;
    int k = idx / npad, i = idx % npad;
    Xs[idx] = (i < n) ? X[(size_t)i * d + k] * winv[k] : 0.0;
}

// materialise a chunk of grid points [mc, d] from the flat index (digit 0 slowest)
__global__ void grid_points_kernel(GridDesc g, long long start, long long count, int mc, double* __restrict__ P) {
    long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= mc) return;
    long long idx = start + (j < count ? j : 0);
    for (int k = g.d - 1; k >= 0; k--) {
        long long dig = idx % g.levels[k];
        idx /= g.levels[k];
        P[(size_t)j * g.d + k] = g.lo[k] + ((double)dig + 0.5) * g.step[k];
    }
}

// K1x: C[k][j] = c * exp(-sum_dim ((x_k - p_j)/delta)^2) for a chunk of mc points (FAMILY_MATERN52: c * R(sum_dim ..)).
// CTA = 64 training rows x 128 points, 256 threads, each thread 8 rows x 4 points.
template <int FAM>
__global__ void __launch_bounds__(256, 3) xcov_kernel(const double* __restrict__ Xs /*[d][npad]*/, const double* __restrict__ P /*[mc][d]*/,
                                                   const double* __restrict__ winv, int n, int d, int npad, int mc, long long count,
                                                   double cscale, double* __restrict__ Cm, int ldc) {
    extern __shared__ __align__(16) double sm[];
    double* Xt = sm;                   // [d][64]
    double* Pt = sm + (size_t)d * 64;  // [d][128+2]
    const int tid = threadIdx.x;
    const int j0 = blockIdx.x * 128, k0 = blockIdx.y * 64;
    for (int e = tid; e < d * 64; e += 256) {
        int k = e / 64, rr = e % 64;
        Xt[k * 64 + rr] = Xs[(size_t)k * npad + k0 + rr];
    }
    {   // point tile without integer division: thread -> (point, k mod 2)
        const int jj = tid >> 1;
        for (int k = tid & 1; k < d; k += 2) Pt[k * 130 + jj] = P[(size_t)(j0 + jj) * d + k] * winv[k];
    }
    __syncthreads();
    const int ty = tid >> 5, tx = tid & 31;   // rows ty + 8a (a<8); points 2tx+{0,1}, 64+2tx+{0,1}
    double D[8][4];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int c = 0; c < 4; c++) D[a][c] = 0.0;
    for (int k = 0; k < d; k++) {
        double xr[8], pj[4];
#pragma unroll
        for (int a = 0; a < 8; a++) xr[a] = Xt[k * 64 + ty + 8 * a];
        double2 v0 = *reinterpret_cast<const double2*>(&Pt[k * 130 + 2 * tx]);
        double2 v1 = *reinterpret_cast<const double2*>(&Pt[k * 130 + 64 + 2 * tx]);
        pj[0] = v0.x; pj[1] = v0.y; pj[2] = v1.x; pj[3] = v1.y;
#pragma unroll
        for (int a = 0; a < 8; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double df = xr[a] - pj[c];
                D[a][c] = fma(df, df, D[a][c]);
            }
    }
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int c = 0; c < 4; c++)      // straight-line: the chains interleave
            if constexpr (FAM == FAMILY_GAUSSIAN) D[a][c] = gpe_exp(-D[a][c]);
#pragma unroll
    for (int a = 0; a < 8; a++) {
        int gk = k0 + ty + 8 * a;
        bool live = gk < n;
        if constexpr (FAM == FAMILY_MATERN52) {      // one row's four chains at a time: 32 at once would spill
#pragma unroll
            for (int c = 0; c < 4; c++) D[a][c] = gpe_matern52(D[a][c]);
        }
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            int gj = j0 + 64 * hh + 2 * tx;
            double2 v;
            v.x = (live && gj < count) ? cscale * D[a][2 * hh] : 0.0;
            v.y = (live && gj + 1 < count) ? cscale * D[a][2 * hh + 1] : 0.0;
            *reinterpret_cast<double2*>(&Cm[(size_t)gk * ldc + gj]) = v;
        }
    }
}


// ---- K1x for tensor-grid points: the Gaussian kernel factorises over the input dimensions,
//     exp(-sum_k ((x_ik - g_k)/delta_k)^2) = prod_k exp(-((x_ik - g_k)/delta_k)^2),
// and a grid point's coordinate in dimension k takes only levels[k] values.  The d * levels one-dimensional factors
// per training point are tabulated once per call (grid_table_kernel: sum(levels) * npad exponentials instead of
// m * npad); an entry of the cross-covariance is then a product of table entries.  Points are consecutive flat
// indices, so inside a CTA's run of points the digits of the leading ("slow") dimensions take at most two
// combinations: their product is formed once per training row, and only the trailing ("fast") dimensions -- the
// shortest suffix whose levels multiply to >= 128 -- cost one multiplication per entry each.
// (n = 2000, d = 8, 10 levels: 2048 x 80 exponentials per call and 3 multiplications per entry, against 8 subtractions,
// 8 FMAs and a 22-instruction exp per entry in xcov_kernel; the cross-covariance was 4.4 % of a chunk on the FP64 pipe
// the TRMM needs.)  Each factor carries its own rounding, so an entry differs from exp(-sum) in the last few ulps --
// the same size as the rounding of the summed exponent in the direct form; parity with the reference is checked on the
// grid path itself (tests/test_gpu_fullsize.py).
// The Matérn kernel does not factorise, but its argument D is still a sum over the dimensions: for FAMILY_MATERN52 the
// table holds the one-dimensional terms df^2, the slow and fast parts are added instead of multiplied, and R(D) is
// applied once per entry.
constexpr int GS_MAXNF = 7;      // fast dimensions (levels >= 2 => at most 7 for a product >= 128)
struct GridSep {
    int d, ks, nf;               // slow dimensions [0, ks), fast dimensions [ks, d)
    int levels[MAXD], toff[MAXD];      // table rows of dimension k start at toff[k]
    int foff[GS_MAXNF];          // offset (doubles) of fast dimension kf's block in shared memory
    long long pfast;             // product of the fast levels
    int ptiles;                  // 128-point tiles per CTA (<= pfast / 128: at most two slow combinations per CTA)
};

template <int FAM>
__global__ void grid_table_kernel(const double* __restrict__ Xs, const double* __restrict__ winv, GridDesc g, GridSep sp, int npad,
                                  int ltot, double* __restrict__ T) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= (long long)ltot * npad) return;
    const int trow = (int)(idx / npad), i = (int)(idx % npad);
    int k = 0;
    while (k + 1 < sp.d && sp.toff[k + 1] <= trow) k++;
    const int l = trow - sp.toff[k];
    const double pt = (g.lo[k] + ((double)l + 0.5) * g.step[k]) * winv[k];      // the coordinate grid_points_kernel gives, scaled
    const double df = Xs[(size_t)k * npad + i] - pt;
    if constexpr (FAM == FAMILY_GAUSSIAN) T[idx] = gpe_exp(-(df * df));
    else T[idx] = df * df;
}

template <int NF, int FAM>
__global__ void __launch_bounds__(256) xcov_grid_kernel(const double* __restrict__ T, GridSep sp, int n, int npad, int mc,
                                                        long long start, long long count, double cscale,
                                                        double* __restrict__ Cm, int ldc) {
    constexpr int ROWS = 128;
    extern __shared__ __align__(16) double sm[];
    double* Ps = sm;                    // [2][ROWS]  cscale * product of the slow factors (Matérn: sum of the slow terms)
    double* Tf = sm + 2 * ROWS;         // fast factors: block kf holds [ROWS][levels + 1]
    __shared__ int sdig[2][MAXD];
    const int tid = threadIdx.x, k0 = blockIdx.y * ROWS;
    const long long jbase = (long long)blockIdx.x * sp.ptiles * 128;
    const long long s0 = (start + jbase) / sp.pfast;
    if (tid < 2) {
        long long sidx = s0 + tid;
        for (int k = sp.ks - 1; k >= 0; k--) {
            sdig[tid][k] = (int)(sidx % sp.levels[k]);
            sidx /= sp.levels[k];
        }
    }
    __syncthreads();
    {
        const int c = tid >> 7, row = tid & (ROWS - 1);
        double prod = (FAM == FAMILY_GAUSSIAN) ? cscale : 0.0;
        for (int k = 0; k < sp.ks; k++) {
            const double tv = T[(size_t)(sp.toff[k] + sdig[c][k]) * npad + k0 + row];
            if constexpr (FAM == FAMILY_GAUSSIAN) prod *= tv;
            else prod += tv;
        }
        Ps[c * ROWS + row] = prod;
    }
#pragma unroll
    for (int kf = 0; kf < NF; kf++) {
        const int L = sp.levels[sp.ks + kf];
        double* blk = Tf + sp.foff[kf];
        for (int e = tid; e < L * ROWS; e += 256) {
            const int l = e >> 7, row = e & (ROWS - 1);
            blk[row * (L + 1) + l] = T[(size_t)(sp.toff[sp.ks + kf] + l) * npad + k0 + row];
        }
    }
    __syncthreads();
    const int ty = tid >> 5, tx = tid & 31;
    for (int pt = 0; pt < sp.ptiles; pt++) {
        const long long j0 = jbase + (long long)pt * 128;
        if (j0 >= mc) break;
        int off[4][NF], combo[4];
        bool livep[4];
#pragma unroll
        for (int q4 = 0; q4 < 4; q4++) {
            const long long j = j0 + 64 * (q4 >> 1) + 2 * tx + (q4 & 1);
            livep[q4] = j < count;
            const long long idx = start + (livep[q4] ? j : 0);
            long long f = idx % sp.pfast;
            combo[q4] = (int)(idx / sp.pfast - s0) & 1;
#pragma unroll
            for (int kf = NF - 1; kf >= 0; kf--) {
                const int L = sp.levels[sp.ks + kf];
                off[q4][kf] = sp.foff[kf] + (int)(f % L);
                f /= L;
            }
        }
#pragma unroll 4
        for (int a = 0; a < ROWS / 8; a++) {
            const int row = ty + 8 * a;
            const bool live = k0 + row < n;
            double v[4];
#pragma unroll
            for (int q4 = 0; q4 < 4; q4++) {
                double x = Ps[combo[q4] * ROWS + row];
#pragma unroll
                for (int kf = 0; kf < NF; kf++) {
                    const double tv = Tf[off[q4][kf] + row * (sp.levels[sp.ks + kf] + 1)];
                    if constexpr (FAM == FAMILY_GAUSSIAN) x *= tv;
                    else x += tv;
                }
                if constexpr (FAM == FAMILY_MATERN52) x = cscale * gpe_matern52(x);
                v[q4] = (live && livep[q4]) ? x : 0.0;
            }
            double* cp = Cm + (size_t)(k0 + row) * ldc + j0 + 2 * tx;
            *reinterpret_cast<double2*>(cp) = make_double2(v[0], v[1]);
            *reinterpret_cast<double2*>(cp + 64) = make_double2(v[2], v[3]);
        }
    }
}

// Plan the slow / fast split for a grid; false when the tables would not fit (fall back to xcov_kernel).
static bool plan_grid_sep(const GridDesc& g, GridSep& sp, size_t& smem, int& ltot) {
    sp.d = g.d;
    ltot = 0;
    for (int k = 0; k < g.d; k++) {
        if (g.levels[k] < 1) return false;
        sp.levels[k] = g.levels[k];
        sp.toff[k] = ltot;
        ltot += g.levels[k];
    }
    long long pf = 1;
    int ks = g.d;
    while (ks > 0 && pf < 128) pf *= g.levels[--ks];
    sp.ks = ks; sp.nf = g.d - ks; sp.pfast = pf;
    if (sp.nf < 1 || sp.nf > GS_MAXNF) return false;
    sp.ptiles = (int)std::max<long long>(1, std::min<long long>(8, pf / 128));
    if (pf < 128 && ks == 0) sp.ptiles = 1;      // the whole grid is shorter than a tile: no slow part, combinations are moot
    size_t off = 0;
    for (int kf = 0; kf < sp.nf; kf++) {
        sp.foff[kf] = (int)off;
        off += (size_t)128 * (g.levels[ks + kf] + 1);
    }
    smem = (2 * 128 + off) * sizeof(double);
    return smem <= 96 * 1024 && ltot <= 4096;
}

template <int NF, int FAM>
static cudaError_t launch_xcov_grid_nf(const double* T, const GridSep& sp, int n, int npad, int mc, long long start, long long count,
                                       double cscale, double* Cm, size_t smem, cudaStream_t st) {
    static SmemOptIn optin;
    if (cudaError_t e = optin.ensure(xcov_grid_kernel<NF, FAM>, smem); e != cudaSuccess) return e;
    const int per = sp.ptiles * 128;
    xcov_grid_kernel<NF, FAM><<<dim3((mc + per - 1) / per, npad / 128), 256, smem, st>>>(T, sp, n, npad, mc, start, count, cscale, Cm, mc);
    return cudaGetLastError();
}

template <int FAM>
static cudaError_t launch_xcov_grid(const double* T, const GridSep& sp, int n, int npad, int mc, long long start, long long count,
                                    double cscale, double* Cm, size_t smem, cudaStream_t st) {
    switch (sp.nf) {
        case 1: return launch_xcov_grid_nf<1, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        case 2: return launch_xcov_grid_nf<2, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        case 3: return launch_xcov_grid_nf<3, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        case 4: return launch_xcov_grid_nf<4, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        case 5: return launch_xcov_grid_nf<5, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        case 6: return launch_xcov_grid_nf<6, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        case 7: return launch_xcov_grid_nf<7, FAM>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

struct GridXcov {        // what predict_chunk needs to build a chunk's cross-covariance from the tables
    const double* T;
    GridSep sp;
    size_t smem;
    long long start;     // flat index of the chunk's first point
};

static cudaError_t launch_xcov_grid(int family, const double* T, const GridSep& sp, int n, int npad, int mc, long long start,
                                    long long count, double cscale, double* Cm, size_t smem, cudaStream_t st) {
    if (family == FAMILY_MATERN52) return launch_xcov_grid<FAMILY_MATERN52>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
    return launch_xcov_grid<FAMILY_GAUSSIAN>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
}

// C [n rows of npad, ldc] = cscale * K(training, P) for the mc points P [mc, d] (columns >= count zero)
template <int FAM>
static cudaError_t launch_xcov_fam(const double* Xs, const double* P, const double* winv, int n, int d, int npad, int mc,
                                   long long count, double cscale, double* Cm, int ldc, cudaStream_t st) {
    static SmemOptIn optin;      // d >= 32 needs more than 48 KB for the two k-major tiles
    const size_t smem = (size_t)d * (64 + 130) * sizeof(double);
    if (cudaError_t e = optin.ensure(xcov_kernel<FAM>, smem); e != cudaSuccess) return e;
    xcov_kernel<FAM><<<dim3(mc / 128, npad / 64), 256, smem, st>>>(Xs, P, winv, n, d, npad, mc, count, cscale, Cm, ldc);
    return cudaGetLastError();
}
static cudaError_t launch_xcov(int family, const double* Xs, const double* P, const double* winv, int n, int d, int npad, int mc,
                               long long count, double cscale, double* Cm, int ldc, cudaStream_t st) {
    if (family == FAMILY_MATERN52) return launch_xcov_fam<FAMILY_MATERN52>(Xs, P, winv, n, d, npad, mc, count, cscale, Cm, ldc, st);
    return launch_xcov_fam<FAMILY_GAUSSIAN>(Xs, P, winv, n, d, npad, mc, count, cscale, Cm, ldc, st);
}

// Implausibility folded into the prediction of one emulator (history_match.py:96-132): instead of mean / variance the
// per-point list of the maxno largest implausibilities over the emulators seen so far, Itop [m][maxno] ascending, is
// updated; the last emulator's pass also produces the keep mask, the counts and the cell statistics, so neither the
// means / variances nor (unless asked for) the final list ever travel through HBM.
constexpr int MAXEM = 16;
struct ImpFuse {
    double z, ve, cm;
    int maxno, first, last;
    double* Itop;                        // chunk's first point; in/out (out may be skipped on the last pass: store_top)
    int store_top;
    long long cell_pts, first_index;     // global flat index of the chunk's first point (cells as in gpe_implausibility)
    unsigned char* keep;                 // chunk's first point, or null
    unsigned long long *count_lt, *cell_min_bits, *cell_count;      // [maxno], [ncell][maxno] (cell 0 = the cell of the call's first point)
    long long cell_base;                 // index of that cell: (call's first_index) / cell_pts
};

// per point: mean, variance from the GEMM outputs
template <bool IMP>
__global__ void __launch_bounds__(128) predict_finalize_kernel(const double* __restrict__ part, int ntile, const double* __restrict__ aux,
                                                               int ld, const double* __restrict__ P, const double* __restrict__ Hs,
                                                               BasisDesc bd, int d, const double* __restrict__ Kf,
                                                               const double* __restrict__ beta, double sigma2, double astar,
                                                               long long count, double* __restrict__ mean, double* __restrict__ var,
                                                               ImpFuse imp) {
    __shared__ double Ks[NR][NR + 1];
    __shared__ double bs[NR];
    const int q = bd.q;
    for (int e = threadIdx.x; e < NR * NR; e += blockDim.x) Ks[e / NR][e % NR] = Kf[e];
    if (threadIdx.x < NR) bs[threadIdx.x] = beta[threadIdx.x];
    __syncthreads();
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool live = j < count;
    if (!IMP && !live) return;
    double mu = 0.0, vj = 1.0;
    if (live) {
        double hv[NR];
#pragma unroll
        for (int a = 0; a < NR; a++) {
            double v = 0.0;
            if (a < q) {
                if (Hs != nullptr) v = Hs[(size_t)j * q + a];
                else if (a == 0) v = 1.0;
                else {
                    double x = P[(size_t)j * d + bd.idx[a]];
                    int pw = bd.pw[a];
                    v = (pw == 1) ? x : pow(x, (double)pw);
                }
            }
            hv[a] = v;
        }
        mu = aux[(size_t)q * ld + j];
#pragma unroll
        for (int a = 0; a < NR; a++)
            if (a < q) mu = fma(hv[a], bs[a], mu);
        if (!IMP) {
            mean[j] = mu;
            if (var == nullptr) return;
        }
        // g = K^-1 h - aux[0:q]
        double gn = 0.0;
        double kv[NR];
#pragma unroll
        for (int a = 0; a < NR; a++) {
            if (a < q) {
                double s = hv[a];
                for (int k = 0; k < a; k++) s = fma(-Ks[a][k], kv[k], s);
                kv[a] = s / Ks[a][a];
                double g = kv[a] - aux[(size_t)a * ld + j];
                gn = fma(g, g, gn);
            } else {
                kv[a] = 0.0;
            }
        }
        double zn = 0.0;
        for (int t = 0; t < ntile; t++) zn += part[(size_t)t * ld + j];
        vj = sigma2 * (astar - zn + gn);
        if (!IMP) {
            var[j] = vj;
            return;
        }
    }
    if (IMP) {
        // this emulator's implausibility into the ascending top-maxno list (np.sort(np.partition(I, -maxno)[-maxno:]), :129)
        double top[MAXEM];
#pragma unroll
        for (int k = 0; k < MAXEM; k++) top[k] = -1.0;
        if (live) {
            if (!imp.first)
                for (int k = 0; k < imp.maxno; k++) top[k] = imp.Itop[(size_t)j * imp.maxno + k];
            const double dz = mu - imp.z;
            const double I = sqrt(dz * dz / (vj + imp.ve));
            if (I > top[0]) {
                top[0] = I;
#pragma unroll
                for (int k = 0; k < MAXEM - 1; k++) {
                    if (k + 1 < imp.maxno && top[k] > top[k + 1]) {
                        double t = top[k];
                        top[k] = top[k + 1];
                        top[k + 1] = t;
                    }
                }
            }
            if (!imp.last || imp.store_top)
                for (int k = 0; k < imp.maxno; k++) imp.Itop[(size_t)j * imp.maxno + k] = top[k];
        }
        if (!imp.last) return;
        // last emulator: the reductions of implaus_kernel on the finished list (warp-aggregated, integer atomics: deterministic)
        if (live && imp.keep != nullptr) imp.keep[j] = (top[0] < imp.cm) ? 1 : 0;
        const long long cell = (imp.cell_pts > 0 && live) ? (imp.first_index + j) / imp.cell_pts - imp.cell_base : -1;
        const long long cell0 = __shfl_sync(0xffffffffu, cell, 0);
        const bool uniform = imp.cell_pts > 0 && __all_sync(0xffffffffu, cell == cell0) && cell0 >= 0;
        for (int k = 0; k < imp.maxno; k++) {
            const double vk = top[imp.maxno - 1 - k];
            const bool lt = live && (vk < imp.cm);
            const unsigned bal = __ballot_sync(0xffffffffu, lt);
            if ((threadIdx.x & 31) == 0 && bal && imp.count_lt != nullptr) atomicAdd(&imp.count_lt[k], (unsigned long long)__popc(bal));
            if (imp.cell_pts <= 0) continue;
            if (uniform) {
                unsigned long long bits = (unsigned long long)__double_as_longlong(vk);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    unsigned long long other = __shfl_xor_sync(0xffffffffu, bits, o);
                    bits = other < bits ? other : bits;
                }
                if ((threadIdx.x & 31) == 0) {
                    if (imp.cell_min_bits != nullptr) atomicMin(&imp.cell_min_bits[(size_t)cell0 * imp.maxno + k], bits);
                    if (bal && imp.cell_count != nullptr) atomicAdd(&imp.cell_count[(size_t)cell0 * imp.maxno + k], (unsigned long long)__popc(bal));
                }
            } else if (live) {
                if (imp.cell_min_bits != nullptr) atomicMin(&imp.cell_min_bits[(size_t)cell * imp.maxno + k], (unsigned long long)__double_as_longlong(vk));
                if (lt && imp.cell_count != nullptr) atomicAdd(&imp.cell_count[(size_t)cell * imp.maxno + k], 1ull);
            }
        }
    }
}

// K5: implausibility per point + reductions.  I >= 0, so the IEEE bit pattern orders like the value
// and min-reductions can use integer atomics (deterministic).
struct ImpDesc {
    int n_emul, maxno;
    double z[MAXEM], ve[MAXEM];
    double cm;
};

__global__ void __launch_bounds__(256) implaus_kernel(const double* __restrict__ mean, const double* __restrict__ var, long long m,
                                                      ImpDesc ds, long long cell_pts, long long first_index, double* __restrict__ Imax,
                                                      unsigned char* __restrict__ keep, unsigned long long* __restrict__ count_lt,
                                                      unsigned long long* __restrict__ cell_min_bits,
                                                      unsigned long long* __restrict__ cell_count) {
    long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool live = r < m;
    double top[MAXEM];   // ascending, top[maxno-1] is the largest
#pragma unroll
    for (int k = 0; k < MAXEM; k++) top[k] = -1.0;
    if (live) {
        for (int o = 0; o < ds.n_emul; o++) {
            double mu = mean[(size_t)o * m + r], v = var[(size_t)o * m + r];
            double dz = mu - ds.z[o];
            double I = sqrt(dz * dz / (v + ds.ve[o]));
            // keep the maxno largest, ascending (np.sort(np.partition(I, -maxno)[-maxno:]))
            if (I > top[0]) {
                top[0] = I;
#pragma unroll
                for (int k = 0; k < MAXEM - 1; k++) {
                    if (k + 1 < ds.maxno && top[k] > top[k + 1]) {
                        double t = top[k];
                        top[k] = top[k + 1];
                        top[k + 1] = t;
                    }
                }
            }
        }
    }
    // outputs
    for (int k = 0; k < ds.maxno; k++) {
        double vk = top[k];
        if (live && Imax != nullptr) Imax[(size_t)r * ds.maxno + k] = vk;
    }
    if (live && keep != nullptr) keep[r] = (top[0] < ds.cm) ? 1 : 0;
    // cells are contiguous runs of cell_pts points, so a warp (32 consecutive points) almost always
    // sits inside one cell: reduce in the warp first, one atomic per warp instead of one per point
    // cells are runs of cell_pts points of the GLOBAL flat index first_index + r; the outputs start at the cell of point 0
    const long long cell = (cell_pts > 0 && live) ? (first_index + r) / cell_pts - first_index / cell_pts : -1;
    const long long cell0 = __shfl_sync(0xffffffffu, cell, 0);
    const bool uniform = cell_pts > 0 && __all_sync(0xffffffffu, cell == cell0) && cell0 >= 0;
    for (int k = 0; k < ds.maxno; k++) {
        // k-th output statistic refers to the (k+1)-th largest: top[maxno-1-k]
        double vk = top[ds.maxno - 1 - k];
        bool lt = live && (vk < ds.cm);
        unsigned bal = __ballot_sync(0xffffffffu, lt);
        if ((threadIdx.x & 31) == 0 && bal && count_lt != nullptr) atomicAdd(&count_lt[k], (unsigned long long)__popc(bal));
        if (cell_pts <= 0) continue;
        if (uniform) {
            unsigned long long bits = (unsigned long long)__double_as_longlong(vk);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                unsigned long long other = __shfl_xor_sync(0xffffffffu, bits, o);
                bits = other < bits ? other : bits;
            }
            if ((threadIdx.x & 31) == 0) {
                if (cell_min_bits != nullptr) atomicMin(&cell_min_bits[(size_t)cell0 * ds.maxno + k], bits);
                if (bal && cell_count != nullptr) atomicAdd(&cell_count[(size_t)cell0 * ds.maxno + k], (unsigned long long)__popc(bal));
            }
        } else if (live) {
            if (cell_min_bits != nullptr) atomicMin(&cell_min_bits[(size_t)cell * ds.maxno + k], (unsigned long long)__double_as_longlong(vk));
            if (lt && cell_count != nullptr) atomicAdd(&cell_count[(size_t)cell * ds.maxno + k], 1ull);
        }
    }
}

// full posterior covariance assembly: V = sigma^2 (A* - Z^T Z + G^T G)
template <int FAM>
__global__ void fullcov_finalize_kernel(const double* __restrict__ ZtZ, int mp, const double* __restrict__ aux, int ld,
                                        const double* __restrict__ P, const double* __restrict__ Hs, BasisDesc bd, int d,
                                        const double* __restrict__ winv, const double* __restrict__ Kf, double sigma2,
                                        double cscale, double astar, const double* __restrict__ r_new, int m,
                                        double* __restrict__ Gbuf /*[q][mp]*/, double* __restrict__ V, int phase) {
    const int q = bd.q;
    if (phase == 0) {   // G[:, j] = K^-1 h_j - aux[0:q][j]
        int j = blockIdx.x * blockDim.x + threadIdx.x;
        if (j >= m) return;
        double kv[NR];
        for (int a = 0; a < q; a++) {
            double hvv;
            if (Hs != nullptr) hvv = Hs[(size_t)j * q + a];
            else if (a == 0) hvv = 1.0;
            else {
                double x = P[(size_t)j * d + bd.idx[a]];
                hvv = (bd.pw[a] == 1) ? x : pow(x, (double)bd.pw[a]);
            }
            double s = hvv;
            for (int k = 0; k < a; k++) s = fma(-Kf[a * NR + k], kv[k], s);
            kv[a] = s / Kf[a * NR + a];
            Gbuf[(size_t)a * mp + j] = kv[a] - aux[(size_t)a * ld + j];
        }
        return;
    }
    size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (idx >= (size_t)m * m) return;
    int i = idx / m, j = idx % m;
    double D = 0.0;
    for (int k = 0; k < d; k++) {
        double df = P[(size_t)i * d + k] * winv[k] - P[(size_t)j * d + k] * winv[k];
        D = fma(df, df, D);
    }
    double prior = (i == j) ? (astar + (r_new ? r_new[i] : 0.0))
                            : cscale * (FAM == FAMILY_MATERN52 ? gpe_matern52(D) : gpe_exp(-D));
    double gg = 0.0;
    for (int a = 0; a < q; a++) gg = fma(Gbuf[(size_t)a * mp + i], Gbuf[(size_t)a * mp + j], gg);
    V[idx] = sigma2 * (prior - ZtZ[(size_t)i * mp + j] + gg);
}

int ensure_predict_ws(gpe_handle* h, long long mc) {
    if (mc <= h->pchunk) return 0;
    auto fr = [](double*& p) { if (p) cudaFree(p); p = nullptr; };
    h->pchunk = 0;
    size_t ntile = h->npad / 128;
    for (auto& sl : h->ps) {
        fr(sl.C); fr(sl.Part); fr(sl.Aux); fr(sl.X); fr(sl.H); fr(sl.Mean); fr(sl.Var);
        CK(cudaMalloc((void**)&sl.C, (size_t)h->npad * mc * sizeof(double)));
        CK(cudaMalloc((void**)&sl.Part, ntile * mc * sizeof(double)));
        CK(cudaMalloc((void**)&sl.Aux, (size_t)NR * mc * sizeof(double)));
        CK(cudaMalloc((void**)&sl.X, (size_t)mc * h->d * sizeof(double)));
        CK(cudaMalloc((void**)&sl.H, (size_t)mc * NR * sizeof(double)));
        CK(cudaMalloc((void**)&sl.Mean, (size_t)mc * sizeof(double)));
        CK(cudaMalloc((void**)&sl.Var, (size_t)mc * sizeof(double)));
    }
    h->pchunk = mc;
    return 0;
}

BasisDesc basis_of(gpe_handle* h) {
    BasisDesc bd;
    bd.q = h->q;
    for (int a = 0; a < NR; a++) { bd.idx[a] = h->basis_idx[a] < 0 ? 0 : h->basis_idx[a]; bd.pw[a] = h->basis_pow[a]; }
    return bd;
}

long long default_chunk(gpe_handle* h) {
    long long c = 65536;     // measured on B200 (n = 2000): 16384 -> 6.46, 65536 -> 6.86 Mpred/s; the slab is npad * c * 8 B (1.07 GB)
    if (const char* e = getenv("GPE_PRED_CHUNK")) c = std::max(128ll, atoll(e));
    return (c + 127) / 128 * 128;
}

// One chunk on stream `st` with the buffers of `sl`: points already in P_dev [mc, d] (rows >= count
// arbitrary but finite).
int predict_chunk(gpe_handle* h, gpe_handle::PredSlot& sl, cudaStream_t st, const double* P_dev, const double* Hs_dev,
                  long long count, int mc, double* mean_dev, double* var_dev, const GridXcov* gx = nullptr, const ImpFuse* imp = nullptr) {
    const int np = h->npad;
    {
        ProfScope ps(h, gpe_handle::CAT_COV, st);
        if (gx != nullptr) CK(launch_xcov_grid(h->family, gx->T, gx->sp, h->n, np, mc, gx->start, count, h->fit_c, sl.C, gx->smem, st));
        else CK(launch_xcov(h->family, h->fXs, P_dev, h->fwinv, h->n, h->d, np, mc, count, h->fit_c, sl.C, mc, st));
    }
    h->launches++;
    int rc;
    // aux = [A^-1 H K^-T | e]^T C     (TN, skinny: the q + 1 live columns of the panel padded to 16 or 32 rows)
    // rows / columns >= n of the padded matrices are identity padding and the slab's rows >= n are zero: the products need
    // only the first kp = n rounded up to the k-tile (n = 2000: 2000 instead of 2048 -- the last, heaviest row tile of the
    // triangular product has 80 live rows, not 128)
    const int kp = std::min(np, (h->n + GEMM_BK - 1) / GEMM_BK * GEMM_BK);
    const int maux = (h->q + 1 <= 16) ? 16 : NR;
    if ((rc = gpe_run_gemm_on(h, st, h->fE, sl.C, sl.Aux, NR, mc, mc, 0, 0, 0, maux, mc, kp, 1.0, 0, KM_FULL, 0, 1, 2, EPI_STORE))) return rc;
    int ntile = 0;
    if (var_dev != nullptr || imp != nullptr) {
        // column norms of Z = Linv C    (NN, Linv lower: k <= i), reduced in the epilogue
        static int ragged = -1;
        if (ragged < 0) {
            const char* e = getenv("GPE_PRED_RAGGED");
            ragged = (e && e[0] == '0') ? 0 : 1;
        }
        int mp = ragged ? kp : np;
        // INT8 tensor-core route (gpe_ozaki.cuh) for chunks it supports: the residue planes of L^-1 are made once per fit and
        // stream (the tag is the generation of the fit state), the padded size is used (rows >= n of Z are zero)
        bool one_row = false;
        if (h->oz_nmod > 0 && np >= h->oz_min && mc >= h->oz_min) {
            GemmP p;
            p.A = h->fLi; p.B = sl.C; p.C = sl.Part; p.lda = np; p.ldb = mc; p.ldc = mc; p.sA = p.sB = p.sC = 0;
            p.M = np; p.N = mc; p.K = np; p.alpha = 1.0; p.accumulate = 0; p.kmode = KM_LE_I; p.lower = 0; p.batch = 1;
            if (oz_supported(p, EPI_SUMSQ) && gpe_oz_reserve(h, st, p)) {
                mp = np;
                h->oz_reuse_a = true;
                h->oz_a_tag = h->fit_gen;
                // every entry of the slab is c exp(-D) or c R(D), in [0, c]: one scale for all points, no pass over the slab for its maxima.
                // (A point far from every training input then keeps fewer significant bits of its tiny column -- its variance
                // is the prior's to the same absolute accuracy, which is what the subtraction prior - |Z|^2 needs.)
                static const int fixed_env = [] { const char* e = getenv("GPE_PRED_FIXED_SCALE"); return e ? atoi(e) : 1; }();
                if (fixed_env) h->oz_b_bound = h->fit_c;
                one_row = oz_sumsq_swapped(p, EPI_SUMSQ);
            }
        }
        if ((rc = gpe_run_gemm_on(h, st, h->fLi, sl.C, sl.Part, np, mc, mc, 0, 0, 0, mp, mc, mp, 1.0, 0, KM_LE_I, 0, 1, 1, EPI_SUMSQ))) return rc;
        ntile = one_row ? 1 : (mp + 127) / 128;
    }
    {
        ProfScope ps(h, gpe_handle::CAT_OTHER, st);
        if (imp != nullptr)
            predict_finalize_kernel<true><<<(unsigned)((count + 127) / 128), 128, 0, st>>>(
                sl.Part, ntile, sl.Aux, mc, P_dev, Hs_dev, basis_of(h), h->d, h->fK, h->fbeta, h->fit_sigma * h->fit_sigma,
                h->fit_astar, count, nullptr, nullptr, *imp);
        else
            predict_finalize_kernel<false><<<(unsigned)((count + 127) / 128), 128, 0, st>>>(
                sl.Part, ntile, sl.Aux, mc, P_dev, Hs_dev, basis_of(h), h->d, h->fK, h->fbeta, h->fit_sigma * h->fit_sigma,
                h->fit_astar, count, mean_dev, var_dev, ImpFuse{});
    }
    h->launches++;
    return 0;
}

}  // namespace

extern "C" {

int gpe_fit_state(gpe_handle* h, const double* delta, double nugget, double sigma, int kind, double r_div,
                  const double* beta_in, double* beta_out, double* sigma_mucm_out, int* status) {
    if (!h || !h->n || !delta) return h ? h->fail_msg("bad argument / no training set") : -2;
    NvtxRange nvtx("gpe_fit_state");
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = gpe_ensure_batch_ws(h, 1))) return rc;
    const int np = h->npad, q = h->q;
    std::vector<double> dl(h->d), bin(NR, 0.0);
    CK(cudaMemcpy(dl.data(), delta, sizeof(double) * h->d, cudaMemcpyDefault));
    if ((rc = gpe_upload_single_par(h, dl.data(), nugget, kind, 1, r_div > 0 ? r_div : 1.0))) return rc;
    if (!h->fLi) {
        CK(cudaMalloc((void**)&h->fLi, (size_t)np * np * sizeof(double)));
        CK(cudaMalloc((void**)&h->fE, (size_t)np * NR * sizeof(double)));
        CK(cudaMalloc((void**)&h->fK, (size_t)NR * NR * sizeof(double)));
        CK(cudaMalloc((void**)&h->fbeta, (size_t)NR * sizeof(double)));
        CK(cudaMalloc((void**)&h->fwinv, (size_t)h->d * sizeof(double)));
        CK(cudaMalloc((void**)&h->fXs, (size_t)h->d * np * sizeof(double)));
    }
    double* bov = nullptr;
    if (beta_in) {
        CK(cudaMemcpy(bin.data(), beta_in, sizeof(double) * q, cudaMemcpyDefault));
        CK(cudaMemcpyAsync(h->fbeta, bin.data(), sizeof(double) * NR, cudaMemcpyHostToDevice, h->st));
        bov = h->fbeta;
    }
    CK(launch_cov_build(h->X, h->r, h->n, h->d, np, h->par, h->winv, h->A, 0, 1, 0, h->st, 0, 0, nullptr, h->family));
    h->launches++;
    CK(cudaMemsetAsync(h->fK, 0, sizeof(double) * NR * NR, h->st));
    CK(cudaMemsetAsync(h->status, 0, sizeof(int), h->st));
    SubBatch sb{0, 1, h->st};
    if ((rc = gpe_factor_and_reduce(h, sb, 0, 0, bov, h->fK))) return rc;
    CK(cudaMemcpyAsync(h->fLi, h->Li, (size_t)np * np * sizeof(double), cudaMemcpyDeviceToDevice, h->st));
    CK(cudaMemcpyAsync(h->fE, h->U, (size_t)np * NR * sizeof(double), cudaMemcpyDeviceToDevice, h->st));
    CK(cudaMemcpyAsync(h->fwinv, h->winv, (size_t)h->d * sizeof(double), cudaMemcpyDeviceToDevice, h->st));
    std::vector<double> bopt(NR, 0.0);
    ItemOut io;
    int st = 0;
    CK(cudaMemcpyAsync(bopt.data(), h->beta, sizeof(double) * NR, cudaMemcpyDeviceToHost, h->st));
    CK(cudaMemcpyAsync(&io, h->out, sizeof io, cudaMemcpyDeviceToHost, h->st));
    CK(cudaMemcpyAsync(&st, h->status, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    if (!beta_in) CK(cudaMemcpyAsync(h->fbeta, h->beta, sizeof(double) * NR, cudaMemcpyDeviceToDevice, h->st));
    scale_train_kernel<<<(h->d * np + 255) / 256, 256, 0, h->st>>>(h->X, h->fwinv, h->n, h->d, np, h->fXs);
    h->launches++;
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    h->fit_kind = kind; h->fit_nugget = nugget; h->fit_sigma = sigma;
    h->fit_c = kind ? 1.0 : (1.0 - nugget);
    h->fit_astar = kind ? (1.0 + nugget * nugget) : 1.0;
    h->fitted = (st == 0);
    h->fit_gen++;
    h->fAinv_valid = false;
    if (beta_out) CK(cudaMemcpy(beta_out, bopt.data(), sizeof(double) * q, cudaMemcpyDefault));
    double sm = std::sqrt(io.quad / ((double)(h->n - q) - 2.0));
    if (sigma_mucm_out) CK(cudaMemcpy(sigma_mucm_out, &sm, sizeof(double), cudaMemcpyDefault));
    if (status) CK(cudaMemcpy(status, &st, sizeof(int), cudaMemcpyDefault));
    return 0;
}

static int predict_common(gpe_handle* h, const double* Xs, const double* Hs, const GridDesc* grid, long long start,
                          long long m, double* mean, double* var, const ImpFuse* imp_call = nullptr) {
    if (!h->fitted) return h->fail_msg("gpe_fit_state has not succeeded on this handle");
    if (!Hs && !h->has_basis) return h->fail_msg("no H* given and no device basis set (gpe_set_basis)");
    NvtxRange nvtx(grid ? "gpe_predict_grid" : "gpe_predict");
    CK(cudaSetDevice(h->device));
    long long chunk = std::min<long long>(default_chunk(h), (m + 127) / 128 * 128);
    int rc;
    if ((rc = ensure_predict_ws(h, chunk))) return rc;
    // Chunks alternate between two (stream, buffer slot) pairs: a slot's staging buffers are reused only
    // by later chunks of the same stream, which orders them.
    const bool x_dev = Xs && gpe_is_device_ptr(Xs), h_dev = Hs && gpe_is_device_ptr(Hs);
    const bool mean_dev = imp_call || gpe_is_device_ptr(mean), var_dev = var && gpe_is_device_ptr(var);
    const int d = h->d, q = h->q;
    // tensor grid: tabulate the one-dimensional kernel factors once (GPE_GRID_SEP=0 keeps the direct kernel)
    GridXcov gx;
    bool use_sep = false;
    TmpDev t_tab(h);
    if (grid) {
        static int sep_on = -1;
        if (sep_on < 0) {
            const char* e = getenv("GPE_GRID_SEP");
            sep_on = (e && e[0] == '0') ? 0 : 1;
        }
        int ltot = 0;
        if (sep_on && plan_grid_sep(*grid, gx.sp, gx.smem, ltot)) {
            double* T = nullptr;
            CK(t_tab.get(&T, (size_t)ltot * h->npad));
            const long long tot = (long long)ltot * h->npad;
            if (h->family == FAMILY_MATERN52)
                grid_table_kernel<FAMILY_MATERN52><<<(unsigned)((tot + 255) / 256), 256, 0, h->st>>>(h->fXs, h->fwinv, *grid, gx.sp, h->npad, ltot, T);
            else
                grid_table_kernel<FAMILY_GAUSSIAN><<<(unsigned)((tot + 255) / 256), 256, 0, h->st>>>(h->fXs, h->fwinv, *grid, gx.sp, h->npad, ltot, T);
            h->launches++;
            gx.T = T;
            use_sep = true;
        }
    }
    const bool two = m > chunk && !h->prof_on;
    if (two) {
        CK(cudaEventRecord(h->ev_fork, h->st));
        for (int k = 0; k < 2; k++) CK(cudaStreamWaitEvent(h->sub_st[k], h->ev_fork, 0));
    }
    int ci = 0;
    for (long long s = 0; s < m; s += chunk, ci++) {
        gpe_handle::PredSlot& sl = h->ps[two ? (ci & 1) : 0];
        cudaStream_t st = two ? h->sub_st[ci & 1] : h->st;
        long long cnt = std::min(chunk, m - s);
        int mc = (int)((cnt + 127) / 128 * 128);
        const double* P = nullptr;
        if (grid) {
            grid_points_kernel<<<(mc + 255) / 256, 256, 0, st>>>(*grid, start + s, cnt, mc, sl.X);
            h->launches++;
            P = sl.X;
        } else if (x_dev && cnt == mc) {
            P = Xs + (size_t)s * d;
        } else {
            if (cnt < mc) CK(cudaMemsetAsync(sl.X, 0, (size_t)mc * d * sizeof(double), st));
            CK(cudaMemcpyAsync(sl.X, Xs + (size_t)s * d, (size_t)cnt * d * sizeof(double), cudaMemcpyDefault, st));
            P = sl.X;
        }
        const double* Hc = nullptr;
        if (Hs) {
            if (h_dev) Hc = Hs + (size_t)s * q;
            else {
                CK(cudaMemcpyAsync(sl.H, Hs + (size_t)s * q, (size_t)cnt * q * sizeof(double), cudaMemcpyDefault, st));
                Hc = sl.H;
            }
        }
        double* mo = imp_call ? nullptr : (mean_dev ? mean + s : sl.Mean);
        double* vo = var ? (var_dev ? var + s : sl.Var) : nullptr;
        gx.start = start + s;
        ImpFuse ic;
        if (imp_call) {          // this chunk's window of the per-point arrays
            ic = *imp_call;
            ic.Itop += (size_t)s * ic.maxno;
            if (ic.keep) ic.keep += s;
            ic.first_index += s;
        }
        if ((rc = predict_chunk(h, sl, st, P, Hc, cnt, mc, mo, vo, use_sep ? &gx : nullptr, imp_call ? &ic : nullptr))) return rc;
        if (!mean_dev) CK(cudaMemcpyAsync(mean + s, sl.Mean, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (var && !var_dev) CK(cudaMemcpyAsync(var + s, sl.Var, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    if (two) {
        for (int k = 0; k < 2; k++) {
            CK(cudaEventRecord(h->ev_join[k], h->sub_st[k]));
            CK(cudaStreamWaitEvent(h->st, h->ev_join[k], 0));
        }
    }
    // asynchronous mode (gpe_set_async): with device-resident points and outputs nothing on the host waits for this call
    const bool all_dev = mean_dev && (!var || var_dev) && (!Xs || x_dev) && (!Hs || h_dev) && !(imp_call && imp_call->last);
    if (!(h->async && all_dev)) CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

int gpe_predict(gpe_handle* h, const double* Xs, const double* Hs, long long m, double* mean, double* var) {
    if (h && m == 0) return 0;                                   // empty chunk: nothing to do
    if (!h || !Xs || !mean || m < 1) return h ? h->fail_msg("bad argument") : -2;
    return predict_common(h, Xs, Hs, nullptr, 0, m, mean, var);
}

int gpe_predict_grid(gpe_handle* h, const int* levels, const double* lo, const double* hi, long long start,
                     long long count, double* mean, double* var) {
    if (h && count == 0) return 0;                               // empty shard of the grid
    if (!h || !levels || !lo || !hi || !mean || count < 1) return h ? h->fail_msg("bad argument") : -2;
    if (h->d > MAXD) return h->fail_msg("grid prediction supports d <= 64");
    GridDesc g;
    g.d = h->d;
    for (int k = 0; k < h->d; k++) {
        g.levels[k] = levels[k];
        g.lo[k] = lo[k];
        g.step[k] = (hi[k] - lo[k]) / (double)levels[k];
    }
    return predict_common(h, nullptr, nullptr, &g, start, count, mean, var);
}

int gpe_predict_implaus(gpe_handle* h, const double* Xs, const double* Hs, const int* levels, const double* lo, const double* hi,
                        long long start, long long m, double z, double var_extra, int maxno, int first, int last, double* Itop,
                        double cm, long long cell_pts, long long first_index, long long ncell, unsigned char* keep,
                        unsigned long long* count_lt, double* cell_min, unsigned long long* cell_count) {
    if (h && m == 0 && !last) return 0;
    if (!h || m < 0 || (!Xs && (!levels || !lo || !hi)) || maxno < 1 || maxno > MAXEM) return h ? h->fail_msg("bad argument") : -2;
    if (!Itop && !(first && last)) return h->fail_msg("Itop is needed to carry the list from one emulator to the next");
    if (Itop && !gpe_is_device_ptr(Itop)) return h->fail_msg("Itop must be device memory");
    if (cell_pts < 0 || first_index < 0 || ncell < 0) return h->fail_msg("cell_pts, first_index and ncell must be non-negative");
    if (cell_pts == 0) ncell = 0;
    if (last && cell_pts > 0 && m > 0 && (first_index + m - 1) / cell_pts - first_index / cell_pts + 1 > ncell)
        return h->fail_msg("the points span more cells than ncell");
    NvtxRange nvtx("gpe_predict_implaus");
    CK(cudaSetDevice(h->device));
    ImpFuse ic{};
    ic.z = z; ic.ve = var_extra; ic.cm = cm; ic.maxno = maxno; ic.first = first != 0; ic.last = last != 0;
    ic.store_top = Itop != nullptr;
    ic.first_index = first_index; ic.cell_pts = last ? cell_pts : 0; ic.cell_base = cell_pts > 0 ? first_index / cell_pts : 0;
    double* top_tmp = nullptr;
    unsigned char* kd = nullptr;
    unsigned long long *cnt = nullptr, *cmin = nullptr, *ccnt = nullptr;
    TmpDev t_top(h), t_k(h), t_cnt(h), t_cmin(h), t_ccnt(h);
    if (!Itop) CK(t_top.get(&top_tmp, (size_t)std::max<long long>(m, 1) * maxno));      // first == last: a one-emulator job
    ic.Itop = Itop ? Itop : top_tmp;
    const bool k_dev = keep && gpe_is_device_ptr(keep);
    if (last) {
        if (keep) { if (k_dev) kd = keep; else CK(t_k.get(&kd, (size_t)std::max<long long>(m, 1))); }
        ic.keep = kd;
        CK(t_cnt.get(&cnt, (size_t)maxno));
        CK(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long) * maxno, h->st));
        ic.count_lt = cnt;
        if (ncell > 0) {
            CK(t_cmin.get(&cmin, (size_t)ncell * maxno));
            CK(t_ccnt.get(&ccnt, (size_t)ncell * maxno));
            CK(cudaMemsetAsync(cmin, 0x7f, sizeof(unsigned long long) * ncell * maxno, h->st));
            CK(cudaMemsetAsync(ccnt, 0, sizeof(unsigned long long) * ncell * maxno, h->st));
            ic.cell_min_bits = cmin; ic.cell_count = ccnt;
        }
    }
    int rc = 0;
    if (m > 0) {
        if (Xs) {
            rc = predict_common(h, Xs, Hs, nullptr, 0, m, nullptr, nullptr, &ic);
        } else {
            if (h->d > MAXD) return h->fail_msg("grid prediction supports d <= 64");
            GridDesc g;
            g.d = h->d;
            for (int k = 0; k < h->d; k++) {
                g.levels[k] = levels[k];
                g.lo[k] = lo[k];
                g.step[k] = (hi[k] - lo[k]) / (double)levels[k];
            }
            rc = predict_common(h, nullptr, nullptr, &g, start, m, nullptr, nullptr, &ic);
        }
        if (rc) return rc;
    }
    if (last) {
        if (keep && !k_dev && m > 0) CK(cudaMemcpyAsync(keep, kd, (size_t)m, cudaMemcpyDeviceToHost, h->st));
        if (count_lt) CK(cudaMemcpyAsync(count_lt, cnt, sizeof(unsigned long long) * maxno, cudaMemcpyDefault, h->st));
        if (ncell > 0 && cell_min) CK(cudaMemcpyAsync(cell_min, cmin, sizeof(double) * ncell * maxno, cudaMemcpyDefault, h->st));
        if (ncell > 0 && cell_count) CK(cudaMemcpyAsync(cell_count, ccnt, sizeof(unsigned long long) * ncell * maxno, cudaMemcpyDefault, h->st));
        CK(cudaStreamSynchronize(h->st));
        CK(cudaGetLastError());
    }
    return 0;
}

int gpe_cross_cov(gpe_handle* h, const double* delta, double nugget, int kind, const double* Xs, int m, double* C_out) {
    if (h && m == 0) return 0;
    if (!h || !h->n || !delta || !Xs || !C_out || m < 1) return h ? h->fail_msg("bad argument") : -2;
    NvtxRange nvtx("gpe_cross_cov");
    CK(cudaSetDevice(h->device));
    const int np = h->npad, d = h->d;
    int mc = (m + 127) / 128 * 128;
    std::vector<double> w(d), dl(d);
    CK(cudaMemcpy(dl.data(), delta, sizeof(double) * d, cudaMemcpyDefault));
    for (int k = 0; k < d; k++) w[k] = 1.0 / dl[k];
    double *wd = nullptr, *xs = nullptr, *P = nullptr, *Cm = nullptr;
    TmpDev t_wd(h), t_xs(h), t_P(h), t_Cm(h);
    CK(t_wd.get(&wd, (size_t)d));
    CK(t_xs.get(&xs, (size_t)d * np));
    CK(t_P.get(&P, (size_t)mc * d));
    CK(t_Cm.get(&Cm, (size_t)np * mc));
    CK(cudaMemcpyAsync(wd, w.data(), sizeof(double) * d, cudaMemcpyHostToDevice, h->st));
    CK(cudaMemsetAsync(P, 0, sizeof(double) * (size_t)mc * d, h->st));
    CK(cudaMemcpyAsync(P, Xs, sizeof(double) * (size_t)m * d, cudaMemcpyDefault, h->st));
    scale_train_kernel<<<(d * np + 255) / 256, 256, 0, h->st>>>(h->X, wd, h->n, d, np, xs);
    CK(launch_xcov(h->family, xs, P, wd, h->n, d, np, mc, m, kind ? 1.0 : 1.0 - nugget, Cm, mc, h->st));
    h->launches += 2;
    bool dev = gpe_is_device_ptr(C_out);
    CK(cudaMemcpy2DAsync(C_out, sizeof(double) * m, Cm, sizeof(double) * mc, sizeof(double) * m, h->n,
                         dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

int gpe_predict_fullcov(gpe_handle* h, const double* Xs, const double* Hs, int m, const double* r_new, double* mean,
                        double* V) {
    if (h && m == 0) return 0;
    if (!h || !Xs || !mean || !V || m < 1) return h ? h->fail_msg("bad argument") : -2;
    if (!h->fitted) return h->fail_msg("gpe_fit_state has not succeeded on this handle");
    if (!Hs && !h->has_basis) return h->fail_msg("no H* given and no device basis set (gpe_set_basis)");
    NvtxRange nvtx("gpe_predict_fullcov");
    CK(cudaSetDevice(h->device));
    const int np = h->npad, d = h->d, q = h->q;
    const int mp = (m + 127) / 128 * 128;
    double *P = nullptr, *Hd = nullptr, *Cm = nullptr, *Zm = nullptr, *ZtZ = nullptr, *aux = nullptr, *G = nullptr, *rn = nullptr,
           *md = nullptr, *Vd = nullptr;
    TmpDev t_P(h), t_Cm(h), t_Zm(h), t_ZtZ(h), t_aux(h), t_G(h), t_md(h), t_Vd(h), t_Hd(h), t_rn(h);
    CK(t_P.get(&P, (size_t)mp * d));
    CK(t_Cm.get(&Cm, (size_t)np * mp));
    CK(t_Zm.get(&Zm, (size_t)np * mp));
    CK(t_ZtZ.get(&ZtZ, (size_t)mp * mp));
    CK(t_aux.get(&aux, (size_t)NR * mp));
    CK(t_G.get(&G, (size_t)NR * mp));
    CK(t_md.get(&md, (size_t)mp));
    CK(t_Vd.get(&Vd, (size_t)m * m));
    CK(cudaMemsetAsync(P, 0, sizeof(double) * (size_t)mp * d, h->st));
    CK(cudaMemcpyAsync(P, Xs, sizeof(double) * (size_t)m * d, cudaMemcpyDefault, h->st));
    if (Hs) {
        CK(t_Hd.get(&Hd, (size_t)m * q));
        CK(cudaMemcpyAsync(Hd, Hs, sizeof(double) * (size_t)m * q, cudaMemcpyDefault, h->st));
    }
    if (r_new) {
        CK(t_rn.get(&rn, (size_t)m));
        CK(cudaMemcpyAsync(rn, r_new, sizeof(double) * m, cudaMemcpyDefault, h->st));
    }
    CK(launch_xcov(h->family, h->fXs, P, h->fwinv, h->n, d, np, mp, m, h->fit_c, Cm, mp, h->st));
    h->launches++;
    int rc = 0;
    if (!rc) rc = gpe_run_gemm(h, h->fE, Cm, aux, NR, mp, mp, 0, 0, 0, NR, mp, np, 1.0, 0, KM_FULL, 0, 1, 2, EPI_STORE);
    if (!rc) rc = gpe_run_gemm(h, h->fLi, Cm, Zm, np, mp, mp, 0, 0, 0, np, mp, np, 1.0, 0, KM_LE_I, 0, 1, 1, EPI_STORE);
    if (!rc) rc = gpe_run_gemm(h, Zm, Zm, ZtZ, mp, mp, mp, 0, 0, 0, mp, mp, np, 1.0, 0, KM_FULL, 0, 1, 2, EPI_STORE);
    if (!rc) {
        BasisDesc bd = basis_of(h);
        double s2 = h->fit_sigma * h->fit_sigma;
        // mean via the diagonal finalize (var == nullptr)
        predict_finalize_kernel<false><<<(m + 127) / 128, 128, 0, h->st>>>(nullptr, 0, aux, mp, P, Hd, bd, d, h->fK, h->fbeta, s2,
                                                                            h->fit_astar, m, md, nullptr, ImpFuse{});
        auto fin = h->family == FAMILY_MATERN52 ? fullcov_finalize_kernel<FAMILY_MATERN52> : fullcov_finalize_kernel<FAMILY_GAUSSIAN>;
        fin<<<(m + 127) / 128, 128, 0, h->st>>>(ZtZ, mp, aux, mp, P, Hd, bd, d, h->fwinv, h->fK, s2, h->fit_c, h->fit_astar, rn, m, G, Vd, 0);
        size_t tot = (size_t)m * m;
        fin<<<(unsigned)((tot + 255) / 256), 256, 0, h->st>>>(ZtZ, mp, aux, mp, P, Hd, bd, d, h->fwinv, h->fK, s2, h->fit_c, h->fit_astar,
                                                            rn, m, G, Vd, 1);
        h->launches += 3;
        CK(cudaMemcpyAsync(mean, md, sizeof(double) * m, cudaMemcpyDefault, h->st));
        CK(cudaMemcpyAsync(V, Vd, sizeof(double) * (size_t)m * m, cudaMemcpyDefault, h->st));
    }
    CK(cudaStreamSynchronize(h->st));
    if (rc) return rc;
    CK(cudaGetLastError());
    return 0;
}

int gpe_implausibility(gpe_handle* h, const double* mean, const double* var, int n_emul, long long m, const double* z,
                       const double* var_extra, double cm, int maxno, long long cell_pts, long long first_index, long long ncell,
                       double* Imax, unsigned char* keep, unsigned long long* count_lt, double* cell_min,
                       unsigned long long* cell_count) {
    if (!h || !z || !var_extra || n_emul < 1 || m < 0 || (m > 0 && (!mean || !var))) return h ? h->fail_msg("bad argument") : -2;
    if (n_emul > MAXEM || maxno < 1 || maxno > n_emul) return h->fail_msg("need 1 <= maxno <= n_emul <= 16");
    if (cell_pts < 0 || first_index < 0 || ncell < 0) return h->fail_msg("cell_pts, first_index and ncell must be non-negative");
    if (cell_pts == 0) ncell = 0;
    if (cell_pts > 0 && m > 0 && (first_index + m - 1) / cell_pts - first_index / cell_pts + 1 > ncell)
        return h->fail_msg("the points span more cells than ncell");
    NvtxRange nvtx("gpe_implausibility");
    CK(cudaSetDevice(h->device));
    ImpDesc ds;
    ds.n_emul = n_emul; ds.maxno = maxno; ds.cm = cm;
    std::vector<double> zz(n_emul), vv(n_emul);
    CK(cudaMemcpy(zz.data(), z, sizeof(double) * n_emul, cudaMemcpyDefault));
    CK(cudaMemcpy(vv.data(), var_extra, sizeof(double) * n_emul, cudaMemcpyDefault));
    for (int o = 0; o < n_emul; o++) { ds.z[o] = zz[o]; ds.ve[o] = vv[o]; }
    const bool in_dev = gpe_is_device_ptr(mean);
    const double *md = mean, *vd = var;
    double *mtmp = nullptr, *vtmp = nullptr, *Id = nullptr;
    unsigned char* kd = nullptr;
    unsigned long long *cnt = nullptr, *cmin = nullptr, *ccnt = nullptr;
    TmpDev t_m(h), t_v(h), t_I(h), t_k(h), t_cnt(h), t_cmin(h), t_ccnt(h);
    if (!in_dev) {
        CK(t_m.get(&mtmp, (size_t)n_emul * m));
        CK(t_v.get(&vtmp, (size_t)n_emul * m));
        CK(cudaMemcpyAsync(mtmp, mean, sizeof(double) * (size_t)n_emul * m, cudaMemcpyHostToDevice, h->st));
        CK(cudaMemcpyAsync(vtmp, var, sizeof(double) * (size_t)n_emul * m, cudaMemcpyHostToDevice, h->st));
        md = mtmp; vd = vtmp;
    }
    const bool I_dev = Imax && gpe_is_device_ptr(Imax), k_dev = keep && gpe_is_device_ptr(keep);
    if (Imax) { if (I_dev) Id = Imax; else CK(t_I.get(&Id, (size_t)m * maxno)); }
    if (keep) { if (k_dev) kd = keep; else CK(t_k.get(&kd, (size_t)m)); }
    CK(t_cnt.get(&cnt, (size_t)maxno));
    CK(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long) * maxno, h->st));
    if (ncell > 0) {
        CK(t_cmin.get(&cmin, (size_t)ncell * maxno));
        CK(t_ccnt.get(&ccnt, (size_t)ncell * maxno));
        CK(cudaMemsetAsync(cmin, 0x7f, sizeof(unsigned long long) * ncell * maxno, h->st));   // large positive double
        CK(cudaMemsetAsync(ccnt, 0, sizeof(unsigned long long) * ncell * maxno, h->st));
    }
    if (m > 0) {                                                 // m == 0: zero counts, +huge cell minima
        implaus_kernel<<<(unsigned)((m + 255) / 256), 256, 0, h->st>>>(md, vd, m, ds, ncell > 0 ? cell_pts : 0, first_index, Id, kd, cnt, cmin, ccnt);
        h->launches++;
    }
    if (Imax && !I_dev && m > 0) CK(cudaMemcpyAsync(Imax, Id, sizeof(double) * (size_t)m * maxno, cudaMemcpyDeviceToHost, h->st));
    if (keep && !k_dev && m > 0) CK(cudaMemcpyAsync(keep, kd, (size_t)m, cudaMemcpyDeviceToHost, h->st));
    if (count_lt) CK(cudaMemcpyAsync(count_lt, cnt, sizeof(unsigned long long) * maxno, cudaMemcpyDefault, h->st));
    if (ncell > 0 && cell_min) CK(cudaMemcpyAsync(cell_min, cmin, sizeof(double) * ncell * maxno, cudaMemcpyDefault, h->st));
    if (ncell > 0 && cell_count) CK(cudaMemcpyAsync(cell_count, ccnt, sizeof(unsigned long long) * ncell * maxno, cudaMemcpyDefault, h->st));
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

}  // extern "C"
