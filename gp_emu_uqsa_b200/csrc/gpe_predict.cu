// K4 posterior mean / variance over large point sets, K4f full covariance, K5 implausibility.
// Reference arithmetic replaced: Posterior.make_covar/make_mean/make_var
// (_emulatorclasses.py:607-631), kernel.covar (_emulatorkernels.py:75-79, :148-152),
// history_match.py:121-136 / :237-250 / :317-329.
//
// Nothing of size m x m or n x m_total is ever materialised: points are processed in chunks (for_chunks);
// per chunk the cross-covariance tile C [n, mc] is generated on device (optionally straight from
// a flat grid index) and a skinny product [A^-1 H K^-T | e]^T C gives the mean and the regression-variance
// term (posterior_cross), and Z = L^-1 C runs with the column norms |L^-1 c_j|^2 reduced in the GEMM
// epilogue (fit_z_product).   v_j = sigma^2 (a*_jj - |L^-1 c_j|^2 + |K^-1 h_j - (Gm K^-T)^T c_j|^2).
// gpe_predict_fullcov, gpe_sens_sample and gpe_predict_grad (a derivative slab in place of C) build on the same steps.
#include "gpe_handle.h"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace gpe;

void gpe_handle::free_fit() {
    dev_free(fLi); dev_free(fE); dev_free(fK); dev_free(fbeta); dev_free(fwinv); dev_free(fXs); dev_free(fAinv);
    fAinv_valid = false;
    for (auto& sl : ps) { dev_free(sl.C); dev_free(sl.Part); dev_free(sl.Aux); dev_free(sl.X); dev_free(sl.H); dev_free(sl.Mean); dev_free(sl.Var); }
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
// CTA = 64 training rows x 128 points, 256 threads, each thread 8 rows x 4 points (the 8 x 4 shape of sqdist_tile).
// GRAD: the derivative slab instead, C[i][k mc + j] = delta_k d/dp_k [c R(D_ij)] = 2 c phi(D_ij) u_ijk with
// u_ijk = (x_ik - p_jk) / delta_k and phi = -dR/dD (exp(-D); Matérn: G(D)); |entry| <= c (DESIGN.md section 9e).  After D, per
// row a second pass over the shared tiles, one input k at a time.  Two CTAs per SM, not three: the second pass keeps more
// registers live than the store loop of C and spills at 80.
template <int FAM, bool GRAD>
__global__ void __launch_bounds__(256, GRAD ? 2 : 3) xcov_kernel(const double* __restrict__ Xs /*[d][npad]*/, const double* __restrict__ P /*[mc][d]*/,
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
    sqdist_tile<8, 8, 64>(Xt, Pt, d, ty, tx, D);
    if constexpr (GRAD) {
        const double c2 = 2.0 * cscale;
#pragma unroll
        for (int a = 0; a < 8; a++) {
            const int row = ty + 8 * a, gk = k0 + row;
            const bool live = gk < n;
            double s[4];
#pragma unroll
            for (int c = 0; c < 4; c++) {      // phi one row's four chains at a time (both families): 32 at once would spill
                double phi;
                if constexpr (FAM == FAMILY_MATERN52) gpe_matern52(D[a][c], phi);
                else phi = gpe_exp(-D[a][c]);
                const int gj = j0 + 64 * (c >> 1) + 2 * tx + (c & 1);
                s[c] = (live && gj < count) ? c2 * phi : 0.0;
            }
            double* crow = Cm + (size_t)gk * d * mc + j0 + 2 * tx;      // row stride d mc (= ldc), formed in 64 bits
            for (int k = 0; k < d; k++) {
                const double xr = Xt[k * 64 + row];
                const double2 v0 = *reinterpret_cast<const double2*>(&Pt[k * 130 + 2 * tx]);
                const double2 v1 = *reinterpret_cast<const double2*>(&Pt[k * 130 + 64 + 2 * tx]);
                *reinterpret_cast<double2*>(crow + (size_t)k * mc) = make_double2(s[0] * (xr - v0.x), s[1] * (xr - v0.y));
                *reinterpret_cast<double2*>(crow + (size_t)k * mc + 64) = make_double2(s[2] * (xr - v1.x), s[3] * (xr - v1.y));
            }
        }
    } else {
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

static cudaError_t launch_xcov_grid(int family, const double* T, const GridSep& sp, int n, int npad, int mc, long long start,
                                    long long count, double cscale, double* Cm, size_t smem, cudaStream_t st) {
    return with_family(family, [&](auto fam) {
        switch (sp.nf) {
            case 1: return launch_xcov_grid_nf<1, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            case 2: return launch_xcov_grid_nf<2, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            case 3: return launch_xcov_grid_nf<3, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            case 4: return launch_xcov_grid_nf<4, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            case 5: return launch_xcov_grid_nf<5, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            case 6: return launch_xcov_grid_nf<6, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            case 7: return launch_xcov_grid_nf<7, fam>(T, sp, n, npad, mc, start, count, cscale, Cm, smem, st);
            default: return cudaErrorInvalidValue;
        }
    });
}

struct GridXcov {        // what predict_chunk needs to build a chunk's cross-covariance from the tables
    const double* T;
    GridSep sp;
    size_t smem;
    long long start;     // flat index of the chunk's first point
};

// C [n rows of npad, ldc] = cscale * K(training, P) for the mc points P [mc, d] (columns >= count zero); GRAD: the derivative
// slab, input k's mc columns at k mc (ldc = d mc)
template <bool GRAD>
static cudaError_t launch_xcov(int family, const double* Xs, const double* P, const double* winv, int n, int d, int npad, int mc,
                               long long count, double cscale, double* Cm, int ldc, cudaStream_t st) {
    return with_family(family, [&](auto fam) {
        static SmemOptIn optin;      // d >= 32 needs more than 48 KB for the two k-major tiles
        const size_t smem = (size_t)d * (64 + 130) * sizeof(double);
        if (cudaError_t e = optin.ensure(xcov_kernel<fam, GRAD>, smem); e != cudaSuccess) return e;
        xcov_kernel<fam, GRAD><<<dim3(mc / 128, npad / 64), 256, smem, st>>>(Xs, P, winv, n, d, npad, mc, count, cscale, Cm, ldc);
        return cudaGetLastError();
    });
}

// K5 implausibility I = |mean - z| / sqrt(var + var_extra) of a point against each emulator's observation z, the per-point
// ascending list of the maxno largest I over the emulators (history_match.py:96-132) and, on the finished lists, the keep mask,
// the counts and the cell statistics.  Two routes share the update and the reduction below, so they give bit-identical results:
// gpe_implausibility (implaus_kernel) on given mean / variance arrays, and gpe_predict_implaus, which folds the update into the
// prediction of one emulator (predict_finalize_kernel<true>: a running list Itop [m][maxno] instead of mean / variance) and the
// reduction into the last emulator's pass, so neither the means / variances nor (unless asked for) the final list travel through HBM.
constexpr int MAXEM = 16;

// What the reduction adds into.  I >= 0, so the IEEE bit pattern orders like the value and the cell minima are integer atomics
// (deterministic).  Cells are runs of cell_pts points of the global flat index; output cell 0 is the cell of the call's first point.
struct ImpStats {
    double cm;
    int maxno;
    long long cell_pts;                  // 0: no cell statistics
    long long cell_base;                 // (call's first_index) / cell_pts
    unsigned char* keep;                 // or null
    unsigned long long *count_lt, *cell_min_bits, *cell_count;      // [maxno], [ncell][maxno]
};

__device__ __forceinline__ double implaus_value(double mean, double var, double z, double ve) {
    const double dz = mean - z;
    return sqrt(dz * dz / (var + ve));
}

// I into the ascending list of the maxno largest, top[maxno-1] the largest (np.sort(np.partition(I, -maxno)[-maxno:]), :129)
__device__ __forceinline__ void top_insert(double (&top)[MAXEM], int maxno, double I) {
    if (I > top[0]) {
        top[0] = I;
#pragma unroll
        for (int k = 0; k < MAXEM - 1; k++) {
            if (k + 1 < maxno && top[k] > top[k + 1]) {
                double t = top[k];
                top[k] = top[k + 1];
                top[k + 1] = t;
            }
        }
    }
}

// The reduction of a point's finished list; every lane of the warp calls it.  local: the point's index in keep, global: its flat index.
// A warp's 32 consecutive points almost always sit in one cell: reduce in the warp first, one atomic per warp instead of one per point.
__device__ __forceinline__ void imp_finish(const double (&top)[MAXEM], bool live, long long local, long long global, const ImpStats& s) {
    if (live && s.keep != nullptr) s.keep[local] = (top[0] < s.cm) ? 1 : 0;
    const long long cell = (s.cell_pts > 0 && live) ? global / s.cell_pts - s.cell_base : -1;
    const long long cell0 = __shfl_sync(0xffffffffu, cell, 0);
    const bool uniform = s.cell_pts > 0 && __all_sync(0xffffffffu, cell == cell0) && cell0 >= 0;
    for (int k = 0; k < s.maxno; k++) {
        const double vk = top[s.maxno - 1 - k];      // the k-th statistic refers to the (k+1)-th largest
        const bool lt = live && (vk < s.cm);
        const unsigned bal = __ballot_sync(0xffffffffu, lt);
        if ((threadIdx.x & 31) == 0 && bal && s.count_lt != nullptr) atomicAdd(&s.count_lt[k], (unsigned long long)__popc(bal));
        if (s.cell_pts <= 0) continue;
        if (uniform) {
            unsigned long long bits = (unsigned long long)__double_as_longlong(vk);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                unsigned long long other = __shfl_xor_sync(0xffffffffu, bits, o);
                bits = other < bits ? other : bits;
            }
            if ((threadIdx.x & 31) == 0) {
                if (s.cell_min_bits != nullptr) atomicMin(&s.cell_min_bits[(size_t)cell0 * s.maxno + k], bits);
                if (bal && s.cell_count != nullptr) atomicAdd(&s.cell_count[(size_t)cell0 * s.maxno + k], (unsigned long long)__popc(bal));
            }
        } else if (live) {
            if (s.cell_min_bits != nullptr) atomicMin(&s.cell_min_bits[(size_t)cell * s.maxno + k], (unsigned long long)__double_as_longlong(vk));
            if (lt && s.cell_count != nullptr) atomicAdd(&s.cell_count[(size_t)cell * s.maxno + k], 1ull);
        }
    }
}

struct ImpFuse {
    double z, ve;
    int first, last;
    double* Itop;                        // chunk's first point; in/out (out may be skipped on the last pass: store_top)
    int store_top;
    long long first_index;               // global flat index of the chunk's first point
    ImpStats st;                         // last pass (keep: the chunk's first point)
};

// h_a(x_j), the a-th mean basis function at point j: the caller's H* [m][q] when given, else the device polynomial basis
__device__ __forceinline__ double basis_value(const double* __restrict__ Hs, int q, const double* __restrict__ P, int d,
                                              const BasisDesc& bd, long long j, int a) {
    if (Hs != nullptr) return Hs[(size_t)j * q + a];
    if (a == 0) return 1.0;
    const double x = P[(size_t)j * d + bd.idx[a]];
    const int pw = bd.pw[a];
    return (pw == 1) ? x : pow(x, (double)pw);
}

// d h_a / d x_k at point j for the device polynomial basis
__device__ __forceinline__ double basis_deriv(const double* __restrict__ P, int d, const BasisDesc& bd, long long j, int k, int a) {
    const int pw = bd.pw[a];
    if (a == 0 || bd.idx[a] != k || pw == 0) return 0.0;
    if (pw == 1) return 1.0;
    const double x = P[(size_t)j * d + k];
    return (pw == 2) ? 2.0 * x : pw * pow(x, (double)(pw - 1));
}

// Row a of the forward substitution kv = K^-1 h with the lower-triangular K (leading dimension LD), from kv[0:a] and h_a.
// One row at a time: the callers use kv[a] as soon as it is ready.
template <int LD>
__device__ __forceinline__ double forward_subst_row(const double* K, const double (&kv)[NR], double h, int a) {
    double s = h;
    for (int k = 0; k < a; k++) s = fma(-K[a * LD + k], kv[k], s);
    return s / K[a * LD + a];
}

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
        for (int a = 0; a < NR; a++) hv[a] = (a < q) ? basis_value(Hs, q, P, d, bd, j, a) : 0.0;
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
                kv[a] = forward_subst_row<NR + 1>(&Ks[0][0], kv, hv[a], a);
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
        // this emulator's implausibility into the running list; the last emulator's pass reduces the finished lists
        const int maxno = imp.st.maxno;
        double top[MAXEM];
#pragma unroll
        for (int k = 0; k < MAXEM; k++) top[k] = -1.0;
        if (live) {
            if (!imp.first)
                for (int k = 0; k < maxno; k++) top[k] = imp.Itop[(size_t)j * maxno + k];
            top_insert(top, maxno, implaus_value(mu, vj, imp.z, imp.ve));
            if (!imp.last || imp.store_top)
                for (int k = 0; k < maxno; k++) imp.Itop[(size_t)j * maxno + k] = top[k];
        }
        if (!imp.last) return;
        imp_finish(top, live, j, imp.first_index + j, imp.st);
    }
}

// per (point j, input k), one thread per column k mc + j of the derivative slab b (b = delta_k dc/dp_k): with a = aux of the
// column and zn = |L^-1 b|^2 (tile partials),
//   dmean = sum_a beta_a dh_a/dp_k + a[q] / delta_k,   dvar = sigma^2 ((c kappa - zn) / delta_k^2 + |K^-1 dh - a[0:q] / delta_k|^2),
// written to dmean / dvar [count][d]
__global__ void __launch_bounds__(128) predict_grad_finalize_kernel(const double* __restrict__ part, int ntile, const double* __restrict__ aux,
                                                                    int mc, const double* __restrict__ P, BasisDesc bd, int d,
                                                                    const double* __restrict__ winv, const double* __restrict__ Kf,
                                                                    const double* __restrict__ beta, double sigma2, double ckappa,
                                                                    long long count, double* __restrict__ dmean, double* __restrict__ dvar) {
    __shared__ double Ks[NR][NR + 1];
    __shared__ double bs[NR];
    const int q = bd.q;
    for (int e = threadIdx.x; e < NR * NR; e += blockDim.x) Ks[e / NR][e % NR] = Kf[e];
    if (threadIdx.x < NR) bs[threadIdx.x] = beta[threadIdx.x];
    __syncthreads();
    const size_t ld = (size_t)d * mc;
    const size_t col = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    const int k = (int)(col / mc);
    const long long j = (long long)(col % mc);
    if (k >= d || j >= count) return;
    const double w = winv[k];
    double dh[NR];
#pragma unroll
    for (int a = 0; a < NR; a++) dh[a] = (a < q) ? basis_deriv(P, d, bd, j, k, a) : 0.0;
    double mu = aux[(size_t)q * ld + col] * w;
#pragma unroll
    for (int a = 0; a < NR; a++)
        if (a < q) mu = fma(dh[a], bs[a], mu);
    dmean[j * d + k] = mu;
    if (dvar == nullptr) return;
    double gn = 0.0;
    double kv[NR];
#pragma unroll
    for (int a = 0; a < NR; a++) {
        if (a < q) {
            kv[a] = forward_subst_row<NR + 1>(&Ks[0][0], kv, dh[a], a);
            const double g = fma(-aux[(size_t)a * ld + col], w, kv[a]);
            gn = fma(g, g, gn);
        } else {
            kv[a] = 0.0;
        }
    }
    double zn = 0.0;
    for (int t = 0; t < ntile; t++) zn += part[(size_t)t * ld + col];
    dvar[j * d + k] = sigma2 * fma(ckappa - zn, w * w, gn);
}

struct ImpDesc {
    int n_emul;
    double z[MAXEM], ve[MAXEM];
};

__global__ void __launch_bounds__(256) implaus_kernel(const double* __restrict__ mean, const double* __restrict__ var, long long m,
                                                      ImpDesc ds, long long first_index, double* __restrict__ Imax, ImpStats st) {
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool live = r < m;
    double top[MAXEM];
#pragma unroll
    for (int k = 0; k < MAXEM; k++) top[k] = -1.0;
    if (live)
        for (int o = 0; o < ds.n_emul; o++)
            top_insert(top, st.maxno, implaus_value(mean[(size_t)o * m + r], var[(size_t)o * m + r], ds.z[o], ds.ve[o]));
    if (live && Imax != nullptr)
        for (int k = 0; k < st.maxno; k++) Imax[(size_t)r * st.maxno + k] = top[k];
    imp_finish(top, live, r, first_index + r, st);
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
            kv[a] = forward_subst_row<NR>(Kf, kv, basis_value(Hs, q, P, d, bd, j, a), a);
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
    double prior = (i == j) ? (astar + (r_new ? r_new[i] : 0.0)) : cov_prior<FAM>(cscale, D);
    double gg = 0.0;
    for (int a = 0; a < q; a++) gg = fma(Gbuf[(size_t)a * mp + i], Gbuf[(size_t)a * mp + j], gg);
    V[idx] = sigma2 * (prior - ZtZ[(size_t)i * mp + j] + gg);
}

int ensure_predict_ws(gpe_handle* h, long long mc) {
    if (mc <= h->pchunk) return 0;
    h->pchunk = 0;
    size_t ntile = h->npad / 128;
    for (auto& sl : h->ps) {
        dev_free(sl.C); dev_free(sl.Part); dev_free(sl.Aux); dev_free(sl.X); dev_free(sl.H); dev_free(sl.Mean); dev_free(sl.Var);
        CK(dev_alloc(&sl.C, (size_t)h->npad * mc));
        CK(dev_alloc(&sl.Part, ntile * mc));
        CK(dev_alloc(&sl.Aux, (size_t)NR * mc));
        CK(dev_alloc(&sl.X, (size_t)mc * h->d));
        CK(dev_alloc(&sl.H, (size_t)mc * NR));
        CK(dev_alloc(&sl.Mean, (size_t)mc));
        CK(dev_alloc(&sl.Var, (size_t)mc));
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

// The fit state a posterior entry point works on; has_H: the caller gives H* for its points
int check_fit(gpe_handle* h, bool has_H) {
    if (!h->fitted) return h->fail_msg("gpe_fit_state has not succeeded on this handle");
    if (!has_H && !h->has_basis) return h->fail_msg("no H* given and no device basis set (gpe_set_basis)");
    return 0;
}

// The caller's points Xs [cnt][d] (host or device memory) into the device buffer P [mc][d], rows >= cnt zero
cudaError_t stage_points(double* P, const double* Xs, long long cnt, int mc, int d, cudaStream_t st) {
    if (cnt < mc)
        if (cudaError_t e = cudaMemsetAsync(P, 0, (size_t)mc * d * sizeof(double), st); e != cudaSuccess) return e;
    return cudaMemcpyAsync(P, Xs, (size_t)cnt * d * sizeof(double), cudaMemcpyDefault, st);
}

// Rows / columns >= n of the padded matrices are identity padding and the slab's rows >= n are zero: the DMMA products over the
// slab need only the first n rounded up to the k-tile (n = 2000: 2000 instead of 2048 -- the last, heaviest row tile of the
// triangular product has 80 live rows, not 128)
int live_k(const gpe_handle* h) { return std::min(h->npad, (h->n + GEMM_BK - 1) / GEMM_BK * GEMM_BK); }

// aux = [A^-1 H K^-T | e]^T C of a slab C [npad][cols] (TN, skinny: the q + 1 live columns of the panel padded to 16 or 32 rows)
int posterior_aux(gpe_handle* h, cudaStream_t st, const double* C, int cols, double* aux) {
    const int maux = (h->q + 1 <= 16) ? 16 : NR;
    return gpe_gemm(h, st, {.A = h->fE, .B = C, .C = aux, .lda = NR, .ldb = cols, .ldc = cols, .M = maux, .N = cols, .K = live_k(h)},
                    GEMM_TN);
}

// The slab C [npad][cols] = c K(training, points) of the points P [cols][d] or of the grid chunk gx (columns >= count zero), and
// its aux
int posterior_cross(gpe_handle* h, cudaStream_t st, const double* P, const GridXcov* gx, int cols, long long count, double* C,
                    double* aux) {
    {
        ProfScope ps(h, gpe_handle::CAT_COV, st);
        if (gx != nullptr) CK(launch_xcov_grid(h->family, gx->T, gx->sp, h->n, h->npad, cols, gx->start, count, h->fit_c, C, gx->smem, st));
        else CK(launch_xcov<false>(h->family, h->fXs, P, h->fwinv, h->n, h->d, h->npad, cols, count, h->fit_c, C, cols, st));
    }
    h->launches++;
    return posterior_aux(h, st, C, cols, aux);
}

// Z = L^-1 C of the fit state (L^-1 lower: k <= i), stored into out (EPI_STORE) or reduced to column norms in the epilogue, tile
// partials out [*ntile][cols] (EPI_SUMSQ).  The route is decided once: the plan below is the route taken.
int fit_z_product(gpe_handle* h, cudaStream_t st, const double* C, int cols, double* out, int epi, int* ntile = nullptr) {
    const int np = h->npad;
    GemmP z{.A = h->fLi, .B = C, .C = out, .lda = np, .ldb = cols, .ldc = cols, .M = np, .N = cols, .K = np, .kmode = KM_LE_I};
    OzHint hint;
    const bool int8 = gpe_int8_route(h, st, z, GEMM_NN, epi);
    if (int8) {
        // INT8 tensor-core route (gpe_ozaki.cuh): the residue planes of L^-1 are made once per fit, stream and layout (the tag is
        // the generation of the fit state), the padded size is used (rows >= n of Z are zero).  Every entry of the slab is
        // c exp(-D) or c R(D), in [0, c]: one scale for all points, no pass over the slab for its maxima.  (A point far from
        // every training input then keeps fewer significant bits of its tiny column -- its variance is the prior's to the same
        // absolute accuracy, which is what the subtraction prior - |Z|^2 needs.)
        hint = OzHint{.reuse_a = true, .a_tag = h->fit_gen, .b_bound = h->fit_c};
    } else if (epi == EPI_SUMSQ) {      // the ragged last row tile exists for the column norms only
        z.M = z.K = live_k(h);
    }
    if (int rc = gpe_gemm_routed(h, st, z, GEMM_NN, epi, int8, hint)) return rc;
    if (ntile != nullptr) *ntile = (int8 && oz_sumsq_swapped(z, epi)) ? 1 : (z.M + 127) / 128;
    return 0;
}

// Chunks alternate between two (stream, buffer slot) pairs when there is more than one and profiling is off: a slot's buffers
// are reused only by later chunks of the same stream, which orders them.
int chunk_slots(const gpe_handle* h, long long nchunk) { return (nchunk > 1 && !h->prof_on) ? 2 : 1; }

// body(ci, slot, stream) for the chunks ci = 0 .. nchunk - 1, forked from the handle's stream and joined back into it
template <class Body>
int for_chunks(gpe_handle* h, long long nchunk, Body body) {
    const bool two = chunk_slots(h, nchunk) == 2;
    if (two) {
        CK(cudaEventRecord(h->ev_fork, h->st));
        for (int k = 0; k < 2; k++) CK(cudaStreamWaitEvent(h->sub_st[k], h->ev_fork, 0));
    }
    for (long long ci = 0; ci < nchunk; ci++) {
        const int k = two ? (int)(ci & 1) : 0;
        if (int rc = body(ci, k, two ? h->sub_st[k] : h->st)) return rc;
    }
    if (two) {
        for (int k = 0; k < 2; k++) {
            CK(cudaEventRecord(h->ev_join[k], h->sub_st[k]));
            CK(cudaStreamWaitEvent(h->st, h->ev_join[k], 0));
        }
    }
    return 0;
}

// One chunk on stream `st` with the buffers of `sl`: points already in P_dev [mc, d] (rows >= count
// arbitrary but finite).
int predict_chunk(gpe_handle* h, gpe_handle::PredSlot& sl, cudaStream_t st, const double* P_dev, const double* Hs_dev,
                  long long count, int mc, double* mean_dev, double* var_dev, const GridXcov* gx = nullptr, const ImpFuse* imp = nullptr) {
    int rc, ntile = 0;
    if ((rc = posterior_cross(h, st, P_dev, gx, mc, count, sl.C, sl.Aux))) return rc;
    if ((var_dev != nullptr || imp != nullptr) && (rc = fit_z_product(h, st, sl.C, mc, sl.Part, EPI_SUMSQ, &ntile))) return rc;
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

// The tensor grid of gpe_predict_grid / gpe_predict_implaus from the caller's levels, lo, hi [d] (host memory)
int make_grid(gpe_handle* h, const int* levels, const double* lo, const double* hi, GridDesc& g) {
    if (h->d > MAXD) return h->fail_msg("grid prediction supports d <= 64");
    g.d = h->d;
    for (int k = 0; k < h->d; k++) {
        g.levels[k] = levels[k];
        g.lo[k] = lo[k];
        g.step[k] = (hi[k] - lo[k]) / (double)levels[k];
    }
    return 0;
}

// The cell arguments of the implausibility entry points; m = 0 skips the check that ncell covers the cells of m points.
int check_cells(gpe_handle* h, long long cell_pts, long long first_index, long long ncell, long long m) {
    if (cell_pts < 0 || first_index < 0 || ncell < 0) return h->fail_msg("cell_pts, first_index and ncell must be non-negative");
    if (cell_pts > 0 && m > 0 && (first_index + m - 1) / cell_pts - first_index / cell_pts + 1 > ncell)
        return h->fail_msg("the points span more cells than ncell");
    return 0;
}

// The implausibility reductions over a call's points: count_lt [maxno] and, with cells, cell_min [ncell][maxno] (bits of I >= 0,
// which order like the value) and cell_count; stats() is what the kernels add into, finish() copies the sums to the caller's
// outputs (host, device or NULL) and waits.
struct ImpAccum {
    gpe_handle* h;
    int maxno;
    long long cell_pts, ncell;      // both 0 without cells
    unsigned long long *count_lt = nullptr, *cell_min = nullptr, *cell_count = nullptr;
    TmpDev t_cnt, t_cmin, t_ccnt;
    ImpAccum(gpe_handle* h_, int maxno_, long long cell_pts_, long long ncell_)
        : h(h_), maxno(maxno_), cell_pts(ncell_ > 0 ? cell_pts_ : 0), ncell(cell_pts_ > 0 ? ncell_ : 0), t_cnt(h_), t_cmin(h_), t_ccnt(h_) {}
    // first_index: global flat index of the call's first point; keep: the call's mask on the device, or null
    ImpStats stats(double cm, long long first_index, unsigned char* keep) const {
        return ImpStats{cm, maxno, cell_pts, cell_pts > 0 ? first_index / cell_pts : 0, keep, count_lt, cell_min, cell_count};
    }
    int init() {
        CK(t_cnt.get(&count_lt, (size_t)maxno));
        CK(cudaMemsetAsync(count_lt, 0, sizeof(unsigned long long) * maxno, h->st));
        if (ncell > 0) {
            CK(t_cmin.get(&cell_min, (size_t)ncell * maxno));
            CK(t_ccnt.get(&cell_count, (size_t)ncell * maxno));
            // 0x7f in every byte is a large positive double: the minimum of a cell that holds no point of the call is +huge
            CK(cudaMemsetAsync(cell_min, 0x7f, sizeof(unsigned long long) * ncell * maxno, h->st));
            CK(cudaMemsetAsync(cell_count, 0, sizeof(unsigned long long) * ncell * maxno, h->st));
        }
        return 0;
    }
    int finish(unsigned long long* count_out, double* min_out, unsigned long long* cnt_out) {
        if (count_out) CK(cudaMemcpyAsync(count_out, count_lt, sizeof(unsigned long long) * maxno, cudaMemcpyDefault, h->st));
        if (ncell > 0 && min_out) CK(cudaMemcpyAsync(min_out, cell_min, sizeof(double) * ncell * maxno, cudaMemcpyDefault, h->st));
        if (ncell > 0 && cnt_out) CK(cudaMemcpyAsync(cnt_out, cell_count, sizeof(unsigned long long) * ncell * maxno, cudaMemcpyDefault, h->st));
        CK(cudaStreamSynchronize(h->st));
        CK(cudaGetLastError());
        return 0;
    }
};

// K4s sampled sensitivity (gpe_sens_sample).  A chunk of Mc samples is evaluated as the (nw + 2) Mc explicit points
// [A | B | AB_which[0] | ... ], Mc consecutive columns each; Z = L^-1 C of all of them is stored, and the posterior covariance of
// a pair of columns is formed from their dot product in Z.
constexpr int SS_MAXW = 16;
constexpr int SS_PG = 4;         // inputs per CTA of the pair-dot pass: A and B are read once per four AB_P columns

// P [(nw + 2) Mc][d]: column block 0 = A, 1 = B, 2 + k = A with input which[k] from B; samples >= cnt are zero rows
__global__ void sens_compose_kernel(const double* __restrict__ XA, const double* __restrict__ XB, long long cnt, int Mc, int d,
                                    const int* __restrict__ which, int nw, double* __restrict__ P) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= (long long)(nw + 2) * Mc) return;
    const int b = (int)(j / Mc), i = (int)(j % Mc);
    const int wk = b >= 2 ? which[b - 2] : -1;
    for (int k = 0; k < d; k++) {
        double v = 0.0;
        if (i < cnt) v = (b == 1 || k == wk) ? XB[(size_t)i * d + k] : XA[(size_t)i * d + k];
        P[j * d + k] = v;
    }
}

// Tile partials of the pair dots over the rows [128 t, 128 t + 128) of Z (live rows < n):
// part [t][3 + 3 nw][Mc] = |z_A|^2, |z_B|^2, z_A.z_B, then per input k |z_X|^2, z_B.z_X, z_A.z_X (X = AB_which[k]).
// One thread per sample: consecutive threads read consecutive columns of Z.  CTA z handles inputs [4z, 4z + 4).
__global__ void __launch_bounds__(128) sens_pairdot_kernel(const double* __restrict__ Z, int n, int Mc, int nw,
                                                           double* __restrict__ part) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    const int t = blockIdx.y, g0 = blockIdx.z * SS_PG;
    const int ng = min(SS_PG, nw - g0), E = 3 + 3 * nw;
    const size_t ld = (size_t)(nw + 2) * Mc;
    const double* za = Z + i;
    const double* zb = Z + Mc + i;
    const double* zx = Z + (size_t)(2 + g0) * Mc + i;
    double aa = 0.0, bb = 0.0, ab = 0.0, xx[SS_PG], bx[SS_PG], ax[SS_PG];
#pragma unroll
    for (int k = 0; k < SS_PG; k++) xx[k] = bx[k] = ax[k] = 0.0;
    const int r1 = min(n, t * 128 + 128);
#pragma unroll 2
    for (int r = t * 128; r < r1; r++) {
        const size_t o = (size_t)r * ld;
        const double a = za[o], b = zb[o];
        aa = fma(a, a, aa);
        bb = fma(b, b, bb);
        ab = fma(a, b, ab);
#pragma unroll
        for (int k = 0; k < SS_PG; k++) {
            if (k < ng) {
                const double x = zx[o + (size_t)k * Mc];
                xx[k] = fma(x, x, xx[k]);
                bx[k] = fma(b, x, bx[k]);
                ax[k] = fma(a, x, ax[k]);
            }
        }
    }
    double* pp = part + (size_t)t * E * Mc + i;
    if (blockIdx.z == 0) {
        pp[0] = aa;
        pp[(size_t)Mc] = bb;
        pp[(size_t)2 * Mc] = ab;
    }
#pragma unroll
    for (int k = 0; k < SS_PG; k++) {
        if (k < ng) {
            const size_t e = 3 + 3 * (size_t)(g0 + k);
            pp[e * Mc] = xx[k];
            pp[(e + 1) * Mc] = bx[k];
            pp[(e + 2) * Mc] = ax[k];
        }
    }
}

// One thread per sample: the estimator terms (t_E, t_V, t_EV, t_S[k], t_T[k]) from the pair dots, the regression vectors
// G [q][cols] (fullcov_finalize_kernel phase 0), the means and the prior of each pair; then the CTA's sums of the terms and of
// their squares, each over its 128 samples in index order, into bpart [blk0 + CTA][2][3 + 2 nw].  Samples >= cnt add zero.
template <int FAM>
__global__ void __launch_bounds__(128) sens_sample_finalize_kernel(const double* __restrict__ part, int ntile, const double* __restrict__ aux,
                                                                   const double* __restrict__ G, const double* __restrict__ P, BasisDesc bd,
                                                                   int d, const double* __restrict__ winv, const double* __restrict__ beta,
                                                                   const int* __restrict__ which, int nw, int Mc, long long cnt, double sigma2, double cscale,
                                                                   double astar, double shift, double* __restrict__ bpart, long long blk0) {
    extern __shared__ double terms[];        // [3 + 2 nw][128]
    __shared__ double bs[NR];
    const int q = bd.q, T = 3 + 2 * nw, E = 3 + 3 * nw;
    const size_t cols = (size_t)(nw + 2) * Mc;
    if (threadIdx.x < NR) bs[threadIdx.x] = beta[threadIdx.x];
    __syncthreads();
    const int i = blockIdx.x * 128 + threadIdx.x;
    auto psum = [&](int e) {                 // tile partials in row-tile order
        double s = 0.0;
        for (int t = 0; t < ntile; t++) s += part[((size_t)t * E + e) * Mc + i];
        return s;
    };
    auto mean = [&](size_t j) {              // as predict_finalize_kernel
        double mu = aux[(size_t)q * cols + j];
        for (int a = 0; a < q; a++) mu = fma(basis_value(nullptr, q, P, d, bd, (long long)j, a), bs[a], mu);
        return mu;
    };
    auto gdot = [&](size_t x, size_t y) {
        double s = 0.0;
        for (int a = 0; a < q; a++) s = fma(G[(size_t)a * cols + x], G[(size_t)a * cols + y], s);
        return s;
    };
    const size_t jA = i, jB = (size_t)Mc + i;
    const double* pa = P + jA * d;
    const double* pb = P + jB * d;
    double Dab = 0.0;
    for (int k = 0; k < d; k++) {
        const double df = (pa[k] - pb[k]) * winv[k];
        Dab = fma(df, df, Dab);
    }
    const double mA = mean(jA), mB = mean(jB);
    const double vA = sigma2 * (astar - psum(0) + gdot(jA, jA)), vB = sigma2 * (astar - psum(1) + gdot(jB, jB));
    const double cAB = sigma2 * (cov_prior<FAM>(cscale, Dab) - psum(2) + gdot(jA, jB));
    double* col = terms + threadIdx.x;
    col[0] = mA;
    col[128] = cAB;
    col[256] = 0.5 * ((mA - mB) * (mA - mB) + vA + vB - 2.0 * cAB);
    for (int k = 0; k < nw; k++) {
        const int w = which[k];
        const size_t jX = (size_t)(2 + k) * Mc + i;
        double Dbx = 0.0;                    // AB_w differs from B in every input but w, from A only in w
        for (int kk = 0; kk < d; kk++) {
            if (kk == w) continue;
            const double df = (pa[kk] - pb[kk]) * winv[kk];
            Dbx = fma(df, df, Dbx);
        }
        const double dfw = (pa[w] - pb[w]) * winv[w];
        const double mX = mean(jX);
        const double vX = sigma2 * (astar - psum(3 + 3 * k) + gdot(jX, jX));
        const double cBX = sigma2 * (cov_prior<FAM>(cscale, Dbx) - psum(4 + 3 * k) + gdot(jB, jX));
        const double cAX = sigma2 * (cov_prior<FAM>(cscale, dfw * dfw) - psum(5 + 3 * k) + gdot(jA, jX));
        col[(3 + k) * 128] = (mB - shift) * (mX - mA) + cBX - cAB;
        col[(3 + nw + k) * 128] = 0.5 * ((mA - mX) * (mA - mX) + vA + vX - 2.0 * cAX);
    }
    if (i >= cnt)
        for (int t = 0; t < T; t++) col[t * 128] = 0.0;
    __syncthreads();
    for (int e = threadIdx.x; e < 2 * T; e += 128) {
        const double* tv = terms + (e < T ? e : e - T) * 128;
        double s = 0.0;
        for (int r = 0; r < 128; r++) s = (e < T) ? s + tv[r] : fma(tv[r], tv[r], s);
        bpart[(size_t)(blk0 + blockIdx.x) * 2 * T + e] = s;
    }
}

// sums [w] = sum over the CTA partials bpart [nblk][w], in CTA order
__global__ void sens_sample_reduce_kernel(const double* __restrict__ bpart, long long nblk, int w, double* __restrict__ sums) {
    const int e = threadIdx.x;
    if (e >= w) return;
    double s = 0.0;
    for (long long b = 0; b < nblk; b++) s += bpart[(size_t)b * w + e];
    sums[e] = s;
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
    if ((rc = gpe_upload_single_par(h, delta, nugget, kind, 1, r_div > 0 ? r_div : 1.0))) return rc;
    if (!h->fLi) {
        CK(dev_alloc(&h->fLi, (size_t)np * np));
        CK(dev_alloc(&h->fE, (size_t)np * NR));
        CK(dev_alloc(&h->fK, (size_t)NR * NR));
        CK(dev_alloc(&h->fbeta, (size_t)NR));
        CK(dev_alloc(&h->fwinv, (size_t)h->d));
        CK(dev_alloc(&h->fXs, (size_t)h->d * np));
    }
    std::vector<double> bin;
    double* bov = nullptr;
    if (beta_in) {
        CK(read_small(bin, beta_in, q));
        bin.resize(NR, 0.0);
        CK(cudaMemcpyAsync(h->fbeta, bin.data(), sizeof(double) * NR, cudaMemcpyHostToDevice, h->st));
        bov = h->fbeta;
    }
    CK(launch_cov_build(h->X, h->r, h->n, h->d, np, h->par, h->winv, h->A, 0, 1, 0, h->st, 0, 0, nullptr, h->family));
    h->launches++;
    CK(cudaMemsetAsync(h->fK, 0, sizeof(double) * NR * NR, h->st));
    CK(cudaMemsetAsync(h->status, 0, sizeof(int), h->st));
    SubBatch sb{0, 1, h->st};
    if ((rc = gpe_factor_and_reduce(h, sb, 0, GRAD_NONE, bov, h->fK))) return rc;
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
    for (int a = 0; a < NR; a++) h->fit_dbeta[a] = beta_in ? bopt[a] - bin[a] : 0.0;
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
    int rc;
    if ((rc = check_fit(h, Hs != nullptr))) return rc;
    NvtxRange nvtx(grid ? "gpe_predict_grid" : "gpe_predict");
    CK(cudaSetDevice(h->device));
    long long chunk = std::min<long long>(default_chunk(h), (m + 127) / 128 * 128);
    if ((rc = ensure_predict_ws(h, chunk))) return rc;
    const bool x_dev = Xs && gpe_is_device_ptr(Xs), h_dev = Hs && gpe_is_device_ptr(Hs);
    const bool mean_dev = imp_call || gpe_is_device_ptr(mean), var_dev = var && gpe_is_device_ptr(var);
    const int d = h->d, q = h->q;
    // tensor grid: tabulate the one-dimensional kernel factors once (the direct kernel when the tables do not fit)
    GridXcov gx;
    bool use_sep = false;
    TmpDev t_tab(h);
    if (grid) {
        int ltot = 0;
        if (plan_grid_sep(*grid, gx.sp, gx.smem, ltot)) {
            double* T = nullptr;
            CK(t_tab.get(&T, (size_t)ltot * h->npad));
            const long long tot = (long long)ltot * h->npad;
            with_family(h->family, [&](auto fam) {
                grid_table_kernel<fam><<<(unsigned)((tot + 255) / 256), 256, 0, h->st>>>(h->fXs, h->fwinv, *grid, gx.sp, h->npad, ltot, T);
            });
            h->launches++;
            gx.T = T;
            use_sep = true;
        }
    }
    rc = for_chunks(h, (m + chunk - 1) / chunk, [&](long long ci, int k, cudaStream_t st) {
        gpe_handle::PredSlot& sl = h->ps[k];
        const long long s = ci * chunk, cnt = std::min(chunk, m - s);
        const int mc = (int)((cnt + 127) / 128 * 128);
        const double* P = nullptr;
        if (grid) {
            grid_points_kernel<<<(mc + 255) / 256, 256, 0, st>>>(*grid, start + s, cnt, mc, sl.X);
            h->launches++;
            P = sl.X;
        } else if (x_dev && cnt == mc) {
            P = Xs + (size_t)s * d;
        } else {
            CK(stage_points(sl.X, Xs + (size_t)s * d, cnt, mc, d, st));
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
            ic.Itop += (size_t)s * ic.st.maxno;
            if (ic.st.keep) ic.st.keep += s;
            ic.first_index += s;
        }
        if ((rc = predict_chunk(h, sl, st, P, Hc, cnt, mc, mo, vo, use_sep ? &gx : nullptr, imp_call ? &ic : nullptr))) return rc;
        if (!mean_dev) CK(cudaMemcpyAsync(mean + s, sl.Mean, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (var && !var_dev) CK(cudaMemcpyAsync(var + s, sl.Var, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
        return 0;
    });
    if (rc) return rc;
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
    GridDesc g;
    if (int rc = make_grid(h, levels, lo, hi, g)) return rc;
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
    int rc;
    if ((rc = check_cells(h, cell_pts, first_index, ncell, last ? m : 0))) return rc;
    NvtxRange nvtx("gpe_predict_implaus");
    CK(cudaSetDevice(h->device));
    TmpDev t_top(h);
    double* top = Itop;
    if (!Itop) CK(t_top.get(&top, (size_t)std::max<long long>(m, 1) * maxno));      // first == last: a one-emulator job
    DevOut<unsigned char> ko(h);
    ImpAccum acc(h, maxno, cell_pts, ncell);
    if (last) {
        CK(ko.stage(keep, (size_t)m));
        if ((rc = acc.init())) return rc;
    }
    const ImpFuse ic{.z = z, .ve = var_extra, .first = first != 0, .last = last != 0, .Itop = top, .store_top = Itop != nullptr,
                     .first_index = first_index, .st = acc.stats(cm, first_index, ko.p)};
    if (m > 0) {
        if (Xs) {
            rc = predict_common(h, Xs, Hs, nullptr, 0, m, nullptr, nullptr, &ic);
        } else {
            GridDesc g;
            if ((rc = make_grid(h, levels, lo, hi, g))) return rc;
            rc = predict_common(h, nullptr, nullptr, &g, start, m, nullptr, nullptr, &ic);
        }
        if (rc) return rc;
    }
    if (!last) return 0;
    CK(ko.flush());
    return acc.finish(count_lt, cell_min, cell_count);
}

int gpe_cross_cov(gpe_handle* h, const double* delta, double nugget, int kind, const double* Xs, int m, double* C_out) {
    if (h && m == 0) return 0;
    if (!h || !h->n || !delta || !Xs || !C_out || m < 1) return h ? h->fail_msg("bad argument") : -2;
    NvtxRange nvtx("gpe_cross_cov");
    CK(cudaSetDevice(h->device));
    const int np = h->npad, d = h->d;
    int mc = (m + 127) / 128 * 128;
    std::vector<double> w;
    CK(read_small(w, delta, d));
    for (double& v : w) v = 1.0 / v;
    double *wd = nullptr, *xs = nullptr, *P = nullptr, *Cm = nullptr;
    TmpDev t_wd(h), t_xs(h), t_P(h), t_Cm(h);
    CK(t_wd.get(&wd, (size_t)d));
    CK(t_xs.get(&xs, (size_t)d * np));
    CK(t_P.get(&P, (size_t)mc * d));
    CK(t_Cm.get(&Cm, (size_t)np * mc));
    CK(cudaMemcpyAsync(wd, w.data(), sizeof(double) * d, cudaMemcpyHostToDevice, h->st));
    CK(stage_points(P, Xs, m, mc, d, h->st));
    scale_train_kernel<<<(d * np + 255) / 256, 256, 0, h->st>>>(h->X, wd, h->n, d, np, xs);
    CK(launch_xcov<false>(h->family, xs, P, wd, h->n, d, np, mc, m, kind ? 1.0 : 1.0 - nugget, Cm, mc, h->st));
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
    int rc;
    if ((rc = check_fit(h, Hs != nullptr))) return rc;
    NvtxRange nvtx("gpe_predict_fullcov");
    CK(cudaSetDevice(h->device));
    const int np = h->npad, d = h->d, q = h->q;
    const int mp = (m + 127) / 128 * 128;
    double *P = nullptr, *Cm = nullptr, *Zm = nullptr, *ZtZ = nullptr, *aux = nullptr, *G = nullptr;
    TmpDev t_P(h), t_Cm(h), t_Zm(h), t_ZtZ(h), t_aux(h), t_G(h);
    DevIn<double> Hd(h), rn(h);
    DevOut<double> md(h), Vd(h);
    CK(t_P.get(&P, (size_t)mp * d));
    CK(t_Cm.get(&Cm, (size_t)np * mp));
    CK(t_Zm.get(&Zm, (size_t)np * mp));
    CK(t_ZtZ.get(&ZtZ, (size_t)mp * mp));
    CK(t_aux.get(&aux, (size_t)NR * mp));
    CK(t_G.get(&G, (size_t)NR * mp));
    CK(md.stage(mean, (size_t)m));
    CK(Vd.stage(V, (size_t)m * m));
    CK(stage_points(P, Xs, m, mp, d, h->st));
    CK(Hd.stage(Hs, (size_t)m * q));
    CK(rn.stage(r_new, (size_t)m));
    rc = posterior_cross(h, h->st, P, nullptr, mp, m, Cm, aux);
    if (!rc)
        rc = gpe_gemm(h, h->st, {.A = h->fLi, .B = Cm, .C = Zm, .lda = np, .ldb = mp, .ldc = mp, .M = np, .N = mp, .K = np, .kmode = KM_LE_I},
                      GEMM_NN);
    if (!rc) rc = gpe_gemm(h, h->st, {.A = Zm, .B = Zm, .C = ZtZ, .lda = mp, .ldb = mp, .ldc = mp, .M = mp, .N = mp, .K = np}, GEMM_TN);
    if (!rc) {
        BasisDesc bd = basis_of(h);
        double s2 = h->fit_sigma * h->fit_sigma;
        // mean via the diagonal finalize (var == nullptr)
        predict_finalize_kernel<false><<<(m + 127) / 128, 128, 0, h->st>>>(nullptr, 0, aux, mp, P, Hd.p, bd, d, h->fK, h->fbeta, s2,
                                                                            h->fit_astar, m, md.p, nullptr, ImpFuse{});
        const size_t tot = (size_t)m * m;
        with_family(h->family, [&](auto fam) {
            fullcov_finalize_kernel<fam><<<(m + 127) / 128, 128, 0, h->st>>>(ZtZ, mp, aux, mp, P, Hd.p, bd, d, h->fwinv, h->fK, s2, h->fit_c,
                                                                             h->fit_astar, rn.p, m, G, Vd.p, 0);
            fullcov_finalize_kernel<fam><<<(unsigned)((tot + 255) / 256), 256, 0, h->st>>>(ZtZ, mp, aux, mp, P, Hd.p, bd, d, h->fwinv, h->fK, s2,
                                                                                          h->fit_c, h->fit_astar, rn.p, m, G, Vd.p, 1);
        });
        h->launches += 3;
        CK(md.flush());
        CK(Vd.flush());
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
    if (int rc = check_cells(h, cell_pts, first_index, ncell, m)) return rc;
    NvtxRange nvtx("gpe_implausibility");
    CK(cudaSetDevice(h->device));
    ImpDesc ds;
    ds.n_emul = n_emul;
    std::vector<double> zz, vv;
    CK(read_small(zz, z, n_emul));
    CK(read_small(vv, var_extra, n_emul));
    for (int o = 0; o < n_emul; o++) { ds.z[o] = zz[o]; ds.ve[o] = vv[o]; }
    DevIn<double> md(h), vd(h);
    DevOut<double> Io(h);
    DevOut<unsigned char> ko(h);
    ImpAccum acc(h, maxno, cell_pts, ncell);
    CK(md.stage(mean, (size_t)n_emul * m));
    CK(vd.stage(var, (size_t)n_emul * m));
    CK(Io.stage(Imax, (size_t)m * maxno));
    CK(ko.stage(keep, (size_t)m));
    if (int rc = acc.init()) return rc;
    if (m > 0) {                                                 // m == 0: zero counts, +huge cell minima
        implaus_kernel<<<(unsigned)((m + 255) / 256), 256, 0, h->st>>>(md.p, vd.p, m, ds, first_index, Io.p, acc.stats(cm, first_index, ko.p));
        h->launches++;
    }
    CK(Io.flush());
    CK(ko.flush());
    return acc.finish(count_lt, cell_min, cell_count);
}

int gpe_sens_sample(gpe_handle* h, const double* XA, const double* XB, long long M, const int* which, int nw, double shift,
                    double* sums) {
    if (h && M == 0) return 0;
    if (!h || !XA || !XB || !which || !sums || M < 0) return h ? h->fail_msg("bad argument") : -2;
    if (nw < 1 || nw > SS_MAXW) return h->fail_msg("gpe_sens_sample takes 1 <= nw <= 16 inputs");
    int rc;
    if ((rc = check_fit(h, false))) return rc;
    NvtxRange nvtx("gpe_sens_sample");
    CK(cudaSetDevice(h->device));
    std::vector<int> wv;
    CK(read_small(wv, which, (size_t)nw));
    for (int k = 0; k < nw; k++) {
        if (wv[k] < 0 || wv[k] >= h->d) return h->fail_msg("which: every input must lie in [0, d)");
        for (int k2 = 0; k2 < k; k2++)
            if (wv[k2] == wv[k]) return h->fail_msg("which: the inputs must be distinct");
    }
    const int np = h->npad, d = h->d, q = h->q, nb = nw + 2, T = 3 + 2 * nw, E = 3 + 3 * nw;
    // samples per chunk: a multiple of 256 (the INT8 route's column tile) with the chunk's nb Mc columns at most the prediction
    // chunk, but never fewer than 256
    const long long Mc = std::min<long long>(std::max<long long>(256, default_chunk(h) / nb / 256 * 256), (M + 255) / 256 * 256);
    const int cols = (int)(nb * Mc);
    const int ntile = (h->n + 127) / 128;
    const long long nchunk = (M + Mc - 1) / Mc, nblk = nchunk * (Mc / 128);
    if ((rc = ensure_predict_ws(h, cols))) return rc;
    DevIn<double> xa(h), xb(h);
    DevIn<int> wd(h);
    DevOut<double> so(h);
    CK(xa.stage(XA, (size_t)M * d));
    CK(xb.stage(XB, (size_t)M * d));
    CK(wd.stage(which, (size_t)nw));
    CK(so.stage(sums, (size_t)2 * T));
    TmpDev t_z[2] = {TmpDev(h), TmpDev(h)}, t_g[2] = {TmpDev(h), TmpDev(h)}, t_part[2] = {TmpDev(h), TmpDev(h)};
    TmpDev t_bp(h);
    double *Zs[2] = {nullptr, nullptr}, *Gs[2] = {nullptr, nullptr}, *Parts[2] = {nullptr, nullptr}, *bpart = nullptr;
    for (int k = 0; k < chunk_slots(h, nchunk); k++) {
        CK(t_z[k].get(&Zs[k], (size_t)np * cols));
        CK(t_g[k].get(&Gs[k], (size_t)q * cols));
        CK(t_part[k].get(&Parts[k], (size_t)ntile * E * Mc));
    }
    CK(t_bp.get(&bpart, (size_t)nblk * 2 * T));
    const BasisDesc bd = basis_of(h);
    const double s2 = h->fit_sigma * h->fit_sigma;
    rc = for_chunks(h, nchunk, [&](long long ci, int k, cudaStream_t st) {
        gpe_handle::PredSlot& sl = h->ps[k];
        const long long s = ci * Mc, cnt = std::min(Mc, M - s);
        {
            ProfScope ps(h, gpe_handle::CAT_OTHER, st);
            sens_compose_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, st>>>(xa.p + (size_t)s * d, xb.p + (size_t)s * d, cnt, (int)Mc,
                                                                               d, wd.p, nw, sl.X);
        }
        h->launches++;
        if ((rc = posterior_cross(h, st, sl.X, nullptr, cols, cols, sl.C, sl.Aux))) return rc;
        if ((rc = fit_z_product(h, st, sl.C, cols, Zs[k], EPI_STORE))) return rc;
        {
            ProfScope ps(h, gpe_handle::CAT_OTHER, st);
            sens_pairdot_kernel<<<dim3((unsigned)(Mc / 128), ntile, (nw + SS_PG - 1) / SS_PG), 128, 0, st>>>(Zs[k], h->n, (int)Mc, nw, Parts[k]);
            fullcov_finalize_kernel<FAMILY_GAUSSIAN><<<(unsigned)((cols + 127) / 128), 128, 0, st>>>(
                nullptr, cols, sl.Aux, cols, sl.X, nullptr, bd, d, h->fwinv, h->fK, s2, h->fit_c, h->fit_astar, nullptr, cols, Gs[k], nullptr, 0);
            with_family(h->family, [&](auto fam) {
                sens_sample_finalize_kernel<fam><<<(unsigned)(Mc / 128), 128, (size_t)T * 128 * sizeof(double), st>>>(
                    Parts[k], ntile, sl.Aux, Gs[k], sl.X, bd, d, h->fwinv, h->fbeta, wd.p, nw, (int)Mc, cnt, s2, h->fit_c, h->fit_astar, shift,
                    bpart, ci * (Mc / 128));
            });
        }
        h->launches += 3;
        return 0;
    });
    if (rc) return rc;
    {
        ProfScope ps(h, gpe_handle::CAT_OTHER, h->st);
        sens_sample_reduce_kernel<<<1, 128, 0, h->st>>>(bpart, nblk, 2 * T, so.p);
    }
    h->launches++;
    CK(so.flush());
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

int gpe_predict_grad(gpe_handle* h, const double* Xs, long long m, double* dmean, double* dvar) {
    if (h && m == 0) return 0;
    if (!h || !Xs || !dmean || m < 0) return h ? h->fail_msg("gpe_predict_grad: Xs and dmean are required and m must be >= 0") : -2;
    int rc;
    if ((rc = check_fit(h, false))) return rc;
    NvtxRange nvtx("gpe_predict_grad");
    CK(cudaSetDevice(h->device));
    const int d = h->d;
    // points per chunk: a multiple of 256 (the INT8 route's column tile) with the chunk's d Mc columns at most the prediction
    // chunk, but never fewer than 256 (the rule of gpe_sens_sample)
    const long long Mc = std::min<long long>(std::max<long long>(256, default_chunk(h) / d / 256 * 256), (m + 255) / 256 * 256);
    const int cols = (int)(d * Mc);
    if ((rc = ensure_predict_ws(h, cols))) return rc;
    const bool x_dev = gpe_is_device_ptr(Xs), mean_dev = gpe_is_device_ptr(dmean), var_dev = dvar && gpe_is_device_ptr(dvar);
    const BasisDesc bd = basis_of(h);
    const double s2 = h->fit_sigma * h->fit_sigma;
    const double kappa = with_family(h->family, [](auto fam) { return FAMILY_KAPPA<fam>; });
    rc = for_chunks(h, (m + Mc - 1) / Mc, [&](long long ci, int k, cudaStream_t st) {
        gpe_handle::PredSlot& sl = h->ps[k];
        const long long s = ci * Mc, cnt = std::min(Mc, m - s);
        const double* P = sl.X;
        if (x_dev && cnt == Mc) P = Xs + (size_t)s * d;
        else CK(stage_points(sl.X, Xs + (size_t)s * d, cnt, (int)Mc, d, st));
        {
            ProfScope ps(h, gpe_handle::CAT_COV, st);
            CK(launch_xcov<true>(h->family, h->fXs, P, h->fwinv, h->n, d, h->npad, (int)Mc, cnt, h->fit_c, sl.C, cols, st));
        }
        h->launches++;
        int ntile = 0;
        if ((rc = posterior_aux(h, st, sl.C, cols, sl.Aux))) return rc;
        if (dvar != nullptr && (rc = fit_z_product(h, st, sl.C, cols, sl.Part, EPI_SUMSQ, &ntile))) return rc;
        double* mo = mean_dev ? dmean + (size_t)s * d : sl.Mean;
        double* vo = dvar ? (var_dev ? dvar + (size_t)s * d : sl.Var) : nullptr;
        {
            ProfScope ps(h, gpe_handle::CAT_OTHER, st);
            predict_grad_finalize_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, st>>>(sl.Part, ntile, sl.Aux, (int)Mc, P, bd, d, h->fwinv,
                                                                                         h->fK, h->fbeta, s2, h->fit_c * kappa, cnt, mo, vo);
        }
        h->launches++;
        if (!mean_dev) CK(cudaMemcpyAsync(dmean + (size_t)s * d, sl.Mean, (size_t)cnt * d * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (dvar && !var_dev) CK(cudaMemcpyAsync(dvar + (size_t)s * d, sl.Var, (size_t)cnt * d * sizeof(double), cudaMemcpyDeviceToHost, st));
        return 0;
    });
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

}  // extern "C"
