// Non-GEMM kernels of the hot path: covariance build (K1), leaf Cholesky+inverse (K2 panels),
// GLS/log-likelihood reductions (K3), fused gradient reduction (K1g), prediction pieces (K4),
// implausibility (K5).  Declarations only; definitions in gpe_kernels.cu / gpe_predict.cu.
#pragma once
#include "gpe_common.cuh"

namespace gpe {

constexpr int NR = 32;        // padded width of the skinny [H | y] panels (q + 1 <= NR)
constexpr int GRAM_SLAB = 128;   // rows per Gram partial (= NB: npad is a multiple); fixed, so sums do not depend on the batch

// Per batch item covariance parameters, built on device from the transformed theta.
struct ItemPar {
    double offs;    // off-diagonal scale  s2_A * c,  c = (1 - nugget) [kernel] or 1 [alt]
    double diagv;   // diagonal without r
    double radd;    // diagonal += radd * r_i
    double s2A;     // sigma^2 folded into A (1 for mucm)
    double c;       // (1 - nugget) or 1
    double nugget;
    double sigma;   // gp4ml: sigma from theta; mucm: filled with sigma_hat by finalize
    double pad_;
};

// Per item scalars produced by llh_finalize_kernel.
struct ItemOut {
    double llh, sig2, f, s2g, logdetA, logdetQ, quad, pad_;
};

// theta [B,p] -> ItemPar[B], winv [B,d] = 1/delta  (kernel.untransform + set_params)
void launch_prep_theta(const double* theta, int B, int p, int d, int mode, double fixed_nugget,
                       ItemPar* par, double* winv, cudaStream_t st);

// K1: A[b] (ld = npad, batch stride sA) from X [n,d]; lower 64x64 tiles only unless full.
// Eout (optional, gmode 0 only): a second matrix per item that receives exp(-D_ij) itself, same tiles and strides as A --
// the factorisation overwrites A, the fused gradient epilogue reads this copy instead of recomputing the exponentials.
cudaError_t launch_cov_build(const double* X, const double* r, int n, int d, int npad, const ItemPar* par,
                             const double* winv, double* A, long long sA, int B, int full, cudaStream_t st,
                             int gmode = 0, int gdim = 0, double* Eout = nullptr, int family = FAMILY_GAUSSIAN);
// (family FAMILY_MATERN52: the entries are R(D) -- G(D) Delta^2 for gmode 1 -- and Eout is ignored)

// copy the n x n top-left of a padded matrix into a dense [n,n] output, mirroring the lower triangle
void launch_unpad_sym(const double* A, int npad, int n, double* out, int mirror, cudaStream_t st);

// identity-padded copies of `batch` dense [n,n] matrices -> [npad,npad], and the lower triangle (zeros above the
// diagonal) of padded matrices back to dense [n,n]  (gpe_potrf: np.linalg.cholesky call sites)
void launch_pad_sym(const double* src, int n, int npad, double* dst, int batch, cudaStream_t st);
void launch_unpad_lower(const double* src, int npad, int n, double* dst, int batch, cudaStream_t st);

// K2 leaf: Cholesky + triangular inverse of the 128x128 diagonal block at `off`.
void launch_leaf(const double* A, double* Linv, int ld, long long sA, long long sL, int off,
                 double* logdet_part, int nleaf, int* status, int B, cudaStream_t st, double* Lfac = nullptr);

// [H | y | 0] -> padded panel HY [npad, NR] (shared by all batch items)
void launch_build_hy(const double* H, const double* y, int n, int q, int npad, double* HY, cudaStream_t st);

// Gram partials of the skinny panel Wy [B, npad, NR]: GP [B, nslab, NR*NR]
void launch_gram(const double* Wy, int npad, int B, double* GP, cudaStream_t st);

// GLS mean, log-likelihood scalars, and the panel Z = [w K^-T | sqrt(f) z].
void launch_llh_finalize(const double* Wy, const double* GP, const double* logdet_part, int nleaf,
                         int n, int q, int npad, int mode, ItemPar* par, ItemOut* out, double* beta,
                         double* Z, int* status, int B, const double* beta_override, double* Kout, cudaStream_t st);

// K1g: per-tile partial sums of  W_ij E_ij Delta_k^2, W_ij E_ij, W_ii, W_ii r_i  (Matérn: W_ij G_ij Delta_k^2, W_ij R_ij, ..).
void launch_grad_partial(const double* X, const double* r, int n, int d, int npad, const double* winv,
                         const double* Ainv, long long sAinv, const double* U, int nu, double* part,
                         int B, cudaStream_t st, const double* E = nullptr, int family = FAMILY_GAUSSIAN);
void launch_grad_finalize(const double* part, int ntile, int n, int d, int npad, int p, int mode, const ItemPar* par,
                          const ItemOut* out, const int* status, double* llh, double* grad,
                          double* sigma_hat, int B, cudaStream_t st);

// K3 + K1g fused: LAUUM (A^-1 = L^-T L^-1) whose 128x128 tiles of W = A^-1 - U U^T stay in registers and are reduced to
// the gradient partials in the epilogue (gpe_lauum_grad.cu).  U [B][np][NR] in; Ut / nUt [B][NR][np] scratch (U^T, -U^T);
// part [B][lauum_grad_ntiles(np)][d + 3] out.  A^-1 is not stored.
bool lauum_grad_supported(int d);
int lauum_grad_ntiles(int npad);
cudaError_t launch_lauum_grad(const double* Li, long long sL, int np, int n, int d, int nu, const double* U, double* Ut, double* nUt,
                              const double* X, const double* r, const double* winv, const double* E, long long sE, double* part,
                              int B, cudaStream_t st, double* Wout = nullptr);
// Wout != nullptr: the same launch with a plain store epilogue -- the lower 128x128 tiles of W = A^-1 - U U^T go to Wout
// (strides as Li) and the reduction is left to launch_grad_partial_we.
cudaError_t launch_grad_partial_we(const double* X, const double* r, int n, int d, int npad, const double* winv, const double* W,
                                   const double* E, long long sM, double* part, int B, cudaStream_t st);

inline int grad_ntiles(int npad) { int t = npad / 64; return t * (t + 1) / 2; }
inline int grad_nvals(int d) { return d + 3; }

}  // namespace gpe
