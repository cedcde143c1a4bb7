/* gpe_b200.h -- C-ABI of the B200-native dense-GP hot path of GP_emu_UQSA.
 *
 * The reference (MathThyMod/GP_emu_UQSA, pure Python) has no FFI: its hot path sits behind
 * the Python object protocol of _emulatorkernels.py / _emulatoroptimise.py /
 * _emulatorclasses.py.  Each entry point below names the reference call site(s) it replaces
 * (file:line relative to gp_emu_uqsa/ in the reference tree); INTEGRATION.md shows the ctypes
 * binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - plain pointers and sizes only; every data pointer may be HOST or DEVICE memory (the
 *    library inspects it with cudaPointerGetAttributes and stages host buffers itself);
 *  - all matrices are row-major float64; all arithmetic is IEEE float64;
 *  - return 0 on success, negative on CUDA/argument error (text via gpe_last_error);
 *    a numerically failed item (non positive-definite covariance, the reference's
 *    LinAlgError -> None path, _emulatoroptimise.py:374-376, :489-491) is reported only
 *    through status[] (index+1 of the first non-positive pivot), never as an error code;
 *  - a unit count of zero (no guesses, no prediction points, an empty grid shard) is a successful
 *    no-op that touches no output, so an empty rank of a partitioned job needs no special case;
 *  - one handle per device per process; a handle is not thread-safe; calls are synchronous
 *    with respect to the returned host-visible results;
 *  - there is NO CPU fallback: every entry point fails if no sm_100 device is present;
 *  - the covariance function is the reference's Gaussian exp(-sum((x_i-x_j)/delta)^2) unless
 *    gpe_set_kernel selects the Matern 5/2 family for the handle (everything else -- nugget forms,
 *    mode bits, likelihoods, posterior formulas -- is shared by both families).
 */
#ifndef GPE_B200_H
#define GPE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpe_handle gpe_handle;

/* mode bits for gpe_llh_grad_batch / gpe_fit_state */
#define GPE_MODE_MUCM 1        /* beliefs.mucm == 'T'      (loglikelihood_mucm)              */
#define GPE_MODE_ALT_NUGGET 2  /* beliefs.alt_nugget == 'T' (kernel_alt_nug)                  */
#define GPE_MODE_NUGGET_FREE 4 /* beliefs.fix_nugget == 'F' (nugget is an optimised parameter) */

/* covariance families for gpe_set_kernel.  With D_ij = sum_k ((x_ik - x_jk) / delta_k)^2 and r = sqrt(D):
 * GAUSSIAN  exp(-D) (the reference's kernel / kernel_alt_nug);
 * MATERN52  (1 + sqrt5 r + 5D/3) exp(-sqrt5 r), Matérn with smoothness 5/2 in the same scaled distance.
 * The nugget / alt-nugget forms (argument `kind` below) and the diagonals are the same for both. */
#define GPE_KERNEL_GAUSSIAN 0
#define GPE_KERNEL_MATERN52 1

int gpe_version(void);
int gpe_create(int device, gpe_handle** out);
int gpe_destroy(gpe_handle* h);
const char* gpe_last_error(gpe_handle* h);
/* number of kernels this library has launched on the handle since creation */
long long gpe_launch_count(gpe_handle* h);

/* The CUDA stream (cudaStream_t) every kernel of this handle is launched on: record CUDA
 * events on it to time the path on the device. */
void* gpe_get_stream(gpe_handle* h);
/* The multistart batch of gpe_llh_grad_batch is split into `nstreams` contiguous groups that run
 * concurrently on their own CUDA streams (default 8, or GPE_STREAMS; 1 = strictly serial launches,
 * which is what per-kernel timing with gpe_profile_* should be read under). */
int gpe_set_streams(gpe_handle* h, int nstreams);

/* Asynchronous mode (off by default).  When on, gpe_llh_grad_batch, gpe_predict and gpe_predict_grid return as soon as
 * their work is enqueued on the handle's stream PROVIDED every input and output pointer of the call is device memory;
 * calls with a host pointer stay synchronous.  gpe_synchronize waits for the handle's stream.  This is what lets one
 * host thread keep several handles busy (the emulators of a history-matching job, history_match.py:96-118) or order
 * its own kernels after a call with events on gpe_get_stream. */
/* Covariance family of the emulator this handle holds (GPE_KERNEL_*; Gaussian by default).  It applies to
 * gpe_cov_build, gpe_cov_grad, gpe_cross_cov, gpe_llh_grad_batch, gpe_fit_state, gpe_predict* and gpe_predict_implaus.
 * A change clears the fit state (gpe_fit_state must run again) and the captured likelihood graphs.  With MATERN52,
 * gpe_sens_contract and gpe_sens_main_effect fail: their closed-form integrals exist for the Gaussian only. */
int gpe_set_kernel(gpe_handle* h, int family);

int gpe_set_async(gpe_handle* h, int on);
int gpe_synchronize(gpe_handle* h);

/* Optional per-launch CUDA-event timing by kernel category (measurement only; the reference's
 * unused @timeit helper, _emulatoroptimise.py:8-17, is the nearest analogue).  ms/count: 10 entries:
 * 0 DMMA GEMM (128-wide tiles; SYRK/TRMM updates of the factorisation and the prediction TRMM),
 * 1 small/skinny GEMM, 2 Cholesky leaf, 3 covariance build, 4 gradient reduction, 5 other,
 * 6 LAUUM (A^-1 = L^-T L^-1) on the DMMA route, 7 / 8 / 9 the INT8 tensor-core route of the large products
 * (csrc/gpe_ozaki.cuh): residue conversion, residue GEMM (tcgen05.mma kind::i8), CRT recombination. */
int gpe_profile_enable(gpe_handle* h, int on);
int gpe_profile_read(gpe_handle* h, double* ms, long long* count, int reset);

/* Training set of one emulator: Data.inputs/outputs/H/r (_emulatorclasses.py:539-584).
 * X [n,d] scaled inputs, y [n], H [n,q] (Data.make_H :558-566), r [n] or NULL (set_r :577-584). */
int gpe_set_training(gpe_handle* h, const double* X, const double* y, const double* H,
                     const double* r, int n, int d, int q);

/* Polynomial mean basis evaluated on device for new points (Basis/make_H,
 * _emulatorclasses.py:263-299, :558-566): column 0 is 1, column j is x[idx[j-1]]^pow[j-1].
 * Needed only when prediction points are not accompanied by an explicit H*. */
int gpe_set_basis(gpe_handle* h, const int* idx, const int* pow, int q);

/* kernel.var / kernel_alt_nug.var + Data.make_A (_emulatorkernels.py:39-50, :112-123;
 * _emulatorclasses.py:572-575): A_out [n,n] = K(X,X) with the nugget/r diagonal.
 * kind 0 = kernel, 1 = kernel_alt_nug; predict as in var(); s2 divides r (alt nugget). */
int gpe_cov_build(gpe_handle* h, const double* delta, double nugget, int kind, int predict,
                  double s2, double* A_out);

/* kernel.grad_delta_A / grad_nugget_A (_emulatorkernels.py:53-71, :126-144) as dense [n,n]
 * matrices, for callers that want them explicitly (the likelihood path never forms them):
 * which = delta index, or -1 for the nugget.  s2 as in the reference's argument. */
int gpe_cov_grad(gpe_handle* h, const double* delta, double nugget, int kind, int which, double s2,
                 double* G_out);

/* kernel.covar (_emulatorkernels.py:75-79, :148-152): C_out [n,m] = K(X, Xs). */
int gpe_cross_cov(gpe_handle* h, const double* delta, double nugget, int kind,
                  const double* Xs, int m, double* C_out);

/* Optimize.loglikelihood_mucm / loglikelihood_gp4ml (_emulatoroptimise.py:305-378, :412-493)
 * for B transformed parameter vectors at once (the multistart batch of Optimize.optimal,
 * :227-247).  theta [B,p] with p = d (+1 nugget) (+1 sigma), ordered [delta.., nugget?, sigma?].
 * Outputs: llh [B] (the minimised value), grad [B,p], sigma_hat [B] (mucm: analytic sigma,
 * :324-327; gp4ml: sigma from theta), status [B]. */
int gpe_llh_grad_batch(gpe_handle* h, const double* theta, int B, int p, int mode,
                       double fixed_nugget, double* llh, double* grad, double* sigma_hat,
                       int* status);

/* Factor once for fixed hyper-parameters and cache the state prediction needs
 * (Data.remake + Optimize.optimalbeta + Optimize.sigma_analytic_mucm,
 * _emulatorclasses.py:553-555, _emulatoroptimise.py:382-408, :497-504).
 * The matrix factored is the one training.remake() leaves: correlation matrix (s2 = 1) plus
 * r / r_div for the alt nugget (r_div = 1 after remake(); = sigma^2 after Optimize.optimal's
 * make_A(s2), :289).  beta_in NULL -> beta = optimalbeta(); else used as given.
 * Outputs (any may be NULL): beta_out [q], sigma_mucm_out (analytic MUCM sigma), status. */
int gpe_fit_state(gpe_handle* h, const double* delta, double nugget, double sigma, int kind,
                  double r_div, const double* beta_in, double* beta_out, double* sigma_mucm_out,
                  int* status);

/* Posterior mean and diagonal variance (Posterior.make_covar/make_mean/make_var,
 * _emulatorclasses.py:607-631, diagonal as consumed at history_match.py:117-118,
 * _emulatorplotting.py:51) for m explicit points Xs [m,d]; Hs [m,q] or NULL (device basis).
 * var may be NULL (mean only). */
int gpe_predict(gpe_handle* h, const double* Xs, const double* Hs, long long m, double* mean,
                double* var);

/* Same over a tensor grid generated on device from the flat index (no input read):
 * point i has coordinate lo[k] + (digit_k(i) + 0.5) * (hi[k]-lo[k]) / levels[k], digit_0 the
 * slowest.  Evaluates flat indices [start, start+count). */
int gpe_predict_grid(gpe_handle* h, const int* levels, const double* lo, const double* hi,
                     long long start, long long count, double* mean, double* var);

/* Full posterior covariance for small m (Posterior.make_var :618-631 as used by
 * posterior_sample, mahalanobis_distance, noise_fit): V [m,m]; r_new [m] or NULL is the
 * new points' r (alt nugget prior diagonal). */
int gpe_predict_fullcov(gpe_handle* h, const double* Xs, const double* Hs, int m,
                        const double* r_new, double* mean, double* V);

/* History-matching arithmetic (history_match.py:121-136, :237-250, :317-329) on per-emulator
 * mean/variance arrays mean [n_emul,m], var [n_emul,m] (device or host):
 * I_o = sqrt((mean_o - z_o)^2 / (var_o + var_extra_o)); Imax [m,maxno] ascending = the maxno
 * largest over emulators; keep [m] = Imax[r,0] < cm; count_lt [maxno] = #(Imax[r,maxno-1-k] < cm).
 * Cells (imp_plot's grid cells, :91-136): if cell_pts > 0, local point r is point first_index + r of a
 * flat global index whose consecutive runs of cell_pts points form the cells; cell_min [ncell,maxno]
 * (min over the cell's points, +huge where the shard holds none) and cell_count [ncell,maxno]
 * (#points below cm) are produced for the ncell cells starting at the cell of point first_index --
 * a shard may begin and end inside a cell; the caller combines shards with min / sum.
 * Any output may be NULL. */
int gpe_implausibility(gpe_handle* h, const double* mean, const double* var, int n_emul,
                       long long m, const double* z, const double* var_extra, double cm,
                       int maxno, long long cell_pts, long long first_index, long long ncell,
                       double* Imax, unsigned char* keep, unsigned long long* count_lt,
                       double* cell_min, unsigned long long* cell_count);

/* The same arithmetic folded into the prediction, one emulator per call (history_match.py:96-132 without the
 * mean / variance arrays): predict m points for THIS handle's emulator -- explicit Xs [m,d] (+ Hs [m,q] or NULL), or, with
 * Xs == NULL, flat indices [start, start+m) of the tensor grid (levels, lo, hi) as in gpe_predict_grid -- and fold
 * I = sqrt((mean - z)^2 / (var + var_extra)) into Itop [m,maxno] (DEVICE memory), the ascending list of the maxno largest
 * implausibilities over the emulators processed so far (first != 0 starts the list; an emulator that must contribute
 * I = 0, reference :99-100, is entered by the caller as a 0 in the initial list).  On the last emulator (last != 0) the
 * keep mask, count_lt and the cell statistics of gpe_implausibility are produced in the same pass (cm, cell_pts,
 * first_index, ncell as there; outputs may be NULL, host or device) and Itop may be NULL when first is set as well.
 * Per point and emulator 8*maxno bytes are read and written instead of 16 written and 16 read. */
int gpe_predict_implaus(gpe_handle* h, const double* Xs, const double* Hs, const int* levels, const double* lo,
                        const double* hi, long long start, long long m, double z, double var_extra, int maxno,
                        int first, int last, double* Itop, double cm, long long cell_pts, long long first_index,
                        long long ncell, unsigned char* keep, unsigned long long* count_lt, double* cell_min,
                        unsigned long long* cell_count);

/* out [n,k] = A^-1 Bm [n,k] for the training matrix factored by gpe_fit_state -- the
 * np.linalg.solve(self.A, .) call sites of the sensitivity code
 * (sensitivity/_sensitivityclasses.py:40-44 e, G; :187 A^-1 Rt; :451, :499 A^-1 T). */
int gpe_solve(gpe_handle* h, const double* Bm, int k, double* out);

/* Product-form n x n integrals of the sensitivity code -- Rtt (:90-102) and Pw (P_prod_calc +
 * Pw_calc, :599-626):  P_kl = scale * u_k u_l * exp(-sum_i gamma_i (x_ki - x_li)^2),
 * u_k = prod_i exp(-acoef_i (x_ki - mvec_i)^2)  (gamma_i = 0 for integrated-out inputs) --
 * contracted without leaving the device:  trace_out = tr(A^-1 P)  (:191, :483-484) and
 * M_out [nv,nv] = V^T P V for V [n,nv], nv <= 32 (V = [G | e]: G^T P G and e^T P e, :192-197, :488-495). */
int gpe_sens_contract(gpe_handle* h, const double* gamma, const double* acoef, const double* mvec,
                      double scale, const double* V, int nv, double* trace_out, double* M_out);

/* Main-effect sweep (main_effect :277-285 with Tw_calc :628-633): for input which[w] and value
 * xw[w,j]:  out[w,j] = sum_k evec_k * scale * prod_{i != P} t1_i exp(-t2_i (x_ki - mvec_i)^2)
 *                                   * exp(-cdiag_P (xw - x_kP)^2)      ( = Tw . e ). */
int gpe_sens_main_effect(gpe_handle* h, const double* t1, const double* t2, const double* cdiag,
                         const double* mvec, const double* evec, double scale, const int* which,
                         int nwhich, const double* xw, int points, double* out);

/* Maximin criterion of the optimised Latin hypercube (design_inputs/design_inputs.py:59-77):
 * argmin_out[k] = np.argmin(pdist(concat(designs[k], extra), 'sqeuclidean')) for N candidate designs
 * designs [N, n, dim] and shared extra points [ne, dim] (fextra; NULL / 0 if none).  Distances are
 * accumulated like scipy's kernel (sequential over dimensions, no FMA), so the indices are identical.
 * Needs no training set.  (The reference compares these *indices* between designs -- a known quirk.) */
int gpe_pdist_argmin(gpe_handle* h, const double* designs, int N, int n, int dim, const double* extra, int ne,
                     long long* argmin_out);

/* Debug/test entry: one batched DMMA GEMM of the family used by the factorisation
 * (gpe_gemm.cuh).  layout 0 NT, 1 NN, 2 TN; device pointers only. */
int gpe_dbg_gemm(gpe_handle* h, const double* A, const double* B, double* C, int lda, int ldb,
                 int ldc, long long sA, long long sB, long long sC, int M, int N, int K,
                 double alpha, int accumulate, int kmode, int lower, int batch, int layout);

/* Debug/test entry: the same product evaluated on the INT8 tensor cores by integer modular arithmetic
 * (csrc/gpe_ozaki.cuh: residues modulo nmod coprime moduli <= 256, one exact tcgen05 u8 GEMM per modulus, CRT) --
 * the route GPE_OZAKI=<nmod> switches the large products of the factorisation to (replaces NumPy's float64 matmul /
 * LAPACK inside np.linalg.cholesky and solve, _emulatoroptimise.py:313-335, 425-441).  M % 128 = N % 256 = K % 128 = 0;
 * device pointers only.  The optional outputs return the intermediate pieces for exact checks: residue planes of
 * op(A) [batch,nmod,M,K] and op(B) [batch,nmod,N,K], of the product [batch,nmod,M,N], and the scale exponents. */
int gpe_dbg_gemm_oz(gpe_handle* h, const double* A, const double* B, double* C, int lda, int ldb,
                    int ldc, long long sA, long long sB, long long sC, int M, int N, int K,
                    double alpha, int accumulate, int kmode, int lower, int batch, int layout, int nmod,
                    unsigned char* planesA, unsigned char* planesB, unsigned char* planesD,
                    int* sexpA, int* sexpB);

/* np.linalg.cholesky for `batch` SPD matrices A [batch,n,n] (device or host) -- the call sites
 * outside the likelihood: posterior_sample (emulatorfunctions.py:283), noise_fit.py:131/:143,
 * and V^-1 in Posterior.mahalanobis_distance (_emulatorclasses.py:672-673).  Outputs (any may be
 * NULL): L_out [batch,n,n] lower Cholesky factor, Linv_out [batch,n,n] = L^-1,
 * logdet [batch] = 2*sum(log L_ii), status [batch] (LAPACK info convention). */
int gpe_potrf(gpe_handle* h, const double* A, int n, int batch, double* L_out, double* Linv_out,
              double* logdet, int* status);

/* Debug/test entry: gpe_potrf with only the inverse factor requested. */
int gpe_dbg_potrf_inv(gpe_handle* h, const double* A, int n, int batch, double* Linv_out,
                      double* logdet, int* status);

/* Debug/test entry: how many products this handle has sent down the INT8 tensor-core route so far (tests use it to
 * assert which route a call took). */
long long gpe_dbg_int8_products(gpe_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* GPE_B200_H */
