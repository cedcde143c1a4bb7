// C-ABI + host orchestration of the B200-native GP hot path (see include/gpe_b200.h).
#include "gpe_handle.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <nvtx3/nvToolsExt.h>

using namespace gpe;

NvtxRange::NvtxRange(const char* name) { nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { nvtxRangePop(); }

// ------------------------------------------------------------------------------------- utils
int gpe_handle::fail(const char* what, cudaError_t e) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    err = buf;
    cudaGetLastError();
    return -1;
}
int gpe_handle::fail_msg(const char* what) {
    err = what;
    return -2;
}

cudaEvent_t gpe_handle::prof_begin(int cat, cudaStream_t s) {
    if (!prof_on) return nullptr;
    cudaEvent_t e;
    if (!prof_pool.empty()) { e = prof_pool.back(); prof_pool.pop_back(); }
    else cudaEventCreate(&e);
    cudaEventRecord(e, s);
    (void)cat;
    return e;
}
void gpe_handle::prof_end(int cat, cudaEvent_t e0, cudaStream_t s) {
    if (!prof_on || !e0) return;
    cudaEvent_t e1;
    if (!prof_pool.empty()) { e1 = prof_pool.back(); prof_pool.pop_back(); }
    else cudaEventCreate(&e1);
    cudaEventRecord(e1, s);
    prof_recs.push_back({cat, e0, e1});
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return h->fail(#call, e__);        \
    } while (0)

bool gpe_is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

template <class T>
static cudaError_t dev_alloc(T** p, size_t count) {
    return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T));
}
template <class T>
static void dev_free(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

void gpe_handle::drop_graphs() {
    for (auto& g : graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    graphs.clear();
}

void gpe_handle::free_batch_ws() {
    drop_graphs();
    dev_free(A); dev_free(S); dev_free(Li); dev_free(Ex); dev_free(Wy); dev_free(Z); dev_free(U); dev_free(GP);
    dev_free(logdet_part); dev_free(par); dev_free(out); dev_free(winv); dev_free(beta);
    dev_free(status); dev_free(gpart); dev_free(theta_d); dev_free(llh_d); dev_free(grad_d); dev_free(sig_d);
    Bcap = 0;
    Bcap_final = false;
}

void gpe_handle::free_training() {
    dev_free(X); dev_free(y); dev_free(H); dev_free(r); dev_free(HY);
    free_batch_ws();
    free_fit();
    n = d = q = npad = nleaf = 0;
}

// Batch workspace: three padded n x n matrices per item (A -> A^-1, S scratch, L^-1) plus the
// skinny panels.  180 GB of HBM3e holds the whole 256-guess batch of config 3 (103 GB), but the
// default cap keeps sub-batches of <= 64 so the factorisation working set stays L2-friendly.
int gpe_ensure_batch_ws(gpe_handle* h, int B) {
    // A workspace that already has the largest obtainable size is kept: batches beyond it run as sub-batches
    // (re-allocating here on every call would also destroy the CUDA graphs before they are ever replayed).
    if (B <= h->Bcap || (h->Bcap > 0 && h->Bcap_final)) return 0;
    size_t per_item = 4ull * h->npad * h->npad * sizeof(double) + 3ull * h->npad * NR * sizeof(double);
    size_t free_b = 0, total_b = 0;
    h->free_batch_ws();
    CK(cudaMemGetInfo(&free_b, &total_b));
    int cap_env = 64;
    if (const char* e = getenv("GPE_BCAP")) cap_env = std::max(1, atoi(e));
    long long fit = (long long)((double)free_b * 0.8 / (double)per_item);
    int want = (int)std::max<long long>(1, std::min<long long>({(long long)B, (long long)cap_env, fit}));
    if (fit < 1) return h->fail_msg("not enough device memory for one n x n factorisation workspace");
    size_t nn = (size_t)h->npad * h->npad;
    CK(dev_alloc(&h->A, want * nn));
    CK(dev_alloc(&h->S, want * nn));
    CK(dev_alloc(&h->Li, want * nn));
    CK(dev_alloc(&h->Ex, want * nn));
    CK(cudaMemsetAsync(h->Li, 0, want * nn * sizeof(double), h->st));
    size_t pn = (size_t)h->npad * NR;
    CK(dev_alloc(&h->Wy, want * pn));
    CK(dev_alloc(&h->Z, want * pn));
    CK(dev_alloc(&h->U, want * pn));
    int nslab = (h->npad + GRAM_SLAB - 1) / GRAM_SLAB;
    CK(dev_alloc(&h->GP, (size_t)want * nslab * NR * NR));
    CK(dev_alloc(&h->logdet_part, (size_t)want * h->nleaf));
    CK(dev_alloc(&h->par, (size_t)want));
    CK(dev_alloc(&h->out, (size_t)want));
    CK(dev_alloc(&h->winv, (size_t)want * h->d));
    CK(dev_alloc(&h->beta, (size_t)want * NR));
    CK(dev_alloc(&h->status, (size_t)want));
    CK(dev_alloc(&h->gpart, (size_t)want * grad_ntiles(h->npad) * grad_nvals(h->d)));
    CK(dev_alloc(&h->theta_d, (size_t)want * (h->d + 2)));
    CK(dev_alloc(&h->llh_d, (size_t)want));
    CK(dev_alloc(&h->grad_d, (size_t)want * (h->d + 2)));
    CK(dev_alloc(&h->sig_d, (size_t)want));
    h->Bcap = want;
    h->Bcap_final = want >= cap_env || want >= fit;
    return 0;
}

// ------------------------------------------------------------------------------------- GEMM helper
// does launch_gemm pick the warp-specialised 128x128 kernel with a machine-filling grid? (mirrors dispatch_tiles)
static bool gemm_is_big(int M, int N, int lower, int batch) {
    if (M % 128 || N % 128 || M == 32 || N == 32) return false;
    long long t128 = (long long)(M / 128) * (N / 128) * batch;
    if (lower) t128 = t128 / 2 + (M / 128) * batch / 2;
    return t128 >= 120;
}

static bool oz_takes(const gpe_handle* h, int M, int N, int K) {
    return h->oz_nmod > 0 && M >= h->oz_min && N >= h->oz_min && K >= h->oz_min && M % OZ_BM == 0 && N % OZ_BN == 0 && K % OZ_BK == 0;
}

static int run_gemm(gpe_handle* h, cudaStream_t st, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                    long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int acc,
                    int kmode, int lower, int batch, int layout, int epi = EPI_STORE, int cat = -1) {
    GemmP p;
    p.A = A; p.B = B; p.C = C; p.lda = lda; p.ldb = ldb; p.ldc = ldc; p.sA = sA; p.sB = sB; p.sC = sC;
    p.M = M; p.N = N; p.K = K; p.alpha = alpha; p.accumulate = acc; p.kmode = kmode; p.lower = lower; p.batch = batch;
    bool big = (M % 128 == 0 || epi == EPI_SUMSQ) && (N % 128 == 0) && N != 32 && M != 32;
    cudaError_t e;
    const bool reuse_a = h->oz_reuse_a;      // a request holds for one product only, whichever route it takes
    const unsigned long long a_tag = h->oz_a_tag;
    const double b_bound = h->oz_b_bound;
    h->oz_reuse_a = false;
    h->oz_a_tag = 0;
    h->oz_b_bound = 0.0;
    if (h->oz_nmod > 0 && M >= h->oz_min && N >= h->oz_min && K >= h->oz_min && oz_supported(p, epi)) {
        // INT8 tensor-core route (gpe_ozaki.cuh): scratch is per stream; growing it is not allowed inside a capture, and
        // every shape has been seen eagerly at least twice before its graph is captured
        OzWs& ws = h->oz_ws[st];
        ws.b_bound = b_bound;
        struct HookCtx { gpe_handle* h; cudaEvent_t e0[3]; } hc{h, {nullptr, nullptr, nullptr}};
        OzHook hook;
        if (h->prof_on) {       // per-phase event pairs: residue conversion, residue GEMM, CRT
            hook.ctx = &hc;
            hook.fn = [](void* c, int phase, bool begin, cudaStream_t s) {
                HookCtx* x = static_cast<HookCtx*>(c);
                const int pc = gpe_handle::CAT_OZ_CONVERT + phase;
                if (begin) x->e0[phase] = x->h->prof_begin(pc, s);
                else x->h->prof_end(pc, x->e0[phase], s);
            };
        }
        e = oz_gemm(p, layout, epi, h->oz_nmod, ws, st, reuse_a, a_tag, hook);
        h->launches += 4;
        h->oz_calls++;
        if (ws.grew) {          // (never during a capture: a shape is captured after it has run eagerly twice)
            ws.grew = false;
            h->graphs_stale = true;
        }
        if (e != cudaSuccess) return h->fail("oz_gemm", e);
        return 0;
    }
    {
        ProfScope ps(h, cat >= 0 ? cat : (big ? gpe_handle::CAT_GEMM_BIG : gpe_handle::CAT_GEMM_SMALL), st);
        e = launch_gemm(p, layout, epi, st);
    }
    h->launches++;
    if (e != cudaSuccess) return h->fail("launch_gemm", e);
    return 0;
}
// Can the INT8 route hold the scratch of product `p` on stream `st`?  Grows the scratch if it must; on an allocation failure the
// error is cleared and the caller stays on the DMMA route (a prediction chunk over a very large training set).
bool gpe_oz_reserve(gpe_handle* h, cudaStream_t st, const GemmP& p) {
    OzWs& ws = h->oz_ws[st];
    bool grew = false;
    const cudaError_t e = oz_reserve(ws, p, h->oz_nmod, grew, false);
    if (grew) { ws.have_a = false; ws.grew = true; }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return true;
}
int gpe_run_gemm_on(gpe_handle* h, cudaStream_t st, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                    long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int acc,
                    int kmode, int lower, int batch, int layout, int epi) {
    return run_gemm(h, st, A, B, C, lda, ldb, ldc, sA, sB, sC, M, N, K, alpha, acc, kmode, lower, batch, layout, epi);
}
int gpe_run_gemm(gpe_handle* h, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                 long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int acc,
                 int kmode, int lower, int batch, int layout, int epi) {
    return run_gemm(h, h->st, A, B, C, lda, ldb, ldc, sA, sB, sC, M, N, K, alpha, acc, kmode, lower, batch, layout, epi);
}

// Recursive Cholesky + triangular inverse of the diagonal block [off, off+m) of every item:
//   F(A11) ; L21 = A21 L11^-T ; A22 -= L21 L21^T ; F(A22) ; Linv21 = -L22^-1 (L21 L11^-1).
// All four updates are DMMA GEMMs with a triangular operand (zero tiles skipped); only the
// 128x128 diagonal leaves are factored by a panel kernel.  2n^3/3 flops, 5 launches per node.
int gpe_handle::ensure_side(int g) {
    if (side_st[g][0]) return 0;
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    for (int k = 0; k < MAX_DEPTH; k++) {
        if (cudaStreamCreateWithPriority(&side_st[g][k], cudaStreamNonBlocking, prio_least) != cudaSuccess) return -1;
        cudaEventCreateWithFlags(&ev_sf[g][k], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ev_sj[g][k], cudaEventDisableTiming);
    }
    return 0;
}

static int potrf_inv_rec(gpe_handle* h, const FactorWs& ws, const SubBatch& sb, int off, int m, int want_L, int depth = 0) {
    const int ld = ws.npad, B = sb.B;
    const long long sM = (long long)ws.npad * ws.npad;
    double* Ab = ws.A + (size_t)sb.b0 * sM;
    double* Sb = ws.S + (size_t)sb.b0 * sM;
    double* Lb = ws.Li + (size_t)sb.b0 * sM;
    if (m == NB) {
        {
            cudaStream_t st = sb.stream(true);
            ProfScope ps(h, gpe_handle::CAT_LEAF, st);
            launch_leaf(Ab, Lb, ld, sM, sM, off, ws.logdet_part + (size_t)sb.b0 * ws.nleaf, ws.nleaf, ws.status + sb.b0, B, st,
                        want_L ? Sb : nullptr);
        }
        h->launches++;
        return 0;
    }
    const int nb = m / NB;
    const int m1 = ((nb + 1) / 2) * NB, m2 = m - m1;
    int rc;
    if ((rc = potrf_inv_rec(h, ws, sb, off, m1, want_L, depth + 1))) return rc;
    double* A21 = Ab + (size_t)(off + m1) * ld + off;
    double* A22 = Ab + (size_t)(off + m1) * ld + off + m1;
    double* S21 = Sb + (size_t)(off + m1) * ld + off;
    double* Li11 = Lb + (size_t)off * ld + off;
    double* Li22 = Lb + (size_t)(off + m1) * ld + off + m1;
    double* Li21 = Lb + (size_t)(off + m1) * ld + off;
    // L21 = A21 * Linv11^T           (NT, Linv11 lower: k <= j)
    if ((rc = run_gemm(h, sb.stream(!gemm_is_big(m2, m1, 0, B)), A21, Li11, S21, ld, ld, ld, sM, sM, sM, m2, m1, m1, 1.0, 0, KM_LE_J, 0, B, 0))) return rc;
    // T = L21 * Linv11  (NN, Linv11 lower: k >= j) -> dead A21 block.  It needs only L21 and Linv11, not the
    // factorisation of A22: with side streams it is launched now, beside the SYRK and the whole A22 sub-recursion
    // (whose leaves and small levels cannot fill the machine), and joined before the last product of the node.
    // On the INT8 route the node's products run in order on one stream: L21 is converted to residues once, for the SYRK, and
    // the planes serve T = L21 Linv11 right after it.
    const bool oz_node = oz_takes(h, m2, m1, m1) && oz_takes(h, m2, m2, m1);
    const bool fork = !oz_node && sb.side != nullptr && depth < gpe_handle::MAX_DEPTH;
    if (fork) {
        cudaStream_t side = sb.side[depth];
        cudaEventRecord(sb.ef[depth], sb.current());
        cudaStreamWaitEvent(side, sb.ef[depth], 0);
        if ((rc = run_gemm(h, side, S21, Li11, A21, ld, ld, ld, sM, sM, sM, m2, m1, m1, 1.0, 0, KM_GE_J, 0, B, 1))) return rc;
        cudaEventRecord(sb.ej[depth], side);
    }
    // A22 -= L21 * L21^T             (SYRK, lower tiles)
    if ((rc = run_gemm(h, sb.stream(!gemm_is_big(m2, m2, 1, B)), S21, S21, A22, ld, ld, ld, sM, sM, sM, m2, m2, m1, -1.0, 1, KM_FULL, 1, B, 0))) return rc;
    if (oz_node) {
        h->oz_reuse_a = true;
        if ((rc = run_gemm(h, sb.current(), S21, Li11, A21, ld, ld, ld, sM, sM, sM, m2, m1, m1, 1.0, 0, KM_GE_J, 0, B, 1))) return rc;
    }
    if ((rc = potrf_inv_rec(h, ws, sb, off + m1, m2, want_L, depth + 1))) return rc;
    if (fork) {
        cudaStreamWaitEvent(sb.current(), sb.ej[depth], 0);
    } else if (!oz_node) {
        if ((rc = run_gemm(h, sb.stream(!gemm_is_big(m2, m1, 0, B)), S21, Li11, A21, ld, ld, ld, sM, sM, sM, m2, m1, m1, 1.0, 0, KM_GE_J, 0, B, 1))) return rc;
    }
    // Linv21 = -Linv22 * T           (NN, Linv22 lower: k <= i)
    if ((rc = run_gemm(h, sb.stream(!gemm_is_big(m2, m1, 0, B)), Li22, A21, Li21, ld, ld, ld, sM, sM, sM, m2, m1, m2, -1.0, 0, KM_LE_I, 0, B, 1))) return rc;
    return 0;
}
int gpe_potrf_inv(gpe_handle* h, const FactorWs& ws, const SubBatch& sb, int want_L) { return potrf_inv_rec(h, ws, sb, 0, ws.npad, want_L); }

static FactorWs handle_ws(gpe_handle* h) { return FactorWs{h->A, h->S, h->Li, h->npad, h->nleaf, h->logdet_part, h->status}; }

// How the gradient reduction of a chunk is done (GPE_FUSED_GRAD = 0 | 1 | 2; all routes sum the same terms, results agree
// to rounding).
//   0: A^-1 by the generic LAUUM GEMM, stored, then the stand-alone reduction kernel that recomputes E and U.U^T
//      (round 1; still used for launches too small for 128x128 tiles).
//   1: LAUUM with the columns of U in its k loop stores W = A^-1 - U U^T; a light kernel reduces W against the
//      covariance build's copy of E.
//   2 (default when 128x128 tiles fill the machine): the reduction in LAUUM's epilogue (gpe_lauum_grad.cu); nothing
//      of size n x n is written after the factorisation.
// Measured on one B200 in one call, n = 4096, d = 16, 32 items, 8 streams, graph replay: 75.41 / 75.79 / 75.38 ms per step
// for routes 0 / 1 / 2, 73.9 ms with the reduction switched off altogether.  The reduction is scalar FP64 work on the pipe
// the DMMAs use: fusing moves it, it does not remove it (DESIGN.md section 8).
static int llh_grad_fused(gpe_handle* h, int B) {
    static int mode = -1;
    if (mode < 0) {
        const char* e = getenv("GPE_FUSED_GRAD");
        mode = e ? atoi(e) : 2;
    }
    h->grad_use_e = false;
    // Matérn: the stand-alone reduction recomputes R and G (the LAUUM epilogue and the E copy are Gaussian-only)
    if (h->family != FAMILY_GAUSSIAN || !gemm_is_big(h->npad, h->npad, 1, B)) return 0;
    if (h->oz_nmod > 0 && h->npad >= h->oz_min && h->npad % OZ_BN == 0) {   // LAUUM on the INT8 route, A^-1 stored: the stand-alone
        static const int use_e = [] { const char* e = getenv("GPE_GRAD_E"); return e ? atoi(e) : 1; }();   // reduction reads the
        h->grad_use_e = use_e != 0;                                          // covariance build's copy of exp(-D)
        return 0;
    }
    if (mode == 2 && !lauum_grad_supported(h->d)) return 1;
    return mode;
}

// Everything after the covariance build for the items of `sb`, already described by h->par / h->winv.
// with_grad = 0 stops after the GLS/likelihood scalars (fit_state path).
int gpe_factor_and_reduce(gpe_handle* h, const SubBatch& sb, int mode, int with_grad, const double* beta_override, double* Kout) {
    const int np = h->npad, ld = np, B = sb.B, b0 = sb.b0;
    const long long sM = (long long)np * np, sP = (long long)np * NR;
    cudaStream_t st;
    const int nslab = (np + GRAM_SLAB - 1) / GRAM_SLAB;
    double* Ab = h->A + (size_t)b0 * sM;
    double* Lb = h->Li + (size_t)b0 * sM;
    double *Wy = h->Wy + (size_t)b0 * sP, *Z = h->Z + (size_t)b0 * sP, *U = h->U + (size_t)b0 * sP;
    double* GP = h->GP + (size_t)b0 * nslab * NR * NR;
    int rc;
    if ((rc = potrf_inv_rec(h, handle_ws(h), sb, 0, np, 0))) return rc;
    // Wy = Linv [H | y]
    st = sb.stream(true);
    if ((rc = run_gemm(h, st, Lb, h->HY, Wy, ld, NR, NR, sM, 0, sP, np, NR, np, 1.0, 0, KM_LE_I, 0, B, 1))) return rc;
    {
        ProfScope ps(h, gpe_handle::CAT_OTHER, st);
        launch_gram(Wy, np, B, GP, st);
        launch_llh_finalize(Wy, GP, h->logdet_part + (size_t)b0 * h->nleaf, h->nleaf, h->n, h->q, np, mode, h->par + b0, h->out + b0,
                            h->beta + (size_t)b0 * NR, Z, h->status + b0, B, beta_override, Kout, st);
    }
    h->launches += 2;
    // U = Linv^T Z = [A^-1 H K^-T | sqrt(f) A^-1 (y - H beta)]
    if ((rc = run_gemm(h, st, Lb, Z, U, ld, NR, NR, sM, sP, sP, np, NR, np, 1.0, 0, KM_GE_I, 0, B, 2))) return rc;
    if (!with_grad) return 0;
    st = sb.stream(false);
    if (h->grad_fused == 2) {
        // LAUUM with the gradient reduction in its epilogue: W = A^-1 - U U^T never leaves the CTA that computed it
        // (gpe_lauum_grad.cu).  Wy and Z are dead by now and hold U^T and -U^T.
        ProfScope ps(h, gpe_handle::CAT_LAUUM, st);
        cudaError_t e = launch_lauum_grad(Lb, sM, np, h->n, h->d, h->q + 1, U, Wy, Z, h->X, h->r, h->winv + (size_t)b0 * h->d,
                                          h->Ex + (size_t)b0 * sM, sM,
                                          h->gpart + (size_t)b0 * lauum_grad_ntiles(np) * grad_nvals(h->d), B, st);
        h->launches += 2;
        if (e != cudaSuccess) return h->fail("launch_lauum_grad", e);
        return 0;
    }
    if (h->grad_fused == 1) {
        // split route (default for machine-filling launches): the same LAUUM launch stores W = A^-1 - U U^T (the columns of
        // U ride along in its k loop) into the dead A buffer; a light reduction kernel combines it with the E copy
        {
            ProfScope ps(h, gpe_handle::CAT_LAUUM, st);
            cudaError_t e = launch_lauum_grad(Lb, sM, np, h->n, h->d, h->q + 1, U, Wy, Z, h->X, h->r, h->winv + (size_t)b0 * h->d,
                                              nullptr, 0, nullptr, B, st, Ab);
            h->launches += 2;
            if (e != cudaSuccess) return h->fail("launch_lauum_grad (store W)", e);
        }
        ProfScope ps(h, gpe_handle::CAT_GRAD, st);
        cudaError_t e = launch_grad_partial_we(h->X, h->r, h->n, h->d, np, h->winv + (size_t)b0 * h->d, Ab, h->Ex + (size_t)b0 * sM, sM,
                                               h->gpart + (size_t)b0 * grad_ntiles(np) * grad_nvals(h->d), B, st);
        h->launches++;
        if (e != cudaSuccess) return h->fail("launch_grad_partial_we", e);
        return 0;
    }
    // small launches (64x64 tiles) and very wide inputs: A^-1 = Linv^T Linv (lower tiles) into the dead A buffer, then
    // the stand-alone reduction kernel
    if ((rc = run_gemm(h, st, Lb, Lb, Ab, ld, ld, ld, sM, sM, sM, np, np, np, 1.0, 0, KM_GE_I, 1, B, 2, EPI_STORE,
                       gpe_handle::CAT_LAUUM))) return rc;
    {
        ProfScope ps(h, gpe_handle::CAT_GRAD, st);
        launch_grad_partial(h->X, h->r, h->n, h->d, np, h->winv + (size_t)b0 * h->d, Ab, sM, U, h->q + 1,
                            h->gpart + (size_t)b0 * grad_ntiles(np) * grad_nvals(h->d), B, st,
                            h->grad_use_e ? h->Ex + (size_t)b0 * sM : nullptr, h->family);
    }
    h->launches++;
    return 0;
}

static void host_item_par(ItemPar& ip, double nugget, int kind, int predict, double s2_for_r, double s2A) {
    ip.c = kind ? 1.0 : (1.0 - nugget);
    ip.offs = s2A * ip.c;
    double diagK = kind ? (predict ? 1.0 + nugget * nugget : 1.0) : (predict ? 1.0 : 1.0 - nugget);
    ip.diagv = s2A * diagK;
    ip.radd = kind ? s2A / s2_for_r : 0.0;
    ip.s2A = s2A; ip.nugget = nugget; ip.sigma = std::sqrt(s2A); ip.pad_ = 0.0;
}

int gpe_upload_single_par(gpe_handle* h, const double* delta, double nugget, int kind, int predict, double s2_for_r) {
    ItemPar ip;
    host_item_par(ip, nugget, kind, predict, s2_for_r, 1.0);
    std::vector<double> w(h->d);
    for (int k = 0; k < h->d; k++) w[k] = 1.0 / delta[k];
    CK(cudaMemcpyAsync(h->par, &ip, sizeof ip, cudaMemcpyHostToDevice, h->st));
    CK(cudaMemcpyAsync(h->winv, w.data(), sizeof(double) * h->d, cudaMemcpyHostToDevice, h->st));
    CK(cudaStreamSynchronize(h->st));   // host vectors go out of scope
    return 0;
}

// ------------------------------------------------------------------------------------- C-ABI
extern "C" {

int gpe_version(void) { return 100; }

int gpe_create(int device, gpe_handle** out) {
    if (!out) return -2;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return -3;   // no CPU fallback
    if (device < 0 || device >= count) return -2;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -3;
    if (prop.major < 10) return -4;                                           // sm_100a only
    if (cudaSetDevice(device) != cudaSuccess) return -3;
    gpe_handle* h = new gpe_handle();
    h->device = device;
    h->sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) != cudaSuccess) { delete h; return -3; }
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (const char* e = getenv("GPE_PRIO")) h->use_prio = e[0] != '0';
    // GPE_SUB_ASYM=1 (experiment): the even sub-batch streams get the highest priority, so that one group runs at full speed and
    // the other fills the gaps its tensor-bound kernels leave, instead of both drifting through the same phases
    const bool asym = [] { const char* e = getenv("GPE_SUB_ASYM"); return e && e[0] != '0'; }();
    for (int s = 0; s < gpe_handle::MAX_SUB; s++) {
        cudaStreamCreateWithPriority(&h->sub_st[s], cudaStreamNonBlocking, (asym && s % 2 == 0) ? prio_greatest : prio_least);
        cudaEventCreateWithFlags(&h->ev_join[s], cudaEventDisableTiming);
        if (h->use_prio) {          // the optional high-priority twin streams (experiment knob, DESIGN.md section 8)
            cudaStreamCreateWithPriority(&h->sub_hi[s], cudaStreamNonBlocking, prio_greatest);
            cudaEventCreateWithFlags(&h->ev_sw[s], cudaEventDisableTiming);
        }
    }
    cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    {   // keep freed temporaries cached in the device's default pool instead of returning them to the driver
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    // the INT8 route is the default for products of 1024 and more in every dimension (GPE_OZAKI=0: DMMA everywhere); its
    // launches fill the machine on their own, so two sub-batch groups are enough there (oz_nsub; eight for the DMMA route)
    if (const char* e = getenv("GPE_OZAKI")) h->oz_nmod = std::max(0, std::min((int)OZ_MAXMOD, atoi(e)));
    if (h->oz_nmod == 1) h->oz_nmod = 2;
    if (const char* e = getenv("GPE_OZAKI_MIN")) h->oz_min = std::max(256, atoi(e));
    if (const char* e = getenv("GPE_OZAKI_STREAMS")) h->oz_nsub = std::max(1, std::min((int)gpe_handle::MAX_SUB, atoi(e)));
    if (const char* e = getenv("GPE_STREAMS")) h->nsub = std::max(1, std::min((int)gpe_handle::MAX_SUB, atoi(e)));
    if (const char* e = getenv("GPE_GRAPHS")) h->use_graphs = e[0] != '0';
    if (const char* e = getenv("GPE_SIDE")) h->use_side = e[0] != '0';
    *out = h;
    return 0;
}

int gpe_destroy(gpe_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->st);
    h->free_training();
    for (int s = 0; s < gpe_handle::MAX_SUB; s++) {
        if (h->sub_st[s]) { cudaStreamSynchronize(h->sub_st[s]); cudaStreamDestroy(h->sub_st[s]); }
        if (h->sub_hi[s]) { cudaStreamSynchronize(h->sub_hi[s]); cudaStreamDestroy(h->sub_hi[s]); }
        if (h->ev_join[s]) cudaEventDestroy(h->ev_join[s]);
        if (h->ev_sw[s]) cudaEventDestroy(h->ev_sw[s]);
    }
    for (int s = 0; s < gpe_handle::MAX_SUB; s++)
        for (int k = 0; k < gpe_handle::MAX_DEPTH; k++) {
            if (h->side_st[s][k]) { cudaStreamSynchronize(h->side_st[s][k]); cudaStreamDestroy(h->side_st[s][k]); }
            if (h->ev_sf[s][k]) cudaEventDestroy(h->ev_sf[s][k]);
            if (h->ev_sj[s][k]) cudaEventDestroy(h->ev_sj[s][k]);
        }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (auto& kv : h->oz_ws) kv.second.release();
    for (auto e : h->prof_pool) cudaEventDestroy(e);
    cudaStreamDestroy(h->st);
    delete h;
    return 0;
}

void* gpe_get_stream(gpe_handle* h) { return h ? (void*)h->st : nullptr; }

int gpe_set_streams(gpe_handle* h, int nstreams) {
    if (!h || nstreams < 1) return -2;
    h->nsub = std::min((int)gpe_handle::MAX_SUB, nstreams);
    h->drop_graphs();
    return 0;
}

int gpe_set_kernel(gpe_handle* h, int family) {
    if (!h) return -2;
    if (family != GPE_KERNEL_GAUSSIAN && family != GPE_KERNEL_MATERN52) return h->fail_msg("unknown kernel family");
    if (family == h->family) return 0;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->st));
    // the fit state and the captured likelihood graphs (keyed on batch and mode only) belong to the old kernel; a new
    // fit generation makes the prediction product re-make its residue planes of L^-1
    h->family = family;
    h->fitted = false;
    h->fAinv_valid = false;
    h->fit_gen++;
    h->drop_graphs();
    return 0;
}

int gpe_set_async(gpe_handle* h, int on) {
    if (!h) return -2;
    h->async = on != 0;
    return 0;
}

int gpe_synchronize(gpe_handle* h) {
    if (!h) return -2;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

int gpe_profile_enable(gpe_handle* h, int on) {
    if (!h) return -2;
    h->prof_on = on != 0;
    return 0;
}

// Drain the recorded event pairs: ms[c] / count[c] per category since the last reset
// (0 big DMMA GEMM tiles, 1 small/skinny GEMM, 2 leaf, 3 covariance build, 4 gradient reduction, 5 other,
// 6 the LAUUM launch A^-1 = L^-T L^-1 on the DMMA route; 7 / 8 / 9 the INT8 route's residue conversion, residue GEMM
// (tcgen05.mma kind::i8) and CRT recombination).
int gpe_profile_read(gpe_handle* h, double* ms, long long* count, int reset) {
    if (!h) return -2;
    cudaStreamSynchronize(h->st);
    for (auto& r : h->prof_recs) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.e0, r.e1) == cudaSuccess) { h->prof_ms[r.cat] += t; h->prof_cnt[r.cat]++; }
        h->prof_pool.push_back(r.e0);
        h->prof_pool.push_back(r.e1);
    }
    h->prof_recs.clear();
    for (int c = 0; c < gpe_handle::NCAT; c++) {
        if (ms) ms[c] = h->prof_ms[c];
        if (count) count[c] = h->prof_cnt[c];
        if (reset) { h->prof_ms[c] = 0; h->prof_cnt[c] = 0; }
    }
    return 0;
}

const char* gpe_last_error(gpe_handle* h) { return h ? h->err.c_str() : "null handle"; }
long long gpe_launch_count(gpe_handle* h) { return h ? h->launches : 0; }
long long gpe_dbg_int8_products(gpe_handle* h) { return h ? h->oz_calls : 0; }

int gpe_set_training(gpe_handle* h, const double* X, const double* y, const double* H, const double* r,
                     int n, int d, int q) {
    if (!h || !X || !y || !H || n < 1 || d < 1 || q < 1) return h ? h->fail_msg("bad argument") : -2;
    if (q + 1 > NR) return h->fail_msg("q + 1 exceeds the skinny panel width (32)");
    // the covariance / gradient kernels keep two k-major 64-row tiles of the scaled inputs (plus the skinny U tiles)
    // in shared memory: d is bounded by the 227 KB a CTA can opt in to
    if ((size_t)(d + NR) * (64 + 66) * sizeof(double) + 8 * (size_t)(d + 3) * sizeof(double) > 227 * 1024)
        return h->fail_msg("d is too large for the shared-memory tiles of the covariance kernels");
    NvtxRange nvtx("gpe_set_training");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->st));
    h->free_training();
    auto upload = [&]() -> int {
        CK(dev_alloc(&h->X, (size_t)n * d));
        CK(dev_alloc(&h->y, (size_t)n));
        CK(dev_alloc(&h->H, (size_t)n * q));
        CK(cudaMemcpyAsync(h->X, X, sizeof(double) * n * d, cudaMemcpyDefault, h->st));
        CK(cudaMemcpyAsync(h->y, y, sizeof(double) * n, cudaMemcpyDefault, h->st));
        CK(cudaMemcpyAsync(h->H, H, sizeof(double) * n * q, cudaMemcpyDefault, h->st));
        if (r) {
            CK(dev_alloc(&h->r, (size_t)n));
            CK(cudaMemcpyAsync(h->r, r, sizeof(double) * n, cudaMemcpyDefault, h->st));
        }
        const int npad = ((n + NB - 1) / NB) * NB;
        CK(dev_alloc(&h->HY, (size_t)npad * NR));
        launch_build_hy(h->H, h->y, n, q, npad, h->HY, h->st);
        h->launches++;
        CK(cudaStreamSynchronize(h->st));
        CK(cudaGetLastError());
        return 0;
    };
    if (int rc = upload()) {        // a half-built training set must not look usable
        h->free_training();
        return rc;
    }
    h->n = n; h->d = d; h->q = q;
    h->npad = ((n + NB - 1) / NB) * NB;
    h->nleaf = h->npad / NB;
    h->has_basis = false;
    return 0;
}

int gpe_set_basis(gpe_handle* h, const int* idx, const int* pw, int q) {
    if (!h || q != h->q) return h ? h->fail_msg("basis size does not match q") : -2;
    h->basis_idx[0] = -1; h->basis_pow[0] = 0;
    for (int j = 1; j < q; j++) {
        if (idx[j - 1] < 0 || idx[j - 1] >= h->d) return h->fail_msg("basis index out of range");
        h->basis_idx[j] = idx[j - 1];
        h->basis_pow[j] = pw[j - 1];
    }
    h->has_basis = true;
    return 0;
}

int gpe_cov_build(gpe_handle* h, const double* delta, double nugget, int kind, int predict, double s2, double* A_out) {
    if (!h || !h->n || !delta || !A_out) return h ? h->fail_msg("bad argument / no training set") : -2;
    NvtxRange nvtx("gpe_cov_build");
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = gpe_ensure_batch_ws(h, 1))) return rc;
    std::vector<double> dl(h->d);
    CK(cudaMemcpy(dl.data(), delta, sizeof(double) * h->d, cudaMemcpyDefault));
    if ((rc = gpe_upload_single_par(h, dl.data(), nugget, kind, predict, s2))) return rc;
    CK(launch_cov_build(h->X, h->r, h->n, h->d, h->npad, h->par, h->winv, h->A, 0, 1, 1, h->st, 0, 0, nullptr, h->family));
    h->launches++;
    size_t nn = (size_t)h->n * h->n;
    double* dst = A_out;
    bool dev = gpe_is_device_ptr(A_out);
    if (!dev) dst = h->S;   // stage through scratch
    launch_unpad_sym(h->A, h->npad, h->n, dst, 0, h->st);
    h->launches++;
    if (!dev) CK(cudaMemcpyAsync(A_out, dst, nn * sizeof(double), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

int gpe_cov_grad(gpe_handle* h, const double* delta, double nugget, int kind, int which, double s2, double* G_out) {
    if (!h || !h->n || !delta || !G_out) return h ? h->fail_msg("bad argument / no training set") : -2;
    if (which < -1 || which >= h->d) return h->fail_msg("which must be a delta index or -1 (nugget)");
    NvtxRange nvtx("gpe_cov_grad");
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = gpe_ensure_batch_ws(h, 1))) return rc;
    std::vector<double> dl(h->d);
    CK(cudaMemcpy(dl.data(), delta, sizeof(double) * h->d, cudaMemcpyDefault));
    ItemPar ip;
    host_item_par(ip, nugget, kind, 1, 1.0, 1.0);
    // grad_delta_A: s2 (1-nu) Delta^2 E  (alt: s2 Delta^2 E);  grad_nugget_A (kernel): -1/2 nu s2 E
    // (Matérn: G in place of E in grad_delta_A, R in place of E in grad_nugget_A)
    ip.offs = (which >= 0) ? s2 * ip.c : -0.5 * nugget * s2;
    std::vector<double> w(h->d);
    for (int k = 0; k < h->d; k++) w[k] = 1.0 / dl[k];
    CK(cudaMemcpyAsync(h->par, &ip, sizeof ip, cudaMemcpyHostToDevice, h->st));
    CK(cudaMemcpyAsync(h->winv, w.data(), sizeof(double) * h->d, cudaMemcpyHostToDevice, h->st));
    CK(cudaStreamSynchronize(h->st));
    size_t nn = (size_t)h->n * h->n;
    bool dev = gpe_is_device_ptr(G_out);
    double* dst = dev ? G_out : h->S;
    if (which == -1 && kind == 1) {
        // kernel_alt_nug.grad_nugget_A: diag(nu^2 s2)
        std::vector<double> host(nn, 0.0);
        for (int i = 0; i < h->n; i++) host[(size_t)i * h->n + i] = nugget * nugget * s2;
        CK(cudaMemcpy(G_out, host.data(), nn * sizeof(double), cudaMemcpyDefault));
        return 0;
    }
    CK(launch_cov_build(h->X, h->r, h->n, h->d, h->npad, h->par, h->winv, h->A, 0, 1, 1, h->st, which >= 0 ? 1 : 2, which,
                        nullptr, h->family));
    launch_unpad_sym(h->A, h->npad, h->n, dst, 0, h->st);
    h->launches += 2;
    if (!dev) CK(cudaMemcpyAsync(G_out, dst, nn * sizeof(double), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    CK(cudaGetLastError());
    return 0;
}

// Device work of one resident sub-batch: theta_d -> (llh_d, grad_d, sig_d, status).  Everything is
// enqueued on h->st and its sub-batch streams (fork/join by events), so the same code path is used
// eagerly and under stream capture.
static int enqueue_llh_chunk(gpe_handle* h, int Bs, int p, int mode, double fixed_nugget, bool capturing) {
    const long long sM = (long long)h->npad * h->npad;
    int rc;
    launch_prep_theta(h->theta_d, Bs, p, h->d, mode, fixed_nugget, h->par, h->winv, h->st);
    h->launches++;
    CK(cudaMemsetAsync(h->status, 0, sizeof(int) * Bs, h->st));
    // contiguous groups of the sub-batch, one stream each (a group needs >= 2 items to be worth a stream)
    // ... and only where the groups pay.  Launched eagerly, an evaluation below npad = 2048 is bound by the launch
    // rate of the host thread: groups multiply the launches (n = 200, 10 guesses: 67 instead of 15; 0.52 -> 0.30 ms
    // with one group; n = 1000, 16 guesses: 2.58 -> 1.74 ms).  Replayed from a CUDA graph the launches are free and the
    // groups overlap one another's latency-bound leaves again (n = 1000, 16 guesses: 1.40 vs 1.77 ms; n = 500, 64
    // guesses: 0.90 vs 1.10 ms); below npad = 512 nothing is left to overlap.
    static int group_npad = -1, group_npad_graph = -1;
    if (group_npad < 0) {
        const char* e = getenv("GPE_GROUP_NPAD");
        group_npad = e ? atoi(e) : 2048;
        e = getenv("GPE_GROUP_NPAD_GRAPH");
        group_npad_graph = e ? atoi(e) : 512;
    }
    int ns = h->npad < (capturing ? group_npad_graph : group_npad) ? 1 : std::max(1, std::min(h->nsub, Bs / 2));
    if (oz_takes(h, h->npad / 2, h->npad / 2, h->npad / 2)) ns = std::min(ns, h->oz_nsub);   // the top level runs on the INT8 route
    // one decision for the whole chunk (every group writes the same partial layout): the smallest group must still
    // fill the machine with 128x128 tiles
    h->grad_fused = llh_grad_fused(h, Bs / ns);
    if (ns > 1) CK(cudaEventRecord(h->ev_fork, h->st));
    for (int g = 0; g < ns; g++) {
        SubBatch sb;
        sb.b0 = (int)((long long)Bs * g / ns);
        sb.B = (int)((long long)Bs * (g + 1) / ns) - sb.b0;
        sb.st = ns > 1 ? h->sub_st[g] : h->st;
        if (ns > 1 && h->use_prio) { sb.hi = h->sub_hi[g]; sb.ev = h->ev_sw[g]; }
        if (h->nsub > 1 && h->use_side) {      // also for a single group (small batches): intra-item overlap only
            if (h->ensure_side(g)) return h->fail_msg("could not create side streams");
            sb.side = h->side_st[g]; sb.ef = h->ev_sf[g]; sb.ej = h->ev_sj[g];
        }
        if (ns > 1) CK(cudaStreamWaitEvent(sb.st, h->ev_fork, 0));
        {
            ProfScope ps(h, gpe_handle::CAT_COV, sb.st);
            CK(launch_cov_build(h->X, h->r, h->n, h->d, h->npad, h->par + sb.b0, h->winv + (size_t)sb.b0 * h->d,
                                h->A + (size_t)sb.b0 * sM, sM, sb.B, 0, sb.st, 0, 0,
                                (h->grad_fused || h->grad_use_e) ? h->Ex + (size_t)sb.b0 * sM : nullptr, h->family));
        }
        h->launches++;
        if ((rc = gpe_factor_and_reduce(h, sb, mode, 1, nullptr, nullptr))) return rc;
        if (ns > 1) {
            CK(cudaEventRecord(h->ev_join[g], sb.stream(false)));
            CK(cudaStreamWaitEvent(h->st, h->ev_join[g], 0));
        }
    }
    {
        ProfScope ps(h, gpe_handle::CAT_OTHER);
        launch_grad_finalize(h->gpart, h->grad_fused == 2 ? lauum_grad_ntiles(h->npad) : grad_ntiles(h->npad), h->n, h->d, h->npad, p, mode,
                             h->par, h->out, h->status, h->llh_d, h->grad_d,
                             h->sig_d, Bs, h->st);
    }
    h->launches++;
    return 0;
}

int gpe_llh_grad_batch(gpe_handle* h, const double* theta, int B, int p, int mode, double fixed_nugget,
                       double* llh, double* grad, double* sigma_hat, int* status) {
    if (h && h->n && B == 0) return 0;                           // a rank that owns no guess of the multistart
    if (!h || !h->n || !theta || B < 1 || !llh || !grad) return h ? h->fail_msg("bad argument / no training set") : -2;
    int p_expect = h->d + ((mode & GPE_MODE_NUGGET_FREE) ? 1 : 0) + ((mode & GPE_MODE_MUCM) ? 0 : 1);
    if (p != p_expect) return h->fail_msg("p does not match d and mode");
    NvtxRange nvtx("gpe_llh_grad_batch");
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = gpe_ensure_batch_ws(h, B))) return rc;
    for (int b0 = 0; b0 < B; b0 += h->Bcap) {
        int Bs = std::min(h->Bcap, B - b0);
        CK(cudaMemcpyAsync(h->theta_d, theta + (size_t)b0 * p, sizeof(double) * Bs * p, cudaMemcpyDefault, h->st));
        gpe_handle::LlhGraph* gr = nullptr;
        if (h->graphs_stale) {      // a scratch buffer of the INT8 route was reallocated since the graphs were captured: the
            for (auto& g : h->graphs) {     // executables go, the sighting counts stay (the buffers grow in the first eager call,
                if (g.exec) cudaGraphExecDestroy(g.exec);       // so the third call of a shape still is the one that captures)
                g.exec = nullptr;
            }
            h->graphs_stale = false;
        }
        if (h->use_graphs && !h->prof_on) {
            for (auto& g : h->graphs)
                if (g.Bs == Bs && g.p == p && g.mode == mode && g.nsub == h->nsub && g.nug == fixed_nugget) gr = &g;
            if (!gr) {
                h->graphs.push_back({Bs, p, mode, h->nsub, fixed_nugget, 0, nullptr, 0});
                gr = &h->graphs.back();
            }
        }
        if (gr && gr->exec) {
            CK(cudaGraphLaunch(gr->exec, h->st));
            h->launches += gr->launches;
        } else if (gr && gr->seen >= 2) {
            // third sighting of this shape (a ragged multistart sees most batch sizes once or twice: those stay
            // eager, capture + instantiate would cost more than it saves): capture the launch sequence (all sub-batch streams join the
            // capture through the fork event), instantiate, replay
            const long long l0 = h->launches;
            cudaGraph_t graph = nullptr;
            CK(cudaStreamBeginCapture(h->st, cudaStreamCaptureModeRelaxed));
            rc = enqueue_llh_chunk(h, Bs, p, mode, fixed_nugget, true);
            cudaError_t ce = cudaStreamEndCapture(h->st, &graph);
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            if (ce != cudaSuccess) return h->fail("cudaStreamEndCapture", ce);
            gr->launches = h->launches - l0;
            ce = cudaGraphInstantiate(&gr->exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ce != cudaSuccess) { gr->exec = nullptr; return h->fail("cudaGraphInstantiate", ce); }
            cudaGraphUpload(gr->exec, h->st);       // (best effort: keeps the upload out of the first replay)
            CK(cudaGraphLaunch(gr->exec, h->st));
        } else {
            if (gr) gr->seen++;
            if ((rc = enqueue_llh_chunk(h, Bs, p, mode, fixed_nugget, false))) return rc;
        }
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(llh + b0, h->llh_d, sizeof(double) * Bs, cudaMemcpyDefault, h->st));
        CK(cudaMemcpyAsync(grad + (size_t)b0 * p, h->grad_d, sizeof(double) * Bs * p, cudaMemcpyDefault, h->st));
        if (sigma_hat) CK(cudaMemcpyAsync(sigma_hat + b0, h->sig_d, sizeof(double) * Bs, cudaMemcpyDefault, h->st));
        if (status) CK(cudaMemcpyAsync(status + b0, h->status, sizeof(int) * Bs, cudaMemcpyDefault, h->st));
    }
    // asynchronous mode: everything is ordered on the handle's stream; with device-resident inputs and outputs the caller
    // may enqueue more work (another handle's, or its own kernels on gpe_get_stream) before waiting
    const bool all_dev = gpe_is_device_ptr(theta) && gpe_is_device_ptr(llh) && gpe_is_device_ptr(grad) &&
                         (!sigma_hat || gpe_is_device_ptr(sigma_hat)) && (!status || gpe_is_device_ptr(status));
    if (!(h->async && all_dev)) CK(cudaStreamSynchronize(h->st));
    return 0;
}

int gpe_dbg_gemm(gpe_handle* h, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                 long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int accumulate,
                 int kmode, int lower, int batch, int layout) {
    if (!h) return -2;
    CK(cudaSetDevice(h->device));
    int rc = run_gemm(h, h->st, A, B, C, lda, ldb, ldc, sA, sB, sC, M, N, K, alpha, accumulate, kmode, lower, batch, layout);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->st));
    return 0;
}

int gpe_dbg_gemm_oz(gpe_handle* h, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                    long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int accumulate,
                    int kmode, int lower, int batch, int layout, int nmod, unsigned char* planesA,
                    unsigned char* planesB, unsigned char* planesD, int* sexpA, int* sexpB) {
    if (!h) return -2;
    CK(cudaSetDevice(h->device));
    GemmP p;
    p.A = A; p.B = B; p.C = C; p.lda = lda; p.ldb = ldb; p.ldc = ldc; p.sA = sA; p.sB = sB; p.sC = sC;
    p.M = M; p.N = N; p.K = K; p.alpha = alpha; p.accumulate = accumulate; p.kmode = kmode; p.lower = lower; p.batch = batch;
    if (!oz_supported(p, EPI_STORE)) return h->fail_msg("gpe_dbg_gemm_oz: shape not supported by the INT8 route");
    OzWs& ws = h->oz_ws[h->st];
    cudaError_t e = oz_gemm(p, layout, EPI_STORE, nmod, ws, h->st);
    if (e != cudaSuccess) return h->fail("oz_gemm", e);
    CK(cudaStreamSynchronize(h->st));
    const bool same = (A == B && lda == ldb && sA == sB && M == N && layout != 1);
    const size_t nA = (size_t)batch * nmod * M * K, nB = (size_t)batch * nmod * N * K, nD = (size_t)batch * nmod * M * N;
    if (planesA) CK(cudaMemcpy(planesA, ws.PA, nA, cudaMemcpyDefault));
    if (planesB) CK(cudaMemcpy(planesB, same ? ws.PA : ws.PB, nB, cudaMemcpyDefault));
    if (planesD) CK(cudaMemcpy(planesD, ws.PD, nD, cudaMemcpyDefault));
    if (sexpA) CK(cudaMemcpy(sexpA, ws.sA, sizeof(int) * (size_t)batch * M, cudaMemcpyDefault));
    if (sexpB) CK(cudaMemcpy(sexpB, same ? ws.sA : ws.sB, sizeof(int) * (size_t)batch * N, cudaMemcpyDefault));
    return 0;
}

int gpe_potrf(gpe_handle* h, const double* A, int n, int batch, double* L_out, double* Linv_out, double* logdet, int* status) {
    if (!h || !A || n < 1 || batch < 1) return h ? h->fail_msg("bad argument") : -2;
    NvtxRange nvtx("gpe_potrf");
    CK(cudaSetDevice(h->device));
    // Self-contained: the padded matrices, the scratch and the inverse factor live in stream-ordered temporaries
    // (cached by the device's memory pool between calls), so the handle's training set, batch workspace and fit
    // state are left alone.  Host inputs/outputs are staged once; padding and un-padding run on the device.
    const int npad = ((n + NB - 1) / NB) * NB, nleaf = npad / NB;
    const size_t nn = (size_t)npad * npad, per = (size_t)n * n;
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const size_t per_item = (3 * nn + 2 * per) * sizeof(double);
    const long long fit = (long long)((double)free_b * 0.6 / (double)per_item);
    if (fit < 1) return h->fail_msg("not enough device memory for one n x n factorisation");
    const int bcap = (int)std::min<long long>({(long long)batch, 64ll, fit});
    const bool a_dev = gpe_is_device_ptr(A), l_dev = L_out && gpe_is_device_ptr(L_out), i_dev = Linv_out && gpe_is_device_ptr(Linv_out);
    double *Ap = nullptr, *Sp = nullptr, *Lp = nullptr, *ldp = nullptr, *src = nullptr, *dst = nullptr;
    int* stp = nullptr;
    TmpDev t_A(h), t_S(h), t_L(h), t_ld(h), t_st(h), t_src(h), t_dst(h);
    CK(t_A.get(&Ap, bcap * nn));
    CK(t_S.get(&Sp, bcap * nn));
    CK(t_L.get(&Lp, bcap * nn));
    CK(t_ld.get(&ldp, (size_t)bcap * nleaf));
    CK(t_st.get(&stp, (size_t)bcap));
    if (!a_dev) CK(t_src.get(&src, bcap * per));
    if ((L_out && !l_dev) || (Linv_out && !i_dev)) CK(t_dst.get(&dst, bcap * per));
    FactorWs ws{Ap, Sp, Lp, npad, nleaf, ldp, stp};
    std::vector<double> ldh((size_t)bcap * nleaf), ldv(bcap);
    int rc;
    for (int b0 = 0; b0 < batch; b0 += bcap) {
        const int bs = std::min(bcap, batch - b0);
        const double* Asrc = A + b0 * per;
        if (!a_dev) {
            CK(cudaMemcpyAsync(src, Asrc, sizeof(double) * bs * per, cudaMemcpyHostToDevice, h->st));
            Asrc = src;
        }
        launch_pad_sym(Asrc, n, npad, Ap, bs, h->st);
        CK(cudaMemsetAsync(Lp, 0, sizeof(double) * bs * nn, h->st));
        CK(cudaMemsetAsync(stp, 0, sizeof(int) * bs, h->st));
        h->launches++;
        SubBatch sb{0, bs, h->st};
        if ((rc = potrf_inv_rec(h, ws, sb, 0, npad, L_out != nullptr))) return rc;
        CK(cudaGetLastError());
        auto emit = [&](const double* padded, double* user, bool user_dev) -> int {
            double* to = user_dev ? user + b0 * per : dst;
            launch_unpad_lower(padded, npad, n, to, bs, h->st);
            h->launches++;
            if (!user_dev) {
                CK(cudaMemcpyAsync(user + b0 * per, dst, sizeof(double) * bs * per, cudaMemcpyDeviceToHost, h->st));
                CK(cudaStreamSynchronize(h->st));       // dst is reused by the next output
            }
            return 0;
        };
        if (Linv_out && (rc = emit(Lp, Linv_out, i_dev))) return rc;
        if (L_out && (rc = emit(Sp, L_out, l_dev))) return rc;
        if (logdet) {
            CK(cudaMemcpyAsync(ldh.data(), ldp, sizeof(double) * bs * nleaf, cudaMemcpyDeviceToHost, h->st));
            CK(cudaStreamSynchronize(h->st));
            for (int b = 0; b < bs; b++) {
                ldv[b] = 0.0;
                for (int l = 0; l < nleaf; l++) ldv[b] += ldh[(size_t)b * nleaf + l];
            }
            CK(cudaMemcpy(logdet + b0, ldv.data(), sizeof(double) * bs, cudaMemcpyDefault));
        }
        if (status) CK(cudaMemcpyAsync(status + b0, stp, sizeof(int) * bs, cudaMemcpyDefault, h->st));
        CK(cudaStreamSynchronize(h->st));
    }
    CK(cudaGetLastError());
    return 0;
}

int gpe_dbg_potrf_inv(gpe_handle* h, const double* A, int n, int batch, double* Linv_out, double* logdet, int* status) {
    return gpe_potrf(h, A, n, batch, nullptr, Linv_out, logdet, status);
}

}  // extern "C"
