// Internal handle layout shared by the C-ABI translation units.
#pragma once
#include <string>
#include <vector>

#include "gpe_b200.h"
#include "gpe_gemm.cuh"
#include "gpe_kernels.cuh"
#include "gpe_ozaki.cuh"
#include <map>

struct gpe_handle {
    int device = 0, sms = 0;
    cudaStream_t st = nullptr;
    std::string err;
    long long launches = 0;
    bool async = false;          // gpe_set_async: calls whose outputs are all device memory return without the final synchronize

    // optional per-category CUDA-event timing of every launch (gpe_profile_*)
    enum { CAT_GEMM_BIG = 0, CAT_GEMM_SMALL = 1, CAT_LEAF = 2, CAT_COV = 3, CAT_GRAD = 4, CAT_OTHER = 5, CAT_LAUUM = 6,
           CAT_OZ_CONVERT = 7, CAT_OZ_GEMM = 8, CAT_OZ_COMBINE = 9, NCAT = 10 };
    bool prof_on = false;
    struct ProfRec { int cat; cudaEvent_t e0, e1; };
    std::vector<ProfRec> prof_recs;
    std::vector<cudaEvent_t> prof_pool;
    double prof_ms[NCAT] = {0};
    long long prof_cnt[NCAT] = {0};
    cudaEvent_t prof_begin(int cat, cudaStream_t s);
    void prof_end(int cat, cudaEvent_t e0, cudaStream_t s);

    // sub-batch streams: the multistart batch is split into contiguous groups that run the
    // factorisation concurrently, so one group's latency-bound leaf panels and small recursion
    // levels overlap the other groups' large DMMA GEMMs
    enum { MAX_SUB = 16 };
    int nsub = 8;
    cudaStream_t sub_st[MAX_SUB] = {nullptr};      // low priority: the large DMMA GEMMs, covariance build, gradient reduction
    cudaStream_t sub_hi[MAX_SUB] = {nullptr};      // high priority: leaf panels, small recursion levels, skinny panels
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_SUB] = {nullptr}, ev_sw[MAX_SUB] = {nullptr};
    bool use_prio = false;
    // side streams, one per (group, recursion depth): the product T = L21 L11^-1 of a node does not depend on
    // the factorisation of its A22 block, so it runs beside that whole sub-recursion (gpe_api.cu:potrf_inv_rec)
    enum { MAX_DEPTH = 10 };
    bool use_side = true;
    cudaStream_t side_st[MAX_SUB][MAX_DEPTH] = {{nullptr}};
    cudaEvent_t ev_sf[MAX_SUB][MAX_DEPTH] = {{nullptr}}, ev_sj[MAX_SUB][MAX_DEPTH] = {{nullptr}};
    int ensure_side(int g);     // measured neutral on B200 (DESIGN.md section 8): off unless GPE_PRIO=1

    // CUDA graphs of the likelihood step: the launch sequence of a (batch size, mode) pair is
    // captured the third time it is seen and replayed afterwards (one cudaGraphLaunch instead of
    // ~650 launches per stream), so the host never limits the small-n, many-stream case
    bool use_graphs = true;
    struct LlhGraph { int Bs, p, mode, nsub; double nug; int seen; cudaGraphExec_t exec; long long launches; };
    std::vector<LlhGraph> graphs;
    void drop_graphs();
    bool graphs_stale = false;

    // training set (device)
    int n = 0, d = 0, q = 0, npad = 0, nleaf = 0;
    double *X = nullptr, *y = nullptr, *H = nullptr, *r = nullptr, *HY = nullptr;
    bool has_basis = false;
    int family = gpe::FAMILY_GAUSSIAN;   // covariance function of every call (gpe_set_kernel)
    int basis_idx[gpe::NR] = {0}, basis_pow[gpe::NR] = {0};

    // batched likelihood workspace
    int Bcap = 0;
    bool Bcap_final = false;
    bool grad_use_e = false;     // classic route with the covariance build's copy of exp(-D) (INT8 route)
    int grad_fused = 0;          // gradient route of the current chunk (gpe_api.cu:llh_grad_fused): 0 classic, 1 split W/E, 2 epilogue     // the workspace already has the largest size obtainable (env cap or device memory)
    double *A = nullptr, *S = nullptr, *Li = nullptr;        // [Bcap][npad][npad]
    double* Ex = nullptr;                                    // [Bcap][npad][npad] exp(-D) kept by the covariance build for the fused gradient epilogue
    double *Wy = nullptr, *Z = nullptr, *U = nullptr;        // [Bcap][npad][NR]
    double *GP = nullptr, *logdet_part = nullptr, *winv = nullptr, *beta = nullptr, *gpart = nullptr;
    gpe::ItemPar* par = nullptr;
    gpe::ItemOut* out = nullptr;
    int* status = nullptr;
    double *theta_d = nullptr, *llh_d = nullptr, *grad_d = nullptr, *sig_d = nullptr;

    // fit state for prediction (gpe_predict.cu)
    bool fitted = false;
    int fit_kind = 0;
    double fit_nugget = 0, fit_sigma = 1, fit_c = 1, fit_astar = 1;
    double *fLi = nullptr;       // [npad][npad]  L^-1 of the training matrix
    double *fE = nullptr;        // [npad][NR]    U = [A^-1 H K^-T | A^-1 (y - H beta)]
    double *fK = nullptr;        // [NR][NR]      Cholesky factor of Q = H^T A^-1 H (host-filled)
    double *fbeta = nullptr;     // [NR]
    double *fwinv = nullptr;     // [d]
    double *fXs = nullptr;       // [d][npad] scaled training inputs, k-major
    double *fAinv = nullptr;     // [npad][npad] A^-1 (lower 128-tiles), built on demand for the sensitivity traces
    bool fAinv_valid = false;
    // prediction chunk workspace
    long long pchunk = 0;
    // two slots: consecutive chunks alternate between two streams so that one chunk's cross-covariance /
    // skinny product / finalize overlap the other's TRMM
    struct PredSlot { double *C = nullptr, *Part = nullptr, *Aux = nullptr, *X = nullptr, *H = nullptr, *Mean = nullptr, *Var = nullptr; };
    PredSlot ps[2];

    // FP64 GEMMs emulated on the INT8 tensor cores (gpe_ozaki.cuh): number of moduli (GPE_OZAKI; 0 = off: DMMA everywhere),
    // smallest dimension that takes the route (GPE_OZAKI_MIN), scratch per stream
    int oz_nmod = 16, oz_min = 1024, oz_nsub = 2;
    std::map<cudaStream_t, gpe::OzWs> oz_ws;
    long long oz_calls = 0;
    unsigned long long oz_a_tag = 0, fit_gen = 0;   // tag of operand A for the next product; generation of the fit state
    double oz_b_bound = 0.0;     // the next product's operand B is bounded by this in magnitude (0: unknown; one product only)
    bool oz_reuse_a = false;     // the next product may use the residue planes of operand A left by the previous one

    int fail(const char* what, cudaError_t e);
    int fail_msg(const char* what);
    void free_batch_ws();
    void free_training();
    void free_fit();
};

struct ProfScope {
    gpe_handle* h; int cat; cudaStream_t s; cudaEvent_t e0;
    ProfScope(gpe_handle* h_, int c, cudaStream_t s_ = nullptr) : h(h_), cat(c), s(s_ ? s_ : h_->st), e0(h_->prof_begin(c, s)) {}
    ~ProfScope() { h->prof_end(cat, e0, s); }
};

// items [b0, b0 + B) of the batch workspace.  A group owns a low-priority stream `st` for its large
// kernels and (optionally) a high-priority stream `hi` for its latency-bound small ones: the block
// scheduler hands freed SMs to high-priority grids first, so one group's leaf panels and small
// recursion levels run inside another group's big GEMM instead of waiting for its tail.  `stream(small)`
// returns the stream for the next launch and orders it after everything the group has enqueued so far.
struct SubBatch {
    int b0, B;
    cudaStream_t st;
    cudaStream_t hi = nullptr;
    cudaEvent_t ev = nullptr;
    mutable bool on_hi = false;
    cudaStream_t* side = nullptr;      // [MAX_DEPTH] side streams of this group (nullptr: everything in order on st)
    cudaEvent_t *ef = nullptr, *ej = nullptr;
    cudaStream_t stream(bool small) const {
        if (!hi || small == on_hi) return on_hi ? hi : st;
        cudaStream_t from = on_hi ? hi : st, to = small ? hi : st;
        cudaEventRecord(ev, from);
        cudaStreamWaitEvent(to, ev, 0);
        on_hi = small;
        return to;
    }
    cudaStream_t current() const { return on_hi ? hi : st; }
};

// Stream-ordered temporary device buffer (cudaMallocAsync / cudaFreeAsync on the handle's stream): released
// on every exit path of the entry point that owns it, after the work already enqueued on that stream; the
// device's default memory pool keeps the memory cached between calls (release threshold set in gpe_create),
// so repeated calls do not pay a device allocation.  Declare at function scope, before the first launch.
struct TmpDev {
    cudaStream_t st;
    void* p = nullptr;
    explicit TmpDev(gpe_handle* h) : st(h->st) {}
    TmpDev(const TmpDev&) = delete;
    TmpDev& operator=(const TmpDev&) = delete;
    ~TmpDev() { if (p) cudaFreeAsync(p, st); }
    template <class T>
    cudaError_t get(T** out, size_t count) {
        cudaError_t e = cudaMallocAsync(&p, count ? count * sizeof(T) : sizeof(T), st);
        *out = (e == cudaSuccess) ? static_cast<T*>(p) : nullptr;
        return e;
    }
};

// The buffers one batched recursive factorisation works on (items are addressed through SubBatch::b0):
// A [B][npad][npad] in (identity padded), overwritten; S scratch (ends up holding the Cholesky factor when asked
// for); Li <- L^-1 (upper blocks must be zero on entry); logdet_part [B][nleaf]; status [B].
struct FactorWs {
    double *A, *S, *Li;
    int npad, nleaf;
    double* logdet_part;
    int* status;
};

// NVTX range over a C-ABI entry point (SURVEY section 5: makes nsys traces of g.train readable)
struct NvtxRange {
    explicit NvtxRange(const char* name);
    ~NvtxRange();
};

bool gpe_is_device_ptr(const void* p);
int gpe_ensure_batch_ws(gpe_handle* h, int B);
int gpe_potrf_inv(gpe_handle* h, const FactorWs& ws, const SubBatch& sb, int want_L);
int gpe_factor_and_reduce(gpe_handle* h, const SubBatch& sb, int mode, int with_grad, const double* beta_override, double* Kout);
int gpe_upload_single_par(gpe_handle* h, const double* delta, double nugget, int kind, int predict, double s2_for_r);
bool gpe_oz_reserve(gpe_handle* h, cudaStream_t st, const gpe::GemmP& p);
int gpe_run_gemm_on(gpe_handle* h, cudaStream_t st, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                    long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int acc,
                    int kmode, int lower, int batch, int layout, int epi);
int gpe_run_gemm(gpe_handle* h, const double* A, const double* B, double* C, int lda, int ldb, int ldc,
                 long long sA, long long sB, long long sC, int M, int N, int K, double alpha, int acc,
                 int kmode, int lower, int batch, int layout, int epi);
