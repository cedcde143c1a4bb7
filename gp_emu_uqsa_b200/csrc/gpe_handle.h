// Internal handle layout shared by the C-ABI translation units.
#pragma once
#include <optional>
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
    cudaStream_t sub_st[MAX_SUB] = {nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_SUB] = {nullptr};
    // side streams, one per (group, recursion depth): the product T = L21 L11^-1 of a node does not depend on
    // the factorisation of its A22 block, so it runs beside that whole sub-recursion (gpe_api.cu:potrf_inv_rec)
    enum { MAX_DEPTH = 10 };
    cudaStream_t side_st[MAX_SUB][MAX_DEPTH] = {{nullptr}};
    cudaEvent_t ev_sf[MAX_SUB][MAX_DEPTH] = {{nullptr}}, ev_sj[MAX_SUB][MAX_DEPTH] = {{nullptr}};
    int ensure_side(int g);     // creates the side streams of group g on first use

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
    bool Bcap_final = false;     // the workspace already has the largest size obtainable (env cap or device memory)
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
    double fit_dbeta[gpe::NR] = {0};     // GLS beta minus the beta the state was fitted with (gpe_loo re-estimates beta)
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
    unsigned long long fit_gen = 0;   // generation of the fit state (tags the prediction product's residue planes of L^-1)

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

// items [b0, b0 + B) of the batch workspace.  A group launches in order on its stream `st`; only the
// products T = L21 L11^-1 of the recursion go to its side streams.
struct SubBatch {
    int b0, B;
    cudaStream_t st;
    cudaStream_t* side = nullptr;      // [MAX_DEPTH] side streams of this group (nullptr: everything in order on st)
    cudaEvent_t *ef = nullptr, *ej = nullptr;
};

// Return h->fail from the enclosing entry point when a CUDA call fails (needs `gpe_handle* h` in scope).
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return h->fail(#call, e__);        \
    } while (0)

// Device buffers the handle keeps between calls
template <class T>
inline cudaError_t dev_alloc(T** p, size_t count) {
    return cudaMalloc((void**)p, (count ? count : 1) * sizeof(T));
}
template <class T>
inline void dev_free(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

bool gpe_is_device_ptr(const void* p);

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

// A caller's input array of `count` elements (host or device memory: each buffer is looked at on its own) as a device pointer
// `p`: the caller's own pointer when it is device memory, else a stream-ordered copy into a temporary.  Null stays null.
template <class T>
struct DevIn {
    TmpDev tmp;
    const T* p = nullptr;
    explicit DevIn(gpe_handle* h) : tmp(h) {}
    cudaError_t stage(const T* src, size_t count) {
        p = src;
        if (!src || gpe_is_device_ptr(src)) return cudaSuccess;
        T* d;
        const cudaError_t e = tmp.get(&d, count);
        p = d;
        return e != cudaSuccess ? e : cudaMemcpyAsync(d, src, count * sizeof(T), cudaMemcpyHostToDevice, tmp.st);
    }
};

// A caller's output array of `count` elements as a device pointer `p` to write through: the caller's own pointer when it is
// device memory, else `scratch` (a device buffer of at least count elements) if given, else a temporary; flush() enqueues
// the copy back to host memory after the writes.  A null pointer leaves p null and flush() a no-op (optional outputs).
template <class T>
struct DevOut {
    TmpDev tmp;
    T* dst = nullptr;
    T* p = nullptr;
    size_t count = 0;
    explicit DevOut(gpe_handle* h) : tmp(h) {}
    cudaError_t stage(T* out, size_t n, T* scratch = nullptr) {
        p = out;
        if (!out || gpe_is_device_ptr(out)) return cudaSuccess;
        dst = out;
        count = n;
        if (scratch) { p = scratch; return cudaSuccess; }
        return tmp.get(&p, n);
    }
    cudaError_t flush() {
        return (dst && count) ? cudaMemcpyAsync(dst, p, count * sizeof(T), cudaMemcpyDeviceToHost, tmp.st) : cudaSuccess;
    }
};

// Appends `count` elements of a short caller array (host or device memory) to the host vector v.
template <class T>
inline cudaError_t read_small(std::vector<T>& v, const T* p, size_t count) {
    v.resize(v.size() + count);
    return cudaMemcpy(v.data() + v.size() - count, p, count * sizeof(T), cudaMemcpyDefault);
}

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

int gpe_ensure_batch_ws(gpe_handle* h, int B);
int gpe_potrf_inv(gpe_handle* h, const FactorWs& ws, const SubBatch& sb, int want_L);
// How the likelihood gradient of a chunk is reduced (gpe_api.cu:grad_route): not at all (fit state), in the LAUUM epilogue, or by
// the stand-alone reduction kernel after A^-1 is stored, recomputing exp(-D) or reading the covariance build's copy of it.
enum GradRoute { GRAD_NONE, GRAD_FUSED, GRAD_CLASSIC, GRAD_CLASSIC_E };
int gpe_factor_and_reduce(gpe_handle* h, const SubBatch& sb, int mode, GradRoute grad, const double* beta_override, double* Kout);
// One item's parameters into h->par / h->winv from the caller's delta [d] (host or device); offs replaces ItemPar::offs.
int gpe_upload_single_par(gpe_handle* h, const double* delta, double nugget, int kind, int predict, double s2_for_r, std::optional<double> offs = {});
// Does product p take the INT8 route on stream st?  Yes when its shape does (route on, every dimension >= oz_min, supported) and
// the stream's residue scratch can hold it; the scratch is grown here, and on an allocation failure the error is cleared and the
// product stays on DMMA.
bool gpe_int8_route(gpe_handle* h, cudaStream_t st, const gpe::GemmP& p, int layout, int epi);
// C = alpha op(A) op(B) (+ C) on the route int8 names, which a caller that plans around the route (the prediction chunk) has
// taken from gpe_int8_route, once.  cat: profile category of a DMMA launch (-1: by shape).
int gpe_gemm_routed(gpe_handle* h, cudaStream_t st, const gpe::GemmP& p, int layout, int epi, bool int8, const gpe::OzHint& hint,
                    int cat = -1);
// Every other dense product: the same on the route gpe_int8_route picks.
inline int gpe_gemm(gpe_handle* h, cudaStream_t st, const gpe::GemmP& p, int layout, int epi = gpe::EPI_STORE,
                    const gpe::OzHint& hint = gpe::OzHint(), int cat = -1) {
    return gpe_gemm_routed(h, st, p, layout, epi, gpe_int8_route(h, st, p, layout, epi), hint, cat);
}
