"""ctypes binding of libgpe_b200.so (include/gpe_b200.h) -- the drop-in boundary.

There is no CPU fallback: importing this module without the built library, or creating a
``Device`` without an sm_100 GPU, raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgpe_b200.so")

MODE_MUCM, MODE_ALT_NUGGET, MODE_NUGGET_FREE = 1, 2, 4
KERNEL_GAUSSIAN, KERNEL_MATERN52 = 0, 1
KM_FULL, KM_LE_J, KM_GE_J, KM_LE_I, KM_GE_I = 0, 1, 2, 3, 4

_dp = C.c_void_p
_lib = None


class GpeError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and declare every prototype of include/gpe_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpeError("libgpe_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "or `make -C gp_emu_uqsa_b200/csrc`); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    i, d, ll, p = C.c_int, C.c_double, C.c_longlong, _dp
    proto = {
        "gpe_version": (i, []),
        "gpe_create": (i, [i, C.POINTER(p)]),
        "gpe_destroy": (i, [p]),
        "gpe_last_error": (C.c_char_p, [p]),
        "gpe_launch_count": (ll, [p]),
        "gpe_dbg_int8_products": (ll, [p]),
        "gpe_get_stream": (p, [p]),
        "gpe_set_streams": (i, [p, i]),
        "gpe_set_async": (i, [p, i]),
        "gpe_set_kernel": (i, [p, i]),
        "gpe_synchronize": (i, [p]),
        "gpe_profile_enable": (i, [p, i]),
        "gpe_profile_read": (i, [p, p, p, i]),
        "gpe_set_training": (i, [p, p, p, p, p, i, i, i]),
        "gpe_set_basis": (i, [p, p, p, i]),
        "gpe_cov_build": (i, [p, p, d, i, i, d, p]),
        "gpe_cov_grad": (i, [p, p, d, i, i, d, p]),
        "gpe_cross_cov": (i, [p, p, d, i, p, i, p]),
        "gpe_llh_grad_batch": (i, [p, p, i, i, i, d, p, p, p, p]),
        "gpe_fit_state": (i, [p, p, d, d, i, d, p, p, p, p]),
        "gpe_predict": (i, [p, p, p, ll, p, p]),
        "gpe_predict_grid": (i, [p, p, p, p, ll, ll, p, p]),
        "gpe_predict_fullcov": (i, [p, p, p, i, p, p, p]),
        "gpe_implausibility": (i, [p, p, p, i, ll, p, p, d, i, ll, ll, ll, p, p, p, p, p]),
        "gpe_predict_implaus": (i, [p, p, p, p, p, p, ll, ll, d, d, i, i, i, p, d, ll, ll, ll, p, p, p, p]),
        "gpe_solve": (i, [p, p, i, p]),
        "gpe_sens_contract": (i, [p, p, p, p, d, p, i, p, p]),
        "gpe_sens_main_effect": (i, [p, p, p, p, p, p, d, p, i, p, i, p]),
        "gpe_dbg_gemm": (i, [p, p, p, p, i, i, i, ll, ll, ll, i, i, i, d, i, i, i, i, i]),
        "gpe_dbg_gemm_oz": (i, [p, p, p, p, i, i, i, ll, ll, ll, i, i, i, d, i, i, i, i, i, i, p, p, p, p, p]),
        "gpe_potrf": (i, [p, p, i, i, p, p, p, p]),
        "gpe_pdist_argmin": (i, [p, p, i, i, i, p, i, p]),
        "gpe_dbg_potrf_inv": (i, [p, p, i, i, p, p, p]),
    }
    for name, (res, args) in proto.items():
        fn = getattr(L, name)          # AttributeError here == header/library mismatch
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


EXPORTS = ["gpe_version", "gpe_create", "gpe_destroy", "gpe_last_error", "gpe_launch_count",
           "gpe_get_stream", "gpe_set_streams", "gpe_set_async", "gpe_set_kernel", "gpe_synchronize", "gpe_profile_enable", "gpe_profile_read",
           "gpe_set_training", "gpe_set_basis", "gpe_cov_build", "gpe_cov_grad", "gpe_cross_cov", "gpe_llh_grad_batch",
           "gpe_fit_state", "gpe_predict", "gpe_predict_grid", "gpe_predict_fullcov", "gpe_implausibility", "gpe_predict_implaus",
           "gpe_solve", "gpe_sens_contract", "gpe_sens_main_effect", "gpe_potrf", "gpe_pdist_argmin",
           "gpe_dbg_gemm", "gpe_dbg_gemm_oz", "gpe_dbg_potrf_inv", "gpe_dbg_int8_products"]


def default_device_index():
    """GPU of this process: GPE_DEVICE, else LOCAL_RANK (one process per GPU under torchrun), else 0."""
    return int(os.environ.get("GPE_DEVICE", os.environ.get("LOCAL_RANK", "0")))


_scratch = None


def scratch_device():
    """A process-wide handle for one-off device work that is not tied to a training set
    (kernel.var on arbitrary points, Cholesky of a small posterior covariance)."""
    global _scratch
    if _scratch is None:
        _scratch = Device(default_device_index())
    return _scratch


def _ptr(a):
    """Raw address of a NumPy array (host) or torch tensor (device/pinned host); None -> NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if a.is_cuda:
        # the handle works on its own non-blocking stream: whatever torch has queued for this tensor (a fill, a clone)
        # must have finished before the library reads or writes it
        import torch
        torch.cuda.current_stream(a.device).synchronize()
    return a.data_ptr()          # torch.Tensor


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Device:
    """One handle per GPU per process (gpe_create / gpe_destroy)."""

    def __init__(self, device=0):
        self.L = load()
        self.h = _dp()
        rc = self.L.gpe_create(int(device), C.byref(self.h))
        if rc != 0:
            why = {-3: "no usable CUDA device", -4: "device is not sm_100 (B200)"}.get(rc, "bad device index")
            raise GpeError("gpe_create failed (%d): %s; there is no CPU fallback" % (rc, why))
        self.device = int(device)
        self.n = self.d = self.q = 0
        self._keep = []

    def close(self):
        if getattr(self, "h", None):
            self.L.gpe_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise GpeError("gpe error %d: %s" % (rc, self.L.gpe_last_error(self.h).decode()))

    @property
    def launches(self):
        return int(self.L.gpe_launch_count(self.h))

    @property
    def int8_products(self):
        """Products sent down the INT8 tensor-core route so far (csrc/gpe_ozaki.cuh)."""
        return int(self.L.gpe_dbg_int8_products(self.h))

    @property
    def stream_ptr(self):
        """cudaStream_t of the handle (wrap with torch.cuda.ExternalStream to record events)."""
        return int(self.L.gpe_get_stream(self.h) or 0)

    PROFILE_CATEGORIES = ("gemm_dmma_128", "gemm_dmma_small", "potrf_leaf", "cov_build", "grad_reduce", "other", "lauum",
                          "int8_residue_conversion", "int8_residue_gemm", "int8_crt_combine")

    def set_streams(self, nstreams):
        """Number of concurrent sub-batch streams of llh_grad_batch (1 = serial launches)."""
        self._ck(self.L.gpe_set_streams(self.h, int(nstreams)))

    def set_kernel(self, family):
        """Covariance family of every later call (KERNEL_GAUSSIAN / KERNEL_MATERN52); a change drops the fit state."""
        self._ck(self.L.gpe_set_kernel(self.h, int(family)))

    def set_async(self, on=True):
        """Calls whose inputs and outputs are all device tensors return once enqueued; ``synchronize()`` waits."""
        self._ck(self.L.gpe_set_async(self.h, int(bool(on))))

    def synchronize(self):
        self._ck(self.L.gpe_synchronize(self.h))

    def profile_enable(self, on=True):
        self._ck(self.L.gpe_profile_enable(self.h, int(bool(on))))

    def profile_read(self, reset=True):
        ms = np.zeros(len(self.PROFILE_CATEGORIES))
        cnt = np.zeros(len(self.PROFILE_CATEGORIES), dtype=np.int64)
        self._ck(self.L.gpe_profile_read(self.h, _ptr(ms), _ptr(cnt), int(bool(reset))))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROFILE_CATEGORIES)}

    # ------------------------------------------------------------------ training set
    def set_training(self, X, y, H, r=None):
        X, y, H = _f64(X), _f64(y), _f64(H)
        if X.ndim == 1:
            X = X.reshape(-1, 1)
        r = None if r is None or np.ndim(r) == 0 else _f64(r)
        n, d = X.shape
        q = H.shape[1]
        self._ck(self.L.gpe_set_training(self.h, _ptr(X), _ptr(y), _ptr(H), _ptr(r), n, d, q))
        self.n, self.d, self.q = n, d, q

    def set_basis(self, idx, powers):
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        powers = np.ascontiguousarray(powers, dtype=np.int32)
        self._ck(self.L.gpe_set_basis(self.h, _ptr(idx), _ptr(powers), 1 + len(idx)))

    # ------------------------------------------------------------------ K1
    def cov_build(self, delta, nugget, kind=0, predict=True, s2=1.0, out=None):
        delta = _f64(delta)
        A = np.empty((self.n, self.n)) if out is None else out
        self._ck(self.L.gpe_cov_build(self.h, _ptr(delta), float(nugget), int(kind), int(bool(predict)), float(s2), _ptr(A)))
        return A

    def cov_grad(self, delta, nugget, kind, which, s2):
        """Dense grad_delta_A (which = dimension) / grad_nugget_A (which = -1)."""
        delta = _f64(delta)
        G = np.empty((self.n, self.n))
        self._ck(self.L.gpe_cov_grad(self.h, _ptr(delta), float(nugget), int(kind), int(which), float(s2), _ptr(G)))
        return G

    def cross_cov(self, delta, nugget, kind, Xs, out=None):
        delta, Xs = _f64(delta), _f64(Xs)
        m = Xs.shape[0]
        Cm = np.empty((self.n, m)) if out is None else out
        self._ck(self.L.gpe_cross_cov(self.h, _ptr(delta), float(nugget), int(kind), _ptr(Xs), m, _ptr(Cm)))
        return Cm

    # ------------------------------------------------------------------ K2/K3/K1g
    def llh_grad_batch(self, theta, mode, fixed_nugget=0.0, out=None):
        """theta: [B,p] NumPy (host) or torch CUDA tensor.  Returns (llh, grad, sigma_hat, status)
        as NumPy arrays, or writes into the torch tensors given in ``out``."""
        if isinstance(theta, np.ndarray) or not hasattr(theta, "data_ptr"):
            theta = _f64(np.atleast_2d(theta))
        B, p = int(theta.shape[0]), int(theta.shape[1])
        if out is None:
            llh, grad = np.empty(B), np.empty((B, p))
            sig, status = np.empty(B), np.zeros(B, dtype=np.int32)
        else:
            llh, grad, sig, status = out
        self._ck(self.L.gpe_llh_grad_batch(self.h, _ptr(theta), B, p, int(mode), float(fixed_nugget),
                                           _ptr(llh), _ptr(grad), _ptr(sig), _ptr(status)))
        return llh, grad, sig, status

    # ------------------------------------------------------------------ K4
    def fit_state(self, delta, nugget, sigma, kind=0, beta=None, r_div=1.0):
        delta = _f64(delta)
        beta_in = None if beta is None else _f64(beta)
        beta_out = np.empty(self.q)
        sig = C.c_double(0.0)
        st = C.c_int(0)
        self._ck(self.L.gpe_fit_state(self.h, _ptr(delta), float(nugget), float(sigma), int(kind), float(r_div), _ptr(beta_in),
                                      _ptr(beta_out), C.addressof(sig), C.addressof(st)))
        return beta_out, float(sig.value), int(st.value)

    def predict(self, Xs, Hs=None, want_var=True, out=None):
        host = isinstance(Xs, np.ndarray) or not hasattr(Xs, "data_ptr")
        if host:
            Xs = _f64(Xs)
            Hs = None if Hs is None else _f64(Hs)
        m = int(Xs.shape[0])
        if out is None:
            mean = np.empty(m)
            var = np.empty(m) if want_var else None
        else:
            mean, var = out
        self._ck(self.L.gpe_predict(self.h, _ptr(Xs), _ptr(Hs), m, _ptr(mean), _ptr(var)))
        return mean, var

    def predict_grid(self, levels, lo, hi, start, count, want_var=True, out=None):
        levels = np.ascontiguousarray(levels, dtype=np.int32)
        lo, hi = _f64(lo), _f64(hi)
        if out is None:
            mean = np.empty(count)
            var = np.empty(count) if want_var else None
        else:
            mean, var = out
        self._ck(self.L.gpe_predict_grid(self.h, _ptr(levels), _ptr(lo), _ptr(hi), int(start), int(count), _ptr(mean), _ptr(var)))
        return mean, var

    def predict_fullcov(self, Xs, Hs=None, r_new=None):
        Xs = _f64(Xs)
        Hs = None if Hs is None else _f64(Hs)
        r_new = None if r_new is None or np.ndim(r_new) == 0 else _f64(r_new)
        m = Xs.shape[0]
        mean, V = np.empty(m), np.empty((m, m))
        self._ck(self.L.gpe_predict_fullcov(self.h, _ptr(Xs), _ptr(Hs), m, _ptr(r_new), _ptr(mean), _ptr(V)))
        return mean, V

    # ------------------------------------------------------------------ K5
    def implausibility(self, mean, var, z, var_extra, cm, maxno=1, ncell=0, want_imax=True, out=None, cell_pts=0, first_index=0):
        """Implausibility of m points from per-emulator mean/var [n_emul, m].  Cells: either ``ncell`` equal
        contiguous cells of the m points, or (``cell_pts`` > 0) runs of cell_pts points of the global flat index
        ``first_index + r`` -- a shard of a larger point set that may start and end inside a cell; cmin / ccnt then
        cover the cells first_index // cell_pts ... (first_index + m - 1) // cell_pts."""
        host = isinstance(mean, np.ndarray)
        if host:
            mean, var = _f64(np.atleast_2d(mean)), _f64(np.atleast_2d(var))
        n_emul, m = int(mean.shape[0]), int(mean.shape[1])
        z, var_extra = _f64(z), _f64(var_extra)
        if out is None:
            Imax = np.empty((m, maxno)) if want_imax else None
            keep = np.empty(m, dtype=np.uint8)
        else:
            Imax, keep = out
        if cell_pts:
            ncell = (first_index + m - 1) // cell_pts - first_index // cell_pts + 1 if m else 0
        elif ncell:
            if m % ncell:
                raise GpeError("m must be a multiple of ncell")
            cell_pts, first_index = m // ncell, 0
        count = np.zeros(maxno, dtype=np.uint64)
        cmin = np.empty((ncell, maxno)) if ncell else None
        ccnt = np.zeros((ncell, maxno), dtype=np.uint64) if ncell else None
        self._ck(self.L.gpe_implausibility(self.h, _ptr(mean), _ptr(var), n_emul, m, _ptr(z), _ptr(var_extra), float(cm),
                                           int(maxno), int(cell_pts), int(first_index), int(ncell), _ptr(Imax), _ptr(keep),
                                           _ptr(count), _ptr(cmin), _ptr(ccnt)))
        return Imax, keep, count, cmin, ccnt

    def predict_implaus(self, z, var_extra, Itop, first, last, points=None, Hs=None, grid=None, maxno=1, cm=0.0, cell_pts=0,
                        first_index=0, keep=None):
        """Prediction of this emulator folded into the running top-``maxno`` implausibility list ``Itop`` [m, maxno]
        (torch CUDA tensor, ascending; see gpe_predict_implaus).  ``points``: NumPy [m,d] or torch CUDA tensor; or
        ``grid`` = (levels, lo, hi, start, m).  On the last emulator returns (count_lt, cell_min, cell_count) and fills
        ``keep`` (torch uint8 tensor or NumPy array) if given; otherwise returns None."""
        if points is not None:
            if isinstance(points, np.ndarray) or not hasattr(points, "data_ptr"):
                points = _f64(points)
                Hs = None if Hs is None else _f64(Hs)
            m, lv, lo, hi, start = int(points.shape[0]), None, None, None, 0
        else:
            lv, lo, hi, start, m = grid
            lv = np.ascontiguousarray(lv, dtype=np.int32)
            lo, hi, start, m = _f64(lo), _f64(hi), int(start), int(m)
        ncell = 0
        if last and cell_pts and m:
            ncell = (first_index + m - 1) // cell_pts - first_index // cell_pts + 1
        count = np.zeros(maxno, dtype=np.uint64) if last else None
        cmin = np.empty((ncell, maxno)) if ncell else None
        ccnt = np.zeros((ncell, maxno), dtype=np.uint64) if ncell else None
        self._ck(self.L.gpe_predict_implaus(self.h, _ptr(points), _ptr(Hs), _ptr(lv), _ptr(lo), _ptr(hi), start, m, float(z),
                                            float(var_extra), int(maxno), int(bool(first)), int(bool(last)), _ptr(Itop), float(cm),
                                            int(cell_pts), int(first_index), int(ncell), _ptr(keep), _ptr(count), _ptr(cmin), _ptr(ccnt)))
        return (count, cmin, ccnt) if last else None

    # ------------------------------------------------------------------ K6
    def solve(self, Bm):
        """A^-1 Bm for the matrix factored by fit_state; Bm [n] or [n,k]."""
        Bm = _f64(Bm)
        one = Bm.ndim == 1
        B2 = Bm.reshape(self.n, -1)
        out = np.empty_like(B2)
        self._ck(self.L.gpe_solve(self.h, _ptr(B2), int(B2.shape[1]), _ptr(out)))
        return out[:, 0] if one else out

    def sens_contract(self, gamma, acoef, mvec, scale, V):
        """(tr(A^-1 P), V^T P V) for the product-form matrix P (see gpe_sens_contract)."""
        gamma, acoef, mvec, V = _f64(gamma), _f64(acoef), _f64(mvec), _f64(V)
        nv = V.shape[1]
        tr = C.c_double(0.0)
        M = np.empty((nv, nv))
        self._ck(self.L.gpe_sens_contract(self.h, _ptr(gamma), _ptr(acoef), _ptr(mvec), float(scale), _ptr(V), nv,
                                          C.addressof(tr), _ptr(M)))
        return float(tr.value), M

    def sens_main_effect(self, t1, t2, cdiag, mvec, evec, scale, which, xw):
        """Tw(x_w) . e for every input in `which` and every x_w value xw [len(which), points]."""
        t1, t2, cdiag, mvec, evec, xw = (_f64(a) for a in (t1, t2, cdiag, mvec, evec, xw))
        which = np.ascontiguousarray(which, dtype=np.int32)
        out = np.empty_like(xw)
        self._ck(self.L.gpe_sens_main_effect(self.h, _ptr(t1), _ptr(t2), _ptr(cdiag), _ptr(mvec), _ptr(evec), float(scale),
                                             _ptr(which), len(which), _ptr(xw), int(xw.shape[1]), _ptr(out)))
        return out

    # ------------------------------------------------------------------ dense Cholesky
    def cholesky(self, A):
        """np.linalg.cholesky(A) on device (lower factor); raises LinAlgError when A is not PD."""
        A = _f64(A)
        n = A.shape[0]
        Lf, st = np.empty_like(A), np.zeros(1, dtype=np.int32)
        self._ck(self.L.gpe_potrf(self.h, _ptr(A), n, 1, _ptr(Lf), None, None, _ptr(st)))
        if st[0] != 0:
            raise np.linalg.LinAlgError("Matrix is not positive definite")
        return Lf

    # ------------------------------------------------------------------ design criterion
    def pdist_argmin(self, designs, extra=None):
        """np.argmin(pdist(concat(design, extra), 'sqeuclidean')) for every design of designs [N, n, dim]."""
        designs = _f64(designs)
        N, n, dim = designs.shape
        extra = None if extra is None else _f64(extra).reshape(-1, dim)
        out = np.empty(N, dtype=np.int64)
        self._ck(self.L.gpe_pdist_argmin(self.h, _ptr(designs), N, n, dim, _ptr(extra), 0 if extra is None else extra.shape[0], _ptr(out)))
        return out

    # ------------------------------------------------------------------ debug
    def dbg_potrf_inv(self, A):
        A = _f64(A)
        if A.ndim == 2:
            A = A[None]
        b, n = A.shape[0], A.shape[1]
        Li, ld, st = np.empty_like(A), np.empty(b), np.zeros(b, dtype=np.int32)
        self._ck(self.L.gpe_dbg_potrf_inv(self.h, _ptr(A), n, b, _ptr(Li), _ptr(ld), _ptr(st)))
        return Li, ld, st

    def dbg_gemm_oz(self, A, B, Cm, M, N, K, lda, ldb, ldc, sA=0, sB=0, sC=0, alpha=1.0, accumulate=0, kmode=0,
                    lower=0, batch=1, layout=0, nmod=18, planesA=None, planesB=None, planesD=None, sexpA=None, sexpB=None):
        """The product of dbg_gemm on the INT8 tensor-core route (device tensors; optional outputs: residue planes, exponents)."""
        self._ck(self.L.gpe_dbg_gemm_oz(self.h, _ptr(A), _ptr(B), _ptr(Cm), lda, ldb, ldc, sA, sB, sC, M, N, K,
                                        float(alpha), int(accumulate), int(kmode), int(lower), int(batch), int(layout), int(nmod),
                                        _ptr(planesA), _ptr(planesB), _ptr(planesD), _ptr(sexpA), _ptr(sexpB)))

    def dbg_gemm(self, A, B, Cm, M, N, K, lda, ldb, ldc, sA=0, sB=0, sC=0, alpha=1.0, accumulate=0, kmode=0,
                 lower=0, batch=1, layout=0):
        self._ck(self.L.gpe_dbg_gemm(self.h, _ptr(A), _ptr(B), _ptr(Cm), lda, ldb, ldc, sA, sB, sC, M, N, K,
                                     float(alpha), int(accumulate), int(kmode), int(lower), int(batch), int(layout)))
