"""Covariance kernels with the reference's interface (gp_emu_uqsa/_emulatorkernels.py):
``kernel`` -- (1-nugget)*exp(-sum((x_i-x_j)/delta)^2), diagonal 1 -- and ``kernel_alt_nug`` --
exp(..), diagonal 1+nugget^2.  ``kernel_matern52`` / ``kernel_matern52_alt_nug`` are the same two
forms with the Matern 5/2 correlation R = (1 + sqrt5 r + 5 D/3) exp(-sqrt5 r), r = sqrt(D), in place of
exp(-D), D = sum((x_i-x_j)/delta)^2 (beliefs key ``kernel matern52``).  Every matrix is produced by the
CUDA kernels behind the C-ABI (K1 ``cov_build_kernel`` / ``xcov_kernel``); the classes only carry the
hyper-parameters, the covariance family and the reference's side effects (``self.A``)."""
import numpy as np

from . import _lib

np.set_printoptions(precision=6)
np.set_printoptions(suppress=True)


class _Kernel:
    kind = 0
    family = _lib.KERNEL_GAUSSIAN

    def __init__(self, dim, par):
        self.d = par.delta
        self.n = par.nugget

    def set_hp(self, d, s, n):
        self.d, self.n = d, n

    def set_params(self, x):
        """delta = leading entries; a trailing entry, if any, is the nugget (reference :20-24)."""
        k = self.d.size
        self.d = x[0:k]
        if x.size > k:
            self.n = x[-1]

    def print_kernel(self):
        print("delta:", self.d)
        print("nugget:", self.n)

    def transform(self, hp):
        return 2.0 * np.log(hp)

    def untransform(self, hp):
        return np.exp(hp / 2.0)

    # -- dense matrices for arbitrary point sets: one-off device calls on the scratch handle ----
    def _loaded_scratch(self, X):
        X = np.ascontiguousarray(X, dtype=float)
        if X.ndim == 1:
            X = X.reshape(-1, 1)
        dev = _lib.scratch_device()
        n = X.shape[0]
        dev.set_training(X, np.zeros(n), np.ones((n, 1)))
        dev.set_kernel(self.family)          # the scratch handle is shared by every kernel object
        return dev, X

    def var(self, X, predict=True):
        """Dense K(X, X).  Like the reference (which keeps ``exp_save``), remembers X for a later
        grad_delta_A / grad_nugget_A call."""
        dev, self._X_last = self._loaded_scratch(X)
        self.A = dev.cov_build(self.d, self.n, self.kind, predict, 1.0)
        return self.A

    def covar(self, XT, XV):
        dev, _ = self._loaded_scratch(XT)
        XV = np.ascontiguousarray(XV, dtype=float)
        if XV.ndim == 1:
            XV = XV.reshape(-1, 1)
        return dev.cross_cov(self.d, self.n, self.kind, XV)

    def grad_delta_A(self, X, di, s2):
        """d(s2 A)/d theta_delta[di]; reference signature (X is the column inputs[:, di]); the point
        set is the one of the last var() call, as the reference's exp_save implies."""
        if getattr(self, "_X_last", None) is None or self._X_last.shape[0] != np.size(X):
            raise _lib.GpeError("grad_delta_A: call var(X) on the same point set first")
        dev, _ = self._loaded_scratch(self._X_last)
        return dev.cov_grad(self.d, self.n, self.kind, int(di), s2)

    def grad_nugget_A(self, X, s2):
        dev, _ = self._loaded_scratch(X)
        return dev.cov_grad(self.d, self.n, self.kind, -1, s2)


class kernel(_Kernel):
    kind = 0


class kernel_alt_nug(_Kernel):
    kind = 1


class kernel_matern52(_Kernel):
    kind = 0
    family = _lib.KERNEL_MATERN52


class kernel_matern52_alt_nug(_Kernel):
    kind = 1
    family = _lib.KERNEL_MATERN52
