"""TEST INFRASTRUCTURE ONLY -- CPU oracle of leave-one-out (LOO) cross-validation.

The reference has no LOO: this states the model the library implements, in NumPy, for both covariance families (the
matrix A of a mode is built with ``gp_oracle.make_A`` / ``matern_oracle.make_A``, exactly as the likelihood of that mode
factors it: MUCM the correlation matrix plus un-scaled r; gp4ml sigma^2 times it, with r).

Closed form (universal kriging, beta re-estimated by GLS on the n - 1 remaining points, flat prior on beta):
    P = A^-1 - A^-1 H (H^T A^-1 H)^-1 H^T A^-1,  alpha = P y,
    e_i = y_i - mu_-i = alpha_i / P_ii,   v_i = s^2 / P_ii,
    L = 1/2 sum_i [ log(2 pi v_i) + e_i^2 / v_i ]     (s^2 = 1 gp4ml; MUCM: s^2 = (1/n) sum_i alpha_i^2 / P_ii, profiled)
    dL/dtheta_k = sum_ab W_ab dA_ab/dtheta_k,  W = F F^T - 1/2 [(P c) alpha^T + alpha (P c)^T],  F = P diag(sqrt w),
    w_i = 1/2 (1/P_ii + alpha_i^2 / (s^2 P_ii^2)),  c_i = alpha_i / (s^2 P_ii).
``loo_brute`` deletes each point in turn, refits beta by GLS on the others and predicts it from the partitioned matrix.
"""
import numpy as np

from . import gp_oracle as _g
from . import matern_oracle as _m

MUCM, ALT, FREE = 1, 2, 4
_FAM = {"gaussian": _g, "matern52": _m}


def _split(theta, d, mode):
    x = _g.untransform(theta)
    delta = x[:d]
    k = d
    nug = None
    if mode & FREE:
        nug = x[k]
        k += 1
    sigma = None if mode & MUCM else x[k]
    return delta, nug, sigma


def make_A(theta, X, mode, family="gaussian", nugget_fixed=1e-4, r=0.0):
    """The matrix the likelihood of ``mode`` factors at the transformed parameters theta."""
    d = X.shape[1]
    delta, nug, sigma = _split(theta, d, mode)
    nugget = nugget_fixed if nug is None else nug
    kind = 1 if mode & ALT else 0
    if mode & MUCM:
        return _FAM[family].make_A(X, delta, nugget, kind, r, 1.0, True)
    s2 = sigma ** 2
    return s2 * _FAM[family].make_A(X, delta, nugget, kind, r, s2, True)


def grad_A(theta, X, mode, family="gaussian", nugget_fixed=1e-4, r=0.0):
    """dA/dtheta for every parameter, in the order [delta.., nugget?, sigma?] (a generator: one n x n matrix at a time,
    so the oracle stays usable at n = 4096)."""
    n, d = X.shape
    delta, nug, sigma = _split(theta, d, mode)
    nugget = nugget_fixed if nug is None else nug
    alt = bool(mode & ALT)
    s2 = 1.0 if mode & MUCM else sigma ** 2
    sq = lambda k: (X[:, k, None] / delta[k] - X[None, :, k] / delta[k]) ** 2
    D = sum(sq(k) for k in range(d))
    if family == "gaussian":
        R = np.exp(-D)
        G = R
    else:
        R, G = _m.R_of_D(D), _m.G_of_D(D)
    del D
    c = 1.0 if alt else 1.0 - nugget
    for k in range(d):
        T = (s2 * c) * G * sq(k)
        np.fill_diagonal(T, 0.0)
        yield T
    if nug is not None:
        if alt:
            yield np.diag(np.full(n, s2 * nugget ** 2))
        else:
            T = (-0.5 * nugget * s2) * R
            np.fill_diagonal(T, 0.0)
            yield T
    if not mode & MUCM:
        # sigma term A - diag(r), as the likelihood's (the reference's form; r is on A's diagonal for the alt nugget only)
        yield make_A(theta, X, mode, family, nugget_fixed, r) - np.diag(np.broadcast_to(np.asarray(r, dtype=float), (n,)))


def loo_closed(A, H, y, profiled):
    """(L, e, v, s2, P, alpha): objective, LOO residuals y - mu_-i, LOO variances, the scale, P and alpha."""
    Ai = np.linalg.inv(A)
    Ai = 0.5 * (Ai + Ai.T)
    AiH = Ai @ H
    P = Ai - AiH @ np.linalg.solve(H.T @ AiH, AiH.T)
    alpha = P @ y
    p = np.diag(P)
    s2 = np.mean(alpha ** 2 / p) if profiled else 1.0
    e, v = alpha / p, s2 / p
    L = 0.5 * np.sum(np.log(2.0 * np.pi * v) + e ** 2 / v)
    return L, e, v, s2, P, alpha


def loo_objective(theta, X, y, H, mode, family="gaussian", nugget_fixed=1e-4, r=0.0):
    """(L, grad, sigma_hat) as gpe_llh_grad_batch returns them with GPE_MODE_LOO."""
    A = make_A(theta, X, mode, family, nugget_fixed, r)
    L, e, v, s2, P, alpha = loo_closed(A, H, y, bool(mode & MUCM))
    p = np.diag(P)
    w = 0.5 * (1.0 / p + alpha ** 2 / (s2 * p ** 2))
    c = alpha / (s2 * p)
    F = P * np.sqrt(w)
    Pc = P @ c
    W = F @ F.T - 0.5 * (np.outer(Pc, alpha) + np.outer(alpha, Pc))
    grad = np.array([np.sum(W * T) for T in grad_A(theta, X, mode, family, nugget_fixed, r)])
    sigma = np.sqrt(s2) if mode & MUCM else _split(theta, X.shape[1], mode)[2]
    return L, grad, sigma


def loo_brute(A, H, y):
    """(mean [n], var [n]) by explicit deletion: for each i, GLS beta on the other points, kriging mean and variance
    (with the GLS term) of y_i from the partitioned A.  Variances in the units of A (multiply by s^2)."""
    n = y.size
    mean, var = np.empty(n), np.empty(n)
    for i in range(n):
        m = np.arange(n) != i
        Am, Hm = A[np.ix_(m, m)], H[m]
        Ai = np.linalg.inv(Am)
        Q = Hm.T @ Ai @ Hm
        b = np.linalg.solve(Q, Hm.T @ Ai @ y[m])
        k = A[m, i]
        mean[i] = H[i] @ b + k @ Ai @ (y[m] - Hm @ b)
        t = H[i] - Hm.T @ Ai @ k
        var[i] = A[i, i] - k @ Ai @ k + t @ np.linalg.solve(Q, t)
    return mean, var


def loo_predict(A, H, y, sigma):
    """gpe_loo: (mean, var) of the training points for the fit-state matrix A with scale sigma."""
    _, e, v, _, _, _ = loo_closed(A, H, y, False)
    return y - e, sigma ** 2 * v
