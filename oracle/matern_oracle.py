"""TEST INFRASTRUCTURE ONLY -- CPU oracle of the Matern 5/2 covariance family.

The reference has no Matern kernel, so there is no code to restate: this is the model the library implements,
written in NumPy/SciPy from its definition.  With D_ij = sum_k ((x_ik - x_jk) / delta_k)^2 and r = sqrt(D):

    R(D) = (1 + sqrt5 r + 5 D / 3) exp(-sqrt5 r)          (Matern, nu = 5/2, in the scaled distance)
    dR/dtheta_k = G(D) ((x_ik - x_jk) / delta_k)^2,   G(D) = (5/6)(1 + sqrt5 r) exp(-sqrt5 r),   delta_k = exp(theta_k / 2)

Everything else is the Gaussian model of ``gp_oracle`` with R in place of exp(-D): ``kernel`` (kind 0) scales the
off-diagonal by (1 - nugget), ``kernel_alt_nug`` (kind 1) puts 1 + nugget^2 on the diagonal; the likelihoods keep the
reference's quirks (MUCM gradient scaled by sigma_hat^2, gp4ml sigma term A - diag(r)).  The likelihoods evaluate
through a Cholesky factor and A^-1, so the oracle stays usable at n = 4096.
"""
import numpy as np
import scipy.spatial.distance as _dist
from scipy import linalg as _sl

from . import gp_oracle as _g

KERNEL, KERNEL_ALT = 0, 1
SQRT5 = np.sqrt(5.0)
transform, untransform = _g.transform, _g.untransform


def R_of_D(D):
    s = SQRT5 * np.sqrt(D)
    return (1.0 + s + 5.0 * D / 3.0) * np.exp(-s)


def G_of_D(D):
    s = SQRT5 * np.sqrt(D)
    return (5.0 / 6.0) * (1.0 + s) * np.exp(-s)


def _sqdist(X, delta):
    return _dist.squareform(_dist.pdist(X / np.asarray(delta, dtype=float), 'sqeuclidean'))


def cov_var(X, delta, nugget, kind=KERNEL, predict=True):
    """var(): R off the diagonal (times 1 - nugget for ``kernel``); diagonal as the Gaussian forms."""
    R = R_of_D(_sqdist(X, delta))
    if kind == KERNEL:
        A = (1.0 - nugget) * R
        np.fill_diagonal(A, 1.0 if predict else 1.0 - nugget)
    else:
        A = R.copy()
        np.fill_diagonal(A, 1.0 + nugget ** 2 if predict else 1.0)
    return A


def make_A(X, delta, nugget, kind=KERNEL, r=0.0, s2=1.0, predict=True):
    A = cov_var(X, delta, nugget, kind, predict)
    if kind == KERNEL_ALT:
        np.fill_diagonal(A, A.diagonal() + np.asarray(r, dtype=float) / s2)
    return A


def covar(XT, XV, delta, nugget, kind=KERNEL):
    w = 1.0 / np.asarray(delta, dtype=float)
    C = R_of_D(_dist.cdist(XT * w, XV * w, 'sqeuclidean'))
    return (1.0 - nugget) * C if kind == KERNEL else C


def grad_delta_A(X, delta, nugget, di, s2, kind=KERNEL):
    """d(s2 A)/d theta_delta[di] = s2 c G Delta_di^2 (c = 1 - nugget for ``kernel``, 1 for the alt nugget)."""
    col = (X[:, di] / delta[di]).reshape(-1, 1)
    f = _dist.squareform(_dist.pdist(col, 'sqeuclidean'))
    pref = (1.0 - nugget) * s2 if kind == KERNEL else s2
    return pref * f * G_of_D(_sqdist(X, delta))


def grad_nugget_A(X, delta, nugget, s2, kind=KERNEL):
    """``kernel``: -1/2 nugget s2 R off the diagonal; alt nugget: diag(nugget^2 s2)."""
    if kind == KERNEL:
        T = (-0.5 * nugget * s2) * R_of_D(_sqdist(X, delta))
        np.fill_diagonal(T, 0.0)
        return T
    return np.diag(np.full(X.shape[0], nugget ** 2 * s2))


def _factor(A, H, y):
    """Cholesky of A and the GLS pieces: (logdet A, A^-1, A^-1 y, A^-1 H, Q = H^T A^-1 H, beta)."""
    cf = _sl.cho_factor(A, lower=True)
    logdetA = 2.0 * np.sum(np.log(np.diag(cf[0])))
    Ainv = _sl.cho_solve(cf, np.eye(A.shape[0]))
    af, aH = Ainv.dot(y), Ainv.dot(H)
    Q = H.T.dot(aH)
    B = np.linalg.solve(Q, H.T.dot(af))
    return logdetA, Ainv, af, aH, Q, B


def _grad_term(T, Ainv, af, aH, Q, B, factor):
    """-1/2 (-tr(A^-1 T) + factor (y^T A^-1 T A^-1 y + (H B - 2 y)^T A^-1 T A^-1 H B) + tr(Q^-1 H^T A^-1 T A^-1 H)):
    the reference's gradient expression (_emulatoroptimise.py:347-357), evaluated from A^-1 in O(n^2 q) per matrix."""
    v = aH.dot(B)
    return -0.5 * (-np.sum(Ainv * T) + factor * (af.dot(T.dot(af)) + (v - 2.0 * af).dot(T.dot(v)))
                   + np.trace(np.linalg.solve(Q, aH.T.dot(T.dot(aH)))))


def _delta_terms(X, delta, nugget, s2, kind):
    """grad_delta_A for every dimension, sharing G(D) (a generator: one n x n matrix at a time)."""
    G = G_of_D(_sqdist(X, delta))
    pref = (1.0 - nugget) * s2 if kind == KERNEL else s2
    for di in range(X.shape[1]):
        col = (X[:, di] / delta[di]).reshape(-1, 1)
        yield pref * G * _dist.squareform(_dist.pdist(col, 'sqeuclidean'))


def loglikelihood_mucm(theta, X, y, H, kind=KERNEL, nugget_fixed=1e-4, r=0.0):
    """(LLH, grad, sigma_hat) of the MUCM likelihood (gradient with the reference's sigma_hat^2 scaling), or None on a
    non-PD matrix."""
    n, d = X.shape
    q = H.shape[1]
    x = untransform(theta)
    delta, nug, _ = _g._split_hp(x, d, has_sigma=False)
    nugget = nugget_fixed if nug is None else nug
    A = make_A(X, delta, nugget, kind, r, 1.0, True)
    try:
        logdetA, Ainv, af, aH, Q, B = _factor(A, H, y)
    except np.linalg.LinAlgError:
        return None
    sig2 = (1.0 / (n - q - 2.0)) * y.dot(af - aH.dot(B))
    LLH = -0.5 * (-(n - q) * np.log(sig2) - logdetA - np.log(np.linalg.det(Q)))
    factor = (n - q) / (sig2 * (n - q - 2))
    grad = [_grad_term(t, Ainv, af, aH, Q, B, factor) for t in _delta_terms(X, delta, nugget, sig2, kind)]
    if x.size == d + 1:
        grad.append(_grad_term(grad_nugget_A(X, delta, nugget, sig2, kind), Ainv, af, aH, Q, B, factor))
    grad = np.array(grad)
    return LLH, grad, np.sqrt(sig2)


def loglikelihood_gp4ml(theta, X, y, H, kind=KERNEL, nugget_fixed=1e-4, r=0.0):
    """(LLH, grad) of the gp4ml likelihood, or None on a non-PD matrix."""
    n, d = X.shape
    q = H.shape[1]
    x = untransform(theta)
    delta, nug, sigma = _g._split_hp(x, d, has_sigma=True)
    nugget = nugget_fixed if nug is None else nug
    s2 = sigma ** 2
    A = s2 * make_A(X, delta, nugget, kind, r, s2, True)
    try:
        logdetA, Ainv, af, aH, Q, B = _factor(A, H, y)
    except np.linalg.LinAlgError:
        return None
    longexp = y.dot(af - aH.dot(B))
    LLH = -0.5 * (-longexp - logdetA - np.log(_sl.det(Q)) - (n - q) * np.log(2.0 * np.pi))
    grad = [_grad_term(t, Ainv, af, aH, Q, B, 1.0) for t in _delta_terms(X, delta, nugget, s2, kind)]
    if x.size == d + 2:
        grad.append(_grad_term(grad_nugget_A(X, delta, nugget, s2, kind), Ainv, af, aH, Q, B, 1.0))
    T = A.copy()                                          # sigma term: A - diag(r) (reference :476-478)
    np.fill_diagonal(T, T.diagonal() - np.asarray(r, dtype=float))
    grad.append(_grad_term(T, Ainv, af, aH, Q, B, 1.0))
    grad = np.array(grad)
    return LLH, grad


def optimalbeta(A, H, y):
    return _g.optimalbeta(A, H, y)


def posterior(Xs, Hs, X, y, H, A, beta, sigma, delta, nugget, kind=KERNEL, r_new=0.0):
    """(mean [m], var [m, m]) given the training matrix A as training.remake() leaves it, via Cholesky solves."""
    cf = _sl.cho_factor(A, lower=True)
    C = covar(X, Xs, delta, nugget, kind)
    mean = Hs.dot(beta) + C.T.dot(_sl.cho_solve(cf, y - H.dot(beta)))
    invA_H = _sl.cho_solve(cf, H)
    temp1 = Hs - C.T.dot(invA_H)
    temp2 = H.T.dot(invA_H)
    Anew = make_A(Xs, delta, nugget, kind, r_new, 1.0, True)
    temp3 = Anew - C.T.dot(_sl.cho_solve(cf, C))
    var = sigma ** 2 * (temp3 + temp1.dot(_sl.solve(temp2, temp1.T, assume_a='pos')))
    return mean, var
