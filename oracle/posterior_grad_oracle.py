"""TEST INFRASTRUCTURE ONLY -- NumPy statement of the posterior gradient (gpe_predict_grad, include/gpe_b200.h) and of the
derivative-based global sensitivity measures built on it (SampledSensitivity.dgsm).

``GradPost`` is ``sens_sample_oracle.Post`` (the explicit posterior of the state gpe_fit_state factors) with the derivatives
of the continuous part of the process: the cross-covariance derivative (2 / delta_k) c phi(D) u_k, phi = -dR/dD, and the
prior derivative variance c kappa / delta_k^2, kappa = -2 R'(0).
"""
import numpy as np
from scipy import linalg as _sl

from . import matern_oracle as _m
from .sens_sample_oracle import Post, rule


class GradPost(Post):
    def kappa(self):
        """-2 R'(0): the prior variance of a derivative is c kappa / delta_k^2."""
        return 2.0 if self.family == 0 else 5.0 / 3.0

    def dcov(self, P):
        """The derivative slab b [d, n, m] = delta_k d/dp_k [c R(D(x_i, p_j))] = 2 c phi(D) u_k, u_k = (x_ik - p_jk) / delta_k,
        phi = -dR/dD."""
        U = (self.X[None, :, :] - np.asarray(P, float)[:, None, :]) / self.delta          # [m, n, d]
        D = (U * U).sum(2)
        phi = np.exp(-D) if self.family == 0 else _m.G_of_D(D)
        return np.moveaxis(2.0 * self.c * phi[:, :, None] * U, 2, 0).transpose(0, 2, 1)

    def dbasis(self, P, k):
        """d h(p) / d p_k [m, q] of the polynomial basis."""
        P = np.asarray(P, float)
        d = P.shape[1]
        inf = list(range(d)) if self.basis_inf is None else list(self.basis_inf)
        pw = [1] * len(inf) if self.powers is None else list(self.powers)
        dH = np.zeros((P.shape[0], 1 + len(inf)))
        for a, (c, p) in enumerate(zip(inf, pw)):
            if c == k and p != 0:
                dH[:, a + 1] = p * P[:, c] ** (p - 1)
        return dH

    def grad(self, P):
        """(dmean [m, d], dvar [m, d]): the gradient of the posterior mean and the posterior variance of each gradient
        component, from the formulas of gpe_predict_grad."""
        P = np.asarray(P, float)
        m, d = P.shape
        B = self.dcov(P)
        dmean, dvar = np.empty((m, d)), np.empty((m, d))
        for k in range(d):
            dC = B[k] / self.delta[k]
            dH = self.dbasis(P, k)
            dmean[:, k] = dH @ self.beta + dC.T @ self.e
            dZ = _sl.solve_triangular(self.L, dC, lower=True)
            dG = _sl.solve_triangular(self.Kq, (dH - dC.T @ self.AiH).T, lower=True)
            dvar[:, k] = self.sigma ** 2 * (self.c * self.kappa() / self.delta[k] ** 2 - (dZ * dZ).sum(0) + (dG * dG).sum(0))
        return dmean, dvar

    def dgsm_terms(self, P, chunk=4096):
        """Per-sample DGSM terms [m, d]: (dm*/dp_k)^2 + Var*(df/dp_k), whose mean over the input distribution is E*[nu_k]."""
        P = np.asarray(P, float)
        out = np.empty(P.shape)
        for s in range(0, P.shape[0], chunk):
            dm, dv = self.grad(P[s:s + chunk])
            out[s:s + chunk] = dm * dm + dv
        return out

    def dgsm_quadrature(self, dists, nodes=64):
        """E*[nu_k] [d] by tensor quadrature over the input distributions (sens_sample_oracle.rule)."""
        rules = [rule(di, nodes) for di in dists]
        P = np.stack([g.reshape(-1) for g in np.meshgrid(*[r[0] for r in rules], indexing="ij")], axis=1)
        W = np.ones(1)
        for _, w in rules:
            W = np.multiply.outer(W, w)
        return W.reshape(-1) @ self.dgsm_terms(P)
