"""TEST INFRASTRUCTURE ONLY -- NumPy statement of the sampled sensitivity estimator (gpe_sens_sample,
include/gpe_b200.h) and a tensor-product quadrature of the integrals it estimates.

``Post`` is the explicit posterior of the state gpe_fit_state factors: A is the training matrix as training.remake()
leaves it (gp_oracle.make_A / matern_oracle.make_A, r included for the alternative nugget), beta and sigma as given.
For two distinct points the posterior covariance takes the off-diagonal (continuous) prior c R(D); the variance of a
point takes the diagonal a* (1, or 1 + nugget^2 for the alternative nugget).
"""
import numpy as np
import scipy.spatial.distance as _dist
from scipy import linalg as _sl

from . import gp_oracle as _g
from . import matern_oracle as _m


class Post:
    def __init__(self, X, y, H, A, beta, sigma, delta, nugget, kind=0, family=0, basis_inf=None, powers=None):
        self.X, self.y, self.H = np.asarray(X, float), np.asarray(y, float), np.asarray(H, float)
        self.beta, self.sigma = np.asarray(beta, float), float(sigma)
        self.delta, self.family = np.asarray(delta, float), int(family)
        self.basis_inf, self.powers = basis_inf, powers
        self.c = (1.0 - nugget) if kind == 0 else 1.0
        self.astar = 1.0 if kind == 0 else 1.0 + nugget * nugget
        self.cf = _sl.cho_factor(A, lower=True)
        self.L = np.tril(self.cf[0])
        self.e = _sl.cho_solve(self.cf, self.y - self.H @ self.beta)
        self.AiH = _sl.cho_solve(self.cf, self.H)
        self.Kq = np.linalg.cholesky(self.H.T @ self.AiH)

    def R(self, D):
        return np.exp(-D) if self.family == 0 else _m.R_of_D(D)

    def D(self, P, Q):
        w = 1.0 / self.delta
        return _dist.cdist(P * w, Q * w, 'sqeuclidean')

    def pieces(self, P):
        """mean [m], z = L^-1 c_x [n, m], g [q, m] with g_x . g_x' the regression term of the covariance."""
        C = self.c * self.R(self.D(self.X, P))
        Hs = _g.make_H_linear(P, self.basis_inf, self.powers)
        mean = Hs @ self.beta + C.T @ self.e
        Z = _sl.solve_triangular(self.L, C, lower=True)
        G = _sl.solve_triangular(self.Kq, (Hs - C.T @ self.AiH).T, lower=True)
        return mean, Z, G

    def var(self, mean_z_g):
        _, Z, G = mean_z_g
        return self.sigma ** 2 * (self.astar - (Z * Z).sum(0) + (G * G).sum(0))

    def pair_cov(self, P, Q, pp, pq):
        """c(P_s, Q_s) for paired rows."""
        D = (((P - Q) / self.delta) ** 2).sum(1)
        return self.sigma ** 2 * (self.c * self.R(D) - (pp[1] * pq[1]).sum(0) + (pp[2] * pq[2]).sum(0))

    def full_cov(self, P):
        """c(P_i, P_j) for every pair, continuous prior on the diagonal too."""
        _, Z, G = self.pieces(P)
        return self.sigma ** 2 * (self.c * self.R(self.D(P, P)) - Z.T @ Z + G.T @ G)


def terms(post, XA, XB, which, shift, chunk=4096):
    """Per-sample terms [M, 3 + 2 nw] = (t_E, t_V, t_EV, t_S[which], t_T[which]) of gpe_sens_sample."""
    XA, XB = np.asarray(XA, float), np.asarray(XB, float)
    M, nw = XA.shape[0], len(which)
    out = np.empty((M, 3 + 2 * nw))
    for s in range(0, M, chunk):
        A, B = XA[s:s + chunk], XB[s:s + chunk]
        pa, pb = post.pieces(A), post.pieces(B)
        vA, vB = post.var(pa), post.var(pb)
        cAB = post.pair_cov(A, B, pa, pb)
        t = out[s:s + chunk]
        t[:, 0] = pa[0]
        t[:, 1] = cAB
        t[:, 2] = 0.5 * ((pa[0] - pb[0]) ** 2 + vA + vB - 2.0 * cAB)
        for k, P in enumerate(which):
            X = A.copy()
            X[:, P] = B[:, P]
            px = post.pieces(X)
            t[:, 3 + k] = (pb[0] - shift) * (px[0] - pa[0]) + post.pair_cov(B, X, pb, px) - cAB
            t[:, 3 + nw + k] = 0.5 * ((pa[0] - px[0]) ** 2 + vA + post.var(px) - 2.0 * post.pair_cov(A, X, pa, px))
    return out


def estimates(T):
    """Means of the terms and their plain Monte Carlo standard errors."""
    M = T.shape[0]
    return T.mean(0), T.std(0, ddof=1) / np.sqrt(M)


def rule(dist, nodes):
    """One input's quadrature nodes and weights (summing to 1): ('normal', m, v) by Gauss-Hermite, ('uniform', lo, hi)
    by Gauss-Legendre."""
    kind, a, b = dist
    if kind == "normal":
        x, w = np.polynomial.hermite_e.hermegauss(nodes)
        return a + np.sqrt(b) * x, w / np.sqrt(2.0 * np.pi)
    x, w = np.polynomial.legendre.leggauss(nodes)
    return a + (b - a) * 0.5 * (x + 1.0), 0.5 * w


def quadrature(post, dists, nodes=64):
    """uE, uV, uEV, E*[V_P] [d] and E*[V_T,P] [d] by tensor quadrature (d <= 2: the full covariance of the nodes^d grid is
    formed)."""
    d = len(dists)
    rules = [rule(di, nodes) for di in dists]
    grids = np.meshgrid(*[r[0] for r in rules], indexing="ij")
    P = np.stack([gk.reshape(-1) for gk in grids], axis=1)
    W = np.ones([nodes] * d)
    for k, (_, w) in enumerate(rules):
        W = W * w.reshape([nodes if j == k else 1 for j in range(d)])
    pc = post.pieces(P)
    mean, var = pc[0].reshape([nodes] * d), post.var(pc).reshape([nodes] * d)
    Cm = post.full_cov(P).reshape([nodes] * (2 * d))
    Wf = W.reshape(-1)
    uE = float((W * mean).sum())
    uV = float(Wf @ Cm.reshape(nodes ** d, nodes ** d) @ Wf)
    uEV = float((W * (mean ** 2 + var)).sum()) - uE ** 2 - uV
    first, total = np.zeros(d), np.zeros(d)
    for k in range(d):
        # axis k first, the other inputs flattened: m2 [nodes, r], C4 [nodes, r, nodes, r]
        rest = nodes ** (d - 1)
        m2 = np.moveaxis(mean, k, 0).reshape(nodes, rest)
        v2 = np.moveaxis(var, k, 0).reshape(nodes, rest)
        C4 = np.moveaxis(np.moveaxis(Cm, d + k, d), k, 0).reshape(nodes, rest, nodes, rest)
        wk = rules[k][1]
        wr = np.moveaxis(W, k, 0).reshape(nodes, rest)[0] / wk[0]
        inner_m = m2 @ wr
        inner_c = np.einsum("iris,r,s->i", C4, wr, wr)
        first[k] = float(wk @ (inner_m ** 2 + inner_c)) - uE ** 2 - uV
        cond_m = wk @ m2
        cond_c = np.einsum("irjr,i,j->r", C4, wk, wk)
        total[k] = float(wr @ (wk @ (m2 ** 2 + v2) - cond_m ** 2 - cond_c))
    return {"uE": uE, "uV": uV, "uEV": uEV, "senseindex": first, "EVTw": total}
