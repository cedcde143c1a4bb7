"""CPU checks of the posterior-gradient formulas of gpe_predict_grad (oracle/posterior_grad_oracle.py, GradPost.grad) against
finite differences of the explicit posterior, of the bound on the derivative slab that keeps the INT8 route's scale valid,
and of the derivative-based sensitivity measures against tensor quadrature and the Poincare bound."""
import numpy as np
import pytest

from oracle import gp_oracle as G
from oracle import matern_oracle as Mo
from oracle import posterior_grad_oracle as GO
from oracle import sens_sample_oracle as SO
from gp_emu_uqsa_b200.sensitivity._sampledsensitivity import sample_points

FORMS = {"mucm": 0, "gp4ml": 0, "alt": 1}      # nugget form -> kind


def _post(family, form, seed=3, n=40, d=3, basis=None):
    """An explicit posterior with the basis [1, x_0 .. x_{d-1}] plus, by default, an x_1**2 term."""
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.5 * X[:, 1] ** 2
    inf, pw = basis if basis is not None else (list(range(d)) + [1], [1] * d + [2])
    H = G.make_H_linear(X, inf, pw)
    kind = FORMS[form]
    r = 1e-3 * (1.0 + rng.random(n)) if kind else 0.0
    delta, nug = 0.3 + 0.4 * rng.random(d), 1e-3
    A = (Mo.make_A if family else G.make_A)(X, delta, nug, kind, r, 1.3 if kind else 1.0)
    beta = G.optimalbeta(A, H, y)
    sigma = 0.7 if form != "mucm" else 1.1
    return rng, GO.GradPost(X, y, H, A, beta, sigma, delta, nug, kind, family, inf, pw)


@pytest.mark.parametrize("family", [0, 1])
@pytest.mark.parametrize("form", ["mucm", "gp4ml", "alt"])
def test_grad_matches_finite_differences(family, form):
    rng, post = _post(family, form)
    P = 0.1 + 0.8 * rng.random((7, 3))
    dmean, dvar = post.grad(P)
    for k in range(3):
        h = 1e-5
        E = np.zeros(3)
        E[k] = h
        fd = (post.pieces(P + E)[0] - post.pieces(P - E)[0]) / (2 * h)
        assert np.all(np.abs(dmean[:, k] - fd) <= 1e-7 * np.abs(dmean).max()), np.abs(dmean[:, k] - fd).max()
        # Var(f(p + h) - f(p - h)) / (2h)^2 from the continuous posterior covariance
        h = 2.5e-4 * post.delta[k]          # Matern's r^3 term makes the error first order in h
        E[k] = h
        prior = post.sigma ** 2 * post.c * post.kappa() / post.delta[k] ** 2
        for j in range(P.shape[0]):
            V = post.full_cov(np.stack([P[j] + E, P[j] - E]))
            fd2 = (V[0, 0] + V[1, 1] - 2.0 * V[0, 1]) / (2 * h) ** 2
            assert abs(dvar[j, k] - fd2) <= 1e-5 * prior, (j, k, dvar[j, k], fd2, prior)
        assert np.all(dvar[:, k] > 0.0) and np.all(dvar[:, k] <= prior * (1 + 1e-12))


@pytest.mark.parametrize("family", [0, 1])
def test_derivative_slab_is_bounded_by_c(family):
    """delta_k |d c / d p_k| <= c for every u_k and every distance r >= |u_k| (the other inputs' share of D)."""
    u = np.linspace(-6.0, 6.0, 2401)
    v = np.linspace(0.0, 6.0, 601)
    X = np.stack(np.meshgrid(u, v, indexing="ij"), axis=-1).reshape(-1, 2)
    post = GO.GradPost.__new__(GO.GradPost)
    post.X, post.delta, post.family, post.c = X, np.ones(2), family, 0.999
    B = post.dcov(np.zeros((1, 2)))
    top = np.abs(B[0]).max()
    assert top <= post.c
    assert top >= (0.85 if family == 0 else 0.62) * post.c      # the maxima: sqrt(2/e) and (sqrt5/3) max s(1+s)e^-s


def _dgsm_case(family):
    rng = np.random.default_rng(6 + family)
    n, d, nug = 60, 2, 1e-3
    X = rng.random((n, d))
    y = np.cos(3 * X[:, 0]) * X[:, 1] + X[:, 1] ** 2
    delta = np.array([0.3, 0.5])
    H = G.make_H_linear(X)
    A = (Mo.make_A if family else G.make_A)(X, delta, nug)
    post = GO.GradPost(X, y, H, A, G.optimalbeta(A, H, y), 0.9, delta, nug, family=family)
    if family == 0:
        m, v = [0.45, 0.55], [0.02, 0.03]
        return post, [("normal", a, b) for a, b in zip(m, v)], dict(m=m, v=v), np.array(v)
    bounds = [[0.1, 0.9], [0.0, 1.0]]
    return post, [("uniform", lo, hi) for lo, hi in bounds], dict(bounds=bounds), np.array([(hi - lo) ** 2 for lo, hi in bounds]) / np.pi ** 2


@pytest.mark.parametrize("family", [0, 1])
def test_dgsm_estimator_matches_quadrature_and_bounds_total_effect(family):
    post, dists, kw, C = _dgsm_case(family)
    ref = post.dgsm_quadrature(dists)
    XA, _ = sample_points(2, 2 ** 14, 0, **kw)
    mu, err = SO.estimates(post.dgsm_terms(XA))
    dev = np.abs(mu - ref)
    assert np.all(dev <= 3.0 * err), dev / err
    assert np.all(dev <= 1e-3 * ref), dev / ref
    # Poincare: the total-effect variance of the continuous part is at most C_k E*[nu_k] (quadrature's EVTw includes the
    # nugget's white-noise share sigma^2 (a* - c))
    Q = SO.quadrature(post, dists)
    total_cont = Q["EVTw"] - post.sigma ** 2 * (post.astar - post.c)
    assert np.all(total_cont > 0.0) and np.all(total_cont <= C * ref), (total_cont, C * ref)
