"""Posterior gradient on the B200 (gpe_predict_grad, Device.predict_grad, posterior_grad, SampledSensitivity.dgsm): the
device against the explicit formulas of oracle/posterior_grad_oracle.py (both families, every nugget form, both product
routes), against central differences of gpe_predict's mean, chunking and reproducibility, buffers, refusals, and the
derivative-based sensitivity measures against the oracle and the Poincare bound on a trained emulator."""
import contextlib
import io
import os
import shutil

import numpy as np
import pytest

from oracle import gp_oracle as G
from oracle import matern_oracle as Mo
from oracle import posterior_grad_oracle as GO
from oracle import sens_sample_oracle as SO

pytestmark = pytest.mark.gpu

FORMS = {"mucm": (0, True), "gp4ml": (0, False), "alt": (1, False)}


@contextlib.contextmanager
def _cwd(path):
    old = os.getcwd()
    os.chdir(path)
    try:
        yield
    finally:
        os.chdir(old)


@contextlib.contextmanager
def _quiet():
    with contextlib.redirect_stdout(io.StringIO()):
        yield


def _device(env=None):
    from gp_emu_uqsa_b200 import _lib
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        return _lib.Device(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v


def _case(n, d, seed, family, form, env=None, square=True, beta=None):
    """A fitted device with the basis [1, x_0 .. x_{d-1}] (+ x_1**2) and the explicit posterior of the same state."""
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * np.abs(X - 0.5).sum(1) + 0.3 * X[:, 1] ** 2
    inf, pw = list(range(d)) + ([1] if square else []), [1] * d + ([2] if square else [])
    H = G.make_H_linear(X, inf, pw)
    kind, mucm = FORMS[form]
    r = 1e-3 * (1.0 + rng.random(n)) if kind else None
    r_div = 1.3 if kind else 1.0
    delta, nug = 0.35 + 0.5 * rng.random(d), 1e-3
    dev = _device(env)
    dev.set_training(X, y, H, r)
    dev.set_basis(inf, pw)
    dev.set_kernel(family)
    sigma = 0.8
    bopt, smucm, st = dev.fit_state(delta, nug, sigma, kind, r_div=r_div, beta=beta)
    if mucm:
        sigma = smucm
        bopt, _, st = dev.fit_state(delta, nug, sigma, kind, r_div=r_div, beta=beta)
    assert st == 0
    A = (Mo.make_A if family else G.make_A)(X, delta, nug, kind, 0.0 if r is None else r, r_div)
    post = GO.GradPost(X, y, H, A, bopt if beta is None else beta, sigma, delta, nug, kind, family, inf, pw)
    return rng, dev, post


def _check(dmean, dvar, post, P, tol):
    rm, rv = post.grad(P)
    assert np.all(np.abs(dmean - rm) <= tol * np.abs(rm).max()), np.abs(dmean - rm).max() / np.abs(rm).max()
    prior = post.sigma ** 2 * post.c * post.kappa() / post.delta ** 2
    assert np.all(np.abs(dvar - rv) <= tol * prior[None, :]), (np.abs(dvar - rv) / prior).max()


@pytest.mark.parametrize("family", [0, 1])
@pytest.mark.parametrize("form", ["mucm", "gp4ml", "alt"])
def test_grad_matches_oracle_dmma(family, form):
    rng, dev, post = _case(300, 4, 1, family, form)
    P = rng.random((1000, 4))
    k0 = dev.int8_products
    dmean, dvar = dev.predict_grad(P)
    assert dev.int8_products == k0
    _check(dmean, dvar, post, P, 1e-10)
    dev.close()


@pytest.mark.parametrize("family", [0, 1])
def test_grad_matches_oracle_int8_and_dmma_routes(family):
    res = {}
    for env in ({}, {"GPE_OZAKI": "0"}):
        rng, dev, post = _case(1500, 6, 2, family, "gp4ml", env)
        P = 0.1 + 0.8 * rng.random((2000, 6))
        k0 = dev.int8_products
        res[bool(env)] = dev.predict_grad(P)
        assert (dev.int8_products > k0) == (not env)
        dev.close()
    _check(*res[False], post, P, 1e-8)
    _check(*res[True], post, P, 1e-10)


@pytest.mark.parametrize("family", [0, 1])
def test_mean_gradient_matches_central_differences_of_predict(family):
    """With a caller's beta and an x**2 term in the basis."""
    beta = np.array([0.2, -0.5, 0.7, 0.1, 1.3, -0.4])
    rng, dev, post = _case(300, 4, 4, family, "gp4ml", beta=beta)
    P = 0.1 + 0.8 * rng.random((500, 4))
    dmean, _ = dev.predict_grad(P, want_var=False)
    h = 1e-5
    for k in range(4):
        E = np.zeros(4)
        E[k] = h
        fd = (dev.predict(P + E, want_var=False)[0] - dev.predict(P - E, want_var=False)[0]) / (2 * h)
        assert np.all(np.abs(dmean[:, k] - fd) <= 1e-7 * np.abs(dmean).max()), np.abs(dmean[:, k] - fd).max()
    dev.close()


def test_reproducible_and_chunk_independent_on_dmma(monkeypatch):
    rng, dev, post = _case(300, 4, 3, 1, "gp4ml", {"GPE_OZAKI": "0"})
    P = rng.random((3000, 4))
    one = dev.predict_grad(P)
    again = dev.predict_grad(P)
    assert np.array_equal(one[0], again[0]) and np.array_equal(one[1], again[1])
    monkeypatch.setenv("GPE_PRED_CHUNK", "1024")          # 256 points (1024 columns) per chunk: 12 chunks on two streams
    many = dev.predict_grad(P)
    assert np.array_equal(one[0], many[0]) and np.array_equal(one[1], many[1])
    _check(*many, post, P, 1e-10)
    dev.close()


def test_buffers_mean_only_and_empty():
    import torch
    rng, dev, post = _case(300, 4, 5, 0, "alt")
    P = rng.random((1000, 4))
    dmean, dvar = dev.predict_grad(P)
    tm = torch.full((1000, 4), 7.0, dtype=torch.float64, device="cuda")
    tv = torch.full((1000, 4), 7.0, dtype=torch.float64, device="cuda")
    dev.predict_grad(torch.from_numpy(P).cuda(), out=(tm, tv))
    assert np.array_equal(tm.cpu().numpy(), dmean) and np.array_equal(tv.cpu().numpy(), dvar)
    m2, v2 = dev.predict_grad(P, want_var=False)
    assert v2 is None and np.array_equal(m2, dmean)
    tm.fill_(7.0)
    dev.predict_grad(torch.from_numpy(P).cuda(), out=(tm, None))
    assert np.array_equal(tm.cpu().numpy(), dmean)
    out = (np.full((0, 4), 7.0), np.full((0, 4), 7.0))
    launches = dev.launches
    dev.predict_grad(P[:0], out=out)
    assert dev.launches == launches
    dev.close()


def _golden_emulator(golden_dir, tmp, basis_str=None, train=True):
    """examples/toy-sim (d = 2, Gaussian kernel, fixed nugget 0.01, MUCM), trained."""
    import gp_emu_uqsa_b200 as g
    os.makedirs(tmp, exist_ok=True)
    for f in os.listdir(os.path.join(golden_dir, "toy-sim")):
        shutil.copyfile(os.path.join(golden_dir, "toy-sim", f), os.path.join(str(tmp), f))
    if basis_str is not None:
        path = os.path.join(str(tmp), "toy-sim_beliefs")
        txt = open(path).read().split("\n")
        open(path, "w").write("\n".join(("basis_str " + basis_str) if ln.startswith("basis_str ") else
                                        ("basis_inf NA 0 1") if ln.startswith("basis_inf ") else
                                        ("beta 1.0 1.0 1.0") if ln.startswith("beta ") else ln for ln in txt))
    with _cwd(tmp), _quiet():
        np.random.seed(0)
        E = g.setup("toy-sim_config")
        if train:
            g.train(E)
    return g, E


def test_refusals(golden_dir, tmp_path):
    from gp_emu_uqsa_b200 import _lib
    rng = np.random.default_rng(8)
    X = rng.random((60, 2))
    y = np.sin(3 * X[:, 0]) + X[:, 1]
    H = np.column_stack([np.ones(60), X])
    P = rng.random((100, 2))
    dev = _device()
    dev.set_training(X, y, H)
    with pytest.raises(_lib.GpeError, match="gpe_fit_state has not succeeded"):
        dev.predict_grad(P)
    assert dev.fit_state(np.array([0.4, 0.5]), 1e-3, 1.0, 0)[2] == 0
    with pytest.raises(_lib.GpeError, match="no device basis"):
        dev.predict_grad(P)
    dev.close()
    g, E = _golden_emulator(golden_dir, tmp_path, basis_str="1.0 np.sin(x) x", train=False)
    with pytest.raises(_lib.GpeError, match="polynomial mean basis"):
        g.posterior_grad(E, P)


def test_posterior_grad_and_dgsm_match_oracle(golden_dir, tmp_path):
    import torch
    import gp_emu_uqsa_b200.sensitivity as s
    g, E = _golden_emulator(golden_dir, tmp_path)
    Xt = E.training.inputs
    A = G.make_A(Xt, E.par.delta, E.par.nugget)
    post = GO.GradPost(Xt, E.training.outputs, E.training.H, A, E.par.beta, E.par.sigma, E.par.delta, E.par.nugget,
                   basis_inf=E.basis.basis_inf, powers=E.basis.poly)
    P = np.random.default_rng(2).random((700, 2))
    dmean, dvar = g.posterior_grad(E, P)
    _check(dmean, dvar, post, P, 1e-10)
    tm, tv = g.posterior_grad(E, torch.from_numpy(P).cuda())
    assert np.array_equal(tm.cpu().numpy(), dmean) and np.array_equal(tv.cpu().numpy(), dvar)
    with _quiet():
        S = s.setup_sampled(E, bounds=[[0.0, 1.0], [0.0, 1.0]], samples=2 ** 12, seed=5)
        S.dgsm()
        S.to_file(str(tmp_path / "sense_file"))
    T = post.dgsm_terms(S._points(S.samples)[0])
    mu, err = SO.estimates(T)
    assert np.all(np.abs(S.dgsm_nu - mu) <= 1e-9 * mu), (S.dgsm_nu, mu)
    assert np.allclose(S.stderr["dgsm_nu"], err, rtol=1e-6)
    assert np.allclose(S.dgsm_bound, S.dgsm_nu / np.pi ** 2, rtol=1e-15)
    txt = open(tmp_path / "sense_file").read().split("\n")
    assert txt[0].startswith("DGSM ") and txt[1].startswith("DGSMbound ")


@pytest.mark.parametrize("inputs", ["normal", "uniform"])
def test_poincare_bound_on_trained_emulator(golden_dir, tmp_path, inputs):
    """E*[V_T,k] of the continuous part (EVTw less the nugget's white-noise share sigma^2 (a* - c)) <= C_k E*[nu_k]."""
    import gp_emu_uqsa_b200.sensitivity as s
    g, E = _golden_emulator(golden_dir, tmp_path)
    kw = dict(m=[0.5, 0.5], v=[0.03, 0.02]) if inputs == "normal" else dict(bounds=[[0.1, 0.9], [0.0, 1.0]])
    with _quiet():
        S = s.setup_sampled(E, samples=2 ** 16, **kw)
        S.totaleffectvariance()
        S.dgsm()
    white = E.par.sigma ** 2 * E.par.nugget          # a* = 1, c = 1 - nugget
    cont = S.EVTw - white
    slack = 3.0 * np.hypot(S.stderr["EVTw"], S.stderr["dgsm_bound"])
    assert np.all(cont > 0.0) and np.all(cont <= S.dgsm_bound + slack), (cont, S.dgsm_bound, slack)
