"""Sampled uncertainty / sensitivity analysis on the B200 (gpe_sens_sample, sensitivity.setup_sampled): the device sums
against the NumPy term table of oracle/sens_sample_oracle.py on identical points (both families, every nugget form, both
product routes, host and device buffers), the estimates against the closed-form integrals and against quadrature, chunking
and reproducibility, and the refusals."""
import contextlib
import io
import os

import numpy as np
import pytest

from oracle import gp_oracle as G
from oracle import matern_oracle as Mo
from oracle import sens_sample_oracle as SO

pytestmark = pytest.mark.gpu


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


def _device(X, y, H, r=None, family=0, env=None):
    from gp_emu_uqsa_b200 import _lib
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        dev = _lib.Device(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v
    dev.set_training(X, y, H, r)
    dev.set_basis(list(range(X.shape[1])), [1] * X.shape[1])
    dev.set_kernel(family)
    return dev


# form: (kind, MUCM sigma?)
FORMS = {"mucm": (0, True), "gp4ml": (0, False), "alt": (1, False)}


def _case(n, d, seed, family, form, env=None):
    """A fitted device and the explicit posterior of the same state."""
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * np.abs(X - 0.5).sum(1)
    H = np.column_stack([np.ones(n), X])
    kind, mucm = FORMS[form]
    r = 1e-3 * (1.0 + rng.random(n)) if kind else None
    r_div = 1.3 if kind else 1.0
    delta, nug = 0.35 + 0.5 * rng.random(d), 1e-3
    dev = _device(X, y, H, r, family, env)
    sigma = 0.8
    beta, smucm, st = dev.fit_state(delta, nug, sigma, kind, r_div=r_div)
    if mucm:
        sigma = smucm
        beta, _, st = dev.fit_state(delta, nug, sigma, kind, r_div=r_div)
    assert st == 0
    mk = Mo.make_A if family else G.make_A
    A = mk(X, delta, nug, kind, 0.0 if r is None else r, r_div)
    post = SO.Post(X, y, H, A, beta, sigma, delta, nug, kind, family)
    return rng, dev, post, y.mean()


def _check_sums(sums, T, tol):
    ref = np.stack([T.sum(0), (T * T).sum(0)])
    scale = np.stack([np.abs(T).sum(0), (T * T).sum(0)])
    assert np.all(np.abs(sums - ref) <= tol * scale), np.max(np.abs(sums - ref) / scale)


@pytest.mark.parametrize("family", [0, 1])
@pytest.mark.parametrize("form", ["mucm", "gp4ml", "alt"])
def test_sums_match_oracle_dmma(family, form):
    import torch
    rng, dev, post, shift = _case(300, 4, 1, family, form)
    M, which = 1024, [2, 0, 3]
    XA, XB = rng.random((M, 4)), rng.random((M, 4))
    T = SO.terms(post, XA, XB, which, shift)
    k0 = dev.int8_products
    _check_sums(dev.sens_sample(XA, XB, which, shift), T, 1e-10)
    assert dev.int8_products == k0
    # device buffers: points, which and sums
    out = torch.empty((2, 3 + 2 * len(which)), dtype=torch.float64, device="cuda")
    dev.sens_sample(torch.from_numpy(XA).cuda(), torch.from_numpy(XB).cuda(), torch.tensor(which, dtype=torch.int32, device="cuda"),
                    shift, out=out)
    _check_sums(out.cpu().numpy(), T, 1e-10)
    dev.close()


@pytest.mark.parametrize("family", [0, 1])
def test_sums_match_oracle_int8_and_dmma_routes(family):
    res = {}
    for env in ({}, {"GPE_OZAKI": "0"}):
        rng, dev, post, shift = _case(1500, 6, 2, family, "gp4ml", env)
        M, which = 4096, list(range(6))
        XA, XB = 0.1 + 0.8 * rng.random((M, 6)), rng.random((M, 6))
        k0 = dev.int8_products
        res[bool(env)] = dev.sens_sample(XA, XB, which, shift)
        assert (dev.int8_products > k0) == (not env)
        dev.close()
    T = SO.terms(post, XA, XB, which, shift)
    _check_sums(res[False], T, 1e-8)
    _check_sums(res[True], T, 1e-10)


def test_chunks_and_reproducibility(monkeypatch):
    rng, dev, post, shift = _case(300, 4, 3, 1, "gp4ml")
    M, which = 3000, [0, 1, 2, 3]
    XA, XB = rng.random((M, 4)), rng.random((M, 4))
    one = dev.sens_sample(XA, XB, which, shift)
    assert np.array_equal(one, dev.sens_sample(XA, XB, which, shift))
    monkeypatch.setenv("GPE_PRED_CHUNK", "1536")          # 256 samples per chunk: 12 chunks on two streams
    many = dev.sens_sample(XA, XB, which, shift)
    assert np.array_equal(many, dev.sens_sample(XA, XB, which, shift))
    assert np.all(np.abs(many - one) <= 1e-12 * np.abs(one))
    _check_sums(many, SO.terms(post, XA, XB, which, shift), 1e-10)
    dev.close()


def _emulator(g, tmp, X, y, delta, nugget, sigma, matern=False, basis_str=None):
    from oracle import ref_loader as RL
    os.makedirs(tmp, exist_ok=True)
    with _cwd(tmp), _quiet():
        cfg = RL.write_emulator_files(str(tmp), X, y, mucm="F", fix_nugget="T", alt_nugget="F", nugget=nugget, name="e")
        txt = open("e_beliefs").read()
        if basis_str is not None:
            txt = "\n".join(("basis_str " + basis_str) if ln.startswith("basis_str ") else ln for ln in txt.split("\n"))
        if matern:
            txt += "kernel matern52\n"
        open("e_beliefs", "w").write(txt)
        E = g.setup(cfg, datashuffle=False, scaleinputs=True)
        E.par.delta = np.array(delta, dtype=float); E.K.d = E.par.delta; E.K.n = E.par.nugget
        E.par.sigma = float(sigma)
        E.training.remake()
        E.opt_T.optimalbeta()
    return E


def _within(est, err, ref, tol):
    dev = np.abs(np.asarray(est) - np.asarray(ref))
    assert np.all(dev <= 3.0 * np.asarray(err)), (dev, err)
    assert np.all(dev <= tol), (dev, tol)


def test_setup_sampled_matches_closed_form(tmp_path):
    """The emulator of test_sensitivity_vs_oracle_larger_n (Gaussian kernel, normal inputs)."""
    import gp_emu_uqsa_b200 as g
    import gp_emu_uqsa_b200.sensitivity as s
    from oracle.sens_oracle import SensOracle
    rng = np.random.default_rng(11)
    n, d = 700, 5
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * (X ** 2).sum(1)
    E = _emulator(g, tmp_path, X, y, 0.3 + 0.4 * rng.random(d), 1e-4, 0.9)
    m, v = list(0.4 + 0.2 * rng.random(d)), list(0.01 + 0.02 * rng.random(d))
    state = np.random.get_state()
    with _quiet():
        S = s.setup_sampled(E, m=m, v=v, samples=2 ** 16)
        S.uncertainty(); S.sensitivity(); S.totaleffectvariance(); S.main_effect(points=20)
        S.to_file(str(tmp_path / "sense_file"))
        table = s.sense_table([S])
    after = np.random.get_state()
    assert np.array_equal(state[1], after[1]) and state[2:] == after[2:]
    O = SensOracle(E.training.inputs, E.training.outputs, E.training.H, E.training.A, E.par.beta, E.par.sigma, E.par.nugget,
                   E.par.delta, m, v)
    uE, uV, uEV = O.uncertainty()
    tol = 1e-3 * abs(uEV)
    for key, ref in (("uE", uE), ("uV", uV), ("uEV", uEV)):
        _within(getattr(S, key), S.stderr[key], ref, tol)
    _within(S.senseindex, S.stderr["senseindex"], O.sensitivity(), tol)
    total = [uEV - O.EVint([k for k in range(d) if k != P]) for P in range(d)]
    _within(S.EVTw, S.stderr["EVTw"], total, tol)
    eff, me = O.main_effect(E.all_data.input_range, points=20)
    assert np.all(np.abs(S.effect - eff) <= 5e-3 * np.sqrt(uEV))
    assert np.all(np.abs(S.mean_effect - me) <= 5e-3 * np.sqrt(uEV))
    txt = open(tmp_path / "sense_file").read().split("\n")
    assert txt[0].startswith("EE ") and txt[3].startswith("EVw ") and txt[4].startswith("EVTw ") and txt[5].startswith("xw ")
    assert table.shape == (1, d + 1)
    # the same seed gives the same results
    with _quiet():
        S2 = s.setup_sampled(E, m=m, v=v, samples=2 ** 16)
        S2.uncertainty(); S2.sensitivity()
    assert (S2.uE, S2.uV, S2.uEV) == (S.uE, S.uV, S.uEV) and np.array_equal(S2.senseindex, S.senseindex)


def test_matern_uniform_inputs_match_quadrature(tmp_path):
    import gp_emu_uqsa_b200 as g
    import gp_emu_uqsa_b200.sensitivity as s
    rng = np.random.default_rng(6)
    X = rng.random((80, 2))
    y = np.cos(3 * X[:, 0]) * X[:, 1] + np.abs(X[:, 1] - 0.4)
    E = _emulator(g, tmp_path, X, y, [0.3, 0.5], 1e-3, 0.9, matern=True)
    bounds = [[0.1, 0.9], [0.0, 1.0]]
    with _quiet():
        S = s.setup_sampled(E, bounds=bounds, samples=2 ** 14, seed=3)
        S.uncertainty(); S.sensitivity(); S.totaleffectvariance()
    Xt = E.training.inputs
    A = Mo.make_A(Xt, E.par.delta, E.par.nugget)
    post = SO.Post(Xt, E.training.outputs, E.training.H, A, E.par.beta, E.par.sigma, E.par.delta, E.par.nugget, family=1)
    Q = SO.quadrature(post, [("uniform", lo, hi) for lo, hi in bounds])
    tol = 1e-3 * abs(Q["uEV"])
    for key in ("uE", "uV", "uEV"):
        _within(getattr(S, key), S.stderr[key], Q[key], tol)
    _within(S.senseindex, S.stderr["senseindex"], Q["senseindex"], tol)
    _within(S.EVTw, S.stderr["EVTw"], Q["EVTw"], tol)


def test_refusals(tmp_path):
    import gp_emu_uqsa_b200 as g
    import gp_emu_uqsa_b200.sensitivity as s
    from gp_emu_uqsa_b200 import _lib
    rng = np.random.default_rng(8)
    X = rng.random((60, 2))
    y = np.sin(3 * X[:, 0]) + X[:, 1]
    E = _emulator(g, tmp_path / "a", X, y, [0.4, 0.5], 1e-3, 1.0)
    for kw, msg in (({"m": [0.5, 0.5]}, "either input means"),
                    ({"m": [0.5, 0.5], "v": [0.01, 0.01], "bounds": [[0, 1], [0, 1]]}, "either input means"),
                    ({"m": [0.5], "v": [0.01]}, "as many finite values"),
                    ({"m": [0.5, 0.5], "v": [0.01, 0.0]}, "variances must be positive"),
                    ({"bounds": [[0, 1], [0.5, 0.5]]}, "lo < hi"),
                    ({"bounds": [[0, 1]]}, "one finite [lo, hi] pair"),
                    ({"bounds": [[0, 1], [0, 1]], "samples": 1000}, "power of two"),
                    ({"bounds": [[0, 1], [0, 1]], "samples": 128}, "power of two")):
        out = io.StringIO()
        with contextlib.redirect_stdout(out):
            assert s.setup_sampled(E, **kw) is None
        assert msg in out.getvalue(), (kw, out.getvalue())
    Enp = _emulator(g, tmp_path / "b", X, y, [0.4, 0.5], 1e-3, 1.0, basis_str="1.0 np.sin(x) x")
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        assert s.setup_sampled(Enp, bounds=[[0, 1], [0, 1]]) is None
    assert "polynomial mean" in out.getvalue()
    # the C-ABI
    H = np.column_stack([np.ones(60), X])
    dev = _device(X, y, H)
    P = rng.random((256, 2))
    with pytest.raises(_lib.GpeError, match="gpe_fit_state has not succeeded"):
        dev.sens_sample(P, P, [0])
    assert dev.fit_state(np.array([0.4, 0.5]), 1e-3, 1.0, 0)[2] == 0
    with pytest.raises(_lib.GpeError, match="1 <= nw <= 16"):
        dev.sens_sample(P, P, [])
    with pytest.raises(_lib.GpeError, match="1 <= nw <= 16"):
        dev.sens_sample(P, P, list(range(17)))
    with pytest.raises(_lib.GpeError, match="distinct"):
        dev.sens_sample(P, P, [1, 1])
    with pytest.raises(_lib.GpeError, match=r"\[0, d\)"):
        dev.sens_sample(P, P, [2])
    sums = np.full((2, 5), 7.0)
    launches = dev.launches
    dev.sens_sample(P[:0], P[:0], [0], out=sums)
    assert np.all(sums == 7.0) and dev.launches == launches
    dev.close()
