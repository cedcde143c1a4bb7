"""Leave-one-out cross-validation on the B200 against oracle/loo_oracle.py: the LOO objective and gradient of
gpe_llh_grad_batch in every mode and both covariance families (both product routes at n = 4096), gpe_loo against
explicit deletion, a failed item beside healthy ones, determinism (graph replay, stream count, likelihood calls around a
LOO call), and the LOO objective through g.setup / g.train."""
import contextlib
import io
import os

import numpy as np
import pytest

from oracle import gp_oracle as O, loo_oracle as LO, matern_oracle as M

pytestmark = pytest.mark.gpu
MODES = [1, 5, 0, 4, 2, 6]          # MUCM, MUCM + free nugget, gp4ml, + free nugget, alt nugget, alt + free nugget
FAMILIES = {"gaussian": 0, "matern52": 1}
LOO = 8


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


def _data(n, d, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * np.abs(X - 0.5).sum(1)
    return rng, X, y, np.column_stack([np.ones(n), X])


def _device(X, y, H, r=None, family="gaussian", env=None):
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
    dev.set_kernel(FAMILIES[family])
    return dev


def _thetas(rng, d, mode, B, lo=0.3, hi=0.9):
    cols = [lo + (hi - lo) * rng.random((B, d))]
    if mode & 4:
        cols.append(0.01 + 0.02 * rng.random((B, 1)))
    if not mode & 1:
        cols.append(0.8 + 0.4 * rng.random((B, 1)))
    return O.transform(np.column_stack(cols))


def _check(dev, theta, mode, X, y, H, r, family, items, nug=1e-3):
    L, g, sig, st = dev.llh_grad_batch(theta, mode | LOO, fixed_nugget=nug)
    assert (st == 0).all()
    for b in items:
        ref_L, ref_g, ref_sig = LO.loo_objective(theta[b], X, y, H, mode, family, nug, r)
        assert abs(L[b] - ref_L) <= 1e-10 * abs(ref_L), (mode, b, L[b], ref_L)
        assert np.max(np.abs(g[b] - ref_g)) <= 1e-9 * np.abs(ref_g).max(), (mode, b, g[b], ref_g)
        assert abs(sig[b] - ref_sig) <= 1e-10 * ref_sig
    return L, g, sig, st


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("mode", MODES)
def test_loo_value_and_gradient_all_modes(family, mode):
    rng, X, y, H = _data(200, 3, 2)
    r = 1e-3 * (1.0 + rng.random(200)) if mode & 2 else None
    dev = _device(X, y, H, r, family)
    theta = _thetas(rng, 3, mode, 6)
    _check(dev, theta, mode, X, y, H, 0.0 if r is None else r, family, range(6))
    dev.close()


@pytest.mark.parametrize("family,mode", [("gaussian", 1), ("gaussian", 4), ("matern52", 4)])
def test_loo_n4096_both_routes(family, mode):
    """n = 4096, d = 16, 32 guesses on the INT8 tensor-core route (default) and the FP64 DMMA route (GPE_OZAKI=0)."""
    rng, X, y, H = _data(4096, 16, 3)
    theta = _thetas(rng, 16, mode, 32, 0.7, 1.0)
    for env, int8 in (({}, True), ({"GPE_OZAKI": "0"}, False)):
        dev = _device(X, y, H, family=family, env=env)
        before = dev.int8_products
        _check(dev, theta, mode, X, y, H, 0.0, family, [0, 31])
        assert (dev.int8_products > before) == int8
        dev.close()


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("given_beta", [False, True])
def test_gpe_loo_matches_explicit_deletion(family, kind, given_beta):
    rng, X, y, H = _data(150, 3, 4)
    r = 1e-3 * (1.0 + rng.random(150)) if kind else None
    dev = _device(X, y, H, r, family)
    delta, nug, sigma = np.array([0.3, 0.5, 0.8]), 1e-3, 1.7
    beta = np.array([0.1, -0.2, 0.3, 0.05]) if given_beta else None
    _, _, st = dev.fit_state(delta, nug, sigma, kind, beta=beta)
    assert st == 0
    mean, var = dev.loo()
    fam = O if family == "gaussian" else M
    A = fam.make_A(X, delta, nug, kind, 0.0 if r is None else r, 1.0, True)
    bm, bv = LO.loo_brute(A, H, y)
    assert np.max(np.abs(mean - bm)) <= 1e-9 * np.abs(y - bm).max()
    assert np.max(np.abs(var - sigma ** 2 * bv)) <= 1e-9 * sigma ** 2 * bv.max()
    # device outputs
    import torch
    mt = torch.empty(150, dtype=torch.float64, device="cuda")
    vt = torch.empty(150, dtype=torch.float64, device="cuda")
    dev.loo(out=(mt, vt))
    assert np.array_equal(mt.cpu().numpy(), mean) and np.array_equal(vt.cpu().numpy(), var)
    dev.close()


def test_loo_non_pd_item_is_flagged_not_fatal():
    rng = np.random.default_rng(1)
    n, d = 150, 2
    X = rng.random((n, d)); X[1] = X[0]          # duplicate point + zero nugget => singular
    y = rng.random(n)
    H = O.make_H_linear(X)
    dev = _device(X, y, H)
    theta = O.transform(np.array([[0.3, 0.3, 1e-3, 1.0], [0.5, 0.5, 1e-17, 1.0], [0.4, 0.6, 2e-3, 1.1]]))
    L, g, sig, st = dev.llh_grad_batch(theta, 4 | LOO, fixed_nugget=0.0)
    assert st[1] != 0 and st[0] == 0 and st[2] == 0
    assert np.isinf(L[1])
    for b in (0, 2):
        ref_L, ref_g, _ = LO.loo_objective(theta[b], X, y, H, 4, "gaussian", 0.0)
        assert abs(L[b] - ref_L) <= 1e-10 * abs(ref_L)
        assert np.max(np.abs(g[b] - ref_g)) <= 1e-9 * np.abs(ref_g).max()
    dev.close()


@pytest.mark.parametrize("n", [300, 2048])
def test_loo_deterministic_graphs_streams_and_neighbouring_llh_calls(n):
    """Eager calls and graph replays give the same bits, so does one stream, and a likelihood call is unchanged by a LOO
    call between two of them."""
    rng, X, y, H = _data(n, 4, 6)
    theta = _thetas(rng, 4, 0, 8)
    dev = _device(X, y, H)
    llh0 = dev.llh_grad_batch(theta, 0, fixed_nugget=1e-3)
    runs = [dev.llh_grad_batch(theta, LOO, fixed_nugget=1e-3) for _ in range(4)]   # eager, eager, capture, replay
    llh1 = dev.llh_grad_batch(theta, 0, fixed_nugget=1e-3)
    for a, b in zip(llh0, llh1):
        assert np.array_equal(a, b)
    for run in runs[1:]:
        for a, b in zip(runs[0], run):
            assert np.array_equal(a, b)
    dev.set_streams(1)
    one = dev.llh_grad_batch(theta, LOO, fixed_nugget=1e-3)
    for a, b in zip(runs[0], one):
        assert np.array_equal(a, b)
    dev.close()


def test_setup_train_loo_matches_sequential_scipy(tmp_path):
    """g.setup on a beliefs file with `objective loo`, then the batched multistart: every start must find what SciPy's
    sequential L-BFGS-B finds on the oracle's LOO objective from the same guesses, and the same best start is selected."""
    import gp_emu_uqsa_b200 as g
    from scipy.optimize import minimize
    from oracle import ref_loader as RL
    rng = np.random.default_rng(21)
    n, d, B = 200, 3, 6
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.3 * np.abs(X[:, 0] - 0.4)
    with _cwd(tmp_path), _quiet():
        cfg = RL.write_emulator_files(str(tmp_path), X, y, mucm="F", fix_nugget="T", alt_nugget="F", nugget=1e-4,
                                      name="m", tries=B, constraints="bounds")
        with open("m_beliefs", "a") as f:
            f.write("objective loo\n")
        E = g.setup(cfg, datashuffle=False, scaleinputs=True)
        np.random.seed(4)
        out = io.StringIO()
        with contextlib.redirect_stdout(out):
            E.opt_T.llh_optimize()
    assert " loo: " in out.getvalue() and " llh: " not in out.getvalue()
    table = E.opt_T.last_table
    Xs, H = E.training.inputs, E.training.H
    bounds_t = 2.0 * np.log(np.array(E.config.bounds))
    np.random.seed(4)
    grid = np.array([bounds_t[R, 0] + (bounds_t[R, 1] - bounds_t[R, 0]) * np.random.random_sample(B) for R in range(bounds_t.shape[0])])
    f = lambda t: LO.loo_objective(t, Xs, y, H, 0, "gaussian", 1e-4)[:2]
    funs = np.array([minimize(f, grid[:, C], method="L-BFGS-B", jac=True, bounds=[list(b) for b in bounds_t]).fun
                     for C in range(B)])
    close = np.abs(table[:, 1] - funs) <= 1e-6 * np.abs(funs)
    assert close.sum() >= B - 1, (table[:, 1], funs)
    assert E.opt_T.best_guess == int(np.argmin(funs))
    assert abs(E.opt_T.best_llh - funs.min()) <= 1e-8 * abs(funs.min())


def test_loo_of_trained_toy_sim_emulator(golden_dir, tmp_path):
    """examples/toy-sim trained with `objective loo` (MUCM), then g.loo: sigma is the profiled LOO sigma at the optimum,
    the checkpoint says `objective loo`, and the LOO predictions match explicit deletion."""
    import shutil
    import gp_emu_uqsa_b200 as g
    for f in os.listdir(os.path.join(golden_dir, "toy-sim")):
        shutil.copyfile(os.path.join(golden_dir, "toy-sim", f), os.path.join(str(tmp_path), f))
    path = os.path.join(str(tmp_path), "toy-sim_beliefs")
    text = open(path).read().rstrip("\n")
    with open(path, "w") as f:
        f.write(text + "\nobjective loo\n")
    with _cwd(tmp_path), _quiet():
        np.random.seed(0)
        E = g.setup("toy-sim_config")
        g.train(E)
        mean, var = g.loo(E)
    assert any("objective loo" in open(os.path.join(str(tmp_path), f)).read()
               for f in os.listdir(str(tmp_path)) if f.startswith("toy-sim_beliefs-"))
    Xt, yt, H = E.training.inputs, E.training.outputs, E.training.H
    theta = O.transform(np.asarray(E.par.delta))
    _, _, ref_sig = LO.loo_objective(theta, Xt, yt, H, 1, "gaussian", E.par.nugget)
    assert abs(E.par.sigma - ref_sig) <= 1e-8 * ref_sig
    A = O.make_A(Xt, E.par.delta, E.par.nugget, 0, 0.0, 1.0, True)
    bm, bv = LO.loo_brute(A, H, yt)
    assert np.max(np.abs(mean - bm)) <= 1e-8 * np.abs(yt - bm).max()
    assert np.max(np.abs(var - E.par.sigma ** 2 * bv)) <= 1e-8 * E.par.sigma ** 2 * bv.max()
    z = (yt - mean) / np.sqrt(var)
    assert abs(np.mean(z ** 2) - 1.0) <= 1e-8          # the profiled sigma makes the standardised errors unit-variance
