"""The Matern 5/2 family on the B200 against oracle/matern_oracle.py: dense matrices, likelihood + gradient in every
mode (both product routes at n = 4096), posterior mean / variance, tensor grids, the fused implausibility pass,
history matching, the multistart optimiser end to end, and the switch back to the Gaussian kernel."""
import contextlib
import io
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import matern_oracle as M

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAT = 1
MODES = [1, 5, 0, 4, 2, 6]          # MUCM, MUCM + free nugget, gp4ml, + free nugget, alt nugget, alt + free nugget


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
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * np.abs(X - 0.5).sum(1)     # a kink: the Matern kernel's use case
    return rng, X, y, np.column_stack([np.ones(n), X])


def _device(X, y, H, r=None, family=MAT, env=None):
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


def _thetas(rng, d, mode, B, lo=0.3, hi=0.9):
    cols = [lo + (hi - lo) * rng.random((B, d))]
    if mode & 4:
        cols.append(0.01 + 0.02 * rng.random((B, 1)))
    if not mode & 1:
        cols.append(0.8 + 0.4 * rng.random((B, 1)))
    return M.transform(np.column_stack(cols))


def _check_llh(dev, theta, mode, X, y, H, r, items):
    kind = 1 if mode & 2 else 0
    llh, grad, sig, st = dev.llh_grad_batch(theta, mode, fixed_nugget=1e-3)
    assert (st == 0).all()
    for b in items:
        if mode & 1:
            ref_llh, ref_g, ref_sig = M.loglikelihood_mucm(theta[b], X, y, H, kind, 1e-3, r)
            assert abs(sig[b] - ref_sig) <= 1e-10 * ref_sig
        else:
            ref_llh, ref_g = M.loglikelihood_gp4ml(theta[b], X, y, H, kind, 1e-3, r)
        assert abs(llh[b] - ref_llh) <= 1e-10 * abs(ref_llh), (mode, b, llh[b], ref_llh)
        assert np.max(np.abs(grad[b] - ref_g)) <= 1e-9 * np.abs(ref_g).max(), (mode, b, grad[b], ref_g)
    return llh, grad


# ----------------------------------------------------------------------------------------------------- dense matrices
@pytest.mark.parametrize("kind", [0, 1])
def test_dense_matrices_match_oracle(kind):
    rng, X, y, H = _data(300, 4, 1)
    from gp_emu_uqsa_b200 import _emulatorkernels as K
    from oracle import gp_oracle as O

    def close(a, b):
        return np.max(np.abs(a - b)) <= 1e-14 * max(1.0, np.abs(b).max())

    dev = _device(X, y, H)
    delta, nug = np.array([0.3, 0.5, 0.8, 1.1]), 0.02
    assert close(dev.cov_build(delta, nug, kind, True, 1.0), M.cov_var(X, delta, nug, kind, True))
    assert close(dev.cov_build(delta, nug, kind, False, 1.0), M.cov_var(X, delta, nug, kind, False))
    for di in range(4):
        assert close(dev.cov_grad(delta, nug, kind, di, 1.7), M.grad_delta_A(X, delta, nug, di, 1.7, kind))
    assert close(dev.cov_grad(delta, nug, kind, -1, 1.7), M.grad_nugget_A(X, delta, nug, 1.7, kind))
    Xs = rng.random((333, 4))
    assert close(dev.cross_cov(delta, nug, kind, Xs), M.covar(X, Xs, delta, nug, kind))
    # the kernel classes go through the shared scratch handle, whose family is set on every call
    par = type("P", (), {"delta": delta, "nugget": nug})()
    k = (K.kernel_matern52 if kind == 0 else K.kernel_matern52_alt_nug)(4, par)
    assert close(k.var(X), M.cov_var(X, delta, nug, kind))
    assert close(k.grad_delta_A(X[:, 0], 0, 1.0), M.grad_delta_A(X, delta, nug, 0, 1.0, kind))
    assert close(K.kernel(4, par).var(X), O.cov_var(X, delta, nug, 0))


# ----------------------------------------------------------------------------------------------------- likelihood
@pytest.mark.parametrize("n", [200, 1000])
@pytest.mark.parametrize("mode", MODES)
def test_llh_grad_all_modes(n, mode):
    rng, X, y, H = _data(n, 3, 2)
    r = 1e-3 * (1.0 + rng.random(n)) if (mode & 2 and n == 200) else None
    dev = _device(X, y, H, r)
    theta = _thetas(rng, 3, mode, 6)
    _check_llh(dev, theta, mode, X, y, H, 0.0 if r is None else r, range(6))


@pytest.mark.parametrize("mode", [1, 4])
def test_llh_grad_n4096_both_routes(mode):
    """n = 4096, d = 16, 32 guesses: the INT8 tensor-core route (default) and the FP64 DMMA route (GPE_OZAKI=0) against
    the oracle, and the gp4ml gradient against central differences of the library's own likelihood."""
    rng, X, y, H = _data(4096, 16, 3)
    theta = _thetas(rng, 16, mode, 32, 0.7, 1.0)
    for env, int8 in (({}, True), ({"GPE_OZAKI": "0"}, False)):
        dev = _device(X, y, H, env=env)
        before = dev.int8_products
        llh, grad = _check_llh(dev, theta, mode, X, y, H, 0.0, [0, 31])
        assert (dev.int8_products > before) == int8
        if not mode & 1:
            h, ks = 1e-4, [0, 7, 16]
            tp = np.repeat(theta[:1], 2 * len(ks), axis=0)
            for j, k in enumerate(ks):
                tp[2 * j, k] += h
                tp[2 * j + 1, k] -= h
            lp = dev.llh_grad_batch(tp, mode, fixed_nugget=1e-3)[0]
            fd = (lp[0::2] - lp[1::2]) / (2 * h)
            assert np.max(np.abs(fd - grad[0, ks])) <= 1e-5 * np.abs(grad[0]).max(), (fd, grad[0, ks])
        dev.close()


# ----------------------------------------------------------------------------------------------------- prediction
@pytest.mark.parametrize("kind", [0, 1])
def test_posterior_mean_and_variance(kind):
    rng, X, y, H = _data(1000, 4, 4)
    r = 1e-3 * (1.0 + rng.random(1000)) if kind else None
    dev = _device(X, y, H, r)
    delta, nug, sigma = np.array([0.4, 0.6, 0.5, 0.9]), 1e-3, 1.3
    beta, _, st = dev.fit_state(delta, nug, sigma, kind)
    assert st == 0
    A = M.make_A(X, delta, nug, kind, 0.0 if r is None else r, 1.0)
    assert np.allclose(beta, M.optimalbeta(A, H, y), rtol=1e-9, atol=1e-10)
    Xs = rng.random((700, 4))
    Hs = np.column_stack([np.ones(700), Xs])
    mref, Vref = M.posterior(Xs, Hs, X, y, H, A, beta, sigma, delta, nug, kind)
    mean, var = dev.predict(Xs)
    scale = np.abs(np.diag(Vref)).max()
    assert np.max(np.abs(mean - mref)) <= 1e-8 * max(1.0, np.abs(mref).max())
    assert np.max(np.abs(var - np.diag(Vref))) <= 1e-8 * scale
    m2, V2 = dev.predict_fullcov(Xs[:300], None, None)
    assert np.max(np.abs(m2 - mref[:300])) <= 1e-8 * max(1.0, np.abs(mref).max())
    assert np.max(np.abs(V2 - Vref[:300, :300])) <= 1e-8 * scale


_GRID_SCRIPT = r"""
import sys, numpy as np
sys.path.insert(0, %r)
from gp_emu_uqsa_b200 import _lib
rng = np.random.default_rng(5)
X = rng.random((500, 3)); y = np.sin(X.sum(1)); H = np.column_stack([np.ones(500), X])
dev = _lib.Device(0); dev.set_training(X, y, H); dev.set_basis([0, 1, 2], [1, 1, 1]); dev.set_kernel(1)
assert dev.fit_state(np.array([0.3, 0.5, 0.7]), 1e-3, 1.2, 0)[2] == 0
lv, lo, hi = np.array([9, 8, 7]), np.array([-0.1, 0.0, 0.2]), np.array([1.1, 1.0, 0.9])
gm, gv = dev.predict_grid(lv, lo, hi, 3, 500)
idx = np.arange(3, 503)
dig = np.stack([idx // 56, (idx // 7) %% 8, idx %% 7], 1).astype(float)
P = lo + (dig + 0.5) * ((hi - lo) / lv)
pm, pv = dev.predict(P)
np.save(sys.argv[1], np.stack([gm, gv, pm, pv]))
"""


def test_grid_matches_explicit_points_both_paths(tmp_path):
    """Tensor grid through the additive table and through the direct kernel (GPE_GRID_SEP=0, read once per process,
    hence the subprocesses) against the same points given explicitly."""
    for sep in ("1", "0"):
        out = str(tmp_path / ("g%s.npy" % sep))
        env = dict(os.environ, GPE_GRID_SEP=sep)
        subprocess.run([sys.executable, "-c", _GRID_SCRIPT % ROOT, out], check=True, env=env)
        gm, gv, pm, pv = np.load(out)
        assert np.max(np.abs(gm - pm)) <= 1e-10 * np.abs(pm).max()
        assert np.max(np.abs(gv - pv)) <= 1e-9 * np.abs(pv).max()


def test_predict_implaus_bit_identical_to_predict_and_implausibility():
    import torch
    rng, X, y, H = _data(1500, 3, 6)
    dev = _device(X, y, H)
    assert dev.fit_state(np.array([0.3, 0.4, 0.6]), 1e-3, 1.1, 0)[2] == 0
    Xs = rng.random((5000, 3))
    z, ve, cm = float(np.median(y)), 1e-3, 2.0
    mean, var = dev.predict(Xs)
    Imax, keep, cnt, _, _ = dev.implausibility(mean[None], var[None], [z], [ve], cm, 1)
    Itop = torch.zeros((5000, 1), dtype=torch.float64, device="cuda")
    keep2 = np.empty(5000, dtype=np.uint8)
    cnt2, _, _ = dev.predict_implaus(z, ve, Itop, True, True, points=Xs, maxno=1, cm=cm, keep=keep2)
    assert np.array_equal(Itop.cpu().numpy(), Imax) and np.array_equal(keep2, keep) and np.array_equal(cnt2, cnt)
    # the same over a tensor grid (additive table)
    lv, lo, hi = [20, 16, 16], [0.0] * 3, [1.0] * 3
    gm, gv = dev.predict_grid(lv, lo, hi, 0, 5120)
    Imax, keep, cnt, _, _ = dev.implausibility(gm[None], gv[None], [z], [ve], cm, 1)
    Itop = torch.zeros((5120, 1), dtype=torch.float64, device="cuda")
    keep2 = np.empty(5120, dtype=np.uint8)
    cnt2, _, _ = dev.predict_implaus(z, ve, Itop, True, True, grid=(lv, lo, hi, 0, 5120), maxno=1, cm=cm, keep=keep2)
    assert np.array_equal(Itop.cpu().numpy(), Imax) and np.array_equal(keep2, keep) and np.array_equal(cnt2, cnt)


# ----------------------------------------------------------------------------------------------------- Python API
def test_nonimp_data_with_two_matern_emulators(golden_dir, tmp_path):
    import gp_emu_uqsa_b200 as g
    import gp_emu_uqsa_b200.history_match as h
    gold = np.load(os.path.join(golden_dir, "hmapi_n100_d3.npz"))
    emuls = []
    with _cwd(tmp_path), _quiet():
        for o in (0, 1):
            for fn in ("hm%d_config_r" % o, "hm%d_beliefs-0f" % o, "hm%d_input-o0-0f" % o, "hm%d_output-o0-0f" % o):
                with open(fn, "wb") as f:
                    f.write(bytes(gold["file_" + fn]))
            with open("hm%d_beliefs-0f" % o, "a") as f:
                f.write("kernel matern52\n")
            emuls.append(g.setup("hm%d_config_r" % o, datashuffle=False, scaleinputs=True))
        zs, ve, cm = list(gold["zs"]), list(gold["var_extra"]), float(gold["cm"])
        sim = gold["sim_in"]
        np.savetxt("sim_in", sim, fmt="%.17g")
        np.savetxt("sim_out", sim[:, :2], fmt="%.17g")
        cnt = h.nonimp_data(emuls, zs, cm, ve, ["sim_in", "sim_out"], maxno=1)
        got = np.atleast_2d(np.loadtxt("nonimp_sim_in"))
    assert all(type(E.K).__name__.startswith("kernel_matern52") for E in emuls)
    # nonimp_data scales the inputs file with the emulators' input_minmax (a later emulator's range wins) and writes the
    # kept rows as scaled
    scaled = sim.copy()
    for E in emuls:
        for idx, (lo, hi) in zip(E.beliefs.active_index, E.beliefs.input_minmax):
            scaled[:, idx] = (sim[:, idx] - lo) / (hi - lo)
    Imax = np.zeros(sim.shape[0])
    for o, E in enumerate(emuls):
        xs = scaled[:, E.beliefs.active_index]
        Xt, yt = E.training.inputs, E.training.outputs
        kind = 1 if E.beliefs.alt_nugget == "T" else 0
        A = M.make_A(Xt, E.par.delta, E.par.nugget, kind, 0.0, 1.0)
        mu, V = M.posterior(xs, E.basis.design_matrix(xs), Xt, yt, E.training.H, A, E.par.beta, E.par.sigma, E.par.delta,
                            E.par.nugget, kind)
        Imax = np.maximum(Imax, np.abs(mu - zs[o]) / np.sqrt(np.diag(V) + ve[o]))
    keep = Imax < cm
    assert cnt == keep.sum()
    assert np.allclose(got, scaled[keep], rtol=0, atol=1e-15)


def test_setup_train_matern_matches_sequential_scipy(tmp_path):
    """g.setup on a beliefs file with `kernel matern52`, then the batched multistart: every start must find what SciPy's
    sequential L-BFGS-B finds on the oracle from the same guesses, and the same best start is selected."""
    import gp_emu_uqsa_b200 as g
    from scipy.optimize import minimize
    from oracle import ref_loader as RL
    rng = np.random.default_rng(21)
    n, d, B = 300, 4, 6
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.3 * np.abs(X[:, 0] - 0.4)
    with _cwd(tmp_path), _quiet():
        cfg = RL.write_emulator_files(str(tmp_path), X, y, mucm="F", fix_nugget="T", alt_nugget="F", nugget=1e-4,
                                      name="m", tries=B, constraints="bounds")
        with open("m_beliefs", "a") as f:
            f.write("kernel matern52\n")
        E = g.setup(cfg, datashuffle=False, scaleinputs=True)
        np.random.seed(4)
        E.opt_T.llh_optimize()
    assert isinstance(E.K, g._emulatorkernels.kernel_matern52)
    table = E.opt_T.last_table
    Xs, H = E.training.inputs, E.training.H
    bounds_t = 2.0 * np.log(np.array(E.config.bounds))
    np.random.seed(4)
    grid = np.array([bounds_t[R, 0] + (bounds_t[R, 1] - bounds_t[R, 0]) * np.random.random_sample(B) for R in range(bounds_t.shape[0])])
    funs = np.array([minimize(lambda t: M.loglikelihood_gp4ml(t, Xs, y, H, 0, 1e-4), grid[:, C], method="L-BFGS-B", jac=True,
                              bounds=[list(b) for b in bounds_t]).fun for C in range(B)])
    close = np.abs(table[:, 1] - funs) <= 1e-6 * np.abs(funs)
    assert close.sum() >= B - 1, (table[:, 1], funs)
    assert E.opt_T.best_guess == int(np.argmin(funs))
    assert abs(E.opt_T.best_llh - funs.min()) <= 1e-8 * abs(funs.min())


def test_switch_back_to_gaussian_is_bit_identical_to_fresh_handle():
    rng, X, y, H = _data(2048, 4, 7)
    theta = _thetas(rng, 4, 0, 4)
    Xs = rng.random((1024, 4))
    delta = np.array([0.4, 0.5, 0.6, 0.7])

    def run(dev):
        out = dev.llh_grad_batch(theta, 0, fixed_nugget=1e-3)[:2]
        dev.fit_state(delta, 1e-3, 1.2, 0)
        return out + dev.predict(Xs) + (dev.cov_build(delta, 1e-3, 0),)

    dev = _device(X, y, H)
    mat = run(dev)
    dev.set_kernel(0)
    back = run(dev)
    fresh = run(_device(X, y, H, family=0))
    for a, b in zip(back, fresh):
        assert np.array_equal(a, b)
    assert not np.array_equal(mat[4], back[4])


def test_sensitivity_is_refused_for_matern(tmp_path):
    import gp_emu_uqsa_b200 as g
    import gp_emu_uqsa_b200.sensitivity as s
    from gp_emu_uqsa_b200 import _lib
    from oracle import ref_loader as RL
    rng, X, y, H = _data(100, 2, 8)
    with _cwd(tmp_path), _quiet():
        cfg = RL.write_emulator_files(str(tmp_path), X, y, mucm="T", fix_nugget="T", alt_nugget="F", name="s")
        with open("s_beliefs", "a") as f:
            f.write("kernel matern52\n")
        E = g.setup(cfg, datashuffle=False, scaleinputs=True)
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        assert s.setup(E, [0.5, 0.5], [0.02, 0.02]) is None
    assert "need the Gaussian kernel" in out.getvalue()
    dev = _device(X, y, H)
    assert dev.fit_state(np.array([0.5, 0.5]), 1e-3, 1.0, 0)[2] == 0
    with pytest.raises(_lib.GpeError, match="sensitivity integrals need the Gaussian kernel"):
        dev.sens_contract(np.ones(2), np.ones(2), np.zeros(2), 1.0, np.ones((100, 1)))
