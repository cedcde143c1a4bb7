"""CPU checks of the Matern 5/2 family: the oracle's correlation against the Bessel form, its gradient against central
differences, and the ``kernel`` key of the beliefs file (read, written, rejected)."""
import contextlib
import io
import os
import types

import numpy as np
import pytest
from scipy import special

from oracle import matern_oracle as M


@contextlib.contextmanager
def _quiet():
    with contextlib.redirect_stdout(io.StringIO()):
        yield


def test_matern52_equals_bessel_form():
    r = np.concatenate([np.linspace(1e-3, 1.0, 500), np.linspace(1.0, 20.0, 500)])
    nu = 2.5
    z = np.sqrt(5.0) * r
    bessel = 2.0 ** (1.0 - nu) / special.gamma(nu) * z ** nu * special.kv(nu, z)
    assert np.max(np.abs(M.R_of_D(r * r) - bessel)) <= 1e-14
    assert M.R_of_D(np.zeros(1))[0] == 1.0


def test_derivative_factor_matches_central_difference():
    rng = np.random.default_rng(3)
    X = rng.random((12, 3))
    delta = np.array([0.4, 0.7, 1.1])
    for k in range(3):
        th = M.transform(delta)
        h = 1e-6
        tp, tm = th.copy(), th.copy()
        tp[k] += h
        tm[k] -= h
        fd = (M.cov_var(X, M.untransform(tp), 0.0) - M.cov_var(X, M.untransform(tm), 0.0)) / (2 * h)
        an = M.grad_delta_A(X, delta, 0.0, k, 1.0)
        assert np.max(np.abs(fd - an)) <= 1e-8


@pytest.mark.parametrize("mucm,alt,free", [(1, 0, 0), (1, 0, 1), (0, 0, 0), (0, 0, 1), (0, 1, 0), (0, 1, 1)])
def test_oracle_llh_gradient_matches_central_difference(mucm, alt, free):
    rng = np.random.default_rng(11)
    n, d = 40, 2
    X = rng.random((n, d))
    y = np.sin(3 * X[:, 0]) + X[:, 1] ** 2
    H = np.column_stack([np.ones(n), X])
    r = 1e-3 * (1 + rng.random(n)) if alt else 0.0
    hp = [0.5, 0.8] + ([0.05] if free else []) + ([] if mucm else [1.3])
    theta = M.transform(np.array(hp))
    f = M.loglikelihood_mucm if mucm else M.loglikelihood_gp4ml
    g = f(theta, X, y, H, alt, 1e-3, r)[1]
    fd = np.empty_like(theta)
    for k in range(theta.size):
        e = np.zeros_like(theta)
        e[k] = 1e-6
        fd[k] = (f(theta + e, X, y, H, alt, 1e-3, r)[0] - f(theta - e, X, y, H, alt, 1e-3, r)[0]) / 2e-6
    if mucm:
        # the MUCM gradient carries the reference's sigma_hat^2 factor (scaled copies of dA/dtheta); the llh itself is
        # the profile likelihood, so compare the direction up to that factor
        sig2 = f(theta, X, y, H, alt, 1e-3, r)[2] ** 2
        g = g / sig2
    assert np.max(np.abs(g - fd)) <= 1e-6 * max(1.0, np.abs(fd).max())


BELIEFS = """active all
output 0
basis_str 1.0 x
basis_inf NA 0
beta 1.0 1.0
delta 1.0 1.0
sigma 1.0
nugget 0.01
fix_nugget T
mucm T
"""


def _fake_emulator(beliefs, path):
    par = types.SimpleNamespace(beta=np.array([0.5, 1.5]), delta=np.array([0.25, 0.75]), sigma=2.0, nugget=0.01)
    return types.SimpleNamespace(config=types.SimpleNamespace(beliefs=path), tv_conf=types.SimpleNamespace(no_of_trains=1),
                                 par=par, all_data=types.SimpleNamespace(input_minmax=[[0.0, 1.0], [0.0, 2.0]]),
                                 beliefs=beliefs)


@pytest.mark.parametrize("kernel", [None, "gaussian", "matern52"])
def test_beliefs_kernel_key_read_and_written(tmp_path, kernel):
    from gp_emu_uqsa_b200 import _emulatorclasses as C
    path = str(tmp_path / "b")
    with open(path, "w") as fh:
        fh.write(BELIEFS + ("kernel %s\n" % kernel if kernel else ""))
    with _quiet():
        bel = C.Beliefs(path)
        assert bel.kernel == (kernel or "gaussian")
        bel.final_beliefs(_fake_emulator(bel, path), final=True)
    written = open(path + "-1f").read()
    expected = ("active_index 0 1\nactive 0 1\noutput_index 0\noutput 0 \nbasis_str 1.0 x\nbasis_inf NA 0\nbeta 0.5 1.5\n"
                "delta 0.25 0.75\nsigma 2.0\nnugget 0.01\nfix_nugget T\nalt_nugget F\nmucm T\n"
                + ("kernel matern52\n" if kernel == "matern52" else "")
                + "input_minmax [[0.0, 1.0], [0.0, 2.0]]\n")
    assert written == expected
    with _quiet():
        again = C.Beliefs(path + "-1f")
    assert again.kernel == bel.kernel


def test_beliefs_unknown_kernel_exits(tmp_path):
    from gp_emu_uqsa_b200 import _emulatorclasses as C
    path = str(tmp_path / "b")
    with open(path, "w") as fh:
        fh.write(BELIEFS + "kernel matern32\n")
    out = io.StringIO()
    with contextlib.redirect_stdout(out), pytest.raises(SystemExit):
        C.Beliefs(path)
    assert "WARNING: kernel should be one of gaussian matern52" in out.getvalue()


def test_kernel_classes_carry_family():
    from gp_emu_uqsa_b200 import _emulatorkernels as K, _lib
    assert (K.kernel.family, K.kernel.kind) == (_lib.KERNEL_GAUSSIAN, 0)
    assert (K.kernel_alt_nug.family, K.kernel_alt_nug.kind) == (_lib.KERNEL_GAUSSIAN, 1)
    assert (K.kernel_matern52.family, K.kernel_matern52.kind) == (_lib.KERNEL_MATERN52, 0)
    assert (K.kernel_matern52_alt_nug.family, K.kernel_matern52_alt_nug.kind) == (_lib.KERNEL_MATERN52, 1)
