"""CPU checks of leave-one-out cross-validation: the oracle's closed form against explicit deletion, its gradient against
central differences of its objective, and the ``objective`` key of the beliefs file (read, written, rejected)."""
import contextlib
import io

import numpy as np
import pytest

from oracle import gp_oracle as O, loo_oracle as LO

MODES = [1, 5, 0, 4, 2, 6]          # MUCM, MUCM + free nugget, gp4ml, + free nugget, alt nugget, alt + free nugget
FAMILIES = ["gaussian", "matern52"]


@contextlib.contextmanager
def _quiet():
    with contextlib.redirect_stdout(io.StringIO()):
        yield


def _case(mode, seed=5, n=30, d=3):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.2 * np.abs(X[:, 0] - 0.5)
    H = np.column_stack([np.ones(n), X])
    r = 1e-3 * (1.0 + rng.random(n)) if mode & 2 else 0.0
    hp = [0.3, 0.5, 0.7][:d] + ([0.05] if mode & 4 else []) + ([] if mode & 1 else [1.3])
    return X, y, H, r, O.transform(np.array(hp))


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("mode", MODES)
def test_closed_form_equals_explicit_deletion(family, mode):
    X, y, H, r, theta = _case(mode)
    A = LO.make_A(theta, X, mode, family, 1e-3, r)
    _, e, v, s2, _, _ = LO.loo_closed(A, H, y, bool(mode & 1))
    mean, var = LO.loo_brute(A, H, y)
    assert np.max(np.abs((y - mean) - e)) <= 1e-10 * np.abs(e).max()
    assert np.max(np.abs(s2 * var - v)) <= 1e-10 * v.max()


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("mode", MODES)
def test_oracle_gradient_matches_central_difference(family, mode):
    X, y, H, r, theta = _case(mode)
    L, g, _ = LO.loo_objective(theta, X, y, H, mode, family, 1e-3, r)
    fd = np.empty_like(theta)
    for k in range(theta.size):
        e = np.zeros_like(theta)
        e[k] = 1e-6
        fd[k] = (LO.loo_objective(theta + e, X, y, H, mode, family, 1e-3, r)[0]
                 - LO.loo_objective(theta - e, X, y, H, mode, family, 1e-3, r)[0]) / 2e-6
    assert np.max(np.abs(g - fd)) <= 1e-6 * np.abs(fd).max()


def test_profiled_sigma_minimises_the_objective():
    """MUCM: s^2 = mean(alpha^2 / P_ii) is the minimiser of the gp4ml-form objective over a free scale."""
    X, y, H, r, theta = _case(1)
    A = LO.make_A(theta, X, 1)
    L, _, _, s2, P, alpha = LO.loo_closed(A, H, y, True)
    p = np.diag(P)
    f = lambda t: 0.5 * np.sum(np.log(2 * np.pi * t / p) + alpha ** 2 / (t * p))
    assert abs(f(s2) - L) <= 1e-12 * abs(L)
    assert f(s2 * 1.01) > L and f(s2 * 0.99) > L


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


def _fake_emulator(path):
    import types
    par = types.SimpleNamespace(beta=np.array([0.5, 1.5]), delta=np.array([0.25, 0.75]), sigma=2.0, nugget=0.01)
    return types.SimpleNamespace(config=types.SimpleNamespace(beliefs=path), tv_conf=types.SimpleNamespace(no_of_trains=1),
                                 par=par, all_data=types.SimpleNamespace(input_minmax=[[0.0, 1.0], [0.0, 2.0]]))


@pytest.mark.parametrize("objective", [None, "llh", "loo"])
def test_beliefs_objective_key_read_and_written(tmp_path, objective):
    from gp_emu_uqsa_b200 import _emulatorclasses as C
    path = str(tmp_path / "b")
    with open(path, "w") as fh:
        fh.write(BELIEFS + ("kernel matern52\n" if objective == "loo" else "")
                 + ("objective %s\n" % objective if objective else ""))
    with _quiet():
        bel = C.Beliefs(path)
        assert bel.objective == (objective or "llh")
        bel.final_beliefs(_fake_emulator(path), final=True)
    written = open(path + "-1f").read()
    expected = ("active_index 0 1\nactive 0 1\noutput_index 0\noutput 0 \nbasis_str 1.0 x\nbasis_inf NA 0\nbeta 0.5 1.5\n"
                "delta 0.25 0.75\nsigma 2.0\nnugget 0.01\nfix_nugget T\nalt_nugget F\nmucm T\n"
                + ("kernel matern52\nobjective loo\n" if objective == "loo" else "")
                + "input_minmax [[0.0, 1.0], [0.0, 2.0]]\n")
    assert written == expected
    with _quiet():
        again = C.Beliefs(path + "-1f")
    assert again.objective == bel.objective


def test_beliefs_unknown_objective_exits(tmp_path):
    from gp_emu_uqsa_b200 import _emulatorclasses as C
    path = str(tmp_path / "b")
    with open(path, "w") as fh:
        fh.write(BELIEFS + "objective kfold\n")
    out = io.StringIO()
    with contextlib.redirect_stdout(out), pytest.raises(SystemExit):
        C.Beliefs(path)
    assert "WARNING: objective should be one of llh loo" in out.getvalue()


def test_optimize_mode_sets_the_loo_bit():
    import types
    from gp_emu_uqsa_b200 import _emulatoroptimise as Opt, _lib
    for objective, bit in (("llh", 0), ("loo", _lib.MODE_LOO)):
        o = Opt.Optimize.__new__(Opt.Optimize)
        o.beliefs = types.SimpleNamespace(mucm="T", alt_nugget="F", fix_nugget="F", objective=objective)
        assert o._mode() == _lib.MODE_MUCM | _lib.MODE_NUGGET_FREE | bit
    assert _lib.MODE_LOO == 8 and "gpe_loo" in _lib.EXPORTS
