"""CPU checks of the sampled sensitivity estimator's conventions (oracle/sens_sample_oracle.py, the term table of
gpe_sens_sample) against independent references: the closed-form integrals (oracle/sens_oracle.py) for a Gaussian kernel
with normal inputs, and tensor quadrature for a Matérn 5/2 kernel with uniform inputs."""
import numpy as np

from oracle import gp_oracle as G
from oracle import matern_oracle as Mo
from oracle import sens_sample_oracle as SO
from oracle.sens_oracle import SensOracle
from gp_emu_uqsa_b200.sensitivity._sampledsensitivity import sample_points


def _check(mu, err, ref, uEV):
    dev = np.abs(mu - ref)
    assert np.all(dev <= 3.0 * err), (dev / err).max()
    assert np.all(dev <= 1e-3 * abs(uEV)), (dev / abs(uEV)).max()


def test_estimator_matches_closed_form_gaussian_normal_inputs():
    rng = np.random.default_rng(5)
    n, d, nug = 150, 4, 1e-3
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.3 * X[:, 0] ** 2
    delta = 0.4 + 0.4 * rng.random(d)
    H, A = G.make_H_linear(X), G.make_A(X, delta, nug)
    beta, sigma = G.optimalbeta(A, H, y), 0.7
    m, v = 0.3 + 0.4 * rng.random(d), 0.01 + 0.03 * rng.random(d)
    O = SensOracle(X, y, H, A, beta, sigma, nug, delta, m, v)
    uE, uV, uEV = O.uncertainty()
    total = np.array([uEV - O.EVint([k for k in range(d) if k != P]) for P in range(d)])   # E*[V_T,P]
    ref = np.concatenate([[uE, uV, uEV], O.sensitivity(), total])
    XA, XB = sample_points(d, 2 ** 14, 0, m=m, v=v)
    T = SO.terms(SO.Post(X, y, H, A, beta, sigma, delta, nug), XA, XB, list(range(d)), y.mean())
    mu, err = SO.estimates(T)
    _check(mu, err, ref, uEV)


def test_estimator_matches_quadrature_matern_uniform_inputs():
    rng = np.random.default_rng(6)
    n, d, nug = 60, 2, 1e-3
    X = rng.random((n, d))
    y = np.cos(3 * X[:, 0]) * X[:, 1] + X[:, 1] ** 2
    delta = np.array([0.3, 0.5])
    H, A = G.make_H_linear(X), Mo.make_A(X, delta, nug)
    post = SO.Post(X, y, H, A, G.optimalbeta(A, H, y), 0.9, delta, nug, family=1)
    bounds = [[0.1, 0.9], [0.0, 1.0]]
    Q = SO.quadrature(post, [("uniform", lo, hi) for lo, hi in bounds])
    ref = np.concatenate([[Q["uE"], Q["uV"], Q["uEV"]], Q["senseindex"], Q["EVTw"]])
    XA, XB = sample_points(d, 2 ** 14, 0, bounds=bounds)
    mu, err = SO.estimates(SO.terms(post, XA, XB, [0, 1], y.mean()))
    _check(mu, err, ref, Q["uEV"])


def test_sample_points_leave_the_global_rng_alone():
    st = np.random.get_state()
    A, B = sample_points(3, 256, 7, m=[0.5, 0.4, 0.6], v=[0.01, 0.02, 0.03])
    after = np.random.get_state()
    assert st[0] == after[0] and np.array_equal(st[1], after[1]) and st[2:] == after[2:]
    A2, B2 = sample_points(3, 256, 7, m=[0.5, 0.4, 0.6], v=[0.01, 0.02, 0.03])
    assert np.array_equal(A, A2) and np.array_equal(B, B2) and np.all(np.isfinite(A)) and not np.array_equal(A, B)
    U, _ = sample_points(2, 1024, 1, bounds=[[0.2, 0.4], [-1.0, 3.0]])
    assert U[:, 0].min() > 0.2 and U[:, 0].max() < 0.4 and U[:, 1].min() > -1.0 and U[:, 1].max() < 3.0


def test_setup_sampled_refuses_malformed_arguments_before_any_device_work():
    import contextlib
    import io
    from types import SimpleNamespace
    from gp_emu_uqsa_b200.sensitivity import setup_sampled
    E = SimpleNamespace(training=SimpleNamespace(inputs=np.zeros((5, 2))), basis=SimpleNamespace(poly=[1, 1]))
    for kw, msg in (({"m": [0.5, 0.5]}, "either input means"),
                    ({"v": [0.01, 0.01]}, "either input means"),
                    ({}, "either input means"),
                    ({"m": [0.5, 0.5], "v": [0.01, 0.01], "bounds": [[0, 1], [0, 1]]}, "either input means"),
                    ({"m": [0.5], "v": [0.01]}, "as many finite values"),
                    ({"m": [0.5, np.nan], "v": [0.01, 0.01]}, "as many finite values"),
                    ({"m": [0.5, 0.5], "v": [0.01, 0.0]}, "variances must be positive"),
                    ({"bounds": [[0, 1], [0.5, 0.5]]}, "lo < hi"),
                    ({"bounds": [[0, 1]]}, "one finite [lo, hi] pair"),
                    ({"bounds": [[0, 1], [0, 1]], "samples": 1000}, "power of two"),
                    ({"bounds": [[0, 1], [0, 1]], "samples": 128}, "power of two")):
        out = io.StringIO()
        with contextlib.redirect_stdout(out):
            assert setup_sampled(E, **kw) is None
        assert msg in out.getvalue(), (kw, out.getvalue())
    E.basis.poly = None
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        assert setup_sampled(E, bounds=[[0, 1], [0, 1]]) is None
    assert "polynomial mean" in out.getvalue()
