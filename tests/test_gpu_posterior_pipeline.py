"""The posterior entry points on the fit state build the cross-covariance slab and the regression product
[A^-1 H K^-T | e]^T C through one step (gpe_predict.cu: posterior_cross), so the mean of predict_fullcov is the mean of predict
bit for bit: on both routes of the L^-1 product, for both covariance families, with the device basis and with explicit H*."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
from oracle import gp_oracle as O  # noqa: E402


@pytest.mark.parametrize("family", [0, 1])
@pytest.mark.parametrize("route", ["dmma", "int8"])
def test_fullcov_mean_is_the_prediction_mean(route, family, monkeypatch):
    from gp_emu_uqsa_b200 import _lib
    if route == "dmma":
        monkeypatch.setenv("GPE_OZAKI", "0")
    else:
        monkeypatch.delenv("GPE_OZAKI", raising=False)
    rng = np.random.default_rng(41 + family)
    n, d, m = 1500, 5, 1000              # m is no multiple of 128; 1024 padded points take the INT8 route when it is on
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * (X ** 2).sum(1)
    H = O.make_H_linear(X)
    Xs = rng.random((m, d))
    Xs[-8:] += 2.0
    dev = _lib.Device(0)
    try:
        dev.set_training(X, y, H)
        dev.set_basis(list(range(d)), [1] * d)
        dev.set_kernel(family)
        _, _, st = dev.fit_state(np.linspace(0.3, 1.2, d), 1e-5, 1.3, 0)
        assert st == 0
        k0 = dev.int8_products
        mean, _ = dev.predict(Xs)                     # with the variance: the product Z = L^-1 C runs
        assert (dev.int8_products > k0) == (route == "int8")
        mf, _ = dev.predict_fullcov(Xs)
        assert np.array_equal(mf, mean)
        Hs = O.make_H_linear(Xs)
        mean_h, _ = dev.predict(Xs, Hs=Hs)
        mf_h, _ = dev.predict_fullcov(Xs, Hs=Hs)
        assert np.array_equal(mf_h, mean_h)
    finally:
        dev.close()
