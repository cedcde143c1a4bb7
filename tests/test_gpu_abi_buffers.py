"""Host and device buffers at the C-ABI: the header lets array arguments be host or device memory, each one on its own.  Every
entry point here is called through dev.L.gpe_* once with NumPy arrays and once with torch CUDA tensors (for
gpe_implausibility also with mean and var in different places) and must return bit-identical results."""
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
PLACES = ("host", "device")


def _place(a, where):
    """NumPy array a as host memory, or copied into a torch CUDA tensor."""
    a = np.ascontiguousarray(a)
    if where == "host":
        return a
    import torch
    return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).cuda()


def _empty(shape, dtype, where):
    return _place(np.zeros(shape, dtype), where)


def _host(a):
    """Host copy of an output, as NumPy with the bits the library wrote (uint64 outputs live in int64 tensors)."""
    if isinstance(a, np.ndarray):
        return a
    return a.cpu().numpy()


def _same(a, b):
    a, b = _host(a), _host(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.fixture(scope="module")
def dev():
    from gp_emu_uqsa_b200 import _lib
    rng = np.random.default_rng(3)
    n, d = 300, 4
    X = rng.random((n, d))
    y = np.sin(X @ rng.normal(size=d)) + 0.1 * (X ** 2).sum(1)
    dev = _lib.Device(0)
    dev.set_training(X, y, np.column_stack([np.ones(n), X]))
    dev.set_basis(list(range(d)), [1] * d)
    delta = 0.3 + 0.5 * rng.random(d)
    _, _, st = dev.fit_state(delta, 1e-4, 0.9)
    assert st == 0
    dev.delta = delta
    yield dev
    dev.close()


def _call(dev, fn, *args):
    from gp_emu_uqsa_b200._lib import _ptr
    dev._ck(getattr(dev.L, fn)(dev.h, *[_ptr(a) if a is None or hasattr(a, "shape") else a for a in args]))


def test_cov_build(dev):
    outs = {}
    for w in PLACES:
        A = _empty((dev.n, dev.n), np.float64, w)
        _call(dev, "gpe_cov_build", _place(dev.delta, w), 1e-4, 0, 1, 1.0, A)
        outs[w] = A
    assert _same(outs["host"], outs["device"])
    assert np.abs(_host(outs["host"])).max() > 0


@pytest.mark.parametrize("which,kind", [(1, 0), (-1, 0), (-1, 1)])
def test_cov_grad(dev, which, kind):
    outs = {}
    for w in PLACES:
        G = _empty((dev.n, dev.n), np.float64, w)
        _call(dev, "gpe_cov_grad", _place(dev.delta, w), 1e-2, kind, which, 1.3, G)
        outs[w] = G
    assert _same(outs["host"], outs["device"])
    assert np.abs(_host(outs["host"])).max() > 0


def test_loo(dev):
    outs = {}
    for w in PLACES:
        mean, var = _empty(dev.n, np.float64, w), _empty(dev.n, np.float64, w)
        _call(dev, "gpe_loo", mean, var)
        outs[w] = (mean, var)
    assert all(_same(a, b) for a, b in zip(outs["host"], outs["device"]))
    assert np.isfinite(_host(outs["host"][1])).all()


def test_pdist_argmin_with_extra(dev):
    rng = np.random.default_rng(5)
    designs, extra = rng.random((6, 40, 3)), rng.random((9, 3))
    outs = {}
    for w in PLACES:
        out = _empty(6, np.int64, w)
        _call(dev, "gpe_pdist_argmin", _place(designs, w), 6, 40, 3, _place(extra, w), 9, out)
        outs[w] = out
    assert _same(outs["host"], outs["device"])


def test_predict_fullcov_with_Hs_and_r_new(dev):
    rng = np.random.default_rng(7)
    m = 70
    Xs = rng.random((m, dev.d))
    Hs, r_new = np.column_stack([np.ones(m), Xs]), 1e-3 * rng.random(m)
    outs = {}
    for w in PLACES:
        mean, V = _empty(m, np.float64, w), _empty((m, m), np.float64, w)
        _call(dev, "gpe_predict_fullcov", _place(Xs, w), _place(Hs, w), m, _place(r_new, w), mean, V)
        outs[w] = (mean, V)
    assert all(_same(a, b) for a, b in zip(outs["host"], outs["device"]))
    mean_ref, _ = dev.predict(Xs, Hs)
    np.testing.assert_allclose(_host(outs["host"][0]), mean_ref, rtol=1e-10, atol=1e-12)


def _implausibility(dev, mean_at, var_at, out_at, mean, var, z, ve, cm, maxno, cell_pts, first_index, ncell):
    n_emul, m = mean.shape
    outs = (_empty((m, maxno), np.float64, out_at), _empty(m, np.uint8, out_at), _empty(maxno, np.uint64, out_at),
            _empty((ncell, maxno), np.float64, out_at), _empty((ncell, maxno), np.uint64, out_at))
    _call(dev, "gpe_implausibility", _place(mean, mean_at), _place(var, var_at), n_emul, m, _place(z, out_at), _place(ve, out_at),
          cm, maxno, cell_pts, first_index, ncell, *outs)
    return outs


def test_implausibility_host_and_device_buffers(dev):
    """mean and var are staged each on its own: all four host / device combinations, with host or device outputs, give the
    all-host result."""
    rng = np.random.default_rng(9)
    n_emul, m, maxno, cell_pts, first_index = 3, 1000, 2, 50, 25
    ncell = (first_index + m - 1) // cell_pts - first_index // cell_pts + 1
    mean, var = rng.normal(size=(n_emul, m)), 0.1 + rng.random((n_emul, m))
    z, ve, cm = rng.normal(size=n_emul), 0.01 * np.ones(n_emul), 1.5
    args = (mean, var, z, ve, cm, maxno, cell_pts, first_index, ncell)
    ref = _implausibility(dev, "host", "host", "host", *args)
    assert 0 < _host(ref[2])[0] < m and _host(ref[4]).sum() > 0
    for mean_at, var_at, out_at in itertools.product(PLACES, PLACES, PLACES):
        got = _implausibility(dev, mean_at, var_at, out_at, *args)
        assert all(_same(a, b) for a, b in zip(got, ref)), (mean_at, var_at, out_at)


def test_predict_implaus_host_and_device_keep(dev):
    import torch
    rng = np.random.default_rng(11)
    m, maxno, cell_pts, first_index = 600, 1, 40, 10
    ncell = (first_index + m - 1) // cell_pts - first_index // cell_pts + 1
    Xs = rng.random((m, dev.d))
    mean, _ = dev.predict(Xs)
    z, cm = float(np.median(mean)), 2.0
    outs = {}
    for w in PLACES:
        Itop = torch.zeros((m, maxno), dtype=torch.float64, device="cuda")
        res = (_empty(m, np.uint8, w), _empty(maxno, np.uint64, w), _empty((ncell, maxno), np.float64, w),
               _empty((ncell, maxno), np.uint64, w))
        _call(dev, "gpe_predict_implaus", _place(Xs, w), None, None, None, None, 0, m, z, 1e-2, maxno, 1, 1, Itop, cm, cell_pts,
              first_index, ncell, *res)
        outs[w] = (Itop,) + res
    assert all(_same(a, b) for a, b in zip(outs["host"], outs["device"]))
    keep = _host(outs["host"][1])
    assert 0 < keep.sum() < m
