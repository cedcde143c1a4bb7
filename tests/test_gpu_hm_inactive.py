"""History matching of points for which no emulator is active (imp_plot on an input pair that no emulator uses): every
emulator contributes I = 0, so every point is kept, every count is the number of points and every cell minimum is 0."""
import contextlib
import io
import os

import numpy as np
import pytest

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


def _rebuild_emulators(g, gold, tmp):
    emuls = []
    with _cwd(tmp), _quiet():
        for o in (0, 1):
            for fn in ("hm%d_config_r" % o, "hm%d_beliefs-0f" % o, "hm%d_input-o0-0f" % o, "hm%d_output-o0-0f" % o):
                with open(fn, "wb") as f:
                    f.write(bytes(gold["file_" + fn]))
            emuls.append(g.setup("hm%d_config_r" % o, datashuffle=False, scaleinputs=True))
    return emuls


@pytest.mark.parametrize("cell_pts,first_index", [(0, 0), (7, 5)])
def test_no_active_emulator_keeps_every_point(golden_dir, tmp_path, cell_pts, first_index):
    import gp_emu_uqsa_b200 as g
    from gp_emu_uqsa_b200.history_match import history_match as hm
    gold = np.load(os.path.join(golden_dir, "hmapi_n100_d3.npz"))
    emuls = _rebuild_emulators(g, gold, tmp_path)
    zs, ve, cm = list(gold["zs"]), list(gold["var_extra"]), float(gold["cm"])
    assert cm > 0
    m, maxno = 200, 2
    x = np.random.default_rng(5).random((m, 3))
    with _quiet():
        keep, count, cmin, ccnt = hm._implausibility_fused(emuls, zs, ve, x, {}, lambda E: False, cm, maxno,
                                                           cell_pts=cell_pts, first_index=first_index)
    assert keep.shape == (m,) and bool((keep == 1).all())
    assert np.array_equal(count, np.full(maxno, m, dtype=np.uint64))
    if not cell_pts:
        assert cmin is None and ccnt is None
        return
    cells = np.arange(first_index, first_index + m) // cell_pts
    sizes = np.bincount(cells - cells[0]).astype(np.uint64)
    assert sizes[0] < cell_pts and sizes[-1] < cell_pts      # the points start and end inside a cell
    assert np.array_equal(cmin, np.zeros((len(sizes), maxno)))
    assert np.array_equal(ccnt, np.repeat(sizes[:, None], maxno, axis=1))
