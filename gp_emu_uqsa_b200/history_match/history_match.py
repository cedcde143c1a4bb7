"""History matching with the reference's call surface (gp_emu_uqsa/history_match/history_match.py):
imp_plot, imp_plot_recon, nonimp_data, new_wave_design.

The reference evaluates a Posterior per grid cell per emulator and then loops over points in
Python.  Here all points of an input pair (grid^2 cells x n_lhc design points) go through ONE
device prediction per emulator whose epilogue folds that emulator's implausibility into a running
top-``maxno`` list (``gpe_predict_implaus``: means and variances never leave the device kernels);
the last emulator's pass also produces the keep mask and the per-cell min / count reductions.  With torch.distributed initialised the flat point index (all cells'
points in cell order, or the rows of the flat routines) is cut into equal tile-aligned ranges, one per
rank -- a cell may straddle two ranks -- and the cell statistics are combined with all-reduce(min / sum)."""
import numpy as _np

from .. import _dist
from .. import _lib
from .. import design_inputs as _gd
from ._hmutilfunctions import check_act, emulsetup, load_datafiles, make_sets, ref_act, ref_plt

__all__ = ["imp_plot", "imp_plot_recon", "nonimp_data", "new_wave_design"]


def _implausibility_fused(emuls, zs, var_extra, x, act_ref, active_fn, cm, maxno, cell_pts=0, first_index=0):
    """(keep, count, cell_min, cell_count) for the points x without the per-emulator mean / variance arrays: every active
    emulator's prediction folds its implausibility into the running top-``maxno`` list on the device
    (``gpe_predict_implaus``); the last one also produces the mask and the reductions.  Emulators for which
    ``active_fn`` is False contribute I = 0 (reference :93, :99-100): they are entered as zeros in the initial list."""
    import torch
    active = [o for o, E in enumerate(emuls) if active_fn(E)]
    m = x.shape[0]
    tdev = torch.device("cuda", _lib.default_device_index())
    keep = torch.empty(m, dtype=torch.uint8, device=tdev)
    if not active:          # no prediction: every emulator enters with mean = z, var = 1, i.e. I = 0
        mean = _np.repeat(_np.asarray(zs, dtype=_np.float64)[:, None], m, axis=1)
        torch.cuda.current_stream(tdev).synchronize()      # the handle works on its own stream
        _, _, count, cmin, ccnt = emuls[0].training.device().implausibility(mean, _np.ones_like(mean), zs, var_extra, cm, maxno=maxno,
                                                                              cell_pts=cell_pts, first_index=first_index,
                                                                              want_imax=False, out=(None, keep))
        return keep, count, cmin, ccnt
    Itop = torch.full((m, maxno), -1.0, dtype=torch.float64, device=tdev)
    n_inactive = len(emuls) - len(active)
    if n_inactive:
        Itop[:, max(0, maxno - n_inactive):] = 0.0
    torch.cuda.current_stream(tdev).synchronize()          # the handles work on their own streams
    res = None
    for pos, o in enumerate(active):
        E = emuls[o]
        cols = [act_ref[str(l)] for l in E.beliefs.active_index]
        dev, _, _, st = E.training.fit(beta=E.par.beta, r_div=E.training._A_args[0])
        if st != 0:
            raise _lib.GpeError("training covariance matrix of emulator %d is not positive definite" % o)
        xe = _np.ascontiguousarray(x[:, cols])
        last = pos == len(active) - 1
        Hs = None if E.basis.poly is not None else E.basis.design_matrix(xe)
        res = dev.predict_implaus(float(zs[o]), float(var_extra[o]), Itop, first=False, last=last, points=xe, Hs=Hs, maxno=maxno,
                                  cm=cm, cell_pts=cell_pts, first_index=first_index, keep=keep if last else None)
    count, cmin, ccnt = res
    return keep, count, cmin, ccnt


def imp_plot(emuls, zs, cm, var_extra, maxno=1, olhcmult=100, grid=10, act=[], fileStr="", plot=True):
    """Implausibility / optical-depth matrices for every pair of active inputs (reference :7-151);
    written to '<fileStr_><m>_IMP_<i>_<j>' and '..._ODP_...' exactly like the reference.  Drawing the
    matrices needs matplotlib and is skipped when it is not installed.  Returns None."""
    sets, minmax, orig_minmax = emulsetup(emuls)
    check_act(act, sets)
    act_ref = ref_act(minmax)
    num_inputs = len(minmax)
    dim = num_inputs - 2
    maxno = int(maxno)
    less_sets = sets if act == [] else [s for s in sets if s[0] in act and s[1] in act]
    print("HM for input pairs:", less_sets)
    rank, world = _dist.rank_world()
    for s in less_sets:
        print("\nset:", s)
        grids = []
        for k in (0, 1):
            lo, hi = minmax[str(s[k])][0], minmax[str(s[k])][1]
            grids.append(_np.linspace(lo, hi, grid, endpoint=False) + 0.5 * (hi - lo) / float(grid))
        X1, X2 = grids
        print("Values of the grid 1:", X1)
        print("Values of the grid 2:", X2)
        n = dim * int(olhcmult)
        N = int(n / 2)
        olhc_range = [it[1] for it in sorted(minmax.items(), key=lambda x: int(x[0])) if int(it[0]) != s[0] and int(it[0]) != s[1]]
        print("olhc_range:", olhc_range)
        filename = "imp_input_" + str(s[0]) + '_' + str(s[1])
        # the reference writes the design and reads it back (:77-84); here rank 0 writes it, everyone gets it in memory
        x_other = _gd.optLatinHyperCube(dim, n, N, olhc_range, filename, _criterion=_gd.device_criterion, _return=True)
        other_dim = [act_ref[str(key)] for key in act_ref if int(key) not in s]
        print("\nCalculating Implausibilities...")
        # flat point index = cell * n + design point, cell = i*grid + j; this rank owns the points [p0, p1)
        ncell = grid * grid
        p0, p1 = _dist.block_aligned(ncell * n, rank, world)
        IMP = _np.full((ncell, maxno), _np.inf)
        ODPc = _np.zeros((ncell, maxno), dtype=_np.uint64)
        if p1 > p0:
            pts = _np.arange(p0, p1)
            cells, lhc = pts // n, pts % n
            x = _np.empty((p1 - p0, num_inputs))
            x[:, act_ref[str(s[0])]] = X1[cells // grid]
            x[:, act_ref[str(s[1])]] = X2[cells % grid]
            x[:, other_dim] = x_other[lhc, :]
            active = lambda E: s[0] in E.beliefs.active_index and s[1] in E.beliefs.active_index
            _, _, cmin, ccnt = _implausibility_fused(emuls, zs, var_extra, x, act_ref, active, cm, maxno, cell_pts=n, first_index=p0)
            c0 = p0 // n
            IMP[c0:c0 + cmin.shape[0]], ODPc[c0:c0 + ccnt.shape[0]] = cmin, ccnt
        IMP = _dist.all_reduce(IMP, "min")
        ODPc = _dist.all_reduce(ODPc, "sum")
        nfileStr = fileStr + "_" if fileStr != "" else fileStr
        if rank == 0:
            for m in range(maxno):
                _np.savetxt(nfileStr + str(m + 1) + "_" + "IMP_" + str(s[0]) + '_' + str(s[1]), IMP[:, m].reshape(grid, grid))
                _np.savetxt(nfileStr + str(m + 1) + "_" + "ODP_" + str(s[0]) + '_' + str(s[1]),
                            (ODPc[:, m].astype(float) / float(n)).reshape(grid, grid))
        _dist.barrier()
    if plot is True:
        print("imp_plot: drawing requires matplotlib (outside the rebuilt hot path); the IMP/ODP files were written")
    return


def imp_plot_recon(cm, maxno=1, act=[], fileStr=""):
    """Reload the IMP/ODP matrices written by imp_plot (reference :154-192).  Returns
    {(i, j): (IMP, ODP)} (the reference only draws them)."""
    if act == []:
        print("WARNING: Please specificy 'act' for active inputs. Return None.")
        return None
    out = {}
    sets = make_sets(act)
    print("HM for input pairs:", sets)
    nfileStr = fileStr + "_" if fileStr != "" else fileStr
    for s in sets:
        print("\nset:", s)
        IMP = _np.loadtxt(nfileStr + str(maxno) + "_" + "IMP_" + str(s[0]) + '_' + str(s[1]))
        ODP = _np.loadtxt(nfileStr + str(maxno) + "_" + "ODP_" + str(s[0]) + '_' + str(s[1]))
        out[(s[0], s[1])] = (IMP, ODP)
    return out


def _flat_keep(emuls, zs, cm, var_extra, x, act_ref, maxno):
    """Non-implausible row mask of x (reference :222-250 / :302-329): rows whose maxno-th largest
    implausibility over the emulators is below cm.  Rows are block-partitioned over the ranks."""
    n = x.shape[0]
    rank, world = _dist.rank_world()
    lo, hi = _dist.block_aligned(n, rank, world)
    keep = _np.zeros(n)
    if hi > lo:
        kd, _, _, _ = _implausibility_fused(emuls, zs, var_extra, x[lo:hi], act_ref, lambda E: True, cm, maxno)
        keep[lo:hi] = kd.cpu().numpy()
    keep = _dist.gather_blocks(keep, n, bounds=_dist.block_aligned)
    return keep > 0.5


def nonimp_data(emuls, zs, cm, var_extra, datafiles, maxno=1, act=[], fileStr=""):
    """Keep the non-implausible rows of an inputs file (and the matching outputs rows); write them to
    '<fileStr_>nonimp_<inputs>' / '<fileStr_>noninp_<outputs>' (sic, reference :257).  Returns the count."""
    sets, minmax, orig_minmax = emulsetup(emuls)
    act_ref = ref_act(minmax)
    check_act(act, sets)
    maxno = int(maxno)
    sim_x, sim_y = load_datafiles(datafiles, orig_minmax)
    print("\nCalculating Implausibilities...")
    keep = _flat_keep(emuls, zs, cm, var_extra, sim_x, act_ref, maxno)
    nimp_inputs, nimp_outputs = sim_x[keep], sim_y[keep]
    nfileStr = fileStr + "_" if fileStr != "" else fileStr
    if _dist.is_writer():
        _np.savetxt(nfileStr + "nonimp_" + datafiles[0], nimp_inputs)
        _np.savetxt(nfileStr + "noninp_" + datafiles[1], nimp_outputs)
    _dist.barrier()
    print(len(nimp_inputs), "data points were non-implausible")
    return len(nimp_inputs)


def new_wave_design(emuls, zs, cm, var_extra, datafiles, maxno=1, olhcmult=100, act=[], fileStr=""):
    """Design new non-implausible inputs: optimised LHC (against the given non-implausible data) filtered
    by implausibility; written to '<fileStr_><inputs>' (reference :264-338).  Returns the count."""
    sets, minmax, orig_minmax = emulsetup(emuls)
    act_ref = ref_act(minmax)
    check_act(act, sets)
    dim = len(minmax)
    maxno = int(maxno)
    sim_x, sim_y = load_datafiles(datafiles, orig_minmax)
    n = dim * int(olhcmult)
    N = int(n / 2)
    olhc_range = [it[1] for it in sorted(minmax.items(), key=lambda x: int(x[0]))]
    print("olhc_range:", olhc_range)
    filename = "olhc_des"
    x = _gd.optLatinHyperCube(dim, n, N, olhc_range, filename, fextra=sim_x, _criterion=_gd.device_criterion, _return=True)
    print("\nCalculating Implausibilities...")
    keep = _flat_keep(emuls, zs, cm, var_extra, x, act_ref, maxno)
    nimp_inputs = x[keep]
    nfileStr = fileStr + "_" if fileStr != "" else fileStr
    if _dist.is_writer():
        _np.savetxt(nfileStr + datafiles[0], nimp_inputs)
    _dist.barrier()
    print("Generated", len(nimp_inputs), "new data points")
    return len(nimp_inputs)
