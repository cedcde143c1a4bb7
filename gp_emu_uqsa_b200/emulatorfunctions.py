"""Public API with the reference's signatures (gp_emu_uqsa/emulatorfunctions.py): setup, train,
plot, posterior, posterior_sample.  Orchestration only -- the arithmetic behind every call
(covariance build, factorisation, likelihood + gradient, posterior mean/variance) runs on the B200
through the C-ABI (``_lib.Device``)."""
import numpy as _np

from . import _emulatorclasses as _emuc
from . import _emulatorkernels as _emuk
from . import _emulatoroptimise as _emuo
from . import _emulatorplotting as _emup
from . import _lib

__all__ = ["setup", "train", "plot", "posterior", "posterior_sample", "posterior_diag"]


def setup(config_file, datashuffle=True, scaleinputs=True):
    """Initialise Config, Beliefs, Hyperparams, Basis, TV_config, All_Data, Data, Posterior, Optimize and
    the kernel; return the Emulator (reference :13-57)."""
    config = _emuc.Config(config_file)
    beliefs = _emuc.Beliefs(config.beliefs)
    par = _emuc.Hyperparams(beliefs)
    basis = _emuc.Basis(beliefs)
    tv_conf = _emuc.TV_config(*(config.tv_config))
    all_data = _emuc.All_Data(config.inputs, config.outputs, tv_conf, beliefs, par, datashuffle, scaleinputs)
    if beliefs.kernel == "matern52":
        print("\n*** Using Matern 5/2 kernel ***")
    if beliefs.alt_nugget != 'T':
        cls = _emuk.kernel_matern52 if beliefs.kernel == "matern52" else _emuk.kernel
    else:
        print("\n*** Using alternative nugget ***")
        cls = _emuk.kernel_matern52_alt_nug if beliefs.kernel == "matern52" else _emuk.kernel_alt_nug
    K = cls(all_data.x_full[0].size, par)
    (x_T, y_T) = all_data.choose_T()
    (x_V, y_V) = all_data.choose_V()
    training = _emuc.Data(x_T, y_T, basis, par, beliefs, K)
    validation = _emuc.Data(x_V, y_V, basis, par, beliefs, K)
    post = _emuc.Posterior(validation, training, par, beliefs, K, lazy=True)
    opt_T = _emuo.Optimize(training, basis, par, beliefs, config)
    return _emuc.Emulator(config, beliefs, par, basis, tv_conf, all_data, training, validation, post, opt_T, K)


def train(E, auto=True, message=False, no_retrain=False):
    """Train the hyper-parameters on the training set, validate, optionally fold validation sets in
    and retrain; write the updated beliefs / data files (reference :61-124)."""
    E.tv_conf.auto_train(auto, no_retrain)
    while E.tv_conf.doing_training():
        print("\n*** Training round", E.tv_conf.no_of_trains, "***")
        print("Training points:", E.training.inputs[:, 0].size)
        E.opt_T.llh_optimize(message)
        E.training.remake()
        E.validation.remake()
        E.post.remake()
        E.post.mahalanobis_distance()
        E.post.indiv_standard_error(ise=2.0)
        E.beliefs.final_beliefs(E, False)
        E.post.final_design_points(E, False)
        if E.tv_conf.check_still_training():
            print("Preparing for next round of training...")
            E.post.incVinT()
            E.tv_conf.next_Vset()
            E.all_data.choose_new_V(E.validation)
            E.training.remake()
            E.validation.remake()
            E.post.remake()
    if E.tv_conf.do_final_build():
        print("\n*** Doing final build ***")
        if E.tv_conf.noV != 0 and E.training.inputs[:, 0].size < E.all_data.numpoints:
            E.post.incVinT()
        E.training.remake()
        E.opt_T.llh_optimize(message)
        E.training.remake()
        E.beliefs.final_beliefs(E, True)
        E.post.final_design_points(E, True)
    return None


def plot(E, plot_dims, fixed_dims=[], fixed_vals=[], mean_or_var="mean", customLabels=[], points=False, predict=True):
    """Posterior over a 30x30 map (two plot_dims) or a 900-point line (one), other inputs fixed
    (reference :128-223).  Returns the Posterior that was evaluated (the reference returns None) so
    the grid values can be used without matplotlib."""
    dim = E.training.inputs[0].size
    minmax, x, y = [], [], []
    print("\n*** Generating plot ***")
    one_d = len(plot_dims) == 1 and dim > 1
    if points and mean_or_var == "mean":
        x = E.training.inputs[:, plot_dims[0]]
        y = E.training.outputs
    col = E.training.inputs[:, plot_dims[0]]
    minmax.append([_np.amin(col), _np.amax(col)])
    if not one_d and dim > 1:
        col = E.training.inputs[:, plot_dims[1]]
        minmax.append([_np.amin(col), _np.amax(col)])
    xlabel = "input " + str(plot_dims[0])
    if one_d:
        ylabel = "output " + str(E.beliefs.output)
    else:
        ylabel = "output " if dim == 1 else "input " + str(plot_dims[1])
    if len(customLabels) > 0:
        xlabel = customLabels[0]
    if len(customLabels) > 1:
        ylabel = customLabels[1]
    pn = 30
    full_xrange = _emup.make_inputs(dim, pn, pn, plot_dims, fixed_dims, fixed_vals, one_d, minmax)
    newinputs = _emuc.Data(full_xrange, None, E.basis, E.par, E.beliefs, E.K)
    print("Estimation (rather than prediction)" if predict is False else "Prediction (rather than estimation)")
    post = _emuc.Posterior(newinputs, E.training, E.par, E.beliefs, E.K, predict, diag_only=True)
    _emup.plotting(dim, post, pn, pn, one_d, mean_or_var, minmax, x, y, labels=[xlabel, ylabel])
    return post


def _as_points(E, x):
    x = _np.asarray(x, dtype=float)
    if x[0].size == 1:
        x = _np.array([x, ]).T if x.ndim == 1 else x
    if x[0, :].size != E.training.inputs[0, :].size:
        print("ERROR: test points have different number of columns"
              "to data in emulator. Exiting.")
        raise SystemExit(1)
    return x


def posterior(E, x, predict=True):
    """(posterior mean [m], posterior covariance [m,m]) at the points x (reference :226-252)."""
    x = _as_points(E, x)
    xs = _emuc.Data(x, None, E.basis, E.par, E.beliefs, E.K)
    p = _emuc.Posterior(xs, E.training, E.par, E.beliefs, E.K, predict=predict)
    return (p.mean, p.var)


def posterior_diag(E, x):
    """(posterior mean [m], posterior variance [m]) for any number of points: what the reference's
    consumers take as ``np.diag(post.var)`` (history_match.py:117-118, _emulatorplotting.py:51)
    without the m x m matrix.  ``x`` may be a NumPy array or a torch CUDA tensor."""
    if hasattr(x, "data_ptr"):
        dev, _, _, st = E.training.fit(beta=E.par.beta, r_div=E.training._A_args[0])
        if st != 0:
            raise _lib.GpeError("training covariance matrix is not positive definite")
        if E.basis.poly is None:
            raise _lib.GpeError("device-resident points need a polynomial mean basis")
        import torch
        m = int(x.shape[0])
        mean = torch.empty(m, dtype=torch.float64, device=x.device)
        var = torch.empty(m, dtype=torch.float64, device=x.device)
        dev.predict(x, None, out=(mean, var))
        return mean, var
    x = _as_points(E, x)
    xs = _emuc.Data(x, None, E.basis, E.par, E.beliefs, E.K)
    p = _emuc.Posterior(xs, E.training, E.par, E.beliefs, E.K, diag_only=True)
    return p.mean, p.var_diag


def posterior_sample(E, x, predict=True):
    """One sample from the posterior at x: mean + chol(V) u with u from the global NumPy RNG
    (reference :255-286); the Cholesky factor of V comes from the device."""
    x = _as_points(E, x)
    xs = _emuc.Data(x, None, E.basis, E.par, E.beliefs, E.K)
    p = _emuc.Posterior(xs, E.training, E.par, E.beliefs, E.K, predict=predict)
    Lf = _lib.scratch_device().cholesky(p.var)
    u = _np.random.randn(x[:, 0].size)
    return p.mean + Lf.dot(u)
