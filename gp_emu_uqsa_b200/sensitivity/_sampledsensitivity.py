"""``SampledSensitivity``: uncertainty and sensitivity analysis of an emulator's posterior by sampling, for either
covariance family, any polynomial mean and independent normal or uniform inputs.

Every quantity the closed-form ``Sensitivity`` reports is an integral of the posterior mean m* and covariance c* over
the input distribution.  Here those integrals are estimated with the pick-freeze (Saltelli / Jansen) estimator on two
scrambled Sobol samples A, B of the inputs: the device evaluates the posterior at A, B and every AB_P (A with input P
from B) and returns the sums of the per-sample terms (``gpe_sens_sample``, include/gpe_b200.h, which lists them).  The
main effects are means of the posterior mean over a sample with one input held at each x_w value (``gpe_predict``).

Unlike the closed-form class, ``EVTw`` here is the true total-effect variance E*[V_T,P] = E*[E[Var(f | x_~P)]], not the
reference's ``uEV - E*[V_P]``.

``dgsm()`` adds the derivative-based global sensitivity measures nu_P = E[(df/dx_P)^2] (Sobol' & Kucherenko 2009) from the
posterior gradient (``gpe_predict_grad``) at sample A, and the Poincare bound C_P nu_P on the total-effect variance of the
continuous part of the process (C_P = v_P for normal inputs, (hi - lo)^2 / pi^2 for uniform ones).
"""
import numpy as np
from scipy.special import ndtri
from scipy.stats import qmc

MAX_GROUP = 16      # inputs per device pass (gpe_sens_sample)
DGSM_SLICE = 65536  # samples per gpe_predict_grad call of dgsm()


def sample_points(d, samples, seed, m=None, v=None, bounds=None):
    """The two input samples A, B [samples, d]: one scrambled Sobol sequence of 2d dimensions (first d columns A, last d
    B) drawn from its own generator, so the global ``np.random`` state does not move.  The points are the centres of the
    Sobol cells (u + 2^-31), which keeps ndtri away from 0.  Normal inputs: m + sqrt(v) ndtri(u); uniform inputs
    ``bounds`` [[lo, hi], ...]: lo + (hi - lo) u."""
    sob = qmc.Sobol(2 * d, scramble=True, seed=np.random.default_rng(seed))
    u = sob.random_base2(int(round(np.log2(samples)))) + 0.5 ** (sob.bits + 1)
    if bounds is None:
        x = np.asarray(m, dtype=float) + np.sqrt(np.asarray(v, dtype=float)) * ndtri(np.concatenate([u[:, :d], u[:, d:]]))
    else:
        lo, hi = np.asarray(bounds, dtype=float).T
        x = lo + (hi - lo) * np.concatenate([u[:, :d], u[:, d:]])
    return np.ascontiguousarray(x[:samples]), np.ascontiguousarray(x[samples:])


def _mean_err(s, s2, M):
    """Mean of M terms from their sum and sum of squares, and its plain Monte Carlo standard error."""
    mu = s / M
    var = np.maximum(s2 - M * mu * mu, 0.0) / max(M - 1, 1)
    return mu, np.sqrt(var / M)


class SampledSensitivity:
    """Sampled counterpart of ``Sensitivity`` (see the module docstring).  Inputs are normal (``m``, ``v``) or uniform
    (``bounds``), one entry per active input, in the scaled training-input units ``Sensitivity`` takes.

    Attributes after the analyses: ``uE``, ``uV``, ``uEV``, ``senseindex`` (E*[V_P]), ``EVTw`` (the true total-effect
    variance E*[V_T,P]), ``effect``, ``mean_effect``, ``dgsm_nu`` and ``dgsm_bound`` (``dgsm()``), and ``stderr``, a dict
    with the plain Monte Carlo standard error of each under the same key (the Sobol points make the actual error smaller)."""

    def __init__(self, emul, m=None, v=None, bounds=None, samples=65536, seed=0):
        self._train = emul.training
        self.beta = np.asarray(emul.par.beta, dtype=float)
        self.input_range = emul.all_data.input_range
        self.minmax = emul.all_data.minmax
        self.x = emul.training.inputs
        self.d = self.x.shape[1]
        self.m = None if m is None else np.asarray(m, dtype=float)
        self.v = None if v is None else np.asarray(v, dtype=float)
        self.bounds = None if bounds is None else np.asarray(bounds, dtype=float)
        self.samples, self.seed = int(samples), int(seed)
        self.shift = float(np.mean(emul.training.outputs))
        self.stderr = {}
        self._est = None
        self._device()
        self.done_uncertainty = self.done_sensitivity = self.done_main_effect = False
        self.done_interaction = self.done_totaleffectvar = self.done_dgsm = False

    def _device(self):
        """The handle with this emulator's fit state (re-factored only if another user of the training set changed it)."""
        dev, _, _, st = self._train.fit(beta=self.beta, r_div=self._train._A_args[0])
        if st != 0:
            raise np.linalg.LinAlgError("Matrix is not positive definite")
        return dev

    def _points(self, samples):
        return sample_points(self.d, samples, self.seed, self.m, self.v, self.bounds)

    def _estimate(self):
        """The one device pass behind uncertainty(), sensitivity() and totaleffectvariance()."""
        if self._est is not None:
            return
        A, B = self._points(self.samples)
        dev, M, d = self._device(), self.samples, self.d
        S, ST = np.zeros(d), np.zeros(d)
        eS, eST = np.zeros(d), np.zeros(d)
        for g0 in range(0, d, MAX_GROUP):
            w = list(range(g0, min(d, g0 + MAX_GROUP)))
            sums = dev.sens_sample(A, B, w, self.shift)
            mu, err = _mean_err(sums[0], sums[1], M)
            if g0 == 0:
                (self.uE, self.uV, self.uEV), e3 = mu[:3], err[:3]
            nw = len(w)
            S[w], eS[w] = mu[3:3 + nw], err[3:3 + nw]
            ST[w], eST[w] = mu[3 + nw:], err[3 + nw:]
        self.uE, self.uV, self.uEV = float(self.uE), float(self.uV), float(self.uEV)
        self.stderr.update(uE=float(e3[0]), uV=float(e3[1]), uEV=float(e3[2]), senseindex=eS, EVTw=eST)
        self._est = (S, ST)

    # ------------------------------------------------------------------ the analyses, printed as Sensitivity prints them
    def uncertainty(self):
        print("\n*** Uncertainty measures ***")
        self._estimate()
        self.done_uncertainty = True
        print("E*[ E[f(X)] ]  :", self.uE)
        print("var*[ E[f(X)] ]:", self.uV)
        print("E*[ var[f(X)] ]:", self.uEV)

    def sensitivity(self):
        print("\n*** Calculate sensitivity indices ***")
        self._estimate()
        self.done_sensitivity = True
        self.senseindex = self._est[0].copy()
        for P in range(self.d):
            if self.done_uncertainty:
                print("E(V" + str([P]) + ")/EV:", self.senseindex[P] / self.uEV)
            else:
                print("E(V" + str([P]) + "):", self.senseindex[P])
        if self.done_uncertainty:
            print("Sum of Sensitivities:", np.sum(self.senseindex / self.uEV))

    def totaleffectvariance(self):
        self._estimate()
        self.done_totaleffectvar = True
        print("\n*** Calculate total effect variance ***")
        self.EVf = self.uEV
        print("E*[ var[f(X)] ]:", self.EVf)
        self.EVTw = self._est[1].copy()
        for P in range(self.d):
            print("E(V[T" + str(P) + "]):", self.EVTw[P])

    def dgsm(self):
        """dgsm_nu[P] = E*[nu_P] = E_x[(dm*/dx_P)^2 + Var*(df/dx_P)], the posterior mean of the derivative-based measure, from
        the posterior gradient at sample A; dgsm_bound[P] = C_P dgsm_nu[P] bounds the total-effect variance of the continuous
        part of the process, E*[V_T,P] - sigma^2 (a* - c) in the terms of ``EVTw`` (which includes the nugget's share)."""
        print("\n*** Derivative-based global sensitivity measures ***")
        A, _ = self._points(self.samples)
        dev, M = self._device(), self.samples
        s, s2 = np.zeros(self.d), np.zeros(self.d)
        for i in range(0, M, DGSM_SLICE):
            dm, dv = dev.predict_grad(A[i:i + DGSM_SLICE])
            t = dm * dm + dv
            s += t.sum(0)
            s2 += (t * t).sum(0)
        nu, err = _mean_err(s, s2, M)
        if self.bounds is None:
            C = self.v.copy()
        else:
            C = (self.bounds[:, 1] - self.bounds[:, 0]) ** 2 / np.pi ** 2
        self.dgsm_nu, self.dgsm_bound = nu, C * nu
        self.stderr.update(dgsm_nu=err, dgsm_bound=C * err)
        self.done_dgsm = True
        for P in range(self.d):
            print("DGSM input " + str(P) + ": E*[nu] " + str(self.dgsm_nu[P]) + ", bound on E*[V_T] " + str(self.dgsm_bound[P]))

    def main_effect(self, plot=False, points=100, w=[], samples=4096):
        """effect[P, j] = mean_s [m*(B_s with x_P = xw_j) - m*(B_s)] and mean_effect[P, j] = mean_s m*(B_s with x_P = xw_j)
        on the x_w grid of ``Sensitivity.main_effect`` (``samples`` points B of the input distribution)."""
        print("\n*** Main effect measures ***")
        self.done_main_effect = True
        self.effect = np.zeros([self.d, points])
        self.mean_effect = np.zeros([self.d, points])
        e_eff, e_mean = np.zeros([self.d, points]), np.zeros([self.d, points])
        w = list(range(self.d)) if list(w) == [] else list(w)
        _, B = self._points(samples)
        dev = self._device()
        base, _ = dev.predict(B, None, want_var=False)
        for P in w:
            print("Main effect measures for input", P, "range", self.input_range[P])
            xw = np.linspace(self.input_range[P][0], self.input_range[P][1], points)
            pts = np.repeat(B[None], points, axis=0)
            pts[:, :, P] = xw[:, None]
            mw, _ = dev.predict(pts.reshape(-1, self.d), None, want_var=False)
            mw = mw.reshape(points, samples)
            self.mean_effect[P], e_mean[P] = _mean_err(mw.sum(1), (mw * mw).sum(1), samples)
            diff = mw - base[None, :]
            self.effect[P], e_eff[P] = _mean_err(diff.sum(1), (diff * diff).sum(1), samples)
        self.stderr.update(effect=e_eff, mean_effect=e_mean)
        if plot:
            print("Plotting main effects requires matplotlib (outside the rebuilt hot path); values are in .effect")

    def to_file(self, filename):
        """The results in the line format of ``Sensitivity.to_file``."""
        print("Sensitivity & Uncertainty results to file...")
        with open(filename, 'w') as f:
            if self.done_uncertainty:
                f.write("EE " + str(self.uE) + "\n")
                f.write("VE " + str(self.uV) + "\n")
                f.write("EV " + str(self.uEV) + "\n")
            if self.done_sensitivity:
                f.write("EVw " + ' '.join(map(str, self.senseindex)) + "\n")
            if self.done_totaleffectvar:
                f.write("EVTw " + ' '.join(map(str, self.EVTw)) + "\n")
            if self.done_main_effect:
                f.write("xw " + ' '.join(map(str, [i for i in np.linspace(0.0, 1.0, self.effect[0].size)])) + "\n")
                for i in range(0, self.d):
                    f.write("ME" + str(i) + " " + ' '.join(map(str, self.effect[i])) + "\n")
            if self.done_dgsm:
                f.write("DGSM " + ' '.join(map(str, self.dgsm_nu)) + "\n")
                f.write("DGSMbound " + ' '.join(map(str, self.dgsm_bound)) + "\n")
