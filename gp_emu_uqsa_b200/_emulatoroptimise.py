"""Hyper-parameter optimisation with the reference's ``Optimize`` interface
(gp_emu_uqsa/_emulatoroptimise.py).  Bounds/constraint construction and SciPy's L-BFGS-B stay on
the host; every log-likelihood + gradient evaluation is served by ``gpe_llh_grad_batch`` on the
B200, all multistart guesses of a round in one call (``_lbfgsb_batch.minimize_batch``); with
``torch.distributed`` initialised the guesses are block-partitioned over the ranks."""
import os

import numpy as np

from . import _dist
from . import _lib
from ._lbfgsb_batch import minimize_batch

np.set_printoptions(precision=6)
np.set_printoptions(suppress=True)


def _fmt_bounds(b):
    return "[{:04.4f} , {:04.4f}]".format(b[0], b[1])


class Optimize:
    def __init__(self, data, basis, par, beliefs, config):
        self.data, self.basis, self.par, self.beliefs, self.config = data, basis, par, beliefs, config
        self.print_message = False
        print("\n*** Optimization options ***")
        X, y = self.data.inputs, self.data.outputs
        ndim = X.shape[1]
        span = lambda i: np.amax(X[:, i]) - np.amin(X[:, i])

        # delta: [0.001, data range] unless the user gave bounds (reference :41-64)
        d_b = []
        if config.delta_bounds == []:
            print("Data-based bounds for delta:")
            for i in range(ndim):
                d_b.append([0.001, span(i)])
                print("    delta", i, _fmt_bounds(d_b[i]))
        else:
            print("User provided bounds for delta:")
            if len(config.delta_bounds) != ndim:
                print("ERROR: Wrong number of delta_bounds specified, exiting.")
                raise SystemExit(1)
            for i in range(ndim):
                user = config.delta_bounds[i] != []
                d_b.append(config.delta_bounds[i] if user else [0.001, span(i)])
                print("    delta", i, _fmt_bounds(d_b[i]), "(user)" if user else "(data)")
        # nugget: small fixed range (reference :69-79)
        if config.nugget_bounds == []:
            print("Data-based bounds for nugget:")
            n_b = [[0.0001, 0.01]]
        else:
            print("User provided bounds for nugget:")
            n_b = config.nugget_bounds
        print("    nugget ", _fmt_bounds(n_b[0]))
        # sigma: [0.001, sqrt(output range)] (reference :81-91)
        if config.sigma_bounds == []:
            print("Data-based bounds for sigma:")
            s_b = [[0.001, np.sqrt(np.amax(y) - np.amin(y))]]
        else:
            print("User provided bounds for sigma:")
            s_b = config.sigma_bounds
        print("    sigma  ", _fmt_bounds(s_b[0]))

        # parameter order [delta.., nugget?, sigma?] (reference :94-103)
        parts = list(d_b)
        if self.beliefs.fix_nugget == "F":
            parts += list(n_b)
        if self.beliefs.mucm != "T":
            parts += list(s_b)
        config.bounds = tuple(parts)
        if config.constraints == "bounds":
            self.bounds_constraint(config.bounds)
        else:
            self.standard_constraint(config.bounds)

    # ---------------------------------------------------------------- constraints
    def _n_params(self):
        p = self.data.K.d.size
        if self.beliefs.fix_nugget == "F":
            p += 1
        if self.beliefs.mucm != "T":
            p += 1
        return p

    def _mode(self):
        m = 0
        if self.beliefs.mucm == "T":
            m |= _lib.MODE_MUCM
        if self.beliefs.alt_nugget == "T":
            m |= _lib.MODE_ALT_NUGGET
        if self.beliefs.fix_nugget == "F":
            m |= _lib.MODE_NUGGET_FREE
        if getattr(self.beliefs, "objective", "llh") == "loo":
            m |= _lib.MODE_LOO
        return m

    def standard_constraint(self, bounds):
        print("Setting up standard constraint")
        K = self.data.K
        self.cons = [[K.transform(0.001), None] for _ in range(K.d.size)]
        self.cons += [[None, None]] * (self._n_params() - K.d.size)

    def bounds_constraint(self, bounds):
        print("Setting up bounds constraint")
        K = self.data.K
        self.cons = [[K.transform(lo), K.transform(hi)] for lo, hi in bounds[:self._n_params()]]

    # ---------------------------------------------------------------- optimisation
    def llh_optimize(self, print_message=False):
        self.print_message = print_message
        print("Optimising hyperparameters...")
        bounds = self.data.K.transform(self.config.bounds)
        self.optimal(self.config.tries, bounds)
        print("best hyperparameters: ")
        self.data.K.print_kernel()
        print("sigma:", np.round(self.par.sigma, decimals=6))
        if self.beliefs.fix_nugget == "F":
            if self.beliefs.alt_nugget == "F":
                print("'noise sigma' estimate from nugget:",
                      np.sqrt(self.par.sigma ** 2 * self.par.nugget / (1.0 - self.par.nugget)))
            else:
                print("'noise sigma' estimate from alt nugget:", self.par.sigma * self.par.nugget)
        self.optimalbeta()
        print("best beta: ", self.par.beta)

    def _eval_batch(self, thetas):
        """(f, g, ok, sigma_hat) for a block of transformed parameter vectors -- one device call."""
        self.data._r_made = self.data.r      # every reference evaluation starts with make_A(): current r
        dev = self.data.device()
        llh, grad, sig, st = dev.llh_grad_batch(thetas, self._mode(), fixed_nugget=float(self.data.K.n))
        return llh, grad, st == 0, sig

    def optimal(self, numguesses, bounds):
        params = self._n_params()
        K = self.data.K
        # initial guesses: one row of uniforms per parameter from the global RNG (reference :206-211)
        guessgrid = np.zeros([params, numguesses])
        print("Calculating initial guesses from bounds")
        _dist.sync_numpy_rng()                     # multi-rank: every rank draws rank 0's guesses
        for R in range(params):
            BL, BU = bounds[R][0], bounds[R][1]
            guessgrid[R, :] = BL + (BU - BL) * np.random.random_sample(numguesses)
        if self.beliefs.fix_nugget == "F":
            print("Training nugget on data")
        mucm = self.beliefs.mucm == "T"
        if mucm:
            print("Using MUCM method for sigma")
        constrained = self.config.constraints != "none"
        print("Using L-BFGS-G method (%s constraints)..." % ("with" if constrained else "no"))

        # the multistart batch: every rank draws the same guesses, owns a contiguous block of them
        rank, world = _dist.rank_world()
        lo, hi = _dist.block(numguesses, rank, world)
        fixed_n = float(K.n)

        def eval_batch(X):
            f, g, ok, _ = self._eval_batch(X)
            return f, g, ok

        x0s = guessgrid.T[lo:hi]
        res_local, rounds, evals = minimize_batch(eval_batch, x0s, self.cons if constrained else None,
                                                    driver=os.environ.get("GPE_LBFGSB_DRIVER") or None) \
            if hi > lo else ([], 0, 0)
        self.last_rounds, self.last_evals = rounds, evals
        # pack (ok, fun, x) per guess and exchange so that every rank sees all of them in guess order
        pack = np.full((numguesses, params + 2), np.nan)
        for k, res in enumerate(res_local):
            if res is not None:
                pack[lo + k, 0], pack[lo + k, 1], pack[lo + k, 2:] = 1.0, res.fun, res.x
            else:
                pack[lo + k, 0] = 0.0
        pack = _dist.gather_blocks(pack, numguesses)
        self.last_table = pack                     # rows [ok, fun, theta...] per guess, in guess order
        K.n = fixed_n if self.beliefs.fix_nugget != "F" else K.n

        # sigma for the printed lines (mucm): one more batched evaluation at the optima (with the LOO objective its sigma_hat
        # is the profiled LOO sigma, which also becomes the emulator's sigma below)
        okrows = np.nonzero(pack[:, 0] == 1.0)[0]
        sig_print = {}
        if mucm and okrows.size:
            _, _, ok2, sig = self._eval_batch(pack[okrows, 2:])
            sig_print = {int(c): float(s) for c, s, o in zip(okrows, sig, ok2) if o}

        loo = self._mode() & _lib.MODE_LOO
        label = "loo" if loo else "llh"
        first_try, best_min, best_x, best_C = True, 10000000.0, None, -1
        for C in range(numguesses):
            if pack[C, 0] != 1.0:
                print("Trying next guess...")
                continue
            fun, x = pack[C, 1], pack[C, 2:]
            if self.print_message:
                print("guess", C, "fun", fun, "x", x, "\n")
            sig_str = ""
            if mucm and C in sig_print:
                self.par.sigma = sig_print[C]
                sig_str = "  sig: " + str(np.around(self.par.sigma, decimals=4))
            print("  hp: ", np.around(K.untransform(x), decimals=4), " %s: " % label, -1.0 * np.around(fun, decimals=4), sig_str)
            if fun < best_min or first_try:
                best_min, best_x, first_try, best_C = fun, K.untransform(x), False, C
        print("********")
        if first_try:
            print("ERROR: No optimization was made due to non-PSD errors. Increase 'tries'. Exiting.")
            raise SystemExit(1)
        if mucm:
            K.set_params(best_x)
            self.par.delta, self.par.nugget = K.d, K.n
            if loo:
                self.par.sigma = sig_print.get(best_C, self.par.sigma)
            else:
                self.sigma_analytic_mucm(best_x)
        else:
            K.set_params(best_x[:-1])
            self.par.delta, self.par.nugget = K.d, K.n
            self.par.sigma = best_x[-1]
        self.best_llh, self.best_guess = best_min, best_C
        self.data.make_A(self.par.sigma ** 2)      # including r still (reference :289)
        self.data.make_H()

    # ---------------------------------------------------------------- single evaluations
    def _single(self, x):
        theta = np.atleast_2d(np.asarray(x, dtype=float))
        llh, grad, ok, sig = self._eval_batch(theta)
        return llh[0], grad[0], bool(ok[0]), sig[0]

    def loglikelihood_mucm(self, x):
        """(LLH, grad) as reference :305-378, or None when the covariance is not PD."""
        hp = self.data.K.untransform(np.asarray(x, dtype=float))
        self.data.K.set_params(hp)
        self.data.make_A()
        llh, grad, ok, sig = self._single(x)
        if not ok:
            print("  Matrix not PSD for", hp, ", try adjusting nugget.")
            return None
        self.par.sigma = sig
        return llh, grad

    def loglikelihood_gp4ml(self, x):
        """(LLH, grad) as reference :412-493, or None when the covariance is not PD."""
        hp = self.data.K.untransform(np.asarray(x, dtype=float))
        self.data.K.set_params(hp[:-1])
        self.par.sigma = hp[-1]
        self.data.make_A(hp[-1] ** 2)
        llh, grad, ok, _ = self._single(x)
        if not ok:
            print("  Matrix not PSD for", hp, ", try adjusting nugget.")
            return None
        return llh, grad

    def sigma_analytic_mucm(self, x):
        """Analytic MUCM sigma for un-transformed hyper-parameters x (reference :382-408)."""
        self.data.K.set_params(np.asarray(x, dtype=float))
        self.data.make_A()
        _, _, sig, st = self.data.fit(beta=None, r_div=1.0)
        if st != 0:
            print("  In sigma_analytic_mucm(): Matrix not PSD for", x, ", try adjusting nugget.")
            raise SystemExit(1)
        self.par.sigma = sig

    def optimalbeta(self):
        """beta = (H^T A^-1 H)^-1 H^T A^-1 y on the current data.A (reference :497-504)."""
        _, bopt, _, st = self.data.fit(beta=None, r_div=self.data._A_args[0])
        if st != 0:
            raise np.linalg.LinAlgError("Matrix is not positive definite")
        self.par.beta = bopt
