"""Host-side object model with the reference's names (Emulator, Config, Beliefs, Hyperparams, Basis,
TV_config, All_Data, Data, Posterior; reference: gp_emu_uqsa/_emulatorclasses.py).

Only the plumbing lives here (text-file parsing, train/validation bookkeeping, file writers).  All
arithmetic on the hot path -- covariance matrices, the factorisation behind the posterior, mean and
variance -- is done on the B200 through ``_lib.Device``; there is no NumPy fallback for it.
"""
import math

import numpy as np

from . import _dist
from . import _lib

_PRED_FULL_LIMIT = 8192     # largest m for which Posterior materialises the full m x m covariance


def _die(msg):
    print(msg)
    raise SystemExit(1)


_CK_W = {}


def _checksum(a):
    """sum_k bits(a_k) * w_k mod 2^64 with fixed odd multipliers w_k (wrap-around uint64 arithmetic)."""
    bits = np.ascontiguousarray(a, dtype=np.float64).reshape(-1).view(np.uint64)
    w = _CK_W.get(bits.size)
    if w is None:
        w = (np.arange(bits.size, dtype=np.uint64) * np.uint64(2) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        if len(_CK_W) < 64:
            _CK_W[bits.size] = w
    return int((bits * w).sum(dtype=np.uint64))


class Emulator:
    """Bundle of the objects that make up one emulator (reference :14-29)."""

    def __init__(self, config, beliefs, par, basis, tv_conf, all_data, training, validation, post, opt_T, K):
        self.config, self.beliefs, self.par, self.basis = config, beliefs, par, basis
        self.tv_conf, self.all_data = tv_conf, all_data
        self.training, self.validation, self.post = training, validation, post
        self.opt_T, self.K = opt_T, K


def _read_keyed_file(path, what):
    """'key value...' lines -> dict (first space splits key from value), as reference :38-46, :109-122."""
    print("*** Reading %s file: %s ***" % (what, path) if what == "config" else "\n*** Reading %s file: %s ***" % (what, path))
    table = {}
    try:
        with open(path, "r") as fh:
            for line in fh:
                key, val = line.split(" ", 1)
                table[key] = val
    except OSError:
        _die("ERROR: Problem reading file.")
    except ValueError:
        _die("ERROR: Some specifications seem to be missing values.")
    return table


class Config:
    """Configuration file (reference :32-98): beliefs/inputs/outputs file names, tv_config,
    bounds, tries, constraints, optional (unused) fix."""

    REQUIRED = ("beliefs", "inputs", "outputs", "tv_config", "delta_bounds", "nugget_bounds", "sigma_bounds",
                "tries", "constraints")

    def __init__(self, config_file):
        self.config_file = config_file
        self.config = _read_keyed_file(config_file, "config")
        for key in self.REQUIRED:
            if key not in self.config:
                _die('WARNING: " %s " specification is missing' % key)
        c = {k: str(v).strip() for k, v in self.config.items()}
        self.beliefs, self.inputs, self.outputs = c["beliefs"], c["inputs"], c["outputs"]
        self.tv_config = [int(t) for t in c["tv_config"].split(" ")]
        if len(self.tv_config) != 3:
            _die("WARNING: tv_config requires 3 entries.")
        print("T-V config:", self.tv_config)
        self.delta_bounds = eval(c["delta_bounds"])
        self.nugget_bounds = eval(c["nugget_bounds"])
        self.sigma_bounds = eval(c["sigma_bounds"])
        self.bounds = tuple(self.delta_bounds + self.nugget_bounds + self.sigma_bounds)
        self.tries = int(c["tries"])
        print("number of tries for optimum:", self.tries)
        if c["constraints"] in ("none", "bounds"):
            self.constraints = c["constraints"]
        else:
            self.constraints = "standard"
            if c["constraints"] != "standard":
                print("unrecognised constraints option, defaulting")
        print("constraints:", self.constraints)
        if "fix" in c:
            self.fix = eval(c["fix"])
            print("Fixing hyperparameters:", self.fix)
        else:
            self.fix = []


class Beliefs:
    """Beliefs file (reference :102-213) and the writer of updated beliefs files (:217-250)."""

    REQUIRED = ("active", "output", "basis_str", "basis_inf", "beta", "delta", "sigma", "nugget", "fix_nugget", "mucm")
    KERNELS = ("gaussian", "matern52")
    OBJECTIVES = ("llh", "loo")

    def __init__(self, beliefs_file):
        self.beliefs_file = beliefs_file
        self.beliefs = _read_keyed_file(beliefs_file, "beliefs")
        for key in self.REQUIRED:
            if key not in self.beliefs:
                _die('WARNING: " %s " specification is missing' % key)
        b = {k: str(v).strip() for k, v in self.beliefs.items()}
        words = lambda k: b[k].split(" ")

        if "active_index" in b:
            w = words("active_index")
            if w[0] == "all":
                self.active_index = []
            else:
                try:
                    self.active_index = [int(t) for t in w]
                except ValueError:
                    print("WARNING: active_index should be 'all' or whitespaced integers,"
                          " setting value to 'unknown' and continuing")
                    self.active_index = "unknown"
        w = words("active")
        self.active = [] if w[0] == "all" else [int(t) for t in w]
        print("active:", self.active)
        if "output_index" in b:
            try:
                self.output_index = int(words("output_index")[0])
            except ValueError:
                print("WARNING: output_index should be an integer, setting value to 'unknown' and continuing")
                self.output_index = "unknown"
        self.output = int(words("output")[0])
        print("output:", self.output)

        self.basis_str = words("basis_str")
        self.basis_inf = [int(t) for t in words("basis_inf")[1:]]
        self.beta = [float(t) for t in words("beta")]
        if len(self.basis_str) != len(self.basis_inf) + 1:
            _die("WARNING: basis_str & basis_inf need an equal number of "
                 "entires, including redundant first entry of basis_inf.")
        if len(self.basis_str) != len(self.beta):
            _die("WARNING: basis_str & beta need an equal number of entries.")
        self.delta = [float(t) for t in words("delta")]
        self.sigma = float(words("sigma")[0])
        self.nugget = float(words("nugget")[0])
        self.fix_nugget = words("fix_nugget")[0]
        self.alt_nugget = words("alt_nugget")[0] if "alt_nugget" in b else "F"
        self.mucm = words("mucm")[0]
        if self.mucm == "T" and self.alt_nugget == "T":
            _die("WARNING: mucm T cannot be used with alt_nugget T")
        # covariance family: absent means the reference's Gaussian kernel, so every existing file keeps its meaning
        self.kernel = words("kernel")[0] if "kernel" in b else "gaussian"
        if self.kernel not in self.KERNELS:
            _die("WARNING: kernel should be one of %s" % " ".join(self.KERNELS))
        # training objective: absent means maximum likelihood; loo minimises the leave-one-out cross-validation objective
        self.objective = words("objective")[0] if "objective" in b else "llh"
        if self.objective not in self.OBJECTIVES:
            _die("WARNING: objective should be one of %s" % " ".join(self.OBJECTIVES))
        self.input_minmax = eval(b["input_minmax"]) if "input_minmax" in b else []

    def final_beliefs(self, E, final=False):
        """Write '<beliefs>-<N>[f]' in the reference's format (:217-250): the checkpoint a rebuilt
        emulator (and history matching) starts from."""
        name = E.config.beliefs + "-" + str(E.tv_conf.no_of_trains) + ("f" if final else "")
        print("New beliefs to file", name)
        ndim = len(E.par.delta)
        seq = " ".join(str(i) for i in range(ndim))
        lines = [
            "active_index " + (seq if self.active == [] else " ".join(map(str, self.active))),
            "active " + seq,
            "output_index " + str(self.output),
            "output 0 ",
            "basis_str " + " ".join(map(str, self.basis_str)),
            "basis_inf NA " + " ".join(map(str, self.basis_inf)),
            "beta " + " ".join(map(str, E.par.beta)),
            "delta " + " ".join(map(str, list(E.par.delta))),
            "sigma " + str(E.par.sigma),
            "nugget " + str(E.par.nugget),
            "fix_nugget " + str(self.fix_nugget),
            "alt_nugget " + str(self.alt_nugget),
            "mucm " + str(self.mucm),
        ] + (["kernel " + self.kernel] if self.kernel != "gaussian" else []) + (
            ["objective loo"] if self.objective == "loo" else []) + [
            "input_minmax " + str(E.all_data.input_minmax),
        ]
        try:
            if _dist.is_writer():             # multi-rank: one writer, everyone waits for the file
                with open(name, "w") as fh:
                    fh.write("\n".join(lines) + "\n")
            _dist.barrier()
        except OSError:
            _die("ERROR: Problem writing to file.")


class Hyperparams:
    """beta, delta, sigma, nugget (reference :254-259)."""

    def __init__(self, beliefs):
        self.beta = np.array(beliefs.beta)
        self.delta = np.array(beliefs.delta)
        self.sigma = beliefs.sigma
        self.nugget = beliefs.nugget


class Basis:
    """Mean-function basis h(x) built from basis_str (reference :263-318).  ``poly`` holds, for a
    pure polynomial basis ('1.0', 'x', 'x**k'), the exponents that let H* be evaluated on device."""

    def __init__(self, beliefs):
        if beliefs.active != []:
            for col in beliefs.basis_inf:
                if col not in beliefs.active:
                    _die("WARNING: basis_inf specifies non-active inputs")
        # stored inputs hold only the active columns: re-index basis_inf to 0..k-1
        beliefs.basis_inf = list(range(len(beliefs.basis_inf)))
        self.h = []
        scope = {"np": np, "math": math}
        for i, expr in enumerate(beliefs.basis_str):
            exec("def h_%d(x):\n    return %s\n" % (i, expr), scope)
            self.h.append(scope["h_%d" % i])
        self.basis_inf = beliefs.basis_inf
        self.poly = self._polynomial_powers(beliefs.basis_str)
        self.print_mean_function(beliefs.basis_inf, beliefs.basis_str, beliefs.active)

    @staticmethod
    def _polynomial_powers(basis_str):
        pw = []
        for expr in basis_str[1:]:
            e = expr.replace(" ", "")
            if e == "x":
                pw.append(1)
            elif e.startswith("x**") and e[3:].isdigit():
                pw.append(int(e[3:]))
            else:
                return None
        try:
            ok = float(eval(basis_str[0], {"x": 1.0})) == 1.0
        except Exception:
            ok = False
        return pw if ok else None

    def print_mean_function(self, basis_inf, basis_str, include):
        txt = "m(x) ="
        for i in range(len(self.h)):
            if i == 0:
                txt += " b"
            else:
                lab = str(basis_inf[i - 1]) if include == [] else str(include[i - 1])
                txt += " + b" + lab + basis_str[i] + "[" + lab + "]"
        self.meanf = txt
        print(txt)

    def design_matrix(self, X):
        """H = (h(x_1), h(x_2), ...) (Data.make_H, reference :558-566), vectorised when possible."""
        X = np.asarray(X, dtype=float)
        n = X.shape[0]
        H = np.empty((n, len(self.h)))
        H[:, 0] = self.h[0](1.0)
        for j in range(1, len(self.h)):
            col = X[:, self.basis_inf[j - 1]]
            try:
                val = np.asarray(self.h[j](col), dtype=float)
                if val.shape != col.shape:
                    raise ValueError
                H[:, j] = val
            except Exception:
                H[:, j] = [self.h[j](v) for v in col]
        return H


class TV_config:
    """Training/validation schedule (reference :321-375)."""

    def __init__(self, k, c, noV):
        self.k, self.c, self.noV = k, c, noV
        self.retrain = "y"
        self.no_of_trains = 0
        self.auto = False
        self.no_retrain = False

    def auto_train(self, auto, no_retrain):
        self.auto = bool(auto)
        self.no_retrain = no_retrain is not False

    def next_train(self):
        self.no_of_trains += 1

    def next_Vset(self):
        self.c += 1

    def _auto_answer(self):
        return "n" if self.no_retrain else "y"

    def check_still_training(self):
        if self.no_of_trains < self.noV:
            if not self.auto and self.no_of_trains >= 1:
                self.retrain = input("Retrain with V in T against new V? y/[n]: ")
            else:
                self.retrain = self._auto_answer()
        else:
            self.retrain = "n"
        return self.retrain == "y"

    def doing_training(self):
        if self.no_of_trains < self.noV and self.retrain == "y":
            self.next_train()
            return True
        return False

    def do_final_build(self):
        self.retrain = self._auto_answer() if self.auto else input("\nRetrain with V in T? y/[n]: ")
        return self.retrain == "y"


class All_Data:
    """Reads the inputs/outputs files, selects active columns, scales inputs to [0,1], shuffles,
    and splits into training / validation sets (reference :379-535)."""

    def __init__(self, all_inputs, all_outputs, tv, beliefs, par, datashuffle, scaleinputs):
        print("\n*** Reading data files ***")
        print("Reading inputs file:", all_inputs)
        try:
            self.x_full = np.loadtxt(all_inputs)
        except OSError:
            _die("ERROR: Problem reading file.")
        if "output_index" in beliefs.beliefs:
            print("Emulator was trained on output_index", beliefs.output_index)
        print("Reading outputs file:", all_outputs)
        try:
            self.y_full = np.loadtxt(all_outputs, usecols=[beliefs.output]).T
            print("Using output", beliefs.output, "(relative to outputs file)")
        except IndexError:
            _die("ERROR: output (column) %s not in outputs file" % beliefs.output)
        except (OSError, ValueError):
            _die("ERROR: Problem reading file.")
        self.dim = self.x_full[0].size
        if self.dim == 1:
            self.x_full = np.array([self.x_full, ]).T
        self.numpoints = self.x_full.shape[0]
        if self.numpoints != self.y_full.size:
            _die("WARNING: different number of data points in input and output files.")
        if "active_index" in beliefs.beliefs:
            print("Emulator was trained on active_index", beliefs.active_index)
        if beliefs.active != []:
            print("Including input dimensions", beliefs.active)
            self.x_full = self.x_full[:, beliefs.active]
        if len(par.delta) != self.x_full.shape[1]:
            _die("WARNING: different number of delta than input dimensions.")
        self.input_minmax = beliefs.input_minmax
        self.map_inputs_0to1(par, scaleinputs)
        self.data_shuffle(datashuffle)
        self.T = self.V = 0
        self.tv = tv
        self.split_T_V_config()

    def map_inputs_0to1(self, par, scaleinputs):
        ncol = self.x_full.shape[1]
        if not scaleinputs:
            print("Input scaling off")
            self.minmax = np.array([(0.0, 1.0)] * ncol)
        elif self.input_minmax == []:
            print("Input scaling based on data")
            mm = [(np.amin(self.x_full[:, i]), np.amax(self.x_full[:, i])) for i in range(ncol)]
            self.minmax = np.array(mm)
            self.input_minmax = [list(t) for t in mm]
        else:
            print('Input scaling based on "input_minmax" in beliefs file')
            self.minmax = np.array(self.input_minmax)
        for i in range(ncol):
            span = self.minmax[i, 1] - self.minmax[i, 0]
            self.x_full[:, i] = (self.x_full[:, i] - self.minmax[i, 0]) / span
            print("Dim", i, "scaled by %", span)
        self.input_range = [[np.amin(self.x_full[:, i]), np.amax(self.x_full[:, i])] for i in range(ncol)]

    def data_shuffle(self, datashuffle):
        if not datashuffle:
            print("Data shuffling turned off")
            return
        print("Shuffling", self.x_full.shape[0], "data points")
        z = np.column_stack([self.x_full, self.y_full])
        _dist.sync_numpy_rng()                    # multi-rank: every rank shuffles with rank 0's generator state
        np.random.shuffle(z)                      # same RNG consumption as the reference (:490)
        ncol = self.x_full.shape[1]
        self.x_full[:, :] = z[:, :ncol]
        self.y_full = z[:, ncol].copy()

    def split_T_V_config(self):
        npts = self.x_full.shape[0]
        print("Split data into", self.tv.k, "sets")
        self.T = int((npts / self.tv.k) * (self.tv.k - self.tv.noV))
        self.V = int((npts / self.tv.k) * 1)
        self.remainder = npts - (self.T + self.tv.noV * self.V)
        print("Remainder", self.remainder, "added to T-set")
        self.T += self.remainder
        print("T-set size:", self.T, ", V-set size:", self.V, ", V sets:", self.tv.noV)

    def _v_rows(self):
        return list(range(self.tv.c * self.V, (self.tv.c + 1) * self.V))

    def choose_T(self):
        rows = list(range(0, self.tv.c * self.V)) \
            + list(range((self.tv.c + self.tv.noV) * self.V, self.tv.k * self.V + self.remainder))
        return self.x_full[rows, :], self.y_full[rows]

    def choose_V(self):
        rows = self._v_rows()
        return self.x_full[rows, :], self.y_full[rows]

    def choose_new_V(self, validation):
        rows = self._v_rows()
        validation.inputs = self.x_full[rows, :]
        validation.outputs = self.y_full[rows]


class Data:
    """A data set with its design matrix H and covariance matrix A (reference :539-584).

    ``A`` is produced on the B200 (``gpe_cov_build``) the first time it is read after the
    hyper-parameters, ``r`` or the inputs changed; training sets own a device handle that also
    serves the likelihood and posterior kernels (``device()``)."""

    def __init__(self, inputs, outputs, basis, par, beliefs, K):
        self.inputs = inputs
        self.outputs = outputs
        self.basis, self.beliefs, self.par, self.K = basis, beliefs, par, K
        self.r = 0
        self._r_made = 0
        self._dev = None
        self._loaded = None
        self._fit_key = None
        self._A = None
        self._A_args = (1.0, True)
        self.make_H()
        self.make_A()

    # ---- matrices -------------------------------------------------------------------------
    def remake(self):
        self.make_H()
        self.make_A()

    def make_H(self):
        self.H = self.basis.design_matrix(self.inputs)

    def make_E(self):
        self.E = self.H.dot(self.par.beta)

    def make_A(self, s2=1.0, predict=True):
        """Record how A is to be built (reference :572-575); the matrix itself is built on device
        when ``A`` is next read.  NB remake() uses s2 = 1, i.e. adds un-scaled r (reference quirk)."""
        self._A_args = (float(s2), bool(predict))
        self._r_made = self.r          # like the reference, A reflects r as of the last make_A()
        self._A = None

    @property
    def kind(self):
        return 1 if self.beliefs.alt_nugget == "T" else 0

    @property
    def A(self):
        if self._A is None:
            s2, predict = self._A_args
            dev = self.device()
            self._A = dev.cov_build(self.K.d, self.K.n, self.kind, predict, s2)
            self.K.A = self._A
        return self._A

    @A.setter
    def A(self, value):
        self._A = value

    def set_r(self, r, message=True):
        if len(r) == self.inputs.shape[0]:
            if message:
                print("\n*** Updating array 'r' of constant variances***")
            self.r = r
        else:
            _die("\nWARNING: length of 'r' does not match number of data points")

    # ---- device side ----------------------------------------------------------------------
    def _fingerprint(self):
        """Content key of what the device holds (inputs, outputs, r, H): a position-weighted 64-bit checksum of
        the raw bits of every array, so permuted rows, swapped entries or a changed sign are seen, not only
        changed moments; costs one pass per array (it is taken before every device call)."""
        X = np.asarray(self.inputs, dtype=float)
        y = np.zeros(X.shape[0]) if self.outputs is None else np.asarray(self.outputs, dtype=float)
        r = np.asarray(self._r_made, dtype=float)
        return tuple((a.shape, _checksum(a)) for a in (X, y, r, np.asarray(self.H, dtype=float)))

    def device(self):
        """The handle holding this data set on the GPU (created and re-uploaded on demand)."""
        if self._dev is None:
            self._dev = _lib.Device(_lib.default_device_index())
        fp = (self.K.family,) + self._fingerprint()
        if fp != self._loaded:
            y = np.zeros(self.inputs.shape[0]) if self.outputs is None else self.outputs
            r = self._r_made if np.ndim(self._r_made) else None
            self._dev.set_training(self.inputs, y, self.H, r)
            if self.basis.poly is not None:
                self._dev.set_basis(self.basis.basis_inf, self.basis.poly)
            self._dev.set_kernel(self.K.family)
            self._loaded = fp
            self._fit_key = None
        return self._dev

    def fit(self, beta=None, r_div=1.0):
        """Factor the training matrix for the current hyper-parameters (cached): returns
        (device, optimal beta, analytic MUCM sigma)."""
        dev = self.device()
        key = (tuple(np.asarray(self.K.d, dtype=float)), float(self.K.n), float(self.par.sigma), self.kind, self.K.family,
               None if beta is None else tuple(np.asarray(beta, dtype=float)), float(r_div))
        if key != self._fit_key:
            bopt, sig, st = dev.fit_state(self.K.d, self.K.n, self.par.sigma, self.kind, beta=beta, r_div=r_div)
            self._fit_key = key
            self._fit_out = (bopt, sig, st)
        return (dev,) + self._fit_out


class Posterior:
    """Posterior of the new points ``Dnew`` given the training set ``Dold`` (reference :588-687).
    mean [m] and var [m,m] are computed on device (``gpe_predict_fullcov``); with
    ``diag_only=True`` only the diagonal is produced (``gpe_predict``, any m) in ``var_diag``.
    The ``predict`` flag is stored and, as in the reference (:595, :621), has no effect."""

    def __init__(self, Dnew, Dold, par, beliefs, K, predict=True, diag_only=False, lazy=False):
        self.Dnew, self.Dold, self.par, self.beliefs, self.K = Dnew, Dold, par, beliefs, K
        self.predict = predict
        self.diag_only = diag_only
        # lazy: g.setup builds a Posterior from the *initial* beliefs before any training; the reference gets
        # through that with LU solves even when those hyper-parameters give a matrix that is not numerically
        # positive definite (train() replaces them).  Here the factorisation is a Cholesky, so the setup-time
        # object defers it to the first read of mean / var / var_diag (or the next remake()).
        self._stale = True
        self._mean = self._var = self._var_diag = None
        if not lazy:
            self.remake()

    def remake(self):
        self._covar = None
        self.make_mean()
        self.make_var()

    def _fresh(self):
        if self._stale:
            self._predict()

    @property
    def mean(self):
        self._fresh()
        return self._mean

    @mean.setter
    def mean(self, value):
        self._mean = value

    @property
    def var(self):
        self._fresh()
        if self._var is None and self._mean is not None and self._mean.size:
            raise _lib.GpeError("the full %d x %d posterior covariance was not formed (more than %d points, or diag_only): "
                                "use var_diag, or predict in smaller blocks" % (self._mean.size, self._mean.size, _PRED_FULL_LIMIT))
        return self._var

    @var.setter
    def var(self, value):
        self._var = value

    @property
    def var_diag(self):
        self._fresh()
        return self._var_diag

    @var_diag.setter
    def var_diag(self, value):
        self._var_diag = value

    @property
    def covar(self):
        if self._covar is None:
            self.make_covar()
        return self._covar

    def make_covar(self):
        self._covar = self.Dold.device().cross_cov(self.K.d, self.K.n, self.Dold.kind, self.Dnew.inputs)

    def _predict(self):
        self._stale = False
        Dn = self.Dnew
        m = Dn.inputs.shape[0]
        if m == 0:
            self.mean, self.var, self.var_diag = np.zeros(0), np.zeros((0, 0)), np.zeros(0)
            return
        dev, _, _, st = self.Dold.fit(beta=self.par.beta, r_div=self.Dold._A_args[0])
        if st != 0:
            _die("ERROR: training covariance matrix is not positive definite (pivot %d). Exiting." % st)
        Hs = None if Dn.basis.poly is not None else Dn.H
        if self.diag_only or m > _PRED_FULL_LIMIT:
            self.mean, self.var_diag = dev.predict(Dn.inputs, Hs)
            self.var = None
        else:
            r_new = np.asarray(Dn._r_made, dtype=float) / Dn._A_args[0] if (np.ndim(Dn._r_made) and Dn.kind == 1) else None
            self.mean, self.var = dev.predict_fullcov(Dn.inputs, Hs, r_new)
            self.var_diag = np.diag(self.var).copy()

    def make_mean(self):
        self._predict()

    def make_var(self):
        pass        # mean and variance come out of the same device pass

    def interval(self):
        half = 1.96 * np.sqrt(np.abs(self.var_diag))
        self.LI, self.UI = self.mean - half, self.mean + half

    def indiv_standard_error(self, ise=2.0):
        retrain = False
        e = (self.Dnew.outputs - self.mean) / np.sqrt(self.var_diag)
        for i in np.nonzero(np.abs(e) >= ise)[0]:
            print("  Bad predictions:", self.Dnew.inputs[i, :], "ise:", np.round(e[i], decimals=4))
            retrain = True
        return retrain

    def mahalanobis_distance(self):
        nV, nT, q = self.Dnew.outputs.size, self.Dold.outputs.size, self.par.beta.size
        try:
            MDvar = 2 * nV * (nV + nT - q - 2.0) / (nT - q - 4.0)
            print("theoretical Mahalanobis_distance (mean, var):(", nV, ",", MDvar, ")")
        except ZeroDivisionError:
            print("theoretical Mahalanobis_distance mean:", nV, "(too few data for variance)")
        if nV:
            # resid^T V^-1 resid = |L_V^-1 resid|^2, V factored on device
            resid = self.Dnew.outputs - self.mean
            Li, _, st = _lib.scratch_device().dbg_potrf_inv(self.var)
            MD = float(np.sum(Li[0].dot(resid) ** 2)) if st[0] == 0 else float("nan")
        else:
            MD = 0.0
        print("calculated Mahalanobis_distance:", MD)
        return True

    def incVinT(self):
        self.Dold.inputs = np.append(self.Dnew.inputs, self.Dold.inputs, axis=0)
        self.Dold.outputs = np.append(self.Dnew.outputs, self.Dold.outputs)
        print("Include V into T, T-set size:", self.Dold.inputs.shape[0])
        self.Dold.H = np.zeros([self.Dold.inputs.shape[0], len(self.Dold.basis.h)])
        self.Dold.A = None

    def final_design_points(self, E, final=False):
        """Write the training set as '<inputs>-o<K>-<N>[f]' / '<outputs>-o<K>-<N>[f]' (reference
        :690-716; '%.8f' text, inputs un-scaled) -- with the beliefs file, the checkpoint format."""
        tag = "-o" + str(E.beliefs.output) + "-" + str(E.tv_conf.no_of_trains) + ("f" if final else "")
        mm = E.all_data.minmax
        unscaled = self.Dold.inputs * (mm[:, 1] - mm[:, 0]) + mm[:, 0]
        for name, arr in ((E.config.inputs + tag, unscaled), (E.config.outputs + tag, self.Dold.outputs)):
            print("Writing T-data to:", name)
            try:
                if _dist.is_writer():
                    np.savetxt(name, arr, delimiter=" ", fmt="%.8f")
                _dist.barrier()
            except OSError:
                _die("ERROR: Problem writing to file.")
