"""User-facing sensitivity functions (reference: gp_emu_uqsa/sensitivity/sensitivityfunctions.py)."""
import numpy as _np

from ._sampledsensitivity import SampledSensitivity
from ._sensitivityclasses import Sensitivity

__all__ = ["setup", "setup_sampled", "sense_table", "Sensitivity", "SampledSensitivity"]


def setup(emul, m, v, case="case2"):
    """Return a Sensitivity instance initialised with input means ``m`` and variances ``v``
    (lists of floats), or None on bad arguments -- same checks and messages as the reference (:7-54)."""
    print("\n*** Initialising Sensitivity class ***")
    if not isinstance(m, list) or not isinstance(v, list):
        print("ERROR: 2nd and 3rd arguments must be lists of floats. "
              "Return None.")
        return None
    if case == "case2":
        if len(emul.par.beta) != emul.training.inputs[0].size + 1 \
                or False in [i == 'x' for i in emul.beliefs.basis_str[1:]]:
            print("The case2 sensitivity routines only work for emulators "
                  "with a gaussian kernel and linear mean. "
                  "This mean function will not work. Return None.")
            return None
        if len(m) != len(emul.par.beta) - 1 or len(v) != len(emul.par.beta) - 1:
            print("Mean and Variance lists must both contain as many items "
                  "as there are input dimensions. Return None.")
            return None
    else:
        print("Only case2 of MUCM's U & S analysis is implemented. Return None.")
        return None
    if emul.K.family != 0:
        print("The sensitivity integrals need the Gaussian kernel; this emulator uses "
              "the Matern 5/2 kernel. Return None.")
        return None
    return Sensitivity(emul, _np.array(m), _np.array(v))


def setup_sampled(emul, m=None, v=None, bounds=None, samples=65536, seed=0):
    """Return a SampledSensitivity instance (any covariance family, any polynomial mean) for independent inputs that are
    either normal -- means ``m`` and variances ``v`` -- or uniform over ``bounds`` = [[lo, hi], ...], one entry per
    active input in the units ``setup`` takes; ``samples`` (a power of two >= 256) Sobol points drawn with ``seed``.
    None on bad arguments, with a message."""
    print("\n*** Initialising SampledSensitivity class ***")
    d = emul.training.inputs.shape[1]
    normal = m is not None and v is not None
    if (m is None) != (v is None) or normal == (bounds is not None):
        print("ERROR: give either input means m and variances v, or uniform input bounds. Return None.")
        return None
    if normal:
        ok = _np.shape(m) == (d,) and _np.shape(v) == (d,)
        if not ok or not (_np.all(_np.isfinite(m)) and _np.all(_np.isfinite(v))):
            print("Mean and Variance lists must both contain as many finite values "
                  "as there are input dimensions. Return None.")
            return None
        if _np.any(_np.asarray(v, dtype=float) <= 0.0):
            print("ERROR: input variances must be positive. Return None.")
            return None
    else:
        if _np.shape(bounds) != (d, 2) or not _np.all(_np.isfinite(bounds)):
            print("ERROR: bounds must hold one finite [lo, hi] pair per input dimension. Return None.")
            return None
        if _np.any(_np.asarray(bounds, dtype=float)[:, 0] >= _np.asarray(bounds, dtype=float)[:, 1]):
            print("ERROR: every input range needs lo < hi. Return None.")
            return None
    if not isinstance(samples, (int, _np.integer)) or samples < 256 or samples & (samples - 1):
        print("ERROR: samples must be a power of two of at least 256. Return None.")
        return None
    if emul.basis.poly is None:
        print("The sampled sensitivity routines need a polynomial mean function "
              "('1.0', 'x', 'x**k' terms). Return None.")
        return None
    return SampledSensitivity(emul, m=m, v=v, bounds=bounds, samples=int(samples), seed=seed)


def sense_table(sense_list, inputNames=[], outputNames=[], rowHeight=6):
    """Table plot of sensitivity indices (reference :57-148).  Drawing needs matplotlib, which is
    outside the hot path this package rebuilds (DESIGN.md section 7); the table of normalised indices
    is returned so callers can still consume the numbers."""
    rows = []
    for s in sense_list:
        rows.append(_np.append(s.senseindex / s.uEV, _np.sum(s.senseindex / s.uEV)))
    table = _np.array(rows)
    try:
        import matplotlib.pyplot  # noqa: F401
    except ImportError:
        print("sense_table: matplotlib is not available; returning the table of indices without plotting")
    return table
