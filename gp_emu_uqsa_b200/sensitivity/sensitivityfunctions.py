"""User-facing sensitivity functions (reference: gp_emu_uqsa/sensitivity/sensitivityfunctions.py)."""
import numpy as _np

from ._sensitivityclasses import Sensitivity

__all__ = ["setup", "sense_table", "Sensitivity"]


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
