"""Posterior gradient (gpe_predict_grad) on one GPU, in one process (the measurement behind DESIGN.md section 9e):

  * gradient points/s at n = 2000, d = 8 (the config-5 generator of bench.py, Gaussian / Matern 5/2 fit state at delta = 0.6,
    nugget 1e-4) on 2^18 uniform points in device memory, both covariance families, the INT8 route (default) and the FP64 DMMA
    route (GPE_OZAKI=0 on a handle of its own), median of 5 after 2 warm-up calls, CUDA events on the handle's stream;
    gpe_predict's points/s on the same points and handle beside it;
  * the per-category serial pass (gpe_profile_read) of one gradient call;
  * one SampledSensitivity.dgsm() at 2^16 samples (normal inputs N(0.5, 0.02), host arrays, wall clock) beside one
    gpe_sens_sample analysis of all 8 inputs at the same M, on the INT8-route handle;
  * card name and power limit before and after.

    python tools/perf_posterior_grad.py profiles/r07_posterior_grad.json
"""
import contextlib
import io
import json
import os
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import bench  # noqa: E402
from gp_emu_uqsa_b200 import _lib  # noqa: E402
from gp_emu_uqsa_b200.sensitivity._sampledsensitivity import SampledSensitivity, sample_points  # noqa: E402
from perf_matern import gpu_info, handle, timed  # noqa: E402

N, D = 2000, 8
M_PTS = 1 << 18
M_DGSM = 1 << 16


def median_ms(dev, fn, warm=2, reps=5):
    for _ in range(warm):
        fn()
    return float(np.median([timed(dev, fn) for _ in range(reps)]))


def wall_ms(fn, warm=1, reps=3):
    for _ in range(warm):
        fn()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out))


def dgsm_vs_sens_sample(dev, y):
    """SampledSensitivity.dgsm() on a stand-in for the object (its points and handle only) and gpe_sens_sample on the same M."""
    m, v = [0.5] * D, [0.02] * D
    S = SimpleNamespace(samples=M_DGSM, d=D, m=np.array(m), v=np.array(v), bounds=None, stderr={},
                        _points=lambda k: sample_points(D, k, 0, m=m, v=v), _device=lambda: dev)

    def run_dgsm():
        with contextlib.redirect_stdout(io.StringIO()):
            SampledSensitivity.dgsm(S)

    A, B = sample_points(D, M_DGSM, 0, m=m, v=v)
    return {"dgsm_ms": round(wall_ms(run_dgsm), 3),
            "sens_sample_all_inputs_ms": round(wall_ms(lambda: dev.sens_sample(A, B, list(range(D)), float(y.mean()))), 3),
            "samples": M_DGSM, "note": "wall clock, host arrays, including sample_points for dgsm()"}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    X, y = bench.synth(N, D)
    H = bench.linear_H(X)
    delta = np.full(D, 0.6)
    P = torch.from_numpy(np.random.default_rng(1).random((M_PTS, D))).cuda()
    res = {"what": "gpe_predict_grad on the config-5 generator (n=%d, d=%d), %d uniform points in device memory, Gaussian / "
                   "Matern 5/2 fit state at delta = 0.6, nugget 1e-4; gpe_predict on the same points and handle" % (N, D, M_PTS),
           "gpu": gpu_info(), "runs": {}}
    for route, env in (("int8", {}), ("dmma", {"GPE_OZAKI": "0"})):
        for fam_name, fam in (("gaussian", _lib.KERNEL_GAUSSIAN), ("matern52", _lib.KERNEL_MATERN52)):
            dev = handle(X, y, H, fam, env)
            assert dev.fit_state(delta, 1e-4, 1.0, 0)[2] == 0
            dm = torch.empty((M_PTS, D), dtype=torch.float64, device="cuda")
            dv = torch.empty((M_PTS, D), dtype=torch.float64, device="cuda")
            mean = torch.empty(M_PTS, dtype=torch.float64, device="cuda")
            var = torch.empty(M_PTS, dtype=torch.float64, device="cuda")
            r = {}
            k0 = dev.int8_products
            ms = median_ms(dev, lambda: dev.predict_grad(P, out=(dm, dv)))
            r["grad"] = {"ms_median": round(ms, 3), "points_per_s": M_PTS / (ms * 1e-3), "int8_products": dev.int8_products - k0}
            ms = median_ms(dev, lambda: dev.predict_grad(P, out=(dm, None)))
            r["grad_mean_only"] = {"ms_median": round(ms, 3), "points_per_s": M_PTS / (ms * 1e-3)}
            ms = median_ms(dev, lambda: dev.predict(P, None, out=(mean, var)))
            r["predict"] = {"ms_median": round(ms, 3), "points_per_s": M_PTS / (ms * 1e-3)}
            r["grad_over_predict_rate"] = r["grad"]["points_per_s"] / r["predict"]["points_per_s"]
            dev.profile_enable(True)
            dev.profile_read(reset=True)
            dev.predict_grad(P, out=(dm, dv))
            prof = dev.profile_read(reset=True)
            dev.profile_enable(False)
            r["serial_pass_grad"] = {k: {"ms": round(v[0], 3), "launches": v[1]} for k, v in prof.items() if v[1]}
            if route == "int8":
                r["dgsm_2^16"] = dgsm_vs_sens_sample(dev, y)
            res["runs"]["%s/%s" % (route, fam_name)] = r
            print(route, fam_name, json.dumps(r), flush=True)
            dev.close()
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
