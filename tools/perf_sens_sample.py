"""Sampled sensitivity analysis (gpe_sens_sample) on one GPU, in one process (the measurement behind DESIGN.md section 9d):

  * ms per analysis of all 8 inputs (10 M posterior columns) on the config-5 generator (n = 2000, d = 8, normal inputs
    N(0.5, 0.02) as in bench.py), M = 2^16 and 2^18 samples, both covariance families, the INT8 route (default) and the FP64
    DMMA route (GPE_OZAKI=0 on a handle of its own), median of 5 after 2 warm-up calls, CUDA events on the handle's stream;
    posterior columns/s beside gpe_predict_grid's points/s on 2^22 grid points with the same handle;
  * the per-category serial pass (gpe_profile_read) of one analysis at 2^18;
  * kernel times of one analysis by name (torch.profiler), from which the pair-dot pass and the product that stores Z;
  * card name and power limit before and after.

    python tools/perf_sens_sample.py profiles/r06_sens_sample.json
"""
import json
import os
import sys
from collections import defaultdict

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import bench  # noqa: E402
from gp_emu_uqsa_b200 import _lib  # noqa: E402
from gp_emu_uqsa_b200.sensitivity._sampledsensitivity import sample_points  # noqa: E402
from perf_matern import gpu_info, handle, timed  # noqa: E402

N, D = 2000, 8
WHICH = list(range(D))


def median_ms(dev, fn, warm=2, reps=5):
    for _ in range(warm):
        fn()
    return float(np.median([timed(dev, fn) for _ in range(reps)]))


def kernel_times(dev, fn):
    """ms per kernel name over one call of fn (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = defaultdict(float)
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0:
            out[ev.name] += ev.device_time_total / 1000.0
    return out


def group(kt):
    g = defaultdict(float)
    for name, ms in kt.items():
        key = ("pair_dot" if "sens_pairdot" in name else "sample_finalize" if "sens_sample_finalize" in name
               else "regression_vectors_G" if "fullcov_finalize" in name else "compose" if "sens_compose" in name
               else "cross_covariance" if "xcov" in name else "int8_product" if "oz_" in name
               else "dmma_product" if "gemm" in name else "other")
        g[key] += ms
    tot = sum(g.values())
    return {k: {"ms": round(v, 3), "share": round(v / tot, 4)} for k, v in sorted(g.items())}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    X, y = bench.synth(N, D)
    H = bench.linear_H(X)
    delta = np.full(D, 0.6)
    res = {"what": "gpe_sens_sample on the config-5 generator (n=%d, d=%d, all %d inputs: %d posterior columns per sample), "
                   "normal inputs N(0.5, 0.02), Gaussian / Matern 5/2 fit state at delta = 0.6, nugget 1e-4" % (N, D, D, D + 2),
           "gpu": gpu_info(), "runs": {}}
    for route, env in (("int8", {}), ("dmma", {"GPE_OZAKI": "0"})):
        for fam_name, fam in (("gaussian", _lib.KERNEL_GAUSSIAN), ("matern52", _lib.KERNEL_MATERN52)):
            dev = handle(X, y, H, fam, env)
            assert dev.fit_state(delta, 1e-4, 1.0, 0)[2] == 0
            r = {}
            for M in (1 << 16, 1 << 18):
                A, B = sample_points(D, M, 0, m=[0.5] * D, v=[0.02] * D)
                A, B = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
                out = torch.empty((2, 3 + 2 * D), dtype=torch.float64, device="cuda")
                k0 = dev.int8_products
                ms = median_ms(dev, lambda: dev.sens_sample(A, B, WHICH, float(y.mean()), out=out))
                r["M=%d" % M] = {"ms_median": round(ms, 3), "posterior_columns_per_s": (D + 2) * M / (ms * 1e-3),
                                 "int8_products": dev.int8_products - k0}
            mg = 1 << 22
            mean = torch.empty(mg, dtype=torch.float64, device="cuda")
            var = torch.empty(mg, dtype=torch.float64, device="cuda")
            lv, lo, hi = np.full(D, 8), np.zeros(D), np.ones(D)
            ms = median_ms(dev, lambda: dev.predict_grid(lv, lo, hi, 0, mg, out=(mean, var)), reps=3)
            r["predict_grid_2^22"] = {"ms_median": round(ms, 3), "points_per_s": mg / (ms * 1e-3)}
            dev.profile_enable(True)
            dev.profile_read(reset=True)
            dev.sens_sample(A, B, WHICH, float(y.mean()), out=out)
            prof = dev.profile_read(reset=True)
            dev.profile_enable(False)
            r["serial_pass_M=2^18"] = {k: {"ms": round(v[0], 3), "launches": v[1]} for k, v in prof.items() if v[1]}
            r["kernels_M=2^18"] = group(kernel_times(dev, lambda: dev.sens_sample(A, B, WHICH, float(y.mean()), out=out)))
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
