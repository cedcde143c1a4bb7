"""Leave-one-out objective against the likelihood on one GPU, in one process (the measurement behind DESIGN.md section 9c):

  * ms per step of the bench workload (n = 4096, d = 16, 32 guesses from bench.py's multistart draw, gp4ml, fixed nugget)
    with and without GPE_MODE_LOO on the INT8 route (default) and the FP64 DMMA route (GPE_OZAKI=0), LOO and likelihood
    steps alternating on one handle, 3 warm-up and 10 timed steps each, CUDA events on the handle's stream;
  * the per-category serial pass (gpe_profile_read, one stream) of one step of each objective on both routes;
  * card name and power limit before and after.

    python tools/perf_loo.py profiles/r05_loo_ab.json
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import bench  # noqa: E402
from gp_emu_uqsa_b200 import _lib  # noqa: E402
from perf_matern import gpu_info, handle, timed  # noqa: E402

OBJECTIVES = (("llh", 0), ("loo", _lib.MODE_LOO))


def step_ab(dev, theta, warm=3, steps=10):
    B, p = theta.shape
    bufs = {name: (torch.empty(B, dtype=torch.float64, device="cuda"), torch.empty(B, p, dtype=torch.float64, device="cuda"),
                   torch.empty(B, dtype=torch.float64, device="cuda"), torch.zeros(B, dtype=torch.int32, device="cuda"))
            for name, _ in OBJECTIVES}
    th0 = torch.tensor(theta, device="cuda")
    ms = {name: [] for name, _ in OBJECTIVES}
    for it in range(warm + steps):
        th = th0 + 1e-3 * it
        for name, mode in OBJECTIVES:           # alternate the two objectives step by step
            t = timed(dev, lambda: dev.llh_grad_batch(th, mode, fixed_nugget=1e-4, out=bufs[name]))
            if it >= warm:
                ms[name].append(t)
    for name, _ in OBJECTIVES:
        assert int(bufs[name][3].abs().sum()) == 0, "failed item"
    return {name: {"ms_per_step_median": float(np.median(v)), "ms_per_step_min": float(np.min(v)),
                   "ms_per_step_max": float(np.max(v)), "ms_all": [round(x, 3) for x in v]} for name, v in ms.items()}


def serial_pass(dev, theta):
    out = {}
    dev.set_streams(1)
    for name, mode in OBJECTIVES:
        dev.llh_grad_batch(theta, mode, fixed_nugget=1e-4)
        dev.profile_enable(True)
        dev.profile_read(reset=True)
        dev.llh_grad_batch(theta, mode, fixed_nugget=1e-4)
        prof = dev.profile_read(reset=True)
        dev.profile_enable(False)
        out[name] = {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in prof.items() if v[1]}
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    n, d, B = bench.N_TRAIN, bench.D_IN, bench.B_PER_GPU
    X, y = bench.synth(n, d)
    H = bench.linear_H(X)
    theta = bench.draw_thetas(B, d, y)
    res = {"what": "LOO objective vs likelihood, llh+grad step (n=%d, d=%d, %d guesses, gp4ml, fixed nugget 1e-4), steps "
                   "alternating on one handle" % (n, d, B), "gpu": gpu_info(), "step": {}, "serial_pass": {}}
    for route, env in (("int8", {}), ("dmma", {"GPE_OZAKI": "0"})):
        dev = handle(X, y, H, _lib.KERNEL_GAUSSIAN, env)
        r = step_ab(dev, theta)
        r["loo_over_llh"] = r["loo"]["ms_per_step_median"] / r["llh"]["ms_per_step_median"]
        res["step"][route] = r
        res["serial_pass"][route] = serial_pass(dev, theta)
        dev.close()
        print(route, json.dumps({k: v for k, v in r.items()}), flush=True)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
