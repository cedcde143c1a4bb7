"""Gaussian against Matern 5/2 on one GPU, in one process (the measurement behind DESIGN.md section 10):

  * ms per llh+grad step of the bench workload (n = 4096, d = 16, 32 guesses from bench.py's multistart draw) for both
    families on the INT8 route (default) and the FP64 DMMA route (GPE_OZAKI=0), the two families alternating step by
    step, 3 warm-up and 10 timed steps each, CUDA events on the handle's stream;
  * the per-category serial pass (gpe_profile_read, one stream) of one step of each family on the INT8 route;
  * grid predictions/s at n = 2000, d = 8 over 2^22 points of the 10^8-point grid, both families alternating.

    python tools/perf_matern.py [out.json]
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from gp_emu_uqsa_b200 import _lib  # noqa: E402

FAMILIES = (("gaussian", _lib.KERNEL_GAUSSIAN), ("matern52", _lib.KERNEL_MATERN52))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))


def handle(X, y, H, family, env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        dev = _lib.Device(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v
    dev.set_training(X, y, H)
    dev.set_basis(list(range(X.shape[1])), [1] * X.shape[1])
    dev.set_kernel(family)
    return dev


def timed(dev, fn):
    """ms of fn() between two CUDA events on the handle's stream."""
    s = torch.cuda.ExternalStream(dev.stream_ptr)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(s)
    fn()
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1)


def llh_ab(X, y, H, theta, env, warm=3, steps=10):
    B, p = theta.shape
    devs = {name: handle(X, y, H, fam, env) for name, fam in FAMILIES}
    bufs = {name: (torch.empty(B, dtype=torch.float64, device="cuda"), torch.empty(B, p, dtype=torch.float64, device="cuda"),
                   torch.empty(B, dtype=torch.float64, device="cuda"), torch.zeros(B, dtype=torch.int32, device="cuda"))
            for name in devs}
    th0 = torch.tensor(theta, device="cuda")
    ms = {name: [] for name in devs}
    for it in range(warm + steps):
        th = th0 + 1e-3 * it
        for name, dev in devs.items():          # alternate the two families step by step
            t = timed(dev, lambda: dev.llh_grad_batch(th, 0, fixed_nugget=1e-4, out=bufs[name]))
            if it >= warm:
                ms[name].append(t)
    for name in devs:
        assert int(bufs[name][3].abs().sum()) == 0, "non-PD item"
    out = {name: {"ms_per_step_median": float(np.median(v)), "ms_per_step_min": float(np.min(v)), "ms_per_step_max": float(np.max(v)),
                  "int8_products": devs[name].int8_products} for name, v in ms.items()}
    return out, devs


def serial_pass(dev, theta):
    dev.set_streams(1)
    dev.llh_grad_batch(theta, 0, fixed_nugget=1e-4)
    dev.profile_enable(True)
    dev.profile_read(reset=True)
    dev.llh_grad_batch(theta, 0, fixed_nugget=1e-4)
    prof = dev.profile_read(reset=True)
    dev.profile_enable(False)
    return {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in prof.items() if v[1]}


def grid_ab(reps=3):
    n, d, m = bench.N_PRED, bench.D_PRED, 1 << 22
    X, y = bench.synth(n, d)
    H = bench.linear_H(X)
    levels = np.full(d, 10, dtype=np.int32)
    mean = torch.empty(m, dtype=torch.float64, device="cuda")
    var = torch.empty(m, dtype=torch.float64, device="cuda")
    devs = {name: handle(X, y, H, fam, {}) for name, fam in FAMILIES}
    for dev in devs.values():
        assert dev.fit_state(np.full(d, 0.5), 1e-4, 1.0, 0)[2] == 0
    ms = {name: [] for name in devs}
    for it in range(1 + reps):
        for name, dev in devs.items():
            t = timed(dev, lambda: dev.predict_grid(levels, np.zeros(d), np.ones(d), it * m, m, out=(mean, var)))
            if it:
                ms[name].append(t)
    res = {name: {"ms_median": float(np.median(v)), "mpred_per_s": m / float(np.median(v)) * 1e-3} for name, v in ms.items()}
    for dev in devs.values():
        dev.close()
    return {"n": n, "d": d, "points": m, "levels": levels.tolist(), **res}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    n, d, B = bench.N_TRAIN, bench.D_IN, bench.B_PER_GPU
    X, y = bench.synth(n, d)
    H = bench.linear_H(X)
    theta = bench.draw_thetas(B, d, y)
    res = {"what": "Gaussian vs Matern 5/2, llh+grad step (n=4096, d=16, 32 guesses, gp4ml, fixed nugget 1e-4) and grid "
                   "prediction (n=2000, d=8, 2^22 points)", "gpu": gpu_info(), "llh_step": {}, "serial_pass_int8": {}}
    for route, env in (("int8", {}), ("dmma", {"GPE_OZAKI": "0"})):
        r, devs = llh_ab(X, y, H, theta, env)
        res["llh_step"][route] = r
        if route == "int8":
            res["serial_pass_int8"] = {name: serial_pass(dev, theta) for name, dev in devs.items()}
        for dev in devs.values():
            dev.close()
        print(route, json.dumps(r), flush=True)
    res["grid"] = grid_ab()
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
