#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native GP_emu_UQSA hot path.

Metric (BASELINE.json): batched llh+grad evaluations/sec at n=4096, d=16 (config 3: 256 multistart
guesses over 8 GPUs = 32 per GPU, weak scaling), plus posterior predictions/sec on the 10^8-point
grid of config 4 and the other BASELINE configs (reported under "extra").  One "step" = one batched
llh+gradient evaluation of 32 hyper-parameter vectors per GPU (theta perturbed every step so nothing
is cached).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun)
    python bench.py --impl reference ...                      (the reference's CPU algorithm, all host cores)

Prints ONE JSON line on rank 0.
"""
import os
import sys


def _host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# The CPU legs must run the BLAS on every host core; torchrun exports OMP_NUM_THREADS=1 to its workers, and OpenBLAS
# sizes its pool when NumPy is first imported -- so this has to happen before `import numpy`.
if ("reference" in sys.argv and os.environ.get("RANK", "0") == "0") or os.environ.get("WORLD_SIZE", "1") == "1":
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = str(_host_cores())

import argparse      # noqa: E402
import contextlib    # noqa: E402
import io            # noqa: E402
import json          # noqa: E402
import subprocess    # noqa: E402
import tempfile      # noqa: E402
import time          # noqa: E402

import numpy as np   # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RESULT_OUT = sys.stdout
METRIC = "llh+grad evals/sec (n=4096,d=16) and posterior preds/sec, 1/2/4/8 B200"
N_TRAIN, D_IN, B_PER_GPU = 4096, 16, 32
N_PRED, D_PRED = 2000, 8
FP64_PEAK_FALLBACK_TFLOPS = 37.19     # tools/ub_fp64.cu on this pool's B200 (profiles/r01_ub_fp64_peaks.json)
HBM_PEAK_FALLBACK_GBS = 6552.0
DUMP_PRED_POINTS = 1 << 18            # grid points whose posterior mean / variance --dump-outputs keeps (6 MB with their indices)


def synth(n, d, seed=0):
    """BASELINE.md section 3 generator."""
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    w = rng.normal(size=d)
    y = np.sin(X @ w) + 0.1 * (X ** 2).sum(1)
    return X, y


def linear_H(X):
    return np.column_stack([np.ones(X.shape[0]), X])


def draw_thetas(B_total, d, y, seed=0):
    """Multistart guesses exactly as Optimize.optimal draws them (_emulatoroptimise.py:206-211):
    row per parameter, uniform in the transformed auto bounds (delta in [1e-3, range=1],
    sigma in [1e-3, sqrt(range y)]), from the global NumPy RNG."""
    np.random.seed(seed)
    bounds = [[0.001, 1.0]] * d + [[0.001, float(np.sqrt(np.amax(y) - np.amin(y)))]]
    tb = 2.0 * np.log(np.array(bounds))
    grid = np.zeros((d + 1, B_total))
    for R in range(d + 1):
        grid[R, :] = tb[R, 0] + (tb[R, 1] - tb[R, 0]) * np.random.random_sample(B_total)
    return np.ascontiguousarray(grid.T)


def bench_config(streams):
    """`config` of the JSON line -- the SAME object for the B200 arm and the reference arm (what differs between
    the arms is said in `impl` and `cpu_baseline.sample`, not here)."""
    return {"workload": "config3: n=4096 d=16 q=17 p=17, gp4ml llh+grad (value + gradient of Optimize.loglikelihood_gp4ml, "
                        "_emulatoroptimise.py:412-493), fixed nugget 1e-4, theta = the multistart draw of _emulatoroptimise.py:206-211 "
                        "from the auto bounds, perturbed each step; 32 guesses per GPU per step (256 over 8 GPUs)",
            "l2": "working set 12.9 GB per step >> 126 MB L2 (inputs larger than L2, no flush needed)",
            "parallelism": "multistart guesses block-partitioned over ranks; one NCCL all_gather of (llh,theta,status) per step",
            "streams": streams}


def flops_llh(n, d, q, p):
    """SURVEY 8(d): F_llh ~ n^3 + n^2 (3d + p + 2q + 4)."""
    return float(n) ** 3 + float(n) ** 2 * (3 * d + p + 2 * q + 4)


def flops_pred(n, d, q):
    """SURVEY 8(d): F_pred ~ n^2 + 2n (d + q + 3)."""
    return float(n) ** 2 + 2.0 * n * (d + q + 3)


def write_emulator_files(workdir, X, y, name, mucm="F", fix_nugget="T", alt_nugget="F", nugget=1e-4, delta=0.5, tries=1,
                         constraints="bounds"):
    """config / beliefs / inputs / outputs text files of a synthetic emulator with a linear mean (the reference's
    on-disk interface, README 'config file' / 'beliefs file')."""
    d = X.shape[1]
    p = lambda f: os.path.join(workdir, f)
    np.savetxt(p(name + "_input"), X, fmt="%.17g")
    np.savetxt(p(name + "_output"), y.reshape(-1, 1), fmt="%.17g")
    with open(p(name + "_beliefs"), "w") as f:
        f.write("active all\noutput 0\nbasis_str 1.0 %s\nbasis_inf NA %s\nbeta %s\n" %
                (" ".join(["x"] * d), " ".join(map(str, range(d))), " ".join(["1.0"] * (d + 1))))
        f.write("delta %s\nsigma 1.0\nnugget %r\nfix_nugget %s\nalt_nugget %s\nmucm %s\n" %
                (" ".join([repr(float(delta))] * d), float(nugget), fix_nugget, alt_nugget, mucm))
    with open(p(name + "_config"), "w") as f:
        f.write("beliefs %s_beliefs\ninputs %s_input\noutputs %s_output\ntv_config 10 0 0\ndelta_bounds [ ]\nsigma_bounds [ ]\n"
                "nugget_bounds [ ]\ntries %d\nconstraints %s\n" % (name, name, name, tries, constraints))
    return name + "_config"


def dump_outputs(outdir, arrays):
    """Write every array as <outdir>/<name>.npy in float64, so that two builds can be compared output for output."""
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, dtype=np.float64))


@contextlib.contextmanager
def quiet_in(workdir):
    old = os.getcwd()
    os.chdir(workdir)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            yield
    finally:
        os.chdir(old)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def fp64_peak():
    p = os.path.join(ROOT, "profiles", "r01_ub_fp64_peaks.json")
    try:
        with open(p) as f:
            j = json.load(f)
        return max(v for k, v in j.items() if k.startswith("dmma884") and isinstance(v, float) and v < 100), "measured (tools/ub_fp64.cu, DMMA.8x8x4)"
    except Exception:
        return FP64_PEAK_FALLBACK_TFLOPS, "fallback"


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        return HBM_PEAK_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ CPU arm
def int8_peak():
    """INT8 tensor-pipe roof for the residue GEMM: twice the measured sustained bf16 rate."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return (2.0 * float(json.load(f)["bf16_tflops_sustained"]),
                    "2 x bf16_tflops_sustained of MEASURED_PEAKS.json (kind::i8 issues at twice the bf16 rate on sm_100a: 4.5 vs 2.25 POP/s nominal)")
    except Exception:
        return 2.0 * 1367.4, "fallback: 2 x 1367.4 TFLOP/s (sustained bf16 of this pool's B200)"


def _blas_info():
    info = {"host_cpus": os.cpu_count(), "usable_cores": _host_cores(), "numpy": np.__version__}
    try:
        import scipy
        info["scipy"] = scipy.__version__
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_info
        pools = threadpool_info()
        info["blas"] = [{k: p_.get(k) for k in ("internal_api", "version", "num_threads", "threading_layer")} for p_ in pools]
        info["threads"] = max([p_.get("num_threads", 1) for p_ in pools] + [1])
    except Exception:
        info["threads"] = _host_cores()
    return info


@contextlib.contextmanager
def all_cores():
    """BLAS pools at every usable host core for the duration (the env fix at the top covers pools created at
    import; this covers a pool that was sized before)."""
    try:
        from threadpoolctl import threadpool_limits
        with threadpool_limits(limits=_host_cores()):
            yield
    except ImportError:
        yield


def cpu_llh_eval(X, y, H, theta, mucm=False):
    """One evaluation of the reference's algorithm (oracle port, NumPy/SciPy/OpenBLAS): seconds."""
    from oracle import gp_oracle as O
    t0 = time.perf_counter()
    res = O.loglikelihood_mucm(theta[:X.shape[1]], X, y, H, 0, 1e-4) if mucm else O.loglikelihood_gp4ml(theta, X, y, H, 0, 1e-4)
    dt = time.perf_counter() - t0
    assert res is not None, "non-PD theta in the CPU leg"
    return dt


def cpu_other_legs():
    """BASELINE.md section 3, items M1 (n = 1000), M2, HM and Sensitivity on the host cores: the oracle port of the
    reference's algorithm on bounded samples.  Returns a dict for `extra.cpu`."""
    from oracle import gp_oracle as O
    from oracle import sens_oracle as SO
    out = {}
    # M1 at config 2's shape: n = 1000, d = 8
    X, y = synth(1000, 8)
    H = linear_H(X)
    th = draw_thetas(4, 8, y)[0]
    th[:8] = 2 * np.log(0.5)
    tg = [cpu_llh_eval(X, y, H, th) for _ in range(3)]
    tm = [cpu_llh_eval(X, y, H, th, mucm=True) for _ in range(3)]
    out["llh_n1000_d8"] = {"gp4ml_s_per_eval_median_of_3": float(np.median(tg)), "mucm_s_per_eval_median_of_3": float(np.median(tm)),
                           "evals_per_s": 1.0 / float(np.median(tg)),
                           "note": "a 64-start llh_optimize needs about 64 x 13 such evaluations one after the other (BASELINE.md section 2)"}
    # M2: g.posterior at n = 2000, d = 8 in m = 1000 chunks (mean + the full m x m covariance: the reference's only API)
    Xp, yp = synth(N_PRED, D_PRED)
    yp2 = np.cos(Xp @ np.random.default_rng(1).normal(size=D_PRED))
    Hp = linear_H(Xp)
    delta = np.full(D_PRED, 0.5)
    A = O.make_A(Xp, delta, 1e-4, 0)
    betas = [O.optimalbeta(A, Hp, yy) for yy in (yp, yp2)]
    rng = np.random.default_rng(7)
    P = (rng.integers(0, 10, size=(5000, D_PRED)) + 0.5) / 10.0          # points of the config-4 grid
    Hs = linear_H(P)
    tp = []
    for c in range(5):
        sl = slice(1000 * c, 1000 * (c + 1))
        t0 = time.perf_counter()
        O.posterior(P[sl], Hs[sl], Xp, yp, Hp, A, betas[0], 1.0, delta, 1e-4, 0)
        tp.append(time.perf_counter() - t0)
    out["posterior_n2000_d8"] = {"preds_per_s": 1000.0 / float(np.median(tp)), "s_per_1000_point_chunk_median_of_5": float(np.median(tp)),
                                 "what": "Posterior.make_covar/make_mean/make_var (_emulatorclasses.py:607-631) per g.posterior call"}
    # HM: the nonimp_data loop (history_match.py:222-250): both emulators' posteriors per chunk + implausibility
    t0 = time.perf_counter()
    mh = 2000
    means, variances = [], []
    for yy, bb in zip((yp, yp2), betas):
        mu, var = O.posterior_diag_chunked(P[:mh], Hs[:mh], Xp, yy, Hp, A, bb, 1.0, delta, 1e-4, 0, chunk=1000)
        means.append(mu); variances.append(var)
    O.implausibility(np.array(means), np.array(variances), [float(np.median(yp)), float(np.median(yp2))], [1e-2, 1e-2], 3.0, 1)
    out["history_match_2_emulators"] = {"points_per_s": mh / (time.perf_counter() - t0), "points": mh}
    # Sensitivity at n = 200, d = 4 (the vectorised port is faster than the reference's Python double loops:
    # BASELINE.md section 2 has 2.7 / 3.3 / 4.5 s for the reference itself at this size)
    Xs_, ys_ = synth(200, 4)
    Hs_ = linear_H(Xs_)
    ds_ = np.full(4, 0.5)
    As_ = O.make_A(Xs_, ds_, 1e-4, 0)
    bs_ = O.optimalbeta(As_, Hs_, ys_)
    t0 = time.perf_counter()
    S = SO.SensOracle(Xs_, ys_, Hs_, As_, bs_, 1.0, 1e-4, ds_, [0.5] * 4, [0.02] * 4)
    tt = {"setup": time.perf_counter() - t0}
    rng_in = [[float(Xs_[:, k].min()), float(Xs_[:, k].max())] for k in range(4)]
    for name, fn in (("uncertainty", S.uncertainty), ("sensitivity", S.sensitivity), ("main_effect", lambda: S.main_effect(rng_in, points=100))):
        t0 = time.perf_counter()
        fn()
        tt[name] = time.perf_counter() - t0
    out["sensitivity_n200_d4_s"] = tt
    return out


def run_reference(args):
    """The reference's own algorithm for the metric's path on the host cores: every timed step is ONE real
    loglikelihood_gp4ml evaluation (value + gradient) at the full n = 4096, d = 16 -- a 1/32 sample of the B200 arm's
    step of 32 guesses, nothing extrapolated.  Warm-up steps run the same code at n = 1024 (they only have to spin
    the BLAS pool up).  --steps timed steps run unless --ref-budget caps the run's wall-clock time; `steps` is what was
    measured."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    t_begin = time.perf_counter()
    K, W = args.steps, args.warmup
    X, y = synth(N_TRAIN, D_IN)
    H = linear_H(X)
    thetas = draw_thetas(B_PER_GPU * max(1, args.gpus), D_IN, y)
    with all_cores():
        info = _blas_info()
        for it in range(W):
            cpu_llh_eval(X[:1024], y[:1024], H[:1024], thetas[it % B_PER_GPU])
        extra_cpu, t_mucm = {}, None
        try:
            extra_cpu = cpu_other_legs()
        except Exception as ex:
            extra_cpu = {"error": repr(ex)}
        times = []
        for it in range(K):
            spent = time.perf_counter() - t_begin
            if args.ref_budget is not None and times and spent + 1.1 * max(times) > args.ref_budget:
                break
            times.append(cpu_llh_eval(X, y, H, thetas[it % B_PER_GPU] + 1e-3 * it))
        spent = time.perf_counter() - t_begin
        if args.ref_budget is None or spent + 1.2 * max(times) < args.ref_budget + 60:      # one full-size MUCM evaluation when it fits
            t_mucm = cpu_llh_eval(X, y, H, thetas[0], mucm=True)
    v = len(times) / float(sum(times))
    extra_cpu["llh_n4096_d16"] = {"gp4ml_s_per_eval": [round(t, 3) for t in times], "gp4ml_s_per_eval_median": float(np.median(times)),
                                  "mucm_s_per_eval": t_mucm}
    cpu = {"value": v, "unit": "evals/s", "cores": int(info["threads"]), "kind": "port",
           "sample": "%d full-size evaluations of loglikelihood_gp4ml (oracle port of _emulatoroptimise.py:412-493), n=4096 d=16, one per step "
                     "(1 of the 32 guesses of the B200 arm's step), %.1f s each; %d warm-up steps at n=1024; nothing extrapolated"
                     % (len(times), float(np.mean(times)), W)}
    cpu.update(info)
    line = {"metric": METRIC, "value": v, "unit": "evals/s", "n_gpus": args.gpus, "steps": len(times), "steps_requested": K, "warmup": W,
            "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference", "config": bench_config(args.streams), "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_begin, "extra": {"cpu": extra_cpu}}
    print(json.dumps(line), file=RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def extra_configs(args, rank, world, local):
    """Driver-run numbers for BASELINE's other configurations through the reference-facing API (N = 1 only for the
    single-emulator ones).  Wall-clock times of whole calls, host work included."""
    import gp_emu_uqsa_b200 as g
    import gp_emu_uqsa_b200.sensitivity as s
    from gp_emu_uqsa_b200 import _lib
    out = {}
    tmp = tempfile.mkdtemp(prefix="gpe_bench_")
    # ---- config 3 as an optimisation: 32 starts per GPU through Optimize.llh_optimize (ragged tail included)
    X, y = synth(N_TRAIN, D_IN)
    with quiet_in(tmp):
        cfg = write_emulator_files(tmp, X, y, "c3", tries=B_PER_GPU * world)
        E = g.setup(cfg, datashuffle=False, scaleinputs=True)
        np.random.seed(0)
        t0 = time.perf_counter()
        E.opt_T.llh_optimize()
        dt = time.perf_counter() - t0
    o = E.opt_T
    out["config3_optimisation"] = {"what": "Optimize.llh_optimize, n=4096 d=16 gp4ml fixed nugget, %d starts (%d per GPU), bounds constraints, "
                                           "batched lock-step L-BFGS-B; first call (no warm-up: workspace allocation and graph capture included)"
                                           % (B_PER_GPU * world, B_PER_GPU),
                                   "seconds": dt, "rounds_this_rank": o.last_rounds, "evals_this_rank": o.last_evals,
                                   "evals_per_s_this_rank": o.last_evals / dt, "best_llh": float(-o.best_llh), "best_guess": int(o.best_guess)}
    dev = E.training.device()
    # ---- steady-state of the other likelihood modes and of small batches at n = 4096 (device-resident theta)
    th = draw_thetas(B_PER_GPU, D_IN, y)
    modes = {"gp4ml_fixed_nugget": (0, th), "mucm_fixed_nugget": (1, th[:, :D_IN]),
             "gp4ml_free_nugget": (4, np.column_stack([th[:, :D_IN], np.full(B_PER_GPU, 2 * np.log(1e-3)), th[:, D_IN]]))}
    ss = {}
    for name, (mode, tt) in modes.items():
        for it in range(4):
            if it == 3:
                t0 = time.perf_counter()
            llh, _, _, st = dev.llh_grad_batch(tt + 1e-3 * it, mode, fixed_nugget=1e-4)
        ms = (time.perf_counter() - t0) * 1e3
        ss[name] = {"ms_per_32": ms, "evals_per_s": B_PER_GPU / ms * 1e3, "all_pd": bool((st == 0).all())}
    out["n4096_steady_state_by_mode"] = ss
    sb = {}
    for Bs in (1, 2, 4, 8):
        ts = []
        for it in range(5):
            t0 = time.perf_counter()
            dev.llh_grad_batch(th[:Bs] + 1e-3 * it, 0, fixed_nugget=1e-4)
            ts.append((time.perf_counter() - t0) * 1e3)
        sb["B=%d" % Bs] = {"ms": float(np.median(ts[2:])), "frac_of_fp64_peak": Bs * flops_llh(N_TRAIN, D_IN, D_IN + 1, D_IN + 1) /
                           (float(np.median(ts[2:])) * 1e-3) * 1e-12 / fp64_peak()[0]}
    out["n4096_small_batches"] = sb
    del E
    if world > 1 or rank != 0:
        return out
    # ---- config 1: examples/toy-sim as shipped (the reference's own example: setup + train + its two plot grids), seed 0
    toy = os.path.join(ROOT, "tests", "golden", "toy-sim")
    if os.path.isdir(toy):
        import shutil
        t1dir = tempfile.mkdtemp(prefix="gpe_bench_toy_")
        for f in os.listdir(toy):
            shutil.copy(os.path.join(toy, f), t1dir)
        best = None
        for rep in range(2):
            with quiet_in(t1dir):
                np.random.seed(0)
                t0 = time.perf_counter()
                E1 = g.setup("toy-sim_config")
                t1 = time.perf_counter()
                g.train(E1)
                t2 = time.perf_counter()
                g.plot(E1, [0], [1], [0.3], "mean")
                g.plot(E1, [0, 1], [2], [0.3], "mean")
                t3 = time.perf_counter()
            best = {"setup_s": t1 - t0, "train_s": t2 - t1, "two_plot_grids_s": t3 - t2, "delta": [float(v) for v in E1.par.delta],
                    "sigma": float(E1.par.sigma), "reference_values": "delta [0.20458, 0.13752], sigma 0.608639 (SURVEY section 4); reference run: 0.71 s"}
        out["config1_toysim_as_shipped"] = best
    # ---- config 2: n = 1000, d = 8, full 64-start optimisation in the four modes
    X2, y2 = synth(1000, 8)
    c2 = {}
    for mucm, fix in (("F", "T"), ("F", "F"), ("T", "T"), ("T", "F")):
        with quiet_in(tmp):
            cfg = write_emulator_files(tmp, X2, y2, "c2_%s%s" % (mucm, fix), mucm=mucm, fix_nugget=fix, tries=64)
            E2 = g.setup(cfg, datashuffle=False, scaleinputs=True)
            np.random.seed(0)
            t0 = time.perf_counter()
            E2.opt_T.llh_optimize()
            cold = time.perf_counter() - t0
            np.random.seed(0)
            t0 = time.perf_counter()
            E2.opt_T.llh_optimize()
            dt = time.perf_counter() - t0
        o = E2.opt_T
        c2["mucm=%s fix_nugget=%s" % (mucm, fix)] = {"seconds": dt, "seconds_first_call": cold, "rounds": o.last_rounds, "evals": o.last_evals,
                                                     "evals_per_s": o.last_evals / dt, "best_llh": float(-o.best_llh), "best_guess": int(o.best_guess)}
    out["config2_optimisation_n1000_d8_64_starts"] = c2
    # ---- config 5: sensitivity at n = 2000, d = 8
    X5, y5 = synth(2000, 8)
    with quiet_in(tmp):
        cfg = write_emulator_files(tmp, X5, y5, "c5")
        E5 = g.setup(cfg, datashuffle=False, scaleinputs=True)
        E5.training.remake(); E5.opt_T.optimalbeta()
        t5 = {}
        for rep in range(2):
            t0 = time.perf_counter(); S = s.setup(E5, [0.5] * 8, [0.02] * 8); t5["setup"] = time.perf_counter() - t0
            t0 = time.perf_counter(); S.uncertainty(); t5["uncertainty"] = time.perf_counter() - t0
            t0 = time.perf_counter(); S.sensitivity(); t5["sensitivity"] = time.perf_counter() - t0
            t0 = time.perf_counter(); S.main_effect(points=100); t5["main_effect_100_points"] = time.perf_counter() - t0
    out["config5_sensitivity_n2000_d8_s"] = t5
    # ---- config 5: noise fit, noisefit2D generator at n = 2000
    if not args.no_noisefit:
        import gp_emu_uqsa_b200.noise_fit as gn
        nf = tempfile.mkdtemp(prefix="gpe_bench_nf_")
        with quiet_in(nf):
            np.random.seed(1)
            x = np.random.rand(2000, 2)
            mean = 3.0 * x[:, 0] ** 3 + np.exp(np.cos(10.0 * x[:, 1]) * np.cos(5.0 * x[:, 0]) ** 2)
            noise = np.abs(0.5 * (x[:, 1] * (np.cos(6 * x[:, 0]) ** 2 + 0.1)))
            np.savetxt("INPUTS", x)
            np.savetxt("OUTPUTS", mean + noise * np.random.randn(2000))
            for name, outputs, alt, cons, db, sbd, nb in (("data", "OUTPUTS", "T", "none", "[[0.05,10.0],[0.05,10.00]]", "[[0.1,3.0]]", "[[0.001,1.05]]"),
                                                         ("noise", "zp-outputs", "F", "bounds", "[[0.05,1.0],[0.05,10.00]]", "[[0.001,10.0]]", "[[0.0001,1.0]]")):
                with open("config-" + name, "w") as f:
                    f.write("beliefs beliefs-%s\ninputs INPUTS\noutputs %s\ntv_config 10 0 0\ndelta_bounds %s\nsigma_bounds %s\n"
                            "nugget_bounds %s\ntries 3\nconstraints %s\n" % (name, outputs, db, sbd, nb, cons))
                with open("beliefs-" + name, "w") as f:
                    f.write("active all\noutput 0\nbasis_str 1.0\nbasis_inf NA\nbeta 1.0\ndelta 1.0 1.0\nsigma 1.0\nnugget 0.00001\n"
                            "fix_nugget F\nalt_nugget %s\nmucm F\n" % alt)
            t0 = time.perf_counter()
            gn.noisefit("config-data", "config-noise", stopat=2, olhcmult=100, samples=200)
            dt = time.perf_counter() - t0
            fit = np.loadtxt("noise-outputs")
            xin = np.loadtxt("noise-inputs")
        true = np.abs(0.5 * (xin[:, 1] * (np.cos(6 * xin[:, 0]) ** 2 + 0.1)))
        out["config5_noisefit_n2000"] = {"seconds": dt, "corr_fit_vs_true_noise": float(np.corrcoef(fit[:, 0], true)[0, 1]),
                                         "what": "noisefit(stopat=2, samples=200): five g.train calls, four 2000x2000 posterior covariances + Cholesky factors"}
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from gp_emu_uqsa_b200 import _dist, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    K, W = args.steps, args.warmup
    n, d, B = N_TRAIN, D_IN, B_PER_GPU
    q, p = d + 1, d + 1

    X, y = synth(n, d)
    H = linear_H(X)
    thetas_all = draw_thetas(B * world, d, y)                 # every rank draws the same global list
    theta_rank = thetas_all[rank * B:(rank + 1) * B].copy()   # block partition of the guess index (SURVEY 8e)

    dev = _lib.Device(local)
    dev.set_streams(args.streams)
    dev.set_training(X, y, H)
    stream = torch.cuda.ExternalStream(dev.stream_ptr, device=torch.device("cuda", local))

    th_d = torch.tensor(theta_rank, device="cuda")
    llh_d = torch.empty(B, dtype=torch.float64, device="cuda")
    grad_d = torch.empty(B, p, dtype=torch.float64, device="cuda")
    sig_d = torch.empty(B, dtype=torch.float64, device="cuda")
    st_d = torch.zeros(B, dtype=torch.int32, device="cuda")
    gather = [torch.empty(B, p + 2, dtype=torch.float64, device="cuda") for _ in range(world)] if world > 1 else None

    def step_device(it):
        th = th_d + 1e-3 * it
        torch.cuda.current_stream().synchronize()
        dev.llh_grad_batch(th, 0, fixed_nugget=1e-4, out=(llh_d, grad_d, sig_d, st_d))
        if world > 1:      # the path's only exchange: gather (llh, theta, status) for the global argmin
            pack = torch.cat([llh_d[:, None], th, st_d.double()[:, None]], dim=1)
            dist.all_gather(gather, pack)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for it in range(W):
        step_device(it)
    barrier()
    assert int(st_d.abs().sum().item()) == 0, "non-PD item in the benchmark batch"
    clocks = ClockSampler(local)
    clocks.start()
    l0 = dev.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for it in range(K):
        step_device(W + it)
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = dev.launches - l0
    # what the last timed step returned, taken before the passes below reuse the buffers: every rank's block of guesses,
    # gathered in guess order
    dumped = None
    if args.dump_outputs:
        mine = torch.cat([llh_d[:, None], grad_d, sig_d[:, None], st_d.double()[:, None]], dim=1)
        blocks = [mine]
        if world > 1:
            blocks = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(blocks, mine)
        step = torch.cat(blocks).cpu().numpy()
        dumped = {"llh": step[:, 0], "grad": step[:, 1:p + 1], "sigma_hat": step[:, p + 1], "status": step[:, p + 2]}
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = B * world * K / (ms_max * 1e-3)

    # ---- e2e: the same step through the public call with HOST buffers (pinned), copies inside
    th_h = torch.empty(B, p, dtype=torch.float64).pin_memory()
    llh_h = torch.empty(B, dtype=torch.float64).pin_memory()
    grad_h = torch.empty(B, p, dtype=torch.float64).pin_memory()
    sig_h = torch.empty(B, dtype=torch.float64).pin_memory()
    st_h = torch.zeros(B, dtype=torch.int32).pin_memory()
    th_np, llh_np, grad_np, sig_np, st_np = (a.numpy() for a in (th_h, llh_h, grad_h, sig_h, st_h))
    Ke = max(2, min(K, 5))
    barrier()
    t0 = time.perf_counter()
    for it in range(Ke):
        th_np[:] = theta_rank + 1e-3 * (W + K + it)
        dev.llh_grad_batch(th_np, 0, fixed_nugget=1e-4, out=(llh_np, grad_np, sig_np, st_np))
        best = float(llh_np.min())          # device->host read of the step's result
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = B * world * Ke / float(te.item())
    clk = clocks.stop()

    # ---- per-kernel CUDA-event timing: the same step with the sub-batch streams switched off, so that
    # every launch runs alone on the handle's stream and its event pair measures that kernel only
    dev.set_streams(1)
    Kp_ = max(2, min(K, 3))
    step_device(W + K)
    barrier()
    dev.profile_enable(True)
    dev.profile_read(reset=True)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for it in range(Kp_):
        step_device(W + K + 1 + it)
    s1.record(stream)
    barrier()
    serial_ms = s0.elapsed_time(s1) / Kp_
    prof = dev.profile_read(reset=True)
    dev.profile_enable(False)
    dev.set_streams(args.streams)

    # ---- posterior predictions/sec over the config-4 grid (10 levels^8 = 10^8 points): the flat index is cut into
    # equal tile-aligned ranges, one per rank (cells of the history-matching statistics may straddle ranks); mean +
    # diagonal variance kept in HBM; then the history-matching pass over two emulators (implausibility, keep mask,
    # per-(dim0,dim1)-cell min and counts, all-reduce of the cell statistics)
    extra = {}
    try:
        Xp, yp = synth(N_PRED, D_PRED)
        rng2 = np.random.default_rng(1)
        yp2 = np.cos(Xp @ rng2.normal(size=D_PRED))
        levels = np.full(D_PRED, 10, dtype=np.int32)
        lo, hi = np.zeros(D_PRED), np.ones(D_PRED)
        total = int(args.grid_points)
        ncell_all = 100
        cell_pts = total // ncell_all
        start, stop = _dist.block_aligned(total, rank, world)
        m = stop - start
        devs = []
        for yy in (yp, yp2):
            dv = _lib.Device(local)
            dv.set_training(Xp, yy, linear_H(Xp))
            dv.set_basis(list(range(D_PRED)), [1] * D_PRED)
            dv.fit_state(np.full(D_PRED, 0.5), 1e-4, 1.0, 0)
            devs.append(dv)
        devp = devs[0]
        mean_d = torch.empty((1, m), dtype=torch.float64, device="cuda")
        var_d = torch.empty((1, m), dtype=torch.float64, device="cuda")
        pstream = torch.cuda.ExternalStream(devp.stream_ptr, device=torch.device("cuda", local))
        warm = min(m, 1 << 18)
        for it in range(3):
            devp.predict_grid(levels, lo, hi, start, warm, out=(mean_d[0, :warm], var_d[0, :warm]))
        barrier()
        lp0 = devp.launches
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(pstream)
        devp.predict_grid(levels, lo, hi, start, m, out=(mean_d[0], var_d[0]))
        p1.record(pstream)
        barrier()
        pred_launches = devp.launches - lp0
        if dumped is not None and m:      # a fixed sample of the shard's points (flat grid indices kept beside the values)
            pick = np.sort(np.random.default_rng(0).choice(m, size=min(m, DUMP_PRED_POINTS), replace=False))
            pick_d = torch.from_numpy(pick).cuda()
            dumped.update(posterior_index=start + pick, posterior_mean=mean_d[0, pick_d].cpu().numpy(),
                          posterior_var=var_d[0, pick_d].cpu().numpy())
        pms = torch.tensor([p0.elapsed_time(p1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(pms, op=dist.ReduceOp.MAX)
        preds = float(total) / (float(pms.item()) * 1e-3)
        # per-kernel event timing: a separate pass over a slice with serial launches (profiling switches the
        # two-stream chunk overlap off so that each event pair brackets one kernel)
        mprof = min(m, 1 << 22)
        devp.profile_enable(True); devp.profile_read(reset=True)
        devp.predict_grid(levels, lo, hi, start, mprof, out=(mean_d[0, :mprof], var_d[0, :mprof]))
        pprof = devp.profile_read(reset=True)
        devp.profile_enable(False)
        # history matching over the same shard, complete pass: both emulators are predicted with their implausibility folded
        # into a running per-point list (gpe_predict_implaus: no mean / variance arrays), the second pass also writes the keep
        # mask and reduces the count and the per-(dim0,dim1)-cell minima / counts
        barrier()
        t0 = time.perf_counter()
        zs = [float(np.median(yp)), float(np.median(yp2))]
        Itop = torch.empty((m, 1), dtype=torch.float64, device="cuda")
        keep_d = torch.empty(m, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        devs[0].predict_implaus(zs[0], 1e-2, Itop, first=True, last=False, grid=(levels, lo, hi, start, m), maxno=1)
        cnt, cmin, ccnt = devs[1].predict_implaus(zs[1], 1e-2, Itop, first=False, last=True, grid=(levels, lo, hi, start, m), maxno=1,
                                                  cm=3.0, cell_pts=cell_pts, first_index=start, keep=keep_d)
        cmin_all = np.full(ncell_all, np.inf)
        ccnt_all = np.zeros(ncell_all + 1, dtype=np.int64)
        c0 = start // cell_pts
        if m:
            cmin_all[c0:c0 + cmin.shape[0]] = cmin[:, 0]
            ccnt_all[c0:c0 + ccnt.shape[0]] = ccnt[:, 0].astype(np.int64)
        ccnt_all[ncell_all] = int(cnt[0])
        if world > 1:      # the path's exchange: all-reduce(min) of the cell minima, all-reduce(sum) of the counts
            tmin = torch.from_numpy(cmin_all).cuda()
            tcnt = torch.from_numpy(ccnt_all).cuda()
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            dist.all_reduce(tcnt, op=dist.ReduceOp.SUM)
            cmin_all, ccnt_all = tmin.cpu().numpy(), tcnt.cpu().numpy()
        torch.cuda.synchronize()
        hm_s = time.perf_counter() - t0
        th = torch.tensor([hm_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(th, op=dist.ReduceOp.MAX)
        # e2e: a slice of the shard through the call with HOST output buffers
        me = min(m, 1 << 22)
        mean_h = np.empty(me); var_h = np.empty(me)
        barrier()
        t0 = time.perf_counter()
        devp.predict_grid(levels, lo, hi, start, me, out=(mean_h, var_h))
        pe = time.perf_counter() - t0
        peak, peak_src = fp64_peak()
        hbm, hbm_src = hbm_peak()
        fpp = flops_pred(N_PRED, D_PRED, D_PRED + 1)
        gms, gcnt = pprof["gemm_dmma_128"]
        i8ms, i8cnt = pprof["int8_residue_gemm"]
        p_int8 = None
        if i8cnt:        # chunks of 1024 points and more over 1024 and more padded training points: the product runs on the INT8 route
            p_nmod = int(os.environ.get("GPE_OZAKI", "16"))
            i8_peak, i8_src = int8_peak()
            i8_ach = p_nmod * float(mprof) * float(N_PRED) ** 2 / (i8ms * 1e-3) * 1e-12
            p_int8 = {"kernel": "oz_gemm_kernel<2> (residue GEMM of Z^T = C^T L^-T, k <= j: TMA, two-CTA multicast clusters, tcgen05.mma kind::i8, "
                                "mod-p epilogue): %d launches" % i8cnt,
                      "bound": "tensor", "unit": "TOP/s", "achieved": i8_ach, "peak": i8_peak, "frac": i8_ach / i8_peak, "peak_source": i8_src,
                      "moduli": p_nmod, "algorithmic": "moduli x n^2 ops per point (the triangular product's FP64 flops)",
                      "ms": i8ms, "residue_conversion_ms": pprof["int8_residue_conversion"][0],
                      "crt_column_norms_ms": pprof["int8_crt_combine"][0]}
        ptraffic = {}
        for tp in ("r02_traffic.json", "r01_traffic.json"):
            tp = os.path.join(ROOT, "profiles", tp)
            if os.path.exists(tp):
                with open(tp) as f:
                    ptraffic = json.load(f)
                break
        cov_ms, cov_cnt = pprof["cov_build"]
        extra = {"posterior_preds_per_s": preds,
                 "posterior_workload": "config4: n=2000 d=8 q=9, %.0e-point tensor grid (10 levels/dim) generated on device from the flat "
                                       "index, cut into %d equal tile-aligned index ranges (one per GPU), mean + diagonal variance written "
                                       "to HBM (%.2f GB per GPU)" % (total, world, 16.0 * m / 1e9),
                 "posterior_ms": float(pms.item()), "posterior_gpu_launches": int(pred_launches),
                 "posterior_e2e_preds_per_s": me * world / pe, "posterior_d2h_bytes_per_pred": 16,
                 "posterior_roofline": {"bound": "tensor", "achieved": preds / world * fpp * 1e-12, "peak": peak,
                                        "unit": "TFLOP/s", "frac": preds / world * fpp * 1e-12 / peak,
                                        "what": "FP64-equivalent: F_pred x preds/s per GPU against the measured FP64 DMMA roof" +
                                                (" -- above 1 because Z = L^-1 C runs as exact INT8 residue GEMMs on the tcgen05 tensor cores "
                                                 "(dominant_kernel carries that kernel's own INT8 roofline)" if p_int8 else ""),
                                        "kernel": "oz_convert_t_kernel + oz_gemm_kernel<2> + oz_combine_rowsumsq_kernel (Z^T = C^T L^-T by residues, row norms in the CRT pass)" if p_int8
                                                  else "gemm_dmma_ws_kernel<NN, EPI_SUMSQ> (Z = L^-1 C with fused column norms)",
                                        "kernel_achieved": ((float(mprof) * float(N_PRED) ** 2 * 1e-12) / (gms * 1e-3) if gms else None) if not p_int8 else
                                                           (float(mprof) * float(N_PRED) ** 2 * 1e-12) / ((i8ms + pprof["int8_residue_conversion"][0] + pprof["int8_crt_combine"][0]) * 1e-3),
                                        "kernel_launches": gcnt if not p_int8 else i8cnt,
                                        "dominant_kernel": p_int8,
                                        "traffic": ptraffic.get("pred_oz_gemm_dram_bytes_per_launch" if p_int8 else "trmm_dram_bytes_per_launch"),
                                        "algorithmic_bytes_per_point": 16,
                                        "by_kernel_ms": {k: v[0] for k, v in pprof.items()},
                                        "cross_covariance": {"ms": cov_ms, "launches": cov_cnt,
                                                             "tflops_alu": mprof * float(N_PRED) * (3 * D_PRED + 1) / (cov_ms * 1e-3) * 1e-12 if cov_ms else None,
                                                             "note": "FP64 ALU + exp work (n (3d + exp) flops per point), not tensor-pipe work"},
                                        "note": "achieved = F_pred (n^2 + 2n(d+q+3)) x preds/s per GPU; kernel_achieved = n^2 flops per "
                                                "point / CUDA-event time of the launches that evaluate Z and its column norms (DMMA: the TRMM; INT8: "
                                                "conversion + residue GEMM + CRT) in a separate serial-launch pass over %d points" % mprof},
                 "history_match": {"points_per_s": float(total) / float(th.item()),
                                   "workload": "complete history-matching pass: 2 emulators predicted over the grid with the implausibility "
                                               "folded into the prediction (cm=3, maxno=1): keep mask, count and per-cell min / count over the "
                                               "10x10 (dim0,dim1) cells; all-reduce(min / sum) of cell statistics; 17 B/point of HBM traffic "
                                               "(8 written + 8 read for the running list, 1 for the mask)",
                                   "emulator_points_per_s": 2.0 * float(total) / float(th.item()),
                                   "non_implausible": int(ccnt_all[ncell_all]), "cells_sum_check": int(ccnt_all[:ncell_all].sum()),
                                   "min_cell_implausibility": float(cmin_all.min()), "seconds": float(th.item())}}
        for dv in devs:
            dv.close()
        del mean_d, var_d
        torch.cuda.empty_cache()
    except Exception as ex:      # the headline metric must still print
        import traceback
        extra = {"posterior_error": repr(ex), "trace": traceback.format_exc()[-600:]}

    dev.close()
    torch.cuda.empty_cache()
    if not args.no_extra:
        try:
            extra.update(extra_configs(args, rank, world, local))
        except BaseException as ex:
            import traceback
            extra["extra_configs_error"] = repr(ex) + " | " + traceback.format_exc()[-600:]

    if rank == 0:
        peak, peak_src = fp64_peak()
        hbm, hbm_src = hbm_peak()
        F = flops_llh(n, d, q, p)
        gemm_ms, gemm_cnt = prof["gemm_dmma_128"]
        lau_ms, lau_cnt = prof["lauum"]
        # dominant kernel: the LAUUM launch (A^-1 = L^-T L^-1, with the gradient reduction in its epilogue): algorithmic n^3/3 flops per item
        lau_flops = B * float(n) ** 3 / 3.0
        kern_ach = lau_flops * lau_cnt / (lau_ms * 1e-3) * 1e-12 if lau_ms else None
        fam_flops = B * float(n) ** 3                       # potrf + trtri + lauum, all DMMA launches of a step
        fam_ms = gemm_ms + lau_ms
        fam_ach = fam_flops * Kp_ / (fam_ms * 1e-3) * 1e-12 if fam_ms else None
        traffic = None
        for tp in ("r02_traffic.json", "r01_traffic.json"):
            tp = os.path.join(ROOT, "profiles", tp)
            if os.path.exists(tp):
                with open(tp) as f:
                    traffic = json.load(f).get("lauum_dram_bytes_per_launch")
                break
        step_ach = B * F / (ms_max / K * 1e-3) * 1e-12
        # streaming kernels (north_star: achieved HBM GB/s for the covariance build; FP64-ALU share beside it)
        npad = (n + 127) // 128 * 128
        streaming = {}
        cov_ms, cov_cnt = prof["cov_build"]
        # the covariance build also keeps E = exp(-D) for the gradient (the LAUUM epilogue on the DMMA route, the stand-alone
        # reduction on the INT8 route unless GPE_GRAD_E=0)
        e_copy = npad >= 1024 and not (prof["int8_residue_gemm"][1] and os.environ.get("GPE_GRAD_E", "1") == "0")
        if cov_ms:
            byt = B * Kp_ * (16.0 if e_copy else 8.0) * (npad * (npad + 64) / 2.0)             # lower 64x64 tiles written once
            flo = B * Kp_ * (n * n / 2.0) * (3 * d + 1)
            streaming["cov_build"] = {"ms_per_step": cov_ms / Kp_, "hbm_GBps": byt / (cov_ms * 1e-3) * 1e-9, "frac_of_hbm": byt / (cov_ms * 1e-3) * 1e-9 / hbm,
                                      "fp64_alu_TFLOPs": flo / (cov_ms * 1e-3) * 1e-12, "frac_of_fp64": flo / (cov_ms * 1e-3) * 1e-12 / peak,
                                      "algorithmic": "%d B x n^2/2 written (A%s), (n^2/2)(3d + exp) flops per item" % (16 if e_copy else 8, " and E = exp(-D)" if e_copy else "")}
        gr_ms, gr_cnt = prof["grad_reduce"]
        if gr_ms:
            byt = B * Kp_ * (16.0 if e_copy else 8.0) * (n * n / 2.0)
            flo = B * Kp_ * (n * n / 2.0) * ((3 * d + 2 * q) if e_copy else (5 * d + 2 * q + 1))
            streaming["grad_reduce"] = {"ms_per_step": gr_ms / Kp_, "hbm_GBps": byt / (gr_ms * 1e-3) * 1e-9, "frac_of_hbm": byt / (gr_ms * 1e-3) * 1e-9 / hbm,
                                        "fp64_alu_TFLOPs": flo / (gr_ms * 1e-3) * 1e-12, "frac_of_fp64": flo / (gr_ms * 1e-3) * 1e-12 / peak,
                                        "algorithmic": ("16 B x n^2/2 read (A^-1 and E), (n^2/2)(3d + 2q) flops per item" if e_copy else
                                                        "8 B x n^2/2 read, (n^2/2)(5d + 2q + exp) flops per item")}
        # ---- the INT8 tensor-core route (default): the large products of the factorisation and LAUUM run as residue GEMMs on
        # tcgen05.mma kind::i8 (csrc/gpe_ozaki.cuh); the dominant kernel of the step is then oz_gemm_kernel
        oz_ms, oz_cnt = prof["int8_residue_gemm"]
        cv_ms, cv_cnt = prof["int8_residue_conversion"]
        cb_ms, cb_cnt = prof["int8_crt_combine"]
        nmod = int(os.environ.get("GPE_OZAKI", "16"))
        oz_min = int(os.environ.get("GPE_OZAKI_MIN", "1024"))
        int8 = None
        if oz_cnt:
            def takes(M, N, K):
                return min(M, N, K) >= oz_min and M % 128 == 0 and N % 256 == 0 and K % 128 == 0

            def rec(m):          # algorithmic FP64 flops of the products of potrf_inv_rec that take the INT8 route
                if m <= 128:
                    return 0.0
                m1 = ((m // 128 + 1) // 2) * 128
                m2 = m - m1
                f = 0.0
                for (M_, N_, K_) in ((m2, m1, m1), (m2, m1, m1), (m2, m2, m1), (m2, m1, m2)):   # each has one triangular factor: M N K flops
                    if takes(M_, N_, K_):
                        f += float(M_) * N_ * K_
                return f + rec(m1) + rec(m2)
            f64_flops = rec(npad) + (float(npad) ** 3 / 3.0 if takes(npad, npad, npad) else 0.0)
            i8_ops = B * nmod * f64_flops                       # one u8 x u8 -> s32 product per modulus
            i8_peak, i8_src = int8_peak()
            i8_ach = i8_ops * Kp_ / (oz_ms * 1e-3) * 1e-12
            i8_traffic = None
            tp = os.path.join(ROOT, "profiles", "r02_traffic_int8.json")
            if os.path.exists(tp):
                with open(tp) as f:
                    i8_traffic = json.load(f)
            int8 = {"kernel": "oz_gemm_kernel<2> (residue GEMM: TMA 128B-swizzled tiles, two-CTA multicast clusters, tcgen05.mma kind::i8, "
                              "TMEM double-buffered accumulator, mod-p epilogue): %d launches per step" % (oz_cnt // Kp_),
                    "bound": "tensor", "unit": "TOP/s", "achieved": i8_ach, "peak": i8_peak, "frac": i8_ach / i8_peak,
                    "peak_source": i8_src,
                    "issue_rate_microbenchmark_TOPs": 4300.0,
                    "issue_rate_source": "profiles/r01_ub_i8_umma.json (tcgen05.mma kind::i8, resident operands, 148 CTAs)",
                    "algorithmic_ops_per_step": i8_ops, "moduli": nmod,
                    "algorithmic": "moduli x FP64 flops of the products it replaces (M N K per triangular product, n^3/3 for LAUUM)",
                    "ms_per_step": oz_ms / Kp_, "traffic": i8_traffic,
                    "residue_conversion_ms_per_step": cv_ms / Kp_, "crt_combine_ms_per_step": cb_ms / Kp_}
        line = {
            "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "b200",
            "config": bench_config(args.streams),
            "gpu_launches": int(launches),
            "clocks": {"sm_mhz": clk["sm_mhz"], "sm_max_mhz": clk["sm_max_mhz"], "reasons": clk["reasons"], "samples": clk["samples"]},
            "e2e": {"value": e2e_val, "unit": "evals/s", "h2d_bytes_per_step": int(B * p * 8),
                    "d2h_bytes_per_step": int(B * (p + 2) * 8 + B * 4), "steps": Ke},
            "roofline": {"bound": "tensor", "achieved": step_ach, "peak": peak, "unit": "TFLOP/s", "frac": step_ach / peak,
                         "what": "the whole llh+grad step in FP64-equivalent terms: 32 x F_llh (n^3 + n^2(3d+p+2q+4)) algorithmic flops / ms_per_step "
                                 "of the timed region, against the measured FP64 DMMA roof" +
                                 (" -- above 1 because the large products run as %d exact INT8 residue GEMMs each on the tcgen05 tensor cores "
                                  "(dominant_kernel below carries that kernel's own INT8 roofline)" % nmod if int8 else ""),
                         "traffic": (int8["traffic"].get("oz_gemm_dram_bytes_per_launch") if int8 and int8["traffic"] else traffic),
                         "peak_source": peak_src + "; MEASURED_PEAKS.json holds no FP64 figure",
                         "dominant_kernel": int8 if int8 else
                                            {"kernel": "lauum_grad_kernel / gemm_dmma_ws_kernel<TN> LAUUM launch (A^-1 = L^-T L^-1, %d items, lower 128x128 tiles)" % B,
                                             "achieved": kern_ach, "frac": (kern_ach / peak) if kern_ach else None,
                                             "algorithmic_flops_per_launch": lau_flops, "algorithmic_bytes_per_launch": B * 8.0 * n * n,
                                             "ms_per_launch": lau_ms / lau_cnt if lau_cnt else None},
                         "kernel_timing": "CUDA-event pair around every launch, measured live in this run in a separate pass of %d steps "
                                          "with the sub-batch streams off (serial launches, %.2f ms/step); the timed region runs %s "
                                          "concurrent sub-batch streams" % (Kp_, serial_ms, "2 (INT8 route)" if int8 else str(args.streams)),
                         "dmma_family": {"what": "all 128x128-tile DMMA launches of a step (on the INT8 route: the levels below %d only)" % oz_min,
                                         "achieved": fam_ach if not int8 else None, "frac": (fam_ach / peak if fam_ach else None) if not int8 else None,
                                         "ms_per_step": fam_ms / Kp_, "launches_per_step": (gemm_cnt + lau_cnt) / Kp_},
                         "step_achieved": step_ach, "step_frac": step_ach / peak,
                         "streaming_kernels": streaming, "hbm_peak_GBps": hbm, "hbm_peak_source": hbm_src,
                         "by_kernel_ms_per_step": {k: v[0] / Kp_ for k, v in prof.items()}},
            "extra": extra,
        }
        if world == 1 and not args.no_cpu:
            with all_cores():
                info = _blas_info()
                thetas = draw_thetas(B, d, y)
                cpu_llh_eval(X[:1024], y[:1024], H[:1024], thetas[0])          # BLAS pool warm-up
                t1 = cpu_llh_eval(X, y, H, thetas[0])
                cpu = {"value": 1.0 / t1, "unit": "evals/s", "cores": int(info["threads"]), "kind": "port",
                       "sample": "1 full-size evaluation of loglikelihood_gp4ml (oracle port of _emulatoroptimise.py:412-493), n=4096 d=16, "
                                 "%.1f s; nothing extrapolated (the --impl reference arm times one per step)" % t1}
                cpu.update(info)
                line["cpu_baseline"] = cpu
                try:
                    line["extra"]["cpu"] = cpu_other_legs()
                except Exception as ex:
                    line["extra"]["cpu"] = {"error": repr(ex)}
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _private_stdout():
    """Library chatter on fd 1 (e.g. NCCL's version banner) must not mix with the ONE JSON line:
    keep a private copy of stdout for the result and point fd 1 at stderr for everything else."""
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(keep, "w")


def main():
    global RESULT_OUT
    RESULT_OUT = _private_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 2 / 3-as-optimisation / 5 legs")
    ap.add_argument("--no-noisefit", action="store_true", help="skip the noise-fit leg of config 5")
    ap.add_argument("--ref-budget", type=float, default=None,
                    help="optional wall-clock cap (s) of the --impl reference run; when given it overrides --steps: timed full-size "
                         "evaluations (about 41 s each on 16 host cores) stop before the cap is passed")
    ap.add_argument("--streams", type=int, default=8, help="concurrent sub-batch streams of gpe_llh_grad_batch")
    ap.add_argument("--grid-points", type=float, default=1e8, help="size of the prediction grid (config 4: 1e8)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (llh, grad, sigma_hat, status of every guess of the step, all "
                         "ranks gathered in guess order) and the posterior mean / variance of a fixed sample of %d grid points with "
                         "their flat indices (under N > 1: of rank 0's shard) as DIR/<name>.npy (float64)" % DUMP_PRED_POINTS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
