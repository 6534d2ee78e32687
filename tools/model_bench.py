"""RK4 step time of the linear, lossy and Westervelt models (DESIGN.md section 4.5a) at the benchmark workload
(64^3 perturbed cells, P4, fp64) and at the same mesh in fp32.

    python tools/model_bench.py [--out DIR] [--windows 7] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU: the three models on the same mesh, each stepped from the same random state with
CUDA-graph replay; timing windows of --steps-per-window steps (one rk4 call each) alternate between the models
(linear, lossy, Westervelt, linear, ...) so that they share the card's state; the median window is reported.
In the run, WesterveltGLLOpt(delta = beta = 0) is checked against LinearGLLOpt bit for bit over 5 steps.

Algorithmic bytes of one RK4 step (s = scalar size, n = dofs): 4 stiffness applies (StiffnessOperator.info()
bytes each) plus the vector passes of the fused stage kernels, VECTOR_PASSES[model] * s * n:
  linear      39  (stages 0..3: 10 + 11 + 11 + 7)
  lossy       40  (stage 3 also writes w = u + s v for the next step)
  westervelt  43  (stages 1..3 read w to rebuild p = w - s vn)
The compact Gamma2 kernel (boundary dofs only) and the w = u + s v pass at the entry of every rk4 call (3 s n per
call, amortised over the window) are not counted.  Share of the HBM peak bench.py uses (bench.measured_peak()).
Writes DIR/models_<config>.json and prints a summary.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

CONFIGS = {"p4_fp64": dict(P=4, cells=64, dtype="float64"), "p4_fp32": dict(P=4, cells=64, dtype="float32")}
VECTOR_PASSES = {"linear": 39, "lossy": 40, "westervelt": 43}
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 4.33e-6, 3.5, 1000.0   # water


def step_bytes(model, apply_bytes, n, s):
    return 4 * apply_bytes + VECTOR_PASSES[model] * s * n


def run_config(name, cfg, args, torch, wfx, peak):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    s = dtype.itemsize
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    t0 = time.perf_counter()
    models = {"linear": wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype),
              "lossy": wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, DELTA, dtype=dtype),
              "westervelt": wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype)}
    setup_s = time.perf_counter() - t0
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    rng = np.random.default_rng(1)
    u0 = (P0 * rng.standard_normal(n)).astype(dtype)
    v0 = (P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    apply_bytes = models["linear"].stiff_op.info()["bytes"]
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15,
           "dt": dt, "delta": DELTA, "beta": BETA, "rho0": RHO0, "setup_s": setup_s,
           "kernel": models["linear"].stiff_op.kernel_info()["variant"], "windows": args.windows,
           "steps_per_window": args.steps_per_window, "hbm_peak_gbs": peak[0], "hbm_peak_source": peak[1],
           "apply_bytes": apply_bytes}

    # in-run check: delta = beta = 0 is the linear model bit for bit
    zero = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, 0.0, 0.0, 1.0, dtype=dtype)
    states = []
    for eqn in (models["linear"], zero):
        eqn.set_state(u0, v0)
        eqn.rk4(0.0, 1.0, dt, max_steps=5)
        states.append(eqn.get_state())
    res["zero_delta_beta_bitwise_linear"] = bool(np.array_equal(states[0][0], states[1][0])
                                                 and np.array_equal(states[0][1], states[1][1]))
    del zero, states
    torch.cuda.empty_cache()

    t_now = {}
    for k, eqn in models.items():
        eqn.set_state(u0, v0)
        t_now[k] = 0.0
        for _ in range(2):   # warm-up: graph capture and first replays
            t_now[k] = eqn.rk4(t_now[k], 1.0, dt, max_steps=args.steps_per_window)[1]
    torch.cuda.synchronize()
    win = {k: [] for k in models}
    for _ in range(args.windows):
        for k, eqn in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t_now[k] = eqn.rk4(t_now[k], 1.0, dt, max_steps=args.steps_per_window)[1]
            e1.record()
            e1.synchronize()
            win[k].append(e0.elapsed_time(e1) / args.steps_per_window)
    for k, eqn in models.items():
        u, v = eqn.get_state()
        ms = float(np.median(win[k]))
        nbytes = step_bytes(k, apply_bytes, n, s)
        res[k] = {"ms_per_step": ms, "windows_ms": win[k], "bytes_per_step": nbytes,
                  "achieved_gbs": nbytes / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak[0],
                  "finite": bool(np.isfinite(u).all() and np.isfinite(v).all())}
    for k in ("lossy", "westervelt"):
        res[k]["over_linear"] = res[k]["ms_per_step"] / res["linear"]["ms_per_step"] - 1.0
        res[k]["over_linear_per_window"] = [a / b - 1.0 for a, b in zip(win[k], win["linear"])]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--steps-per-window", type=int, default=20)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if args.windows < 5 or args.steps_per_window < 10:
        raise SystemExit("model_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("model_bench: no CUDA device")
    import wave_fenics_b200 as wfx
    import bench
    from ensemble_bench import card
    peak = bench.measured_peak()
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    gpu["torch_name"] = torch.cuda.get_device_name(0)
    ok = True
    for name in args.configs.split(","):
        r = run_config(name, CONFIGS[name], args, torch, wfx, peak)
        r["gpu"] = gpu
        with open(os.path.join(args.out, f"models_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        ok = ok and r["zero_delta_beta_bitwise_linear"] and all(r[k]["finite"] for k in VECTOR_PASSES)
        print(f"{name} ({r['ndofs']} dofs, {gpu.get('name')}, {gpu.get('power_limit')}): "
              f"delta=beta=0 bitwise linear: {r['zero_delta_beta_bitwise_linear']}")
        for k in VECTOR_PASSES:
            e = r[k]
            extra = f", {100 * e['over_linear']:+.2f} % over linear" if "over_linear" in e else ""
            print(f"  {k:10s} {e['ms_per_step']:.4f} ms/step, {e['frac_of_hbm_peak']:.3f} of peak{extra}")
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("model_bench: a check failed")


if __name__ == "__main__":
    main()
