"""RK4 step time with and without a source profile (DESIGN.md section 4.5c) for the linear and Westervelt models at
the benchmark workload (64^3 perturbed cells, P4) in fp64 and fp32.

    python tools/source_profile_bench.py [--out DIR] [--windows 7] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU: four models on the same mesh (linear and Westervelt, each unprofiled and with a
focusing profile of random amplitudes on the x = 0 face), each stepped from the same random state with CUDA-graph
replay; timing windows of --steps-per-window steps (one rk4 call each) alternate between the four so that they
share the card's state; the median window is reported, and the increment of the profiled step over the unprofiled
one per window.  The profiled boundary term touches the (P N + 1)^2 tag-1 dofs only and adds fp64 trigonometry
there at every stage.  In the run, a profile with a = 1 and tau = 0 is checked against the unprofiled model over 5
steps (relative L2 difference of u).  Writes DIR/source_profile_<config>.json and prints a summary.
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
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 4.33e-6, 3.5, 1000.0   # water


def run_config(name, cfg, args, torch, wfx):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    X = wfx.dof_coordinates(mesh)
    face = np.abs(X[:, 0]) < 1e-12
    rng = np.random.default_rng(2)
    amp = 0.5 + rng.random(n)
    delay = np.zeros(n)
    delay[face] = wfx.focus_delays(X[face], (L / 2, L / 2, L / 2), C0)
    t0 = time.perf_counter()
    models = {"linear": wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype),
              "linear_profiled": wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype),
              "westervelt": wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype),
              "westervelt_profiled": wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype)}
    setup_s = time.perf_counter() - t0
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    u0 = (P0 * rng.standard_normal(n)).astype(dtype)
    v0 = (P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "source_dofs": int(face.sum()), "dtype": str(dtype),
           "perturb": 0.15, "dt": dt, "delta": DELTA, "beta": BETA, "rho0": RHO0, "setup_s": setup_s,
           "windows": args.windows, "steps_per_window": args.steps_per_window}

    # in-run check: the identity profile against the unprofiled model
    eqn = models["linear_profiled"]
    states = []
    for prof in (False, True):
        eqn.set_source_profile(np.ones(n) if prof else None, None)
        eqn.set_state(u0, v0)
        eqn.rk4(0.0, 1.0, dt, max_steps=5)
        states.append(eqn.get_state()[0].astype(np.float64))
    res["identity_profile_rel_l2"] = float(np.linalg.norm(states[1] - states[0]) / np.linalg.norm(states[0]))
    del states
    for k in ("linear_profiled", "westervelt_profiled"):
        models[k].set_source_profile(amp, delay)

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
        res[k] = {"ms_per_step": float(np.median(win[k])), "windows_ms": win[k],
                  "finite": bool(np.isfinite(u).all() and np.isfinite(v).all())}
    for k in ("linear", "westervelt"):
        p = res[k + "_profiled"]
        p["over_unprofiled"] = p["ms_per_step"] / res[k]["ms_per_step"] - 1.0
        p["over_unprofiled_per_window"] = [a / b - 1.0 for a, b in zip(win[k + "_profiled"], win[k])]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--steps-per-window", type=int, default=20)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if args.windows < 5 or args.steps_per_window < 10:
        raise SystemExit("source_profile_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("source_profile_bench: no CUDA device")
    import wave_fenics_b200 as wfx
    from ensemble_bench import card
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    gpu["torch_name"] = torch.cuda.get_device_name(0)
    ok = True
    for name in args.configs.split(","):
        r = run_config(name, CONFIGS[name], args, torch, wfx)
        r["gpu"] = gpu
        with open(os.path.join(args.out, f"source_profile_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        tol = 1e-13 if name.endswith("fp64") else 1e-5
        ok = ok and r["identity_profile_rel_l2"] < tol and all(r[k]["finite"] for k in r if isinstance(r[k], dict)
                                                               and "finite" in r[k])
        print(f"{name} ({r['ndofs']} dofs, {r['source_dofs']} source dofs, {gpu.get('name')}, "
              f"{gpu.get('power_limit')}): identity profile rel. L2 {r['identity_profile_rel_l2']:.2e}")
        for k in ("linear", "linear_profiled", "westervelt", "westervelt_profiled"):
            e = r[k]
            extra = f", {100 * e['over_unprofiled']:+.2f} % over unprofiled" if "over_unprofiled" in e else ""
            print(f"  {k:20s} {e['ms_per_step']:.4f} ms/step{extra}")
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("source_profile_bench: a check failed")


if __name__ == "__main__":
    main()
