"""RK4 step time in layered media (DESIGN.md section 4.5e), 64^3 perturbed cells, P4, fp64 and fp32.

    python tools/medium_bench.py [--out DIR] [--windows 7] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU, four models on the same mesh, each stepped with CUDA-graph replay from a small random
state:
  westervelt         WesterveltGLLOpt with its scalar kappa
  westervelt_kappa   the same model with a per-dof kappa (set_nonlinearity): the stage kernels read kappa_i
  linear             LinearGLLOpt
  linear_medium      LinearGLLOpt in a water | tissue | bone layered medium (weighted mass and facet masses, scaled G)
Timing windows of --steps-per-window steps (one rk4 call each) alternate between the four models so that they share
the card's state; the median window is reported, and each pair's ratio per window.  The card's name and power limit
are read in the same run.

Algorithmic bytes per step beyond the four stiffness applies (s = scalar size, n = dofs): the Westervelt step makes
43 vector passes with a scalar kappa and 47 with a per-dof kappa (kappa_i read once per stage); the linear step makes
39 with or without a medium (the medium only changes the values of m, m1, m2 and G).  Writes DIR/medium_<config>.json
and DIR/medium.md and prints a summary.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

CONFIGS = {"p4_fp64": dict(P=4, cells=64, dtype="float64"), "p4_fp32": dict(P=4, cells=64, dtype="float32")}
PASSES = {"westervelt": 43, "westervelt_kappa": 47, "linear": 39, "linear_medium": 39}
PAIRS = (("westervelt_kappa", "westervelt"), ("linear_medium", "linear"))
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 1e-2, 3.5, 1000.0
LAYERS = ((1000.0, 1500.0, 3.5), (1050.0, 1580.0, 6.0), (1900.0, 2800.0, 4.5))   # water, tissue, bone


def layered_medium(wfx, mesh, N):
    cx = np.arange(mesh.ncells) // (N * N)
    layer = np.minimum(3 * cx // N, 2)
    rho, c, beta = (np.array([lay[k] for lay in LAYERS])[layer] for k in range(3))
    return wfx.Medium(rho, c, beta)


def run_config(name, cfg, args, torch, wfx):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    s = dtype.itemsize
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    med = layered_medium(wfx, mesh, N)
    models = {"westervelt": wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype),
              "westervelt_kappa": wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype),
              "linear": wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype),
              "linear_medium": wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, medium=med)}
    kappa = 2 * BETA / (RHO0 * C0 ** 2) * np.random.default_rng(2).uniform(0.5, 2.0, n)
    models["westervelt_kappa"].set_nonlinearity(kappa)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    apply_bytes = models["linear"].stiff_op.info()["bytes"]
    rng = np.random.default_rng(1)
    u0 = (1e3 * rng.standard_normal(n)).astype(dtype)
    v0 = (1e3 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15, "dt": dt,
           "kernel": models["linear"].stiff_op.kernel_info()["variant"], "windows": args.windows,
           "steps_per_window": args.steps_per_window, "apply_bytes": apply_bytes}
    t_now = {}
    for k, eqn in models.items():
        eqn.set_state(u0, v0)
        t_now[k] = 0.0
        for _ in range(2):   # warm-up: graph capture and first replays
            t_now[k] = eqn.rk4(t_now[k], 1e9, dt, max_steps=args.steps_per_window)[1]
    torch.cuda.synchronize()
    win = {k: [] for k in models}
    for _ in range(args.windows):
        for k, eqn in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t_now[k] = eqn.rk4(t_now[k], 1e9, dt, max_steps=args.steps_per_window)[1]
            e1.record()
            e1.synchronize()
            win[k].append(e0.elapsed_time(e1) / args.steps_per_window)
    for k, eqn in models.items():
        u, v = eqn.get_state()
        ms = float(np.median(win[k]))
        nbytes = 4 * apply_bytes + PASSES[k] * s * n
        res[k] = {"ms_per_step": ms, "windows_ms": win[k], "bytes_per_step": nbytes,
                  "achieved_gbs": nbytes / (ms * 1e-3) / 1e9,
                  "finite": bool(np.isfinite(u).all() and np.isfinite(v).all())}
    for a, b in PAIRS:
        per = [x / y - 1.0 for x, y in zip(win[a], win[b])]
        res[a]["over_" + b] = float(np.median(per))
        res[a]["over_" + b + "_per_window"] = per
    return res


def write_md(path, results, gpu):
    lines = ["# RK4 step time in layered media", "",
             f"Written by `tools/medium_bench.py` on {gpu.get('name')} at a power limit of {gpu.get('power_limit')}; "
             "64^3 perturbed cells, P4, one GPU, CUDA-graph replay, the four models alternated in one run, median of "
             "the windows (the ratio: median of the per-window ratios).  Bytes are algorithmic (see the tool's "
             "docstring).", "",
             "| config | model | ms / step | GB / step | GB/s | against |",
             "|---|---|---|---|---|---|"]
    for r in results:
        for k in PASSES:
            e = r[k]
            over = "".join(f"{100 * e['over_' + b]:+.2f} % over {b}" for a, b in PAIRS if a == k)
            lines.append(f"| {r['config']} | {k} | {e['ms_per_step']:.4f} | {e['bytes_per_step'] / 1e9:.3f} | "
                         f"{e['achieved_gbs']:.0f} | {over} |")
    lines.append("")
    with open(path, "w") as fh:
        fh.write("\n".join(lines))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--steps-per-window", type=int, default=20)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if args.windows < 5 or args.steps_per_window < 10:
        raise SystemExit("medium_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("medium_bench: no CUDA device")
    import wave_fenics_b200 as wfx
    from ensemble_bench import card
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    gpu["torch_name"] = torch.cuda.get_device_name(0)
    results, ok = [], True
    for name in args.configs.split(","):
        r = run_config(name, CONFIGS[name], args, torch, wfx)
        r["gpu"] = gpu
        results.append(r)
        with open(os.path.join(args.out, f"medium_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        ok = ok and all(r[k]["finite"] for k in PASSES)
        print(f"{name} ({r['ndofs']} dofs, {gpu.get('name')}, {gpu.get('power_limit')})")
        for k in PASSES:
            e = r[k]
            extra = "".join(f", {100 * e['over_' + b]:+.2f} % over {b}" for a, b in PAIRS if a == k)
            print(f"  {k:17s} {e['ms_per_step']:.4f} ms/step{extra}")
    write_md(os.path.join(args.out, "medium.md"), results, gpu)
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("medium_bench: a run went non-finite")


if __name__ == "__main__":
    main()
