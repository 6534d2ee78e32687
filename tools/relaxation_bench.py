"""RK4 step time of the Westervelt model with relaxation absorption (DESIGN.md section 4.5f), 64^3 perturbed cells, P4,
fp64 and fp32.

    python tools/relaxation_bench.py [--out DIR] [--windows 7] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU, four WesterveltGLLOpt models on the same mesh with M = 0, 1, 2, 3 relaxation processes
(soft tissue, 0.5 dB/cm/MHz^1.1 fitted over 0.25 .. 1.5 MHz), each stepped with CUDA-graph replay from a small random
state.  Timing windows of --steps-per-window steps (one rk4 call each) alternate between the four models so that they
share the card's state; the median window is reported.  The increment per process is the least-squares slope of the
step time over M.  The card's name and power limit, and the HBM bandwidth of a 4 GiB device-to-device copy, are
measured in the same run.

Counted bytes per process and step: RELAX_PASSES = 21 vector passes of s bytes (s = scalar size) over the dofs -- the
stage kernel reads and writes the memory variables with the tableau of u and v (stage 0: q read, q, q0, qn written,
eps read: 5; stages 1-2: q, qn, q0, eps read, q, qn written: 6 each; stage 3: q, qn, eps read, q written: 4).  The
target is an increment per process at 0.8 or more of the measured copy bandwidth on those bytes.  Writes
DIR/relaxation_<config>.json and DIR/relaxation.md and prints a summary.
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
RELAX_PASSES = 21
TARGET = 0.8
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 1e-2, 3.5, 1000.0
ALPHA0, Y = 0.5 * np.log(10.0) / 20.0 * 100.0, 1.1      # 0.5 dB/cm/MHz^1.1 in Np/m at 1 MHz


def copy_bandwidth(torch, nbytes=4 << 30, reps=10):
    """bytes / s of a device-to-device copy (read + write) of nbytes, median of reps"""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    del a, b
    return 2 * nbytes / float(np.median(times))


def run_config(name, cfg, args, torch, wfx):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    s = dtype.itemsize
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    med = wfx.Medium(1000.0, C0, alpha0=ALPHA0, y=Y)
    models, rels = {}, {}
    for M in (0, 1, 2, 3):
        rels[M] = med.relaxation(0.5 * F0, 3.0 * F0, M) if M else None
        models[M] = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype,
                                         relaxation=rels[M])
    dt = min([wfx.cfl_timestep(mesh.h_min, C0, P, F0)] + [r.max_dt() for r in rels.values() if r is not None])
    rng = np.random.default_rng(1)
    u0 = (1e3 * rng.standard_normal(n)).astype(dtype)
    v0 = (1e3 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15, "dt": dt,
           "windows": args.windows, "steps_per_window": args.steps_per_window,
           "relax_bytes_per_process": RELAX_PASSES * s * n,
           "fit_error": {M: r.fit_error for M, r in rels.items() if r is not None}}
    t_now = {}
    for M, eqn in models.items():
        eqn.set_state(u0, v0)
        t_now[M] = 0.0
        for _ in range(2):   # warm-up: graph capture and first replays
            t_now[M] = eqn.rk4(t_now[M], 1e9, dt, max_steps=args.steps_per_window)[1]
    torch.cuda.synchronize()
    win = {M: [] for M in models}
    for _ in range(args.windows):
        for M, eqn in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t_now[M] = eqn.rk4(t_now[M], 1e9, dt, max_steps=args.steps_per_window)[1]
            e1.record()
            e1.synchronize()
            win[M].append(e0.elapsed_time(e1) / args.steps_per_window)
    for M, eqn in models.items():
        u, v = eqn.get_state()
        res[f"M{M}"] = {"ms_per_step": float(np.median(win[M])), "windows_ms": win[M],
                        "finite": bool(np.isfinite(u).all() and np.isfinite(v).all())}
    ms = np.array([res[f"M{M}"]["ms_per_step"] for M in models])
    slope = float(np.polyfit(np.arange(4), ms, 1)[0])
    res["ms_per_process"] = slope
    res["process_gbs"] = RELAX_PASSES * s * n / (slope * 1e-3) / 1e9 if slope > 0 else float("inf")
    return res


def write_md(path, results, gpu):
    lines = ["# Relaxation absorption: step time per relaxation process", "",
             f"Written by `tools/relaxation_bench.py` on {gpu.get('name')} at a power limit of {gpu.get('power_limit')}; "
             "64^3 perturbed cells, P4, one GPU, WesterveltGLLOpt with CUDA-graph replay, M = 0..3 alternated in one "
             "run, median of the windows.  Per process: the slope of the step time over M, on "
             f"{RELAX_PASSES} counted vector passes (see the tool's docstring), against the "
             f"{gpu.get('copy_gbs', 0):.0f} GB/s of a device-to-device copy measured in the same run "
             f"(target: {TARGET:g} of it).", "",
             "| config | M = 0 ms | M = 1 ms | M = 2 ms | M = 3 ms | ms / process | GB / process | GB/s | of copy |",
             "|---|---|---|---|---|---|---|---|---|"]
    for r in results:
        ms = " | ".join(f"{r[f'M{M}']['ms_per_step']:.4f}" for M in range(4))
        lines.append(f"| {r['config']} | {ms} | {r['ms_per_process']:.4f} | {r['relax_bytes_per_process'] / 1e9:.3f} | "
                     f"{r['process_gbs']:.0f} | {r['process_gbs'] / gpu.get('copy_gbs', np.nan):.2f} |")
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
        raise SystemExit("relaxation_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("relaxation_bench: no CUDA device")
    import wave_fenics_b200 as wfx
    from ensemble_bench import card
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    gpu["torch_name"] = torch.cuda.get_device_name(0)
    gpu["copy_gbs"] = copy_bandwidth(torch) / 1e9
    results, ok = [], True
    for name in args.configs.split(","):
        r = run_config(name, CONFIGS[name], args, torch, wfx)
        r["gpu"] = gpu
        results.append(r)
        with open(os.path.join(args.out, f"relaxation_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        ok = ok and all(r[f"M{M}"]["finite"] for M in range(4))
        print(f"{name} ({r['ndofs']} dofs, {gpu.get('name')}, {gpu.get('power_limit')}, copy {gpu['copy_gbs']:.0f} GB/s)")
        for M in range(4):
            print(f"  M = {M}: {r[f'M{M}']['ms_per_step']:.4f} ms/step")
        print(f"  per process: {r['ms_per_process']:.4f} ms, {r['process_gbs']:.0f} GB/s "
              f"({r['process_gbs'] / gpu['copy_gbs']:.2f} of the copy)")
    write_md(os.path.join(args.out, "relaxation.md"), results, gpu)
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("relaxation_bench: a run went non-finite")


if __name__ == "__main__":
    main()
