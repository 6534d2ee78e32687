"""RK4 step time of the Pennes thermal model (DESIGN.md section 4.5d) against the linear wave model's step on the same
mesh and operators (64^3 perturbed cells, P4), fp64 and fp32.

    python tools/thermal_bench.py [--out DIR] [--windows 7] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU: a LinearGLLOpt and a PennesGLL built on its operators (PennesGLL.from_wave), each
stepped with CUDA-graph replay from a random state (the thermal model at 0.8 of its power-iteration step, with a
random heat source and the dose accumulating); timing windows of --steps-per-window steps (one rk4 call each)
alternate between the two models so that they share the card's state; the median window is reported.  The card's
name and power limit are read in the same run.

Algorithmic bytes of one thermal RK4 step (s = scalar size, n = dofs): 4 stiffness applies (StiffnessOperator.info()
bytes each) plus the fused stage kernels' vector passes, VECTOR_PASSES * s * n with
  29 = 7 + 8 + 8 + 6   (stage 0: reads b r f th, writes th0 th thn; stages 1, 2: read b r f thn th th0, write th thn;
                         stage 3: reads b r f thn th, writes th)
plus, in stage 3, DOSE_BYTES_PER_DOF = 16 (CEM43 read and write, fp64) and 2 s n (theta_max read and write).  The
linear step's bytes are those of tools/model_bench.py (39 vector passes).  Share of the HBM peak bench.py uses
(bench.measured_peak()).  Writes DIR/thermal_<config>.json and DIR/thermal.md and prints a summary.
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
VECTOR_PASSES = 29
DOSE_BYTES_PER_DOF = 16
LINEAR_VECTOR_PASSES = 39
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
K_T, RHOC, WBCB = 0.5, 3.6e6, 2.0e3   # soft tissue


def thermal_step_bytes(apply_bytes, n, s):
    return 4 * apply_bytes + (VECTOR_PASSES + 2) * s * n + DOSE_BYTES_PER_DOF * n


def linear_step_bytes(apply_bytes, n, s):
    return 4 * apply_bytes + LINEAR_VECTOR_PASSES * s * n


def run_config(name, cfg, args, torch, wfx, peak):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    s = dtype.itemsize
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    t0 = time.perf_counter()
    wave = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype)
    th = wfx.PennesGLL.from_wave(wave, K_T, RHOC, WBCB)
    setup_s = time.perf_counter() - t0
    rng = np.random.default_rng(1)
    u0 = (P0 * rng.standard_normal(n)).astype(dtype)
    v0 = (P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    th.set_heat_source(1e6 * rng.random(n))
    T0 = 37.0 + 8.0 * rng.random(n)
    lam, dt_max = th.max_eigenvalue(200)
    dts = {"linear": wfx.cfl_timestep(mesh.h_min, C0, P, F0), "thermal": 0.8 * dt_max}
    apply_bytes = wave.stiff_op.info()["bytes"]
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15,
           "dt_linear": dts["linear"], "dt_thermal": dts["thermal"], "lambda_max_estimate": lam,
           "kernel": wave.stiff_op.kernel_info()["variant"], "windows": args.windows,
           "steps_per_window": args.steps_per_window, "hbm_peak_gbs": peak[0], "hbm_peak_source": peak[1],
           "apply_bytes": apply_bytes, "setup_s": setup_s}
    wave.set_state(u0, v0)
    th.set_state(T0)
    models = {"linear": wave, "thermal": th}
    t_now = {k: 0.0 for k in models}
    for k, eqn in models.items():
        for _ in range(2):   # warm-up: graph capture and first replays
            t_now[k] = eqn.rk4(t_now[k], 1e9, dts[k], max_steps=args.steps_per_window)[1]
    torch.cuda.synchronize()
    win = {k: [] for k in models}
    for _ in range(args.windows):
        for k, eqn in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t_now[k] = eqn.rk4(t_now[k], 1e9, dts[k], max_steps=args.steps_per_window)[1]
            e1.record()
            e1.synchronize()
            win[k].append(e0.elapsed_time(e1) / args.steps_per_window)
    u, v = wave.get_state()
    d = th.dose()
    finite = {"linear": bool(np.isfinite(u).all() and np.isfinite(v).all()),
              "thermal": bool(np.isfinite(th.get_state()).all() and np.isfinite(d.cem43).all())}
    for k, fn in (("linear", linear_step_bytes), ("thermal", thermal_step_bytes)):
        ms = float(np.median(win[k]))
        nbytes = fn(apply_bytes, n, s)
        res[k] = {"ms_per_step": ms, "windows_ms": win[k], "bytes_per_step": nbytes,
                  "achieved_gbs": nbytes / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak[0],
                  "finite": finite[k]}
    res["thermal"]["over_linear"] = res["thermal"]["ms_per_step"] / res["linear"]["ms_per_step"] - 1.0
    res["thermal"]["over_linear_per_window"] = [a / b - 1.0 for a, b in zip(win["thermal"], win["linear"])]
    res["thermal"]["dose_steps"] = d.steps
    return res


def write_md(path, results, gpu):
    lines = ["# Thermal (Pennes) RK4 step against the linear wave step", "",
             f"Written by `tools/thermal_bench.py` on {gpu.get('name')} at a power limit of {gpu.get('power_limit')}; "
             "64^3 perturbed cells, P4, one GPU, CUDA-graph replay, the two models alternated in one run, median of "
             "the windows.  Bytes are algorithmic (see the tool's docstring); the share is of the measured HBM peak "
             "bench.py uses.", "",
             "| config | model | ms / step | GB / step | GB/s | share of HBM peak | thermal over linear |",
             "|---|---|---|---|---|---|---|"]
    for r in results:
        for k in ("linear", "thermal"):
            e = r[k]
            over = f"{100 * e['over_linear']:+.2f} %" if "over_linear" in e else ""
            lines.append(f"| {r['config']} | {k} | {e['ms_per_step']:.4f} | {e['bytes_per_step'] / 1e9:.3f} | "
                         f"{e['achieved_gbs']:.0f} | {e['frac_of_hbm_peak']:.3f} | {over} |")
    lines += ["", f"HBM peak used: {results[0]['hbm_peak_gbs']:.0f} GB/s ({results[0]['hbm_peak_source']}).", ""]
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
        raise SystemExit("thermal_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("thermal_bench: no CUDA device")
    import wave_fenics_b200 as wfx
    import bench
    from ensemble_bench import card
    peak = bench.measured_peak()
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    gpu["torch_name"] = torch.cuda.get_device_name(0)
    results, ok = [], True
    for name in args.configs.split(","):
        r = run_config(name, CONFIGS[name], args, torch, wfx, peak)
        r["gpu"] = gpu
        results.append(r)
        with open(os.path.join(args.out, f"thermal_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        ok = ok and r["linear"]["finite"] and r["thermal"]["finite"]
        print(f"{name} ({r['ndofs']} dofs, {gpu.get('name')}, {gpu.get('power_limit')})")
        for k in ("linear", "thermal"):
            e = r[k]
            extra = f", {100 * e['over_linear']:+.2f} % over linear" if "over_linear" in e else ""
            print(f"  {k:8s} {e['ms_per_step']:.4f} ms/step, {e['frac_of_hbm_peak']:.3f} of peak{extra}")
    write_md(os.path.join(args.out, "thermal.md"), results, gpu)
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("thermal_bench: a check failed")


if __name__ == "__main__":
    main()
