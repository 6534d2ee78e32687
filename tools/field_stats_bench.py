"""Cost of the field statistics (DESIGN.md section 4.5b) at the benchmark workload (64^3 perturbed cells, P4) in fp64
and fp32.

    python tools/field_stats_bench.py [--out DIR] [--windows 9] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU: the linear model with the statistics off and on with H = 0, 3 and 8 harmonics (the
window open from t = 0, so every step is sampled), plus the Westervelt model off and at H = 3; one model object
per variant on the same mesh, each stepped from the same random state with CUDA-graph replay.  Timing windows of
--steps-per-window steps (one rk4 call each) alternate between the variants so that they share the card's state;
the median window is reported.  The increment of a variant is its median step time minus that of the same model
with the statistics off, and also the median of the per-window differences (adjacent windows).

Bytes of one sampled step (s = scalar size, n = dofs): read u (s), read-modify-write pmax and pmin (4 s), and
read-modify-write H fp64 (re, im) pairs (32 H):  (5 s + 32 H) n.  Share of the HBM peak bench.py uses
(bench.measured_peak()) = those bytes over the increment.  Writes DIR/field_stats_<config>.json and prints a summary.
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
# variant -> (model, harmonics or None for off)
VARIANTS = {"linear_off": ("linear", None), "linear_h0": ("linear", 0), "linear_h3": ("linear", 3),
            "linear_h8": ("linear", 8), "westervelt_off": ("westervelt", None), "westervelt_h3": ("westervelt", 3)}
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 4.33e-6, 3.5, 1000.0   # water


def stats_bytes(nharm, n, s):
    return (5 * s + 32 * nharm) * n


def run_config(name, cfg, args, torch, wfx, peak):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    s = dtype.itemsize
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    t0 = time.perf_counter()
    models = {}
    for k, (model, nharm) in VARIANTS.items():
        if model == "linear":
            eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype)
        else:
            eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype)
        if nharm is not None:
            eqn.set_field_stats(0.0, harmonics=nharm)
        models[k] = eqn
    setup_s = time.perf_counter() - t0
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    rng = np.random.default_rng(1)
    u0 = (P0 * rng.standard_normal(n)).astype(dtype)
    v0 = (P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15, "dt": dt,
           "setup_s": setup_s, "windows": args.windows, "steps_per_window": args.steps_per_window,
           "hbm_peak_gbs": peak[0], "hbm_peak_source": peak[1]}

    t_now = {}
    for k, eqn in models.items():
        eqn.set_state(u0, v0)   # also resets the statistics
        t_now[k] = 0.0
        for _ in range(2):      # warm-up: graph capture and first replays
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
    for k, (model, nharm) in VARIANTS.items():
        eqn = models[k]
        u, v = eqn.get_state()
        e = {"ms_per_step": float(np.median(win[k])), "windows_ms": win[k],
             "finite": bool(np.isfinite(u).all() and np.isfinite(v).all())}
        if nharm is not None:
            fs = eqn.field_stats()
            e["samples"] = fs.samples
            e["maps_finite"] = bool(np.isfinite(fs.pmax).all() and np.isfinite(fs.harmonics).all())
            # the maps bound the final state
            e["peaks_bound_state"] = bool((fs.pmax >= u).all() and (fs.pmin <= u).all())
            off = model + "_off"
            nbytes = stats_bytes(nharm, n, s)
            inc = e["ms_per_step"] - float(np.median(win[off]))
            inc_paired = float(np.median([a - b for a, b in zip(win[k], win[off])]))
            e.update({"harmonics": nharm, "increment_ms": inc, "increment_paired_ms": inc_paired,
                      "over_off": e["ms_per_step"] / float(np.median(win[off])) - 1.0, "stats_bytes": nbytes,
                      "stats_bytes_per_entry": nbytes / n,
                      "ideal_ms_at_peak": nbytes / (peak[0] * 1e9) * 1e3,
                      "frac_of_hbm_peak": nbytes / (inc * 1e-3) / 1e9 / peak[0] if inc > 0 else None,
                      "frac_of_hbm_peak_paired": (nbytes / (inc_paired * 1e-3) / 1e9 / peak[0]
                                                  if inc_paired > 0 else None)})
        res[k] = e
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--windows", type=int, default=9)
    ap.add_argument("--steps-per-window", type=int, default=20)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if args.windows < 5 or args.steps_per_window < 10:
        raise SystemExit("field_stats_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("field_stats_bench: no CUDA device")
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
        with open(os.path.join(args.out, f"field_stats_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        print(f"{name} ({r['ndofs']} dofs, {gpu.get('name')}, {gpu.get('power_limit')}, "
              f"peak {peak[0]:.1f} GB/s {peak[1]})")
        for k in VARIANTS:
            e = r[k]
            ok = ok and e["finite"] and e.get("maps_finite", True) and e.get("peaks_bound_state", True)
            line = f"  {k:15s} {e['ms_per_step']:.4f} ms/step"
            if "increment_ms" in e:
                frac = e["frac_of_hbm_peak"]
                line += (f", +{1e3 * e['increment_ms']:.1f} us (paired +{1e3 * e['increment_paired_ms']:.1f} us, "
                         f"ideal {1e3 * e['ideal_ms_at_peak']:.1f} us), {e['stats_bytes_per_entry']:.0f} B/dof, "
                         f"{'n/a' if frac is None else f'{frac:.3f}'} of peak, {100 * e['over_off']:+.2f} %")
            print(line)
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("field_stats_bench: a check failed")


if __name__ == "__main__":
    main()
