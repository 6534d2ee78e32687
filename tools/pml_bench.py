"""RK4 step time of the linear and Westervelt models with a perfectly matched layer (DESIGN.md section 4.5g), 64^3
perturbed cells, P4, fp64 and fp32.

    python tools/pml_bench.py [--out DIR] [--windows 7] [--steps-per-window 20] [--configs p4_fp64,p4_fp32]

Per configuration, on one GPU, four models on the same mesh: LinearGLLOpt and WesterveltGLLOpt, each without a layer
and with a two-cell PML.box on the five faces other than the source face, stepped with CUDA-graph replay from a small
random state.  Timing windows of --steps-per-window steps (one rk4 call each) alternate between the four so that they
share the card's state; the median window is reported, and the increment of the layer is the difference of the
medians.  The card's name and power limit, and the HBM bandwidth of a 4 GiB device-to-device copy, are measured in the
same run.

Counted bytes of the two layer kernels per step (pml_bytes, from shapes; s = scalar size, nq = 125 points per cell):
  per layer point and stage: J^-1 9s, |detJ| w s, the two dofmap indices 8 B, r written s and read back s, the
    inverse-map entry 4 B, and phi with the RK4 tableau: 12s (stage 0), 15s (stages 1, 2), 9s (stage 3);
  per layer dof and stage: the cell kernel's w, psi and zeta gathers 5s (once per dof; the Westervelt model also reads
    vn for p: s more), the dof kernel's b read-modify-write 2s, p and p_t 2s, zeta sums 3s, m~ s, psi with the tableau
    4s (stage 0), 5s (1, 2), 3s (3), the dof index and the inverse map's offset 8 B.
The share of the copy rate is pml_bytes / increment / copy rate (target 0.6).  Writes DIR/pml_<config>.json and
DIR/pml.md and prints a summary.
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
TARGET = 0.6
L, C0, F0, P0 = 0.1, 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 1e-2, 3.5, 1000.0
FACES = [(0, 1), (1, 0), (1, 1), (2, 0), (2, 1)]
PHI_STAGE = (12, 15, 15, 9)      # phi traffic per point and stage, in scalars
PSI_STAGE = (4, 5, 5, 3)         # psi traffic per dof and stage, in scalars


def pml_bytes(ncells, npd, nq, s, westervelt):
    """algorithmic bytes of the two layer kernels per RK4 step (see the docstring)"""
    total = 0
    for st in range(4):
        per_point = 9 * s + s + 8 + 2 * s + 4 + PHI_STAGE[st] * s
        per_dof = (5 + (1 if westervelt else 0)) * s + 2 * s + 2 * s + 3 * s + s + PSI_STAGE[st] * s + 8
        total += ncells * nq * per_point + npd * per_dof
    return total


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
    pml = wfx.PML.box(mesh, 2 * L / N, FACES, C0)
    models = {}
    for kind in ("linear", "westervelt"):
        for layer in (False, True):
            key = f"{kind}{'_pml' if layer else ''}"
            if kind == "linear":
                models[key] = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, pml=pml if layer else None)
            else:
                models[key] = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype,
                                                   pml=pml if layer else None)
    info = models["linear_pml"].pml_info()
    dt = min(wfx.cfl_timestep(mesh.h_min, C0, P, F0), pml.max_dt())
    rng = np.random.default_rng(1)
    u0 = (1e3 * rng.standard_normal(n)).astype(dtype)
    v0 = (1e3 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype)
    nq = (P + 1) ** 3
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15, "dt": dt,
           "windows": args.windows, "steps_per_window": args.steps_per_window, "faces": FACES,
           "pml_cells": info["cells"], "pml_dofs": info["dofs"], "zeta_max": info["zeta_max"],
           "pml_bytes_linear": pml_bytes(info["cells"], info["dofs"], nq, s, False),
           "pml_bytes_westervelt": pml_bytes(info["cells"], info["dofs"], nq, s, True)}
    t_now = {}
    for key, eqn in models.items():
        eqn.set_state(u0, v0)
        t_now[key] = 0.0
        for _ in range(2):   # warm-up: graph capture and first replays
            t_now[key] = eqn.rk4(t_now[key], 1e9, dt, max_steps=args.steps_per_window)[1]
    torch.cuda.synchronize()
    win = {key: [] for key in models}
    for _ in range(args.windows):
        for key, eqn in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t_now[key] = eqn.rk4(t_now[key], 1e9, dt, max_steps=args.steps_per_window)[1]
            e1.record()
            e1.synchronize()
            win[key].append(e0.elapsed_time(e1) / args.steps_per_window)
    for key, eqn in models.items():
        u, v = eqn.get_state()
        res[key] = {"ms_per_step": float(np.median(win[key])), "windows_ms": win[key],
                    "finite": bool(np.isfinite(u).all() and np.isfinite(v).all())}
    for kind in ("linear", "westervelt"):
        inc = res[f"{kind}_pml"]["ms_per_step"] - res[kind]["ms_per_step"]
        res[f"{kind}_increment_ms"] = inc
        res[f"{kind}_pml_gbs"] = res[f"pml_bytes_{kind}"] / (inc * 1e-3) / 1e9 if inc > 0 else float("inf")
    return res


def write_md(path, results, gpu):
    lines = ["# Perfectly matched layer: step time of the layer", "",
             f"Written by `tools/pml_bench.py` on {gpu.get('name')} at a power limit of {gpu.get('power_limit')}; "
             "64^3 perturbed cells, P4, one GPU, CUDA-graph replay, a two-cell `PML.box` on the five faces other "
             "than the source face, the four models alternated in one run, median of the windows.  The increment is "
             "the step with the layer minus the step without; its counted bytes (see the tool's docstring) over the "
             f"increment are compared with the {gpu.get('copy_gbs', 0):.0f} GB/s of a device-to-device copy measured "
             f"in the same run (target: {TARGET:g} of it; a share below it is a miss).", "",
             "| config | model | layer cells | layer dofs | ms / step | with layer | increment ms | GB counted | GB/s "
             "| of copy |",
             "|---|---|---|---|---|---|---|---|---|---|"]
    for r in results:
        for kind in ("linear", "westervelt"):
            gbs = r[f"{kind}_pml_gbs"]
            lines.append(f"| {r['config']} | {kind} | {r['pml_cells']} | {r['pml_dofs']} | "
                         f"{r[kind]['ms_per_step']:.4f} | {r[kind + '_pml']['ms_per_step']:.4f} | "
                         f"{r[kind + '_increment_ms']:.4f} | {r['pml_bytes_' + kind] / 1e9:.3f} | {gbs:.0f} | "
                         f"{gbs / gpu.get('copy_gbs', np.nan):.2f} |")
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
        raise SystemExit("pml_bench: at least 5 windows of 10 steps")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pml_bench: no CUDA device")
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
        with open(os.path.join(args.out, f"pml_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        ok = ok and all(r[k]["finite"] for k in ("linear", "linear_pml", "westervelt", "westervelt_pml"))
        print(f"{name} ({r['ndofs']} dofs, layer {r['pml_cells']} cells / {r['pml_dofs']} dofs, {gpu.get('name')}, "
              f"{gpu.get('power_limit')}, copy {gpu['copy_gbs']:.0f} GB/s)")
        for kind in ("linear", "westervelt"):
            print(f"  {kind}: {r[kind]['ms_per_step']:.4f} ms/step, with the layer "
                  f"{r[kind + '_pml']['ms_per_step']:.4f}; increment {r[kind + '_increment_ms']:.4f} ms, "
                  f"{r[kind + '_pml_gbs']:.0f} GB/s ({r[kind + '_pml_gbs'] / gpu['copy_gbs']:.2f} of the copy)")
    write_md(os.path.join(args.out, "pml.md"), results, gpu)
    print(json.dumps({"gpu": gpu}))
    if not ok:
        raise SystemExit("pml_bench: a run went non-finite")


if __name__ == "__main__":
    main()
