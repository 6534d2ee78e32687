"""Ensemble stiffness apply and RK4 step against single-field runs, at the benchmark workload (64^3 perturbed
cells, P4, fp64) and at P7 fp32 (37^3 cells, 17.6 M dofs).

    python tools/ensemble_bench.py [--out DIR] [--windows 7] [--per-window 20] [--configs p4_fp64,p7_fp32]

Per configuration, on one GPU, in bench.py's manner (CUDA events, warm-up inside the run, median over
windows, vectors far larger than L2):
  - separate: the fused stiffness + 1/m apply (apply_scaled) on plain vectors, one member at a time;
  - ensemble: one apply_ensemble with scale = 1/m on member-interleaved (ndofs, nv) vectors, nv in 1, 2, 4, 8;
  - an RK4 step of an nv-member LinearGLLEnsemble against a single-field LinearGLLOpt step.
Every ensemble result is checked in the run against the separate applies of the same inputs (relative L2
per member <= 1e-12 fp64, <= 1e-5 fp32).  Algorithmic bytes of an ensemble apply:
ncells*nd*(6s+4) + ndofs*(2*nv+1)*s (G and the int32 dofmap once, x and y per member, 1/m once), as a share
of the HBM peak bench.py uses.  Writes DIR/ensemble_<config>.json and prints a summary.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {"p4_fp64": dict(P=4, cells=64, dtype="float64"), "p7_fp32": dict(P=7, cells=37, dtype="float32")}
NVS = (1, 2, 4, 8)
L = 0.1


def card():
    """Name, power limit and max SM clock of GPU 0 (query only)."""
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def register_usage(lib_path):
    """Registers / spill stores of every stiff_ens_kernel instantiation from the library's resource table."""
    try:
        out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", lib_path], capture_output=True,
                             text=True, timeout=120).stdout
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}
    res, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        if name and "stiff_ens_kernel" in name and "REG:" in line:
            demangled = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip() or name
            res[demangled] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    return res


def timed(torch, fn, windows, per_window, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(windows + 1)]
    ev[0].record()
    for w in range(windows):
        for _ in range(per_window):
            fn()
        ev[w + 1].record()
    torch.cuda.synchronize()
    ms = [ev[w].elapsed_time(ev[w + 1]) / per_window for w in range(windows)]
    return float(np.median(ms)), ms


def run_config(name, cfg, args, torch, wfx, peak):
    P, N = cfg["P"], cfg["cells"]
    dtype = np.dtype(cfg["dtype"])
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    s = dtype.itemsize
    tol = 1e-12 if dtype == np.float64 else 1e-5
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    n = mesh.ndofs
    t0 = time.perf_counter()
    geo = wfx.Geometry(mesh, P, dtype)
    op = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo, ensemble=True)
    mass = wfx.MassOperator(mesh, P, dtype=dtype, geometry=geo)
    setup_s = time.perf_counter() - t0
    minv = mass.inverse_diagonal_ptr()
    info = op.info()
    nmax = max(NVS)
    g = torch.Generator(device="cuda").manual_seed(42)
    xs = [torch.randn(n, dtype=tdt, device="cuda", generator=g) for _ in range(nmax)]
    ys = [torch.empty_like(xs[0]) for _ in range(nmax)]
    res = {"config": name, "P": P, "cells": N ** 3, "ndofs": n, "dtype": str(dtype), "perturb": 0.15,
           "single_kernel": op.kernel_info()["variant"], "setup_s": setup_s, "windows": args.windows,
           "applies_per_window": args.per_window, "hbm_peak_gbs": peak[0], "hbm_peak_source": peak[1]}

    # separate fused applies, one member after another (members 0..7 cycled so that no vector stays in L2)
    state = {"i": 0}

    def sep():
        i = state["i"] % nmax
        op.apply_scaled(xs[i], minv, ys[i])
        state["i"] += 1

    for i in range(nmax):
        op.apply_scaled(xs[i], minv, ys[i])
    ms_sep, win_sep = timed(torch, sep, args.windows, args.per_window)
    bytes_single = info["bytes"]
    res["separate"] = {"ms_per_member": ms_sep, "windows_ms": win_sep, "gdofs_per_member": n / (ms_sep * 1e-3) / 1e9,
                       "bytes": bytes_single, "frac_of_hbm_peak": bytes_single / (ms_sep * 1e-3) / 1e9 / peak[0]}
    res["ensemble"] = {}
    for nv in NVS:
        X = torch.stack(xs[:nv], dim=1).contiguous()
        Y = torch.full_like(X, float("nan"))
        op.apply_ensemble(X, Y, scale_ptr=minv)
        torch.cuda.synchronize()
        err = max(float(torch.linalg.norm((Y[:, m] - ys[m]).double()) / torch.linalg.norm(ys[m].double()))
                  for m in range(nv))
        ms, win = timed(torch, lambda: op.apply_ensemble(X, Y, scale_ptr=minv), args.windows, args.per_window)
        nbytes = info["num_cells"] * info["num_dofs"] * (6 * s + 4) + n * (2 * nv + 1) * s
        res["ensemble"][str(nv)] = {
            "ms_per_apply": ms, "ms_per_member": ms / nv, "windows_ms": win,
            "gdofs_per_member": n / (ms / nv * 1e-3) / 1e9, "speedup_vs_separate": ms_sep / (ms / nv),
            "bytes": nbytes, "achieved_gbs": nbytes / (ms * 1e-3) / 1e9,
            "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak[0],
            "max_member_rel_l2_vs_separate": err, "check_ok": err <= tol}
        del X, Y
    del xs, ys
    torch.cuda.empty_cache()

    # RK4: an nv-member ensemble step against a single-field step (fresh models on the same mesh)
    res["rk4"] = {}
    c0 = 1500.0
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, 0.5e6)
    one = wfx.LinearGLLOpt(mesh, None, P, c0, 0.5e6, 6e4, dtype=dtype)
    one.init()
    ms1, _ = timed(torch, lambda: one.rk4(0.0, 1.0, dt, max_steps=1), args.windows, args.per_window // 2 or 1)
    res["rk4"]["single_ms_per_step"] = ms1
    del one
    for nv in (4, 8):
        ens = wfx.LinearGLLEnsemble(mesh, None, P, c0, np.linspace(0.3e6, 0.6e6, nv), np.full(nv, 6e4), dtype=dtype)
        ens.init()
        ms, _ = timed(torch, lambda: ens.rk4(0.0, 1.0, dt, max_steps=1), args.windows, args.per_window // 2 or 1)
        res["rk4"][str(nv)] = {"ms_per_step": ms, "ms_per_member": ms / nv, "speedup_vs_single": ms1 / (ms / nv)}
        del ens
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--per-window", type=int, default=20)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if args.windows < 5 or args.per_window < 20:
        raise SystemExit("ensemble_bench: at least 5 windows of 20 applies")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_bench: no CUDA device")
    import wave_fenics_b200 as wfx
    import bench
    peak = bench.measured_peak()
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    gpu["torch_name"] = torch.cuda.get_device_name(0)
    regs = register_usage(wfx.capi.LIB_PATH)
    ok = True
    for name in args.configs.split(","):
        r = run_config(name, CONFIGS[name], args, torch, wfx, peak)
        r["gpu"] = gpu
        r["registers"] = regs
        with open(os.path.join(args.out, f"ensemble_{name}.json"), "w") as fh:
            json.dump(r, fh, indent=1)
        print(f"{name}: separate {r['separate']['ms_per_member']:.4f} ms/member "
              f"({r['separate']['gdofs_per_member']:.2f} GDoF/s, {r['separate']['frac_of_hbm_peak']:.3f} of peak)")
        for nv, e in r["ensemble"].items():
            ok = ok and e["check_ok"]
            print(f"  nv={nv}: {e['ms_per_apply']:.4f} ms/apply, {e['ms_per_member']:.4f} ms/member, "
                  f"{e['gdofs_per_member']:.2f} GDoF/s/member, x{e['speedup_vs_separate']:.2f}, "
                  f"{e['frac_of_hbm_peak']:.3f} of peak, rel L2 {e['max_member_rel_l2_vs_separate']:.1e}")
        print(f"  rk4: single {r['rk4']['single_ms_per_step']:.4f} ms/step; "
              + "; ".join(f"nv={k}: {v['ms_per_member']:.4f} ms/member/step" for k, v in r["rk4"].items() if k != "single_ms_per_step"))
    print(json.dumps({"gpu": gpu, "registers": regs}))
    if not ok:
        raise SystemExit("ensemble_bench: an ensemble result differs from the separate applies")


if __name__ == "__main__":
    main()
