#!/usr/bin/env python
"""Benchmark of the waveFEniCS hot path on B200 (see the contract in DESIGN.md section 5).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--scaling weak|strong]
                  [--dump-outputs DIR]

N = 1 workload: BASELINE.json configs[1] -- single-B200 stiffness + mass operator apply,
64^3 hex cells, P4 (16 974 593 dofs), fp64.  One "step" = one fused apply
kv = M^-1 (-c0^2 K u).  `value` = GDoF/s with all inputs resident in HBM; `e2e` = the same
apply through the C-ABI host entry point (pinned host x -> device -> apply -> host y).
N > 1 (weak, the default): the same per-GPU block on every rank of a cartesian partition, the
interface dofs of K u reduced with the halo exchange before the mass inverse.
--scaling strong: BASELINE configs[3], a fixed 128^3-cell global mesh split over the N ranks.

Timing: the K timed applies run back to back, split by CUDA events on the launching stream into
R = min(--windows, K // MIN_WINDOW_STEPS) windows (at least one), with barrier + synchronize before the
first and after the last; max over ranks per window; `value` comes from the MEDIAN window's time per
apply (all windows are reported).  The default K = 140 is 7 windows of 20 applies.  A second,
>= 0.6 s window gives the sustained (power-capped) figure with its own clock record.  The nvidia-smi
sampler starts before the first barrier and the warm-up, so no rank does host work inside another
rank's window.

--dump-outputs DIR writes what the last timed step computed, kv (rank 0's vector when N > 1), to
DIR/kv.npy in float64: all of it, or the entries at a fixed, seeded sample of DUMP_MAX_VALUES dof
indices (sorted) when it is longer.  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.

--impl reference times the CPU restatement of the reference operator (oracle/, built with the
reference's own compiler flags) on the box's host cores, on a bounded sample of the workload;
it never imports the product package.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GDoF/s stiffness+mass apply (P4 hex, fp64)"
UNIT = "GDoF/s"
L = 0.1
DUMP_MAX_VALUES = 1 << 22  # 32 MiB of float64 per dumped array
MIN_WINDOW_STEPS = 20  # ~9 ms at the default size: the window length of the recorded measurements (profiles/)


def dump_sample_index(n):
    """None (the whole vector) or the sorted dof indices of the fixed sample that --dump-outputs writes."""
    if n <= DUMP_MAX_VALUES:
        return None
    return np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_VALUES, replace=False))


def dump_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_threads():
    """Host cores this process may use.  Not OMP_NUM_THREADS: torch.distributed.run sets it to 1."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    return max(1, min(n, 32))  # thread-private y copies: bound the memory


class ClockSampler:
    """nvidia-smi SM clock / throttle-reason sampler; rows are time-stamped so that one sampler
    serves several timed regions (summary(t0, t1) = the rows that fall inside a region)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0, period_ms=50):
        self.rows, self.proc, self.index, self.period = [], None, index, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", str(self.period)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t_end = time.time() + 3.0
            while not self.rows and time.time() < t_end:  # wait until it is really sampling
                time.sleep(0.02)
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            time.sleep(1.5 * self.period / 1e3)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        rows = [r for (t, r) in self.rows if len(r) >= 7 and (t0 is None or t >= t0) and (t1 is None or t <= t1)]
        num = lambda s: float(s) if s.replace(".", "", 1).isdigit() else None
        sm = [num(r[0]) for r in rows if num(r[0]) is not None]
        mx = [num(r[1]) for (_, r) in self.rows if len(r) >= 7 and num(r[1]) is not None]
        pw = [num(r[2]) for r in rows if num(r[2]) is not None]
        reasons = sorted({self.NAMES[i] for r in rows for i in range(4) if r[3 + i].startswith("Active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "reasons": reasons, "samples": len(sm)}


# ---- CPU reference arm (oracle only; no product import) ------------------------------------------
CPU_KIND = {"kind": "port", "how": "dense skernel + b/m, {t} OpenMP threads, -Ofast -march=native"}


def reference_operator_sample(mesh, P, G, m, x, threads, repeats):
    """The REFERENCE's own StiffnessOperator::operator() / skernel (oracle/_ref/libwfref_cpu_fast.so, cut out of
    common/operators.hpp and compiled at the reference's -Ofast) followed by b / m.  The reference is serial per
    MPI rank; the ranks are host threads here, each applying the operator to its own range of cells into a
    private vector (ghost contributions), summed afterwards like scatter_rev(add).  -> (seconds, kv); None: library
    not built."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle
    lib = oracle.ref_cpu(fast=True)
    if lib is None:
        return None
    nd = (P + 1) ** 3
    f64p, i32p = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    dphi = np.ascontiguousarray(oracle.tabulate_dphi(P)).reshape(-1)
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    G = np.ascontiguousarray(G, dtype=np.float64)
    bounds = np.linspace(0, mesh.ncells, threads + 1).astype(np.int64)
    ys = [np.zeros(mesh.ndofs) for _ in range(threads)]
    # the dofs a rank's cells touch (a slab of the lexicographic numbering): only those are summed
    span = [(int(dm[bounds[r]:bounds[r + 1]].min()), int(dm[bounds[r]:bounds[r + 1]].max()) + 1) if bounds[r + 1] > bounds[r]
            else (0, 0) for r in range(threads)]

    def rank(r):
        c0, c1 = int(bounds[r]), int(bounds[r + 1])
        if c1 > c0:
            lib.wfref_stiffness_apply(c1 - c0, mesh.ndofs, nd, dm[c0:].ctypes.data_as(i32p), G[c0:].ctypes.data_as(f64p),
                                      dphi.ctypes.data_as(f64p), x.ctypes.data_as(f64p), ys[r].ctypes.data_as(f64p))

    best = 1e300
    with ThreadPoolExecutor(threads) as ex:
        for it in range(repeats + 1):  # first pass: warm-up
            for y in ys:
                y[:] = 0
            t0 = time.perf_counter()
            list(ex.map(rank, range(threads)))
            b = np.zeros(mesh.ndofs)
            for r in range(threads):  # scatter_rev(add) of the ranks' contributions
                b[span[r][0]:span[r][1]] += ys[r][span[r][0]:span[r][1]]
            kv = b / m
            if it:
                best = min(best, time.perf_counter() - t0)
    assert np.isfinite(kv).all()
    return best, kv


def cpu_operator_sample(cells, P, threads, repeats=1):
    """Times the reference CPU operator (dense skernel + b/m) on a cells^3 sample mesh: the reference's own
    code when oracle/_ref holds it (kind "reference"), else the oracle's restatement (kind "port").
    -> (ndofs, seconds, kv)"""
    from oracle import oracle, refmesh
    mesh = refmesh.box(cells, P, (L, L, L))
    G, detJ = oracle.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    oracle.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    t_ref = reference_operator_sample(mesh, P, G, m, x, threads, repeats)
    if t_ref is not None:
        CPU_KIND.update(kind="reference", how="the reference's own StiffnessOperator::operator() / skernel (oracle/_ref, "
                        "-Ofast -march=x86-64-v3) + b/m, {t} ranks = host threads over cell ranges, private vectors summed")
        return (mesh.ndofs, *t_ref)
    y = np.zeros(mesh.ndofs)
    oracle.stiffness_apply(mesh, P, G, x, y, dense=True, nthreads=threads, fast=True)  # warm-up
    best = 1e300
    for _ in range(repeats):
        y[:] = 0
        t0 = time.perf_counter()
        oracle.stiffness_apply(mesh, P, G, x, y, dense=True, nthreads=threads, fast=True)
        kv = y / m
        best = min(best, time.perf_counter() - t0)
    assert np.isfinite(kv).all()
    return mesh.ndofs, best, kv


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    cells = args.ref_cells
    for _ in range(args.warmup):
        cpu_operator_sample(min(cells, 8), args.P, threads)
    # bounded: if K steps of the requested sample would not end within ~2.5 minutes, shrink the sample
    # mesh (the cost is proportional to the number of cells; the rate in DoF/s is what is reported) -- except
    # under --dump-outputs, whose output must depend on the arguments only, not on the speed of the host
    ndofs, dt, kv = cpu_operator_sample(cells, args.P, threads)
    budget = 150.0
    if dt * args.steps > budget and cells > 8 and not args.dump_outputs:
        cells = max(8, int(cells * (budget / (dt * args.steps)) ** (1.0 / 3.0)))
        ndofs, dt, kv = cpu_operator_sample(cells, args.P, threads)
    t = [dt]
    for _ in range(args.steps - 1):
        ndofs, dt, kv = cpu_operator_sample(cells, args.P, threads)
        t.append(dt)
    if args.dump_outputs:
        idx = dump_sample_index(kv.size)
        dump_outputs(args.dump_outputs, {"kv": kv if idx is None else kv[idx]})
    ms = 1e3 * float(np.mean(t))
    value = ndofs / (ms * 1e-3) / 1e9
    sample = f"{cells}^3 cells P{args.P} ({ndofs} dofs) " + CPU_KIND["how"].format(t=threads)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"stiffness+mass apply, P{args.P} hex, fp64 (the reference's CPU operator; bounded sample)",
                       "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": CPU_KIND["kind"], "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---- product arm ------------------------------------------------------------------------------------
def run_b200(args):
    import ctypes as C

    import torch
    import torch.distributed as dist
    import wave_fenics_b200 as wfx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = wfx.Context.get(local_rank)
    P, N = args.P, args.cells
    from wave_fenics_b200 import partition
    grid = partition.rank_grid(world)

    halo = None
    if args.scaling == "strong":
        gshape = (args.global_cells,) * 3
        glen = (L, L, L)
    else:
        gshape = tuple(N * g for g in grid)
        glen = tuple(L * g for g in grid)
    if world == 1:
        mesh = wfx.create_box_hex(gshape, P, glen, perturb=args.perturb)
    else:
        mesh = partition.create_box_hex_partition(gshape, P, glen, grid, rank, perturb=args.perturb)
        halo = partition.make_halo(mesh, ctx, np.float64)
    t_setup = time.perf_counter()
    geo = wfx.Geometry(mesh, P, ctx=ctx)
    stiff = wfx.StiffnessOperator(mesh, P, ctx=ctx, geometry=geo)
    mass = wfx.MassOperator(mesh, P, ctx=ctx, geometry=geo)
    t_setup = time.perf_counter() - t_setup
    info = stiff.info()
    kernel_info = stiff.kernel_info()
    halo_transport = halo.transport if halo is not None else None
    if halo is not None:
        mass.assemble(halo)
    minv_ptr = mass.inverse_diagonal_ptr()

    dev = torch.device("cuda", local_rank)
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    x = torch.randn(mesh.ndofs, dtype=torch.float64, device=dev, generator=g)
    if halo is not None:
        halo.update_fwd(x)  # ghost copies of the input agree with their owners (scatter_fwd, LinearGLL.hpp:164)
    y = torch.empty_like(x)

    # high priority: the small pack / exchange / unpack kernels must not queue behind the interior batches
    comm_stream = torch.cuda.Stream(device=dev, priority=-1) if halo is not None else None

    def step():
        if halo is None:
            stiff.apply_scaled(x, minv_ptr, y)
        else:
            # interface cells -> their ghost reduction (+ 1/m on the owner) on a side stream while
            # the interior cells run with the fused 1/m; shared dofs are never scaled in-kernel
            main = torch.cuda.current_stream()
            stiff.apply_part(x, y, 0, beta=0, scale_ptr=minv_ptr)
            comm_stream.wait_stream(main)
            halo.update_rev_fwd_scaled(y, minv_ptr, stream=comm_stream.cuda_stream)
            stiff.apply_part(x, y, 1, beta=0, scale_ptr=minv_ptr)
            main.wait_stream(comm_stream)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def global_h_min(m):
        """mesh::h minimum over all ranks (MPI_Reduce MIN + Bcast, demo/cpu_planar3d/main.cpp:57-58)"""
        t = torch.tensor([m.h_min], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t.item())

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def windows(fn, sizes):
        """sum(sizes) calls of fn back to back, an event after each window of sizes[i] calls, barrier +
        synchronize before the first and after the last: device time of each window on this rank in ms"""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(sizes) + 1)]
        sync_all()
        ev[0].record()
        for i, k in enumerate(sizes):
            for _ in range(k):
                fn()
            ev[i + 1].record()
        sync_all()
        return [ev[i].elapsed_time(ev[i + 1]) for i in range(len(sizes))]

    win_steps = [len(s) for s in np.array_split(np.arange(args.steps), args.windows)]
    # the sampler (a forked nvidia-smi) starts BEFORE the first barrier of the timed windows, the warm-up after
    # it, directly before the timed applies: with the warm-up first, the first window measured slower than the
    # next (DESIGN.md section 5)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    sync_all()
    for _ in range(args.warmup):
        step()
    tw0 = time.time()
    win_local = windows(step, win_steps)
    tw1 = time.time()
    if args.dump_outputs and rank == 0:
        idx = dump_sample_index(mesh.ndofs)
        kv = y if idx is None else y[torch.from_numpy(idx).to(dev)]
        dump_outputs(args.dump_outputs, {"kv": kv.cpu().numpy()})
    win_ms = max_over_ranks(win_local)
    ms = float(np.median([w / k for w, k in zip(win_ms, win_steps)]))
    ndofs_global = mesh.ndofs_global
    value = ndofs_global / (ms * 1e-3) / 1e9

    # sustained: one window of >= args.sustain_s seconds of back-to-back applies (power cap territory)
    sustained = None
    if args.sustain_s > 0:
        k_sus = max(args.steps, int(np.ceil(args.sustain_s * 1e3 / ms)))
        ts0 = time.time()
        ms_sus = max_over_ranks(windows(step, [k_sus]))[0] / k_sus
        ts1 = time.time()
        sustained = {"ms_per_step": ms_sus, "steps": k_sus, "value": ndofs_global / (ms_sus * 1e-3) / 1e9}
    if rank == 0:
        sampler.stop()
    clocks = sampler.summary(tw0, tw1) if rank == 0 else None
    if rank == 0 and sustained:
        sustained["clocks"] = sampler.summary(ts0 + 0.1, ts1)

    # correctness of what was just timed, inside the run: the product path against an independent
    # second GPU implementation (per-cell kernel, coloured cells, global read-modify-write; plain
    # ghost reduction, then b/m), and bitwise agreement of all copies of a rank-shared dof.
    parity = None
    if not args.no_parity:
        simple = wfx.StiffnessOperator(mesh, P, ctx=ctx, geometry=geo, mode=wfx.capi.STIFF_CELL_COLOUR)
        step()
        y2 = torch.empty_like(x)
        simple.apply(x, y2, beta=0)
        if halo is not None:
            halo.update_rev_fwd(y2)
        minv = torch.from_numpy(mass.inverse_diagonal()).to(dev)
        y2 *= minv
        sl = mesh.size_local
        num = torch.stack([((y[:sl] - y2[:sl]) ** 2).sum(), (y2[:sl] ** 2).sum()])
        ghosts_equal = 1
        if halo is not None:
            dist.all_reduce(num)
            z = y.clone()
            halo.update_fwd(z)
            ge = torch.tensor([int(torch.equal(z, y))], device=dev)
            dist.all_reduce(ge, op=dist.ReduceOp.MIN)
            ghosts_equal = int(ge.item())
        rel = float(torch.sqrt(num[0] / num[1]).item())
        parity = {"rel_l2_vs_cell_kernel": rel, "tol": 1e-12, "ghost_copies_bitwise_equal": bool(ghosts_equal),
                  "ok": bool(rel < 1e-12 and ghosts_equal)}
        del simple, y2, minv
        assert parity["ok"], f"in-run parity check failed: {parity}"

    # structured fast path (SURVEY 8f-2): the same mesh without the vertex perturbation -- every cell a
    # parallelepiped, G = w_q * A_cell, 6 scalars per cell, per-point G never read.  Separate roofline
    # with its own algorithmic bytes.
    affine = None
    if world == 1 and not args.no_affine and args.perturb > 0:
        mesh_a = wfx.create_box_hex(gshape, P, glen, perturb=0.0)
        geo_a = wfx.Geometry(mesh_a, P, ctx=ctx)
        stiff_a = wfx.StiffnessOperator(mesh_a, P, ctx=ctx, geometry=geo_a)
        mass_a = wfx.MassOperator(mesh_a, P, ctx=ctx, geometry=geo_a)
        minv_a = mass_a.inverse_diagonal_ptr()
        ki_a, info_a = stiff_a.kernel_info(), stiff_a.info()
        for _ in range(args.warmup):
            stiff_a.apply_scaled(x, minv_a, y)
        wa = [w / k for w, k in zip(windows(lambda: stiff_a.apply_scaled(x, minv_a, y), win_steps), win_steps)]
        ms_a = float(np.median(wa))
        # parity of the fast path inside the run: against the per-cell kernel on the per-point G
        simple_a = wfx.StiffnessOperator(mesh_a, P, ctx=ctx, geometry=geo_a, mode=wfx.capi.STIFF_CELL_COLOUR)
        ya = torch.empty_like(x)
        simple_a.apply(x, ya, beta=0)
        ya *= torch.from_numpy(mass_a.inverse_diagonal()).to(dev)
        rel_a = float(((y - ya).norm() / ya.norm()).item())
        assert rel_a < 1e-12, f"affine fast path differs from the general kernel: {rel_a}"
        affine = {"ms_per_step": ms_a, "value": mesh_a.ndofs / (ms_a * 1e-3) / 1e9, "unit": UNIT,
                  "kernel": ki_a, "bytes_per_step": info_a["bytes"], "windows_ms_per_step": wa,
                  "rel_l2_vs_cell_kernel_general_G": rel_a}
        del simple_a, ya, stiff_a, mass_a, geo_a, mesh_a

    # end-to-end through the C-ABI host entry point, pinned host buffers, copies in the timed region
    xh = torch.empty(mesh.ndofs, dtype=torch.float64).pin_memory()
    yh = torch.empty(mesh.ndofs, dtype=torch.float64).pin_memory()
    xh.copy_(x)
    n_e2e = max(3, min(args.steps, 10))
    if world == 1:
        call = lambda: wfx.capi.call("wfx_stiffness_mass_apply_host", stiff.handle, mass.handle,
                                     C.c_void_p(xh.data_ptr()), C.c_void_p(yh.data_ptr()))
        for _ in range(3):
            call()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            call()
        dt1 = (time.perf_counter() - t0) / n_e2e
        step()
        assert torch.equal(yh, y.cpu()), "host-path result differs from device path"
        # the same through the multi-vector entry point: n_e2e DIFFERENT host vectors (one per step), every
        # step's input copied host -> device and its result device -> host inside the timed call; copy-in,
        # apply and copy-out of consecutive vectors are pipelined on three streams
        nv = n_e2e
        xs = [torch.empty(mesh.ndofs, dtype=torch.float64).pin_memory() for _ in range(nv)]
        ys = [torch.empty(mesh.ndofs, dtype=torch.float64).pin_memory() for _ in range(nv)]
        for i, t in enumerate(xs):
            t.copy_(xh)
            t[:1000] += float(i)  # distinct inputs
        xp = (C.c_void_p * nv)(*[t.data_ptr() for t in xs])
        yp = (C.c_void_p * nv)(*[t.data_ptr() for t in ys])
        batch = lambda: wfx.capi.call("wfx_stiffness_mass_apply_host_batch", stiff.handle, mass.handle, nv, xp, yp)
        batch()
        t0 = time.perf_counter()
        batch()
        dtb = (time.perf_counter() - t0) / nv
        assert torch.equal(ys[0], yh), "pipelined host path differs from the single-vector host path"
        x.copy_(xs[nv - 1])
        step()
        assert torch.equal(ys[nv - 1], y.cpu()), "pipelined host path differs from the device path"
        x.copy_(xh)
        e2e = {"value": mesh.ndofs / dtb / 1e9, "unit": UNIT, "h2d_bytes_per_step": mesh.ndofs * 8,
               "d2h_bytes_per_step": mesh.ndofs * 8, "ms_per_step": dtb * 1e3,
               "api": f"wfx_stiffness_mass_apply_host_batch: {nv} host vectors per call, H2D | apply | D2H pipelined over "
                      "three streams (PCIe full duplex); every vector is copied in and its result copied out",
               "single_vector_call": {"value": mesh.ndofs / dt1 / 1e9, "ms_per_step": dt1 * 1e3,
                                      "api": "wfx_stiffness_mass_apply_host (H2D, apply, D2H strictly in order)"}}
        del xs, ys
    else:
        # every rank: its part of x from pinned host memory, the distributed apply (halo included),
        # its part of the result back to pinned host memory
        def host_step():
            x.copy_(xh, non_blocking=True)
            step()
            yh.copy_(y, non_blocking=True)
            torch.cuda.synchronize()

        for _ in range(3):
            host_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            host_step()
        sync_all()
        dt = max_over_ranks([(time.perf_counter() - t0) / n_e2e])[0]
        nb = torch.tensor([mesh.ndofs * 8], dtype=torch.int64, device=dev)
        dist.all_reduce(nb)
        e2e = {"value": ndofs_global / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(nb.item()),
               "d2h_bytes_per_step": int(nb.item()), "ms_per_step": dt * 1e3,
               "note": "per-rank pinned buffers; bytes summed over ranks"}

    # second half of the BASELINE metric: one full RK4 step (4 x stiffness + boundary term +
    # halo + fused stage update) of the wave model on the same mesh, through wfx_wave_rk4
    rk4 = None
    if not args.no_rk4:
        del x, y
        eqn = wfx.LinearGLLOpt(mesh, None, P, 1500.0, 0.5e6, 6e4, ctx=ctx, halo=halo)
        eqn.init()
        dt_w = wfx.cfl_timestep(global_h_min(mesh), 1500.0, P, 0.5e6)
        eqn.rk4(0.0, 1.0, dt_w, max_steps=2)
        k_rk = max(3, min(args.steps, 10))
        rk_local = []
        for w in range(3):
            sync_all()
            ev0.record()
            eqn.rk4((2 + w * k_rk) * dt_w, 1.0, dt_w, max_steps=k_rk)
            ev1.record()
            sync_all()
            rk_local.append(ev0.elapsed_time(ev1) / k_rk)
        rk_ms = max_over_ranks(rk_local)
        ms_rk = float(np.median(rk_ms))
        u_chk, _ = eqn.get_state()
        # (the wave starts at x = 0: ranks away from the source face are still at rest)
        assert np.isfinite(u_chk).all() and (rank != 0 or np.abs(u_chk).max() > 0)
        # algorithmic bytes per step (DESIGN.md section 5): 4 stages x (G + dofmap + read un +
        # write b) + the fused stage updates (10 + 11 + 11 + 7 vector passes)
        s8 = 8
        b_step = 4 * (info["num_cells"] * info["num_dofs"] * (6 * s8 + 4) + mesh.ndofs * 2 * s8) + 39 * mesh.ndofs * s8
        rk4 = {"ms_per_step": ms_rk, "windows_ms_per_step": rk_ms, "steps": k_rk, "dofs_global": int(ndofs_global),
               "gdof_steps_per_s": ndofs_global / (ms_rk * 1e-3) / 1e9,
               "bytes_per_step_per_gpu": b_step, "achieved_gbs_per_gpu": b_step / (ms_rk * 1e-3) / 1e9}

    # BASELINE configs[3] inside the default run, so that the driver's 1/2/4/8 series carries the
    # strong-scaling numbers too: the full RK4 step on a FIXED 128^3-cell global mesh (135 M dofs) split
    # over the N ranks.  At N = 8 with the default 64^3 cells per GPU it is the weak-scaling mesh itself.
    strong = None
    if not args.no_strong and not args.no_rk4 and args.scaling == "weak":
        sshape = (args.global_cells,) * 3
        if sshape == tuple(gshape) and rk4:
            strong = {"global_cells": list(sshape), "dofs_global": int(ndofs_global), "rk4_ms_per_step": rk4["ms_per_step"],
                      "note": "same mesh and run as the weak-scaling rk4 figure"}
        elif all(sshape[a] % grid[a] == 0 for a in range(3)):
            del eqn, stiff, mass, geo
            torch.cuda.empty_cache()
            if world == 1:
                smesh, shalo = wfx.create_box_hex(sshape, P, (L, L, L), perturb=args.perturb), None
            else:
                smesh = partition.create_box_hex_partition(sshape, P, (L, L, L), grid, rank, perturb=args.perturb)
                shalo = partition.Halo(smesh, ctx, np.float64, comm=halo.comm)
            seqn = wfx.LinearGLLOpt(smesh, None, P, 1500.0, 0.5e6, 6e4, ctx=ctx, halo=shalo)
            seqn.init()
            dt_s = wfx.cfl_timestep(global_h_min(smesh), 1500.0, P, 0.5e6)
            seqn.rk4(0.0, 1.0, dt_s, max_steps=2)
            k_s = 5
            loc = []
            for w in range(3):
                sync_all()
                ev0.record()
                seqn.rk4((2 + w * k_s) * dt_s, 1.0, dt_s, max_steps=k_s)
                ev1.record()
                sync_all()
                loc.append(ev0.elapsed_time(ev1) / k_s)
            s_ms = max_over_ranks(loc)
            u_s, _ = seqn.get_state()
            assert np.isfinite(u_s).all()
            strong = {"global_cells": list(sshape), "dofs_global": int(smesh.ndofs_global),
                      "rk4_ms_per_step": float(np.median(s_ms)), "windows_ms_per_step": s_ms,
                      "cells_per_gpu": list(smesh.shape), "halo_transport": shalo.transport if shalo is not None else None}
            del seqn, smesh

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peak()
    if rk4:
        rk4["frac_of_hbm_peak"] = rk4["achieved_gbs_per_gpu"] / peak
    # dominant kernel = stiff_brick_kernel: the step is its `nlaunches` colour launches, so the
    # kernel's average launch duration is ms / nlaunches and its algorithmic bytes per launch are
    # bytes / nlaunches (DESIGN.md section 5); achieved = bytes per step / step time.
    nc_nd = info["num_cells"] * info["num_dofs"]
    bytes_no_dofmap = info["bytes"] - 4.0 * nc_nd
    achieved = info["bytes"] / (ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and args.cells == 64 and P == 4 and args.scaling == "weak":
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "kernel": "stiff_brick_kernel",
                "bytes_per_step": info["bytes"], "launches_per_step": info["nlaunches"],
                # the regular-brick kernel never reads a per-point dofmap (positions are arithmetic; it reads
                # one int32 per brick DOF instead): the same time against the bytes without the +4 B/point term
                "frac_no_dofmap": bytes_no_dofmap / (ms * 1e-3) / 1e9 / peak,
                "limiter": "HBM is the bounding roofline; the measured DRAM traffic over this step time is "
                           "dram_traffic_gbs (about 0.8 of the copy bandwidth: ~2400 concurrent 6-KB streams plus "
                           "scattered 136-byte rows); the rest is the 1.14x traffic overhead and load latency at "
                           "16 warps per SM (DESIGN.md section 6)"}
    if traffic:
        # what DRAM actually moved per step (ncu bytes of one launch x launches) over the measured step time
        roofline["dram_traffic_gbs"] = traffic * info["nlaunches"] / (ms * 1e-3) / 1e9
        roofline["dram_traffic_frac"] = roofline["dram_traffic_gbs"] / peak
    if sustained:
        roofline["sustained"] = {"ms_per_step": sustained["ms_per_step"], "steps": sustained["steps"],
                                 "achieved": info["bytes"] / (sustained["ms_per_step"] * 1e-3) / 1e9,
                                 "frac": info["bytes"] / (sustained["ms_per_step"] * 1e-3) / 1e9 / peak,
                                 "peak": peak, "clocks": sustained.get("clocks")}
    if affine:
        ach_a = affine["bytes_per_step"] / (affine["ms_per_step"] * 1e-3) / 1e9
        affine["roofline"] = {"bound": "hbm", "achieved": ach_a, "peak": peak, "unit": "GB/s", "frac": ach_a / peak,
                              "note": "algorithmic bytes of the fast path: 6 scalars of G per cell + x, 1/m, y once"}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        nd_cpu, t_cpu, _ = cpu_operator_sample(args.ref_cells, P, threads)
        cpu = {"value": nd_cpu / t_cpu / 1e9, "unit": UNIT, "cores": threads, "kind": CPU_KIND["kind"],
               "sample": f"{args.ref_cells}^3 cells P{P} ({nd_cpu} dofs), " + CPU_KIND["how"].format(t=threads)}
    s = 8
    g_bytes, vec_bytes = 6 * s * nc_nd, 3 * s * mesh.ndofs
    shape = "x".join(map(str, mesh.shape))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"stiffness+mass apply kv=M^-1(-c0^2 K u), {shape} hex cells per GPU, P{P}, fp64, "
                                   f"{'perturbed (non-affine)' if args.perturb else 'affine'} geometry, general 6-entry G per point",
                       "cells_per_gpu": int(info["num_cells"]), "dofs_global": int(ndofs_global), "degree": P,
                       "l2_policy": f"inputs larger than L2 (G {g_bytes / 1e9:.2f} GB + vectors {vec_bytes / 1e9:.2f} GB per apply "
                                    f"vs 126 MB L2); no flush needed",
                       "dofmap": "brick-implicit (one int32 per brick dof, no per-point dofmap is read): see roofline.frac_no_dofmap",
                       "timing": f"{args.steps} applies back to back in {len(win_steps)} windows of {win_steps} applies, "
                                 "median window time per apply, max over ranks per window",
                       "partition": "x".join(map(str, grid)), "setup_s": round(t_setup, 2),
                       "kernel": kernel_info, "halo_transport": halo_transport},
            "windows_ms": win_ms, "window_steps": win_steps, "window_ms_min": min(win_ms), "window_ms_max": max(win_ms),
            "clocks": clocks, "sustained": sustained, "parity": parity, "affine_fast_path": affine,
            "e2e": e2e,
            # per apply: the colour launches of the brick kernel + the ghost reduction (one fused kernel over
            # peer memory; pack, unpack-add, pack, unpack around two NCCL groups otherwise)
            "gpu_launches": args.steps * (info["nlaunches"] + (0 if halo is None else (1 if halo_transport == "p2p" else 4))),
            "roofline": roofline, "cpu_baseline": cpu, "rk4": rk4, "strong_scaling": strong}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed applies; default 140 (b200 arm), 5 (reference arm)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--windows", type=int, default=7,
                    help=f"windows the timed applies are split into, each of at least {MIN_WINDOW_STEPS} applies "
                         "(one when --steps is smaller); the median is reported")
    ap.add_argument("--sustain-s", type=float, default=0.6, help="length of the sustained window in seconds (0 = skip)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cells", type=int, default=64, help="weak scaling: cells per axis per GPU")
    ap.add_argument("--global-cells", type=int, default=128, help="strong scaling: cells per axis of the global mesh")
    ap.add_argument("--P", type=int, default=4)
    ap.add_argument("--perturb", type=float, default=0.15)
    ap.add_argument("--ref-cells", type=int, default=48, help="CPU sample mesh (cells per axis)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-rk4", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-affine", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the 128^3 strong-scaling RK4 sub-measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output kv to DIR/kv.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 140 if args.impl == "b200" else 5
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.windows = max(1, min(args.windows, args.steps // MIN_WINDOW_STEPS))
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
