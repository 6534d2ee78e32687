#!/usr/bin/env python
"""The cpu_planar3d demo (demo/cpu_planar3d/main.cpp:14-98) on the B200 path.

Same physical set-up and control flow as the reference driver: speed of sound 1500 m/s, source
0.5 MHz, amplitude 60 kPa, domain length 0.1 m, degree 4, CFL time step snapped to whole steps
per period, final time L/c0 + 8/f0, LinearGLLOpt.init() then .rk4(t0, tf, dt), "Solve time".
--model lossy / westervelt runs the lossy or Westervelt model instead (DESIGN.md section 4.5a) with water-like
defaults: diffusivity of sound 4.33e-6 m^2/s, coefficient of nonlinearity 3.5, density 1000 kg/m^3.
--stats-periods K accumulates field statistics on the device over the last K periods of the run (DESIGN.md
section 4.5b) and prints, along the x axis, the peak positive and negative pressure and, at the absorbing end, the
fundamental's amplitude and the second harmonic's share of it.  The harmonics are exact Fourier components only
over whole periods of whole steps, so the run then stops on the last whole step before the final time (a shortened
last step would be a sample off the uniform grid) and exactly K * (steps per period) steps are sampled.
--focus DEPTH focuses the source (DESIGN.md section 4.5c): per-dof delays from focus_delays for a focus at x = DEPTH
on the axis through the centre of the source face, and the four lateral faces absorbing (tag 2) instead of rigid;
--aperture R switches the source off outside radius R of the face centre.  With --stats-periods the field statistics
are then reported along that axis: the position and value of the maximum of |p1| and of pmax.  For a small
aperture (Fresnel number a^2 / (lambda DEPTH) of a few) that maximum lies short of DEPTH, as the Rayleigh integral
predicts.
--heat-seconds S (with --stats-periods) heats tissue with the acoustic field (DESIGN.md section 4.5d): a Pennes thermal
model on the same mesh and operators takes its heat source Q = sum_h alpha0 (h f0 / 1 MHz)^y |p_h|^2 / (rho0 c0) from
the harmonic maps, is heated for S seconds and cools for --cool-seconds C with the source off, and reports the peak
temperature rise, the maximum CEM43 thermal dose, and the number of dofs and the volume at or above 240 min.
--absorption alpha0 [Np/m at 1 MHz] and --absorption-power y set the tissue absorption.
--layer X0 X1 --layer-rho R --layer-c C [--layer-beta B] puts a slab of another medium across the beam (DESIGN.md
section 4.5e): the cells whose centres lie in X0 < x < X1 get density R, speed of sound C and, for the Westervelt
model, coefficient of nonlinearity B (default --beta); the rest is water (1000 kg/m^3, 1500 m/s, --beta).  The time
step comes from the largest speed of sound.  With --stats-periods the on-axis |p1| is reported before and after the
slab; with --heat-seconds the thermal model is built on its own operators and heated with the per-dof 1 / (rho c).
--relaxation M [--band F_LO F_HI] (lossy / westervelt) makes the wave itself lose energy with the same power law that
heats (DESIGN.md section 4.5f): M relaxation processes fitted to --absorption (f / 1 MHz)^--absorption-power over the
band (default f0 / 2 .. 3 f0) in the tissue -- the slab with --layer (water keeps delta), else the whole domain.  It
reports the fit error and the phase speed at f0; the time step is also kept below the relaxation's bound.
--pml WIDTH replaces every absorbing face -- the far end and, with --focus, the four lateral faces -- by a perfectly
matched layer (DESIGN.md section 4.5g) WIDTH deep inside the domain (PML.box, R0 = 1e-4) with rigid outer faces, so
that a focused beam's side lobes leave the domain instead of coming back into the maps; it prints the layer's cells,
dofs and largest damping, and keeps the time step below the layer's bound.
--time-reversal (with --focus and --stats-periods; linear or lossy model) focuses by time reversal (DESIGN.md section
4.5h): an emission run from a point source at the focus with the array silent (profile amplitude 0), the first
harmonic on tag 1 conjugated (phase_conjugate_delays), then a treatment run with those delays and one with the
geometric delays of --focus.  It prints the focal |p1| (the point source's weights as a sensor) of both treatments and
the reciprocity prediction of each from the emission, sum_i m1_i a_i exp(-i w tau_i) (1 + i w delta / c0^2) p1_i.
The reference reads `../mesh.xdmf` (not in its repository); here the mesh is a structured
n x m x m hexahedral box with tag 1 on x = 0 (source) and tag 2 on x = L (absorbing).

    python demo/planar3d.py [--nx 32] [--nyz 4] [--length 0.1] [--steps N] [--check]
                            [--model linear|lossy|westervelt] [--stats-periods K] [--focus DEPTH] [--aperture R]
                            [--heat-seconds S] [--cool-seconds C] [--absorption ALPHA0] [--absorption-power Y]
                            [--layer X0 X1 --layer-rho R --layer-c C [--layer-beta B]]
                            [--relaxation M [--band F_LO F_HI]] [--pml WIDTH] [--time-reversal]
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wave_fenics_b200 as wfx  # noqa: E402


def stats_window(t0, tf, dt, k, periods, max_steps=0):
    """(run_tf, run_steps, t_start) for field statistics over the last `periods` periods of k steps each: the run
    takes nw whole steps (the last whole step at or before tf, or max_steps) and stops there, and the last
    periods * k of them are sampled.  t_start - dt/2, the threshold of the sampling rule, lies half a step past
    the step before the window, so rounding in the accumulated time cannot move the window's edge."""
    nw = int(np.floor((tf - t0) / dt + 1e-9))
    if max_steps > 0:
        nw = min(nw, max_steps)
    nsamples = min(periods * k, nw)
    return t0 + (nw + 0.5) * dt, nw, t0 + (nw - nsamples + 1) * dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=32, help="cells along the propagation direction")
    ap.add_argument("--nyz", type=int, default=4, help="cells across")
    ap.add_argument("--steps", type=int, default=0, help="stop after this many steps (0: run to the final time)")
    ap.add_argument("--check", action="store_true", help="compare with the CPU oracle (small meshes)")
    ap.add_argument("--model", choices=("linear", "lossy", "westervelt"), default="linear")
    ap.add_argument("--delta", type=float, default=4.33e-6, help="diffusivity of sound [m^2/s] (lossy, westervelt)")
    ap.add_argument("--beta", type=float, default=3.5, help="coefficient of nonlinearity (westervelt)")
    ap.add_argument("--rho0", type=float, default=1000.0, help="density [kg/m^3] (westervelt)")
    ap.add_argument("--stats-periods", type=int, default=0,
                    help="field statistics (peaks, harmonics) over the last K periods of the run (0: off)")
    ap.add_argument("--length", type=float, default=0.1, help="domain length along x [m]")
    ap.add_argument("--focus", type=float, default=0.0,
                    help="focal depth [m] on the axis through the centre of the source face (0: plane source)")
    ap.add_argument("--aperture", type=float, default=0.0,
                    help="with --focus: source radius [m] around the face centre (0: the whole face)")
    ap.add_argument("--heat-seconds", type=float, default=0.0,
                    help="with --stats-periods: heat tissue with the field's harmonic maps for S seconds (0: off)")
    ap.add_argument("--cool-seconds", type=float, default=0.0, help="cooling after the heating, source off")
    ap.add_argument("--absorption", type=float, default=5.0, help="tissue absorption alpha0 [Np/m at 1 MHz]")
    ap.add_argument("--absorption-power", type=float, default=1.1, help="frequency power law y of the absorption")
    ap.add_argument("--layer", type=float, nargs=2, metavar=("X0", "X1"), default=None,
                    help="a slab of another medium across the beam between x = X0 and x = X1 [m]")
    ap.add_argument("--layer-rho", type=float, default=1900.0, help="with --layer: the slab's density [kg/m^3]")
    ap.add_argument("--layer-c", type=float, default=2800.0, help="with --layer: the slab's speed of sound [m/s]")
    ap.add_argument("--layer-beta", type=float, default=None,
                    help="with --layer: the slab's coefficient of nonlinearity (default --beta)")
    ap.add_argument("--relaxation", type=int, default=0, choices=(0, 1, 2, 3),
                    help="absorb the wave in the tissue with M relaxation processes (lossy, westervelt; 0: off)")
    ap.add_argument("--band", type=float, nargs=2, metavar=("F_LO", "F_HI"), default=None,
                    help="with --relaxation: the fitted band [Hz] (default f0 / 2 .. 3 f0)")
    ap.add_argument("--pml", type=float, default=0.0, metavar="WIDTH",
                    help="a perfectly matched layer WIDTH [m] deep in place of the absorbing faces (0: off)")
    ap.add_argument("--time-reversal", action="store_true",
                    help="with --focus and --stats-periods: time-reversal delays from a point source at the focus")
    args = ap.parse_args()
    if args.time_reversal and (args.focus <= 0 or args.stats_periods <= 0):
        ap.error("--time-reversal needs --focus (the target) and --stats-periods (the harmonic maps)")
    if args.time_reversal and (args.model == "westervelt" or args.check or args.heat_seconds > 0):
        ap.error("--time-reversal needs a linear model (--model linear or lossy) and takes no --check or --heat-seconds")
    if args.pml < 0:
        ap.error("--pml WIDTH needs WIDTH > 0")
    if args.pml > 0 and args.check:
        ap.error("--check compares with the oracle without a layer; it does not take --pml")
    if args.relaxation and args.model == "linear":
        ap.error("--relaxation needs --model lossy or westervelt (for linear tissue: --model lossy --delta 0)")
    if args.relaxation and args.check:
        ap.error("--check compares with the oracle without relaxation; it does not take --relaxation")
    if args.layer is not None and args.check:
        ap.error("--check compares with the homogeneous oracle; it does not take --layer")
    if args.layer is not None and not args.layer[0] < args.layer[1]:
        ap.error("--layer X0 X1 needs X0 < X1")
    if args.heat_seconds > 0 and args.stats_periods <= 0:
        ap.error("--heat-seconds needs --stats-periods (the heat source comes from the harmonic maps)")

    speedOfSound, sourceFrequency, pressureAmplitude = 1500.0, 0.5e6, 60000.0   # main.cpp:25-30
    period = 1.0 / sourceFrequency
    domainLength = args.length                                                   # :33
    degreeOfBasis = 4                                                            # :36
    side = domainLength / args.nx
    width = side * args.nyz
    absorbing = [(0, 1)]
    if args.focus > 0:
        absorbing += [(1, 0), (1, 1), (2, 0), (2, 1)]
    # with --pml the absorbing faces are rigid and the layer takes their place
    tags = ((0, 0, 1),) + (() if args.pml > 0 else tuple((a, s, 2) for a, s in absorbing))
    mesh = wfx.create_box_hex((args.nx, args.nyz, args.nyz), degreeOfBasis, (domainLength, width, width), tags=tags)
    pml = wfx.PML.box(mesh, args.pml, absorbing, speedOfSound) if args.pml > 0 else None
    medium = None
    if args.layer is not None:
        xc = mesh.x[mesh.xdofs, 0].mean(axis=1)                          # cell centres along x
        slab = (xc > args.layer[0]) & (xc < args.layer[1])
        beta_slab = args.beta if args.layer_beta is None else args.layer_beta
        medium = wfx.Medium(np.where(slab, args.layer_rho, 1000.0), np.where(slab, args.layer_c, speedOfSound),
                            np.where(slab, beta_slab, args.beta))
        print(f"layer: {int(slab.sum())} cells in {args.layer[0]:.4f} < x < {args.layer[1]:.4f} with rho = "
              f"{args.layer_rho:g}, c = {args.layer_c:g}, beta = {beta_slab:g}; Z ratio to water "
              f"{args.layer_rho * args.layer_c / (1000.0 * speedOfSound):.4f}")
    relaxation = None
    if args.relaxation:
        # the tissue: the slab (water elsewhere keeps delta), else every cell
        tissue = slab if args.layer is not None else np.ones(mesh.ncells, dtype=bool)
        rho = medium.rho if medium is not None else 1000.0
        c = medium.c if medium is not None else speedOfSound
        medium = wfx.Medium(rho, c, None if medium is None else medium.beta, alpha0=np.where(tissue, args.absorption, 0.0),
                            y=args.absorption_power)
        band = args.band or (0.5 * sourceFrequency, 3.0 * sourceFrequency)
        relaxation = medium.relaxation(band[0], band[1], args.relaxation)
        cell = int(np.argmax(tissue))
        print(f"relaxation: {relaxation.M} processes fitted to {args.absorption:g} (f / 1 MHz)^{args.absorption_power:g}"
              f" Np/m over {band[0]:.4g} .. {band[1]:.4g} Hz, fit error {relaxation.fit_error:.3e}; in the tissue "
              f"alpha(f0) = {relaxation.alpha(sourceFrequency)[cell]:.6e} Np/m, phase speed at f0 "
              f"{relaxation.phase_speed(sourceFrequency)[cell]:.4f} m/s (c = {np.broadcast_to(c, (mesh.ncells,))[cell]:g})")
    c_max = speedOfSound if medium is None else medium.c_max
    timeStepSize = wfx.cfl_timestep(mesh.h_min, c_max, degreeOfBasis, sourceFrequency)  # :61-66
    if relaxation is not None and timeStepSize >= relaxation.max_dt():
        timeStepSize = period / np.ceil(period / relaxation.max_dt())                  # whole steps per period
    if pml is not None and timeStepSize >= pml.max_dt():
        timeStepSize = period / np.ceil(period / pml.max_dt())
    startTime, finalTime = 0.0, domainLength / speedOfSound + 8.0 / sourceFrequency            # :63-64
    print(f"Number of step per period: {int(round(period / timeStepSize))}")
    print(f"dt = {timeStepSize:.15g}")
    nstep = int((finalTime - startTime) / timeStepSize + 1)
    delta = 0.0 if args.model == "linear" else args.delta
    beta = args.beta if args.model == "westervelt" else 0.0
    if args.model == "linear":
        eqn = wfx.LinearGLLOpt(mesh, None, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                               medium=medium, pml=pml)                                                     # :75
    else:
        if medium is not None and args.model == "lossy":
            # the lossy model stays linear
            medium = wfx.Medium(medium.rho, medium.c, alpha0=medium.alpha0, y=medium.y)
        eqn = wfx.WesterveltGLLOpt(mesh, None, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                                   delta, beta, args.rho0, medium=medium, relaxation=relaxation, pml=pml)
    print(f"Number of steps: {nstep}")
    if pml is not None:
        info = eqn.pml_info()
        print(f"pml: {info['cells']} cells, {info['dofs']} dofs, {args.pml:.4f} m deep on {len(absorbing)} faces, "
              f"zeta_max = {info['zeta_max']:.6e} 1/s")
    print(f"Degrees of freedom: {mesh.ndofs_global}")
    X = wfx.dof_coordinates(mesh)
    if args.focus > 0:
        face = np.abs(X[:, 0]) < 1e-12
        delay = np.zeros(mesh.ndofs)
        delay[face] = wfx.focus_delays(X[face], (args.focus, width / 2, width / 2), speedOfSound)
        amp = None
        if args.aperture > 0:
            amp = (np.hypot(X[:, 1] - width / 2, X[:, 2] - width / 2) <= args.aperture).astype(np.float64)
        eqn.set_source_profile(amp, delay)
        print(f"focused source: focus at x = {args.focus:.4f} on the face axis, "
              f"delays up to {delay.max():.4e} s, aperture {'whole face' if amp is None else args.aperture}")
    if args.time_reversal:
        k = int(round(period / timeStepSize))
        window = stats_window(startTime, finalTime, timeStepSize, k, args.stats_periods, args.steps)
        time_reversal(eqn, mesh, X, (args.focus, width / 2, width / 2), amp, delay, delta / speedOfSound ** 2,
                      sourceFrequency, startTime, timeStepSize, window)
        return
    eqn.init()                                                                   # :83
    run_tf, run_steps = finalTime, args.steps
    if args.stats_periods > 0:
        k = int(round(period / timeStepSize))
        run_tf, run_steps, t_start = stats_window(startTime, finalTime, timeStepSize, k, args.stats_periods, args.steps)
        eqn.set_field_stats(t_start, harmonics=2)
    eqn.ctx.synchronize()
    t0 = time.perf_counter()
    steps, t_end = eqn.rk4(startTime, run_tf, timeStepSize, max_steps=run_steps)  # :88
    eqn.ctx.synchronize()
    print(f"Solve time: {time.perf_counter() - t0:.6f}  ({steps} steps, t = {t_end:.6e})")   # :92
    u, v = eqn.get_state()
    if args.stats_periods > 0:
        fs = eqn.field_stats()
        # the dofs on the x axis (y = z = 0; with --focus the axis through the face centre), source to absorbing end
        yz = width / 2 if args.focus > 0 else 0.0
        line = np.where((np.abs(X[:, 1] - yz) < 1e-9 * width) & (np.abs(X[:, 2] - yz) < 1e-9 * width))[0]
        line = line[np.argsort(X[line, 0])]
        x = X[line, 0]
        pmax, pmin, p1, p2 = fs.pmax[line], fs.pmin[line], np.abs(fs.harmonics[0, line]), np.abs(fs.harmonics[1, line])
        whole = fs.samples == args.stats_periods * k
        print(f"field statistics over {fs.samples} steps ({fs.samples / k:g} periods of {k} steps"
              f"{'' if whole else ', fewer than asked: the run is shorter than the window'}), "
              f"t = {fs.t_first:.6e} .. {fs.t_last:.6e}")
        if fs.samples:
            print(f"along x: max pmax = {pmax.max():.6e} at x = {x[pmax.argmax()]:.4f}, "
                  f"min pmin = {pmin.min():.6e} at x = {x[pmin.argmin()]:.4f}")
            print(f"at the absorbing end (x = {x[-1]:.4f}): |p1| = {p1[-1]:.6e}, |p2|/|p1| = {p2[-1] / p1[-1]:.6e}")
            if args.layer is not None:
                before, after = x < args.layer[0], x > args.layer[1]
                for name, sel in (("before the layer", before), ("after the layer", after)):
                    if sel.any():
                        print(f"{name}: on-axis |p1| mean {p1[sel].mean():.6e}, max {p1[sel].max():.6e} "
                              f"({int(sel.sum())} dofs)")
            if args.focus > 0:
                print(f"on-axis maximum: |p1| = {p1.max():.6e} at x = {x[p1.argmax()]:.5f}, "
                      f"pmax = {pmax.max():.6e} at x = {x[pmax.argmax()]:.5f} (focus requested at x = {args.focus:.5f})")
        if args.heat_seconds > 0 and fs.samples == 0:
            print("thermal: skipped, the statistics window holds no samples (no heat source without harmonics)")
        elif args.heat_seconds > 0:
            heat(args, eqn, speedOfSound, medium)
    else:
        print(f"max |p| = {np.abs(u).max():.6e} at x = {X[np.abs(u).argmax(), 0]:.4f}")
    if args.check:
        from oracle import oracle
        G, detJ = oracle.precompute_geometric_data(mesh, degreeOfBasis)
        m = np.zeros(mesh.ndofs)
        oracle.mass_apply(mesh, degreeOfBasis, detJ, np.ones(mesh.ndofs), m)
        m1, m2 = oracle.boundary_facet_mass(mesh, degreeOfBasis)
        uo, vo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
        if args.focus > 0:
            from model_oracle import model_oracle
            model_oracle.rk4_westervelt_profile(mesh, degreeOfBasis, G, m, m1, m2, speedOfSound, sourceFrequency,
                                                pressureAmplitude, delta, beta, args.rho0, amp, delay, startTime,
                                                run_tf, timeStepSize, uo, vo, max_steps=run_steps, sumfact=True,
                                                nthreads=oracle.max_threads())
        elif args.model == "linear":
            oracle.rk4(mesh, degreeOfBasis, G, m, m1, m2, speedOfSound, sourceFrequency, pressureAmplitude,
                       startTime, run_tf, timeStepSize, uo, vo, max_steps=run_steps, sumfact=True,
                       nthreads=oracle.max_threads())
        else:
            from model_oracle import model_oracle
            model_oracle.rk4_westervelt(mesh, degreeOfBasis, G, m, m1, m2, speedOfSound, sourceFrequency,
                                        pressureAmplitude, delta, beta, args.rho0, startTime, run_tf,
                                        timeStepSize, uo, vo, max_steps=run_steps, sumfact=True,
                                        nthreads=oracle.max_threads())
        print(f"relative L2 difference to the CPU oracle: u {np.linalg.norm(u - uo) / np.linalg.norm(uo):.3e}"
              f"  v {np.linalg.norm(v - vo) / np.linalg.norm(vo):.3e}")


def time_reversal(eqn, mesh, X, focus, amp, delay, s_src, f0, t0, dt, window):
    """Emission from a point source at `focus` with the array silent, then treatments with the geometric delays and
    with the conjugate delays of the emission's first harmonic on tag 1; prints each focal |p1| and its reciprocity
    prediction from the emission (DESIGN.md section 4.5h)."""
    run_tf, run_steps, t_start = window
    fdofs, fq = wfx.point_source(mesh, focus)
    m1 = eqn.bnd_op.facet_masses()[0]
    face = m1 > 0
    a = np.ones(mesh.ndofs) if amp is None else amp

    def first_harmonic():
        eqn.init()
        eqn.set_field_stats(t_start, harmonics=1)
        eqn.rk4(t0, run_tf, dt, max_steps=run_steps)
        return eqn.field_stats().harmonics[0]

    eqn.set_source_profile(np.zeros(mesh.ndofs))
    eqn.set_volume_source(fdofs, fq)
    emission = first_harmonic()
    eqn.set_volume_source()
    w = 2.0 * np.pi * f0
    print(f"time reversal: emission from a point source at x = {focus[0]:.5f} ({len(fdofs)} dofs), "
          f"|p1| on tag 1 up to {np.abs(emission[face]).max():.6e}")
    conjugate = np.where(face, wfx.phase_conjugate_delays(emission, f0), 0.0)
    focal = {}
    for name, tau in (("geometric", delay), ("time-reversal", conjugate)):
        eqn.set_source_profile(amp, tau)
        focal[name] = fq @ first_harmonic()[fdofs]
        pred = np.sum(m1 * a * np.exp(-1j * w * tau) * (1.0 + 1j * w * s_src) * emission)
        print(f"time reversal: {name} delays: focal |p1| = {abs(focal[name]):.6e}, reciprocity prediction "
              f"{abs(pred):.6e} (difference {abs(focal[name] - pred):.3e})")
    print(f"time reversal: gain over the geometric delays {abs(focal['time-reversal']) / abs(focal['geometric']):.4f}")


def heat(args, eqn, c0, medium=None, k=0.5, rhoc=3.6e6, perfusion=2.0e3, T_art=37.0):
    """HIFU heating from the wave model's harmonic maps: soft-tissue-like k [W/(m K)], rhoC [J/(m^3 K)] and
    perfusion wbCb [W/(m^3 K)], all faces insulated.  In a layered medium the thermal model has operators of its own
    (the wave model's geometry is scaled) and the heat source uses the per-dof 1 / (rho c)."""
    if medium is None:
        th = wfx.PennesGLL.from_wave(eqn, k, rhoc, perfusion, T_art)
    else:
        th = wfx.PennesGLL(eqn.V, eqn.k_, k, rhoc, perfusion, T_art, dtype=eqn.dtype, ctx=eqn.ctx)
    if medium is not None and medium.alpha0 is not None:
        th.heat_from_wave(eqn, None, medium=medium)       # the absorption the wave relaxes with (--relaxation)
    else:
        th.heat_from_wave(eqn, args.absorption, args.absorption_power, args.rho0, c0, medium=medium)
    dt = th.stable_dt()
    th.init()
    eqn.ctx.synchronize()
    t0 = time.perf_counter()
    th.set_heat_scale(1.0)
    n1, t = th.rk4(0.0, args.heat_seconds, dt)
    T_heat = th.get_state()
    n2 = 0
    if args.cool_seconds > 0:
        th.set_heat_scale(0.0)
        n2, t = th.rk4(t, args.heat_seconds + args.cool_seconds, dt)
    eqn.ctx.synchronize()
    d = th.dose()
    lesion = d.cem43 >= 240.0
    m = eqn.mass_op.diagonal().astype(np.float64)
    print(f"thermal: Q max {th.heat_source().max():.6e} W/m^3, dt = {dt:.6e} s, {n1} heating + {n2} cooling steps "
          f"in {time.perf_counter() - t0:.3f} s")
    print(f"thermal: peak rise {d.T_max.max() - T_art:.6e} K (at the end of heating {T_heat.max() - T_art:.6e} K), "
          f"max CEM43 {d.cem43.max():.6e} min, {int(lesion.sum())} dofs >= 240 min, "
          f"volume {m[lesion].sum():.6e} m^3 >= 240 min")


if __name__ == "__main__":
    main()
