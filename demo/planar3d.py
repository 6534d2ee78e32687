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
The reference reads `../mesh.xdmf` (not in its repository); here the mesh is a structured
n x m x m hexahedral box with tag 1 on x = 0 (source) and tag 2 on x = L (absorbing).

    python demo/planar3d.py [--nx 32] [--nyz 4] [--length 0.1] [--steps N] [--check]
                            [--model linear|lossy|westervelt] [--stats-periods K] [--focus DEPTH] [--aperture R]
                            [--heat-seconds S] [--cool-seconds C] [--absorption ALPHA0] [--absorption-power Y]
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
    args = ap.parse_args()
    if args.heat_seconds > 0 and args.stats_periods <= 0:
        ap.error("--heat-seconds needs --stats-periods (the heat source comes from the harmonic maps)")

    speedOfSound, sourceFrequency, pressureAmplitude = 1500.0, 0.5e6, 60000.0   # main.cpp:25-30
    period = 1.0 / sourceFrequency
    domainLength = args.length                                                   # :33
    degreeOfBasis = 4                                                            # :36
    side = domainLength / args.nx
    width = side * args.nyz
    tags = ((0, 0, 1), (0, 1, 2))
    if args.focus > 0:
        tags += ((1, 0, 2), (1, 1, 2), (2, 0, 2), (2, 1, 2))
    mesh = wfx.create_box_hex((args.nx, args.nyz, args.nyz), degreeOfBasis, (domainLength, width, width), tags=tags)
    timeStepSize = wfx.cfl_timestep(mesh.h_min, speedOfSound, degreeOfBasis, sourceFrequency)  # :61-66
    startTime, finalTime = 0.0, domainLength / speedOfSound + 8.0 / sourceFrequency            # :63-64
    print(f"Number of step per period: {int(round(period / timeStepSize))}")
    print(f"dt = {timeStepSize:.15g}")
    nstep = int((finalTime - startTime) / timeStepSize + 1)
    delta = 0.0 if args.model == "linear" else args.delta
    beta = args.beta if args.model == "westervelt" else 0.0
    if args.model == "linear":
        eqn = wfx.LinearGLLOpt(mesh, None, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude)  # :75
    else:
        eqn = wfx.WesterveltGLLOpt(mesh, None, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                                   delta, beta, args.rho0)
    print(f"Number of steps: {nstep}")
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
            if args.focus > 0:
                print(f"on-axis maximum: |p1| = {p1.max():.6e} at x = {x[p1.argmax()]:.5f}, "
                      f"pmax = {pmax.max():.6e} at x = {x[pmax.argmax()]:.5f} (focus requested at x = {args.focus:.5f})")
        if args.heat_seconds > 0 and fs.samples == 0:
            print("thermal: skipped, the statistics window holds no samples (no heat source without harmonics)")
        elif args.heat_seconds > 0:
            heat(args, eqn, speedOfSound)
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


def heat(args, eqn, c0, k=0.5, rhoc=3.6e6, perfusion=2.0e3, T_art=37.0):
    """HIFU heating from the wave model's harmonic maps: soft-tissue-like k [W/(m K)], rhoC [J/(m^3 K)] and
    perfusion wbCb [W/(m^3 K)], all faces insulated"""
    th = wfx.PennesGLL.from_wave(eqn, k, rhoc, perfusion, T_art)
    th.heat_from_wave(eqn, args.absorption, args.absorption_power, args.rho0, c0)
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
