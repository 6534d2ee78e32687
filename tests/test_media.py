"""Layered acoustic media (DESIGN.md section 4.5e): per-cell density, sound speed and nonlinearity.

The model (1 / (rho c^2)) p_tt - div((1 / rho) grad p) [- loss] = (beta / (rho^2 c^4)) (p^2)_tt, multiplied by
rho_ref c0^2, maps onto weights of the existing operators: the stiffness rho_ref / rho_c (Geometry.scale_cells), a
weighted lumped mass rho_ref c0^2 / (rho_c c_c^2), weighted facet masses (rho_ref / rho_f on the source tag, Z_ref /
Z_f on the absorbing tag) and a per-dof kappa.  The restatement (model_oracle) takes G, m, m1, m2 as given and kappa
per dof.

CPU: the premises of the bitwise checks (identity medium, the power-of-two special case, kappa as a direct sum), two
known answers on the restatement -- the lowest mode of a water | bone rigid box and normal-incidence transmission
through a duct -- and the restatement against a textbook RK4.
GPU: the weighted operators against the oracle, the identity medium and the power-of-two case bit for bit, parity of
every model with random media, the per-dof kappa path, ensembles, the duct on the device, heating.
"""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL64 = 1e-12
TOL32_RUN = 1e-4      # fp32 model runs against the fp64 restatement (as test_heterogeneous)
C0, F0, P0 = 1500.0, 0.5e6, 6e4
RHO_REF = 1000.0
DELTA, BETA, RHO0 = 1e-2, 900.0, 1000.0
KAPPA = 2.0 * BETA / (RHO0 * C0 * C0)       # the scalar of wfx_wave_create_westervelt, same rounding


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


def loguniform(rng, lo, hi, n):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), n))


def random_medium(wfx, ncells, seed, beta=True):
    """rho in [900, 2000], c in [1400, 3000], beta in [0, 8] (log-uniform, with some exact zeros)"""
    rng = np.random.default_rng(seed)
    rho, c = loguniform(rng, 900.0, 2000.0, ncells), loguniform(rng, 1400.0, 3000.0, ncells)
    b = None
    if beta:
        b = loguniform(rng, 0.1, 8.0, ncells)
        b[rng.random(ncells) < 0.2] = 0.0
    return wfx.Medium(rho, c, b, rho_ref=RHO_REF)


def weighted_inputs(orc, mo, mesh, P, medium, c0=C0):
    """(G * sigma, m~, m1~, m2~) of the restatement for a medium"""
    G, detJ = orc.precompute_geometric_data(mesh, P)
    Gs = np.ascontiguousarray(G * medium.stiffness_weight(mesh.ncells)[:, None, None, None])
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, np.ascontiguousarray(detJ * medium.mass_weight(mesh.ncells, c0)[:, None]),
                   np.ones(mesh.ndofs), m)
    m1, m2 = mo.boundary_facet_mass_weighted(mesh, P, medium.facet_weight(mesh, c0))
    return Gs, m, m1, m2


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


# ---- CPU: premises -----------------------------------------------------------------------------------------------
def test_identity_medium_weights_are_exactly_one(wfx, orc):
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = wfx.Medium(np.full(mesh.ncells, RHO_REF), np.full(mesh.ncells, C0), np.full(mesh.ncells, BETA), RHO_REF)
    assert np.all(med.stiffness_weight(mesh.ncells) == 1.0)
    assert np.all(med.mass_weight(mesh.ncells, C0) == 1.0)
    assert np.all(med.facet_weight(mesh, C0) == 1.0)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    assert np.all(med.kappa(mesh, detJ, C0, BETA) == KAPPA)
    assert wfx.Medium(RHO_REF, C0).c_max == C0


def test_power_of_two_medium_is_the_scaled_form(wfx):
    """rho = rho_ref (c0 / c)^2 with c / c0 a power of two: sigma = (c / c0)^2 and mu = 1 exactly, kappa_c the scalar"""
    ncells = 40
    c = C0 * np.random.default_rng(3).choice([0.5, 1.0, 2.0, 4.0], ncells)
    med = wfx.Medium(RHO_REF * (C0 / c) ** 2, c, BETA, RHO_REF)
    assert np.array_equal(med.stiffness_weight(ncells), (c / C0) ** 2)
    assert np.all(med.mass_weight(ncells, C0) == 1.0)
    assert np.all(med.cell_kappa(ncells) == KAPPA)


def test_kappa_is_the_weighted_sum(wfx, orc):
    """kappa_i from Medium against a direct loop over cells and points"""
    P = 2
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15, renumber=5)
    med = random_medium(wfx, mesh.ncells, 1)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    mu = med.mass_weight(mesh.ncells, C0)
    kc = 2.0 * med.beta / (med.rho * med.c ** 2)
    perm = wfx.capi.compute_permutations(P)
    num, den = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    for cell in range(mesh.ncells):
        for t in range(len(perm)):
            i = mesh.dofmap[cell, perm[t]]
            num[i] += kc[cell] * mu[cell] * detJ[cell, t]
            den[i] += mu[cell] * detJ[cell, t]
    got = med.kappa(mesh, detJ, C0)
    assert np.abs(got - num / den).max() <= 1e-15 * kc.max()
    assert np.any(got == 0) and np.any(got > 0)


def test_medium_refuses_bad_parameters(wfx):
    for args in ((0.0, C0), (RHO_REF, -1.0), (np.array([1.0, np.nan]), C0), (RHO_REF, C0, -1.0),
                 (np.ones(3), np.ones(4)), (np.ones((2, 2)), C0)):
        with pytest.raises(wfx.WfxError):
            wfx.Medium(*args)
    with pytest.raises(wfx.WfxError):
        wfx.Medium(np.ones(3), C0).stiffness_weight(4)


# ---- CPU: known answers --------------------------------------------------------------------------------------------
L = 0.1
WATER, BONE = (1000.0, 1500.0), (1900.0, 2800.0)
NX, NA, WIDTH = 8, 3, 0.02
# Measured on the CPU (P4, 8 x 1 x 1 cells, fp64), before the bounds were set:
#   lowest nonzero generalised eigenvalue of (-A_sigma, M~):  |w_h^2 / w^2 - 1| = 6.6e-12
#   Rayleigh quotient of the exact mode's interpolant:       |lam / w^2 - 1|   = 6.6e-12
# The root of the scaled form (rho ~ c^-2) lies 4.8 % below it.
KNOWN_BOUNDS = dict(eig=1e-9, rayleigh=1e-9)


def _lowest_root(f, hi):
    from scipy.optimize import brentq
    ws = np.linspace(1.0, hi, 40001)
    v = f(ws)
    i = np.nonzero(np.sign(v[:-1]) != np.sign(v[1:]))[0][0]
    return brentq(f, ws[i], ws[i + 1], xtol=1e-14, rtol=1e-15)


def two_layer_omega(a, z1, z2, c1, c2):
    """lowest root of (1/Z1) sin(k1 a) cos(k2 (L - a)) + (1/Z2) sin(k2 (L - a)) cos(k1 a) = 0"""
    f = lambda w: (np.sin(w * a / c1) * np.cos(w * (L - a) / c2) / z1  # noqa: E731
                   + np.sin(w * (L - a) / c2) * np.cos(w * a / c1) / z2)
    return _lowest_root(f, 4 * np.pi * c2 / L)


def test_two_layer_box_with_independent_density(wfx, orc, mo):
    """water | bone rigid box: the lowest nonzero generalised eigenvalue of (-A_sigma, M~) is w^2 of the exact mode
    (p and (1/rho) dp/dn continuous), and so is the exact mode's Rayleigh quotient."""
    P = 4
    mesh = wfx.create_box_hex((NX, 1, 1), P, (L, WIDTH, WIDTH), tags=())
    a = NA * L / NX
    cx = np.arange(mesh.ncells)
    rho = np.where(cx < NA, WATER[0], BONE[0])
    c = np.where(cx < NA, WATER[1], BONE[1])
    med = wfx.Medium(rho, c, rho_ref=RHO_REF)
    Gs, m, _, _ = weighted_inputs(orc, mo, mesh, P, med)
    n = mesh.ndofs
    A = np.empty((n, n))
    e = np.zeros(n)
    for j in range(n):
        e[:] = 0.0
        e[j] = 1.0
        y = np.zeros(n)
        orc.stiffness_apply(mesh, P, Gs, e, y, dense=True)
        A[:, j] = y                                              # A = -c0^2 K_sigma
    s = 1.0 / np.sqrt(m)
    ev = np.linalg.eigvalsh(-(A * s[:, None]) * s[None, :])
    z1, z2 = WATER[0] * WATER[1], BONE[0] * BONE[1]
    w = two_layer_omega(a, z1, z2, WATER[1], BONE[1])
    assert abs(ev[0]) < 1e-6 * ev[1]
    assert abs(ev[1] / w ** 2 - 1) < KNOWN_BOUNDS["eig"], ev[1] / w ** 2 - 1
    k1, k2 = w / WATER[1], w / BONE[1]
    x = wfx.dof_coordinates(mesh)[:, 0]
    B = np.cos(k1 * a) / np.cos(k2 * (L - a))
    u0 = np.where(x <= a, np.cos(k1 * x), B * np.cos(k2 * (L - x)))
    lam = -(u0 @ (A @ u0)) / (u0 @ (m * u0))
    assert abs(lam / w ** 2 - 1) < KNOWN_BOUNDS["rayleigh"], lam / w ** 2 - 1
    # the scaled form (density ~ c^-2, Z ~ 1 / c) has its lowest root elsewhere
    w_old = two_layer_omega(a, 1.0 / WATER[1], 1.0 / BONE[1], WATER[1], BONE[1])
    assert abs(w_old / w - 1) > 0.02


# Normal-incidence transmission: a duct (rigid lateral walls), source dp/dn = g on x = 0 in water, an interface at
# x = a, the absorbing end (tag 2) in medium 2 at x = LD.  Steady state, time factor e^{i w t}:
#   p = A e^{-i k1 x} + B e^{i k1 x} (x < a),  C e^{-i k2 (x - a)} (x > a)
#   i k1 (A - B) = G,  A e^{-i k1 a} + B e^{i k1 a} = C,  (k1 / rho1)(A e^{-i k1 a} - B e^{i k1 a}) = (k2 / rho2) C
# with G = p0 w / c0, the amplitude of g after its ramp.
DUCT_MEDIUM2 = (1500.0, 2000.0)   # Z2 / Z1 = 2: R = 1/3, the source-interface cavity settles as 3^-n
DUCT_NX, DUCT_NA, DUCT_H, DUCT_P = 16, 4, 0.75e-3, 4
DUCT_SETTLE, DUCT_WINDOW = 24, 2   # periods before the statistics window, periods in it
# Measured on the CPU restatement (P4, 16 x 1 x 1 cells, fp64), before the bounds were set:
#   max over the axis |(|p1_h| - |p1_exact|)| / max |p1_exact| = 2.0e-5
#   with the absorbing facet weight left at 1:               = 0.90
DUCT_BOUND = 1e-4


def duct_case(wfx):
    mesh = wfx.create_box_hex((DUCT_NX, 1, 1), DUCT_P, (DUCT_NX * DUCT_H, DUCT_H, DUCT_H))
    cx = np.arange(mesh.ncells)
    rho = np.where(cx < DUCT_NA, WATER[0], DUCT_MEDIUM2[0])
    c = np.where(cx < DUCT_NA, WATER[1], DUCT_MEDIUM2[1])
    med = wfx.Medium(rho, c, rho_ref=RHO_REF)
    a = DUCT_NA * DUCT_H
    w = 2 * np.pi * F0
    k1, k2 = w / WATER[1], w / DUCT_MEDIUM2[1]
    G = P0 * w / C0
    M = np.array([[1j * k1, -1j * k1, 0],
                  [np.exp(-1j * k1 * a), np.exp(1j * k1 * a), -1],
                  [k1 / WATER[0] * np.exp(-1j * k1 * a), -k1 / WATER[0] * np.exp(1j * k1 * a), -k2 / DUCT_MEDIUM2[0]]])
    A, B, Cc = np.linalg.solve(M, np.array([G, 0, 0], dtype=complex))
    xyz = wfx.dof_coordinates(mesh)
    axis = np.nonzero((np.abs(xyz[:, 1]) < 1e-12) & (np.abs(xyz[:, 2]) < 1e-12))[0]
    axis = axis[np.argsort(xyz[axis, 0])]
    x = xyz[axis, 0]
    exact = np.where(x <= a, A * np.exp(-1j * k1 * x) + B * np.exp(1j * k1 * x), Cc * np.exp(-1j * k2 * (x - a)))
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, DUCT_P, F0)
    t_start = DUCT_SETTLE / F0 + dt          # the window holds whole periods: samples t_n in (24 T, 26 T]
    nsteps = int(round((DUCT_SETTLE + DUCT_WINDOW) / F0 / dt))
    return mesh, med, axis, np.abs(exact), dt, t_start, nsteps


def duct_error(p1, exact):
    return np.abs(np.abs(p1) - exact).max() / exact.max()


def _duct_restatement(wfx, orc, mo, absorbing_weight=True):
    mesh, med, axis, exact, dt, t_start, nsteps = duct_case(wfx)
    P = DUCT_P
    G, m, m1, m2 = weighted_inputs(orc, mo, mesh, P, med)
    if not absorbing_weight:
        m2 = orc.boundary_facet_mass(mesh, P)[1]
    u, v = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    kappa = np.zeros(mesh.ndofs)
    t, acc, nsamp = 0.0, np.zeros(len(axis), dtype=complex), 0
    w = 2 * np.pi * F0
    for _ in range(nsteps):
        _, t = mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, kappa, C0, F0, P0, 0.0, t, 1.0, dt, u, v, max_steps=1,
                                        sumfact=True)
        if t >= t_start - 0.5 * dt:
            acc += u[axis] * np.exp(-1j * w * t)
            nsamp += 1
    return duct_error(2.0 / nsamp * acc, exact)


def test_duct_transmission_known_answer(wfx, orc, mo):
    """|p1(x)| on the axis after the cavity has settled, against the closed form; with the absorbing facet weight
    left at 1 (the end then reflects) the bound fails."""
    err = _duct_restatement(wfx, orc, mo)
    assert err < DUCT_BOUND, err
    bad = _duct_restatement(wfx, orc, mo, absorbing_weight=False)
    assert bad > 10 * DUCT_BOUND, bad


# Two-layer nonlinearity: the planar case of test_field_stats (10 mm x 0.6 mm x 0.6 mm, 33 x 2 x 2 cells of P4, source
# at x = 0, absorbing end at x = L, delta = 0, p0 = 1 MPa) in water with beta = 0 in the first 11 cells (x < a) and
# beta = 3.5 beyond.  The second harmonic stays small in layer 1 and grows from the interface with the Fubini
# small-distance slope, |p_2(x)| = beta w p0^2 (x - a) / (2 rho c^3).  Two whole periods sampled from 9 periods on.
# Measured on the CPU restatement (fp64, kappa_i from Medium.kappa), before the bounds were set:
#   max | |p_1| / p0 - 1 |                 = 5.9e-5
#   layer 1: max |p_2| / |p_1|             = 2.9e-4
#   |p_2(L)| / Fubini(L - a) - 1           = -6.1e-3   (Fubini(L) from a uniform beta would be 50 % higher)
BETA2_NX, BETA2_NA, BETA2_L, BETA2_P0, BETA2 = 33, 11, 0.01, 1e6, 3.5
BETA2_BOUNDS = dict(p1=3e-4, layer1_p2_over_p1=1e-3, fubini=2e-2)


def beta2_case(wfx):
    P = 4
    side = BETA2_L / BETA2_NX
    mesh = wfx.create_box_hex((BETA2_NX, 2, 2), P, (BETA2_L, 2 * side, 2 * side))
    cx = np.arange(mesh.ncells) // 4
    med = wfx.Medium(RHO_REF, C0, np.where(cx < BETA2_NA, 0.0, BETA2), rho_ref=RHO_REF)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    k = int(round(1.0 / F0 / dt))
    X = wfx.dof_coordinates(mesh)
    line = np.where((np.abs(X[:, 1]) < 1e-12) & (np.abs(X[:, 2]) < 1e-12))[0]
    line = line[np.argsort(X[line, 0])]
    return mesh, P, med, dt, 9 * k, 2 * k, line, X[line, 0], BETA2_NA * side


def check_beta2(a1, a2, x, a):
    b = BETA2_BOUNDS
    assert np.abs(a1 / BETA2_P0 - 1).max() < b["p1"], np.abs(a1 / BETA2_P0 - 1).max()
    assert (a2 / a1)[x <= a].max() < b["layer1_p2_over_p1"], (a2 / a1)[x <= a].max()
    fubini = BETA2 * 2 * np.pi * F0 * BETA2_P0 ** 2 * (x[-1] - a) / (2 * RHO_REF * C0 ** 3)
    assert abs(a2[-1] / fubini - 1) < b["fubini"], (a2[-1], fubini)
    assert a2[-1] > 20 * a2[x <= a].max()


def test_two_layer_nonlinearity_known_answer(wfx, orc, mo):
    mesh, P, med, dt, n0, n, line, x, a = beta2_case(wfx)
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    kap = med.kappa(mesh, detJ, C0)
    assert kap.max() == 2.0 * BETA2 / (RHO_REF * C0 * C0) and kap.min() == 0.0
    u, v, t = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs), 0.0
    acc, w = np.zeros((2, len(line)), dtype=complex), 2 * np.pi * F0
    for s in range(n0 + n):
        _, t = mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, kap, C0, F0, BETA2_P0, 0.0, t, 1.0, dt, u, v,
                                        max_steps=1, sumfact=True, nthreads=orc.max_threads())
        if s >= n0:
            for h in (1, 2):
                acc[h - 1] += u[line] * np.exp(-1j * h * w * t)
    check_beta2(np.abs(2.0 / n * acc[0]), np.abs(2.0 / n * acc[1]), x, a)


# ---- CPU: the restatement ------------------------------------------------------------------------------------------
def test_restatement_matches_textbook_rk4(wfx, orc, mo):
    """wo_rk4_westervelt_medium against a textbook RK4 of the lumped system with a dense stiffness and a per-dof kappa
    (random medium, both tags); with kappa_i = kappa it is wo_rk4_westervelt bit for bit."""
    P = 2
    mesh = wfx.create_box_hex(2, P, (0.02, 0.02, 0.02), perturb=0.1)
    med = random_medium(wfx, mesh.ncells, 7)
    G, m, m1, m2 = weighted_inputs(orc, mo, mesh, P, med)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    kap = med.kappa(mesh, detJ, C0)
    n = mesh.ndofs
    A = np.zeros((n, n))
    for j in range(n):
        e, col = np.zeros(n), np.zeros(n)
        e[j] = 1.0
        orc.stiffness_apply(mesh, P, G, e, col, dense=True)
        A[:, j] = col
    s = DELTA / 1500.0 ** 2

    def acc(t, p, pd):
        g, gd = mo.source(t, F0, P0, C0)
        num = A @ p + s * (A @ pd) + kap * m * pd ** 2 + (C0 ** 2 * g + DELTA * gd) * m1 - C0 * m2 * pd
        return num / (m * (1.0 - kap * p) + DELTA / C0 * m2)

    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    t0, nsteps = 1.0e-6, 8
    rng = np.random.default_rng(5)
    p, pd = 0.3 * P0 * rng.standard_normal(n), 0.3 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)
    uo, vo = p.copy(), pd.copy()
    steps, _ = mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, t0, 1.0, dt, uo, vo,
                                        max_steps=nsteps)
    assert steps == nsteps
    t = t0
    for _ in range(nsteps):
        k1p, k1v = pd, acc(t, p, pd)
        k2p, k2v = pd + dt / 2 * k1v, acc(t + dt / 2, p + dt / 2 * k1p, pd + dt / 2 * k1v)
        k3p, k3v = pd + dt / 2 * k2v, acc(t + dt / 2, p + dt / 2 * k2p, pd + dt / 2 * k2v)
        k4p, k4v = pd + dt * k3v, acc(t + dt, p + dt * k3p, pd + dt * k3v)
        p = p + dt / 6 * (k1p + 2 * k2p + 2 * k3p + k4p)
        pd = pd + dt / 6 * (k1v + 2 * k2v + 2 * k3v + k4v)
        t += dt
    assert rel_l2(uo, p) < 1e-13 and rel_l2(vo, pd) < 1e-13
    # kappa_i = kappa: the scalar restatement, bit for bit
    u1, v1, u2, v2 = (a.copy() for a in (uo, vo, uo, vo))
    r1 = mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, np.full(n, KAPPA), C0, F0, P0, DELTA, t0, 1.0, dt, u1, v1,
                                  max_steps=5)
    r2 = mo.rk4_westervelt(mesh, P, G, m, m1, m2, C0, F0, P0, DELTA, BETA, RHO0, t0, 1.0, dt, u2, v2, max_steps=5)
    assert r1 == r2 and np.array_equal(u1, u2) and np.array_equal(v1, v2)


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_weighted_operators(wfx, orc, mo, torch, dtype):
    """m~ and 1/m~ bitwise against the oracle's mass on detJ * mu; the facet masses against the restatement to
    1e-14; NULL weights bitwise the unweighted operators; refused weights refused."""
    P = 3
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.15, renumber=3)
    med = random_medium(wfx, mesh.ncells, 11)
    mu = med.mass_weight(mesh.ncells, C0)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    geo = wfx.Geometry(mesh, P, dtype)
    m_want = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, np.ascontiguousarray(detJ * mu[:, None]), np.ones(mesh.ndofs), m_want)
    mass = wfx.MassOperator(mesh, P, dtype, geometry=geo, cell_weight=mu)
    assert np.array_equal(mass.diagonal(), m_want.astype(dtype))
    inv = (1.0 / m_want).astype(dtype)
    assert np.array_equal(mass.inverse_diagonal(), inv)
    plain = wfx.MassOperator(mesh, P, dtype, geometry=geo)
    m0 = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m0)
    assert np.array_equal(plain.diagonal(), m0.astype(dtype))
    assert np.array_equal(wfx.MassOperator(mesh, P, dtype, geometry=geo, cell_weight=np.ones(mesh.ncells)).diagonal(),
                          plain.diagonal())
    fw = med.facet_weight(mesh, C0)
    m1w, m2w = mo.boundary_facet_mass_weighted(mesh, P, fw)
    b1, b2 = wfx.BoundaryOperator(mesh, P, dtype, facet_weight=fw).facet_masses()
    np.testing.assert_allclose(b1, m1w, rtol=1e-14, atol=0)
    np.testing.assert_allclose(b2, m2w, rtol=1e-14, atol=0)
    assert np.abs(b2 - orc.boundary_facet_mass(mesh, P)[1]).max() > 1e-3 * np.abs(b2).max()
    p1, p2 = wfx.BoundaryOperator(mesh, P, dtype).facet_masses()
    o1, o2 = wfx.BoundaryOperator(mesh, P, dtype, facet_weight=np.ones(len(fw))).facet_masses()
    assert np.array_equal(p1, o1) and np.array_equal(p2, o2)
    for bad in (np.zeros(mesh.ncells), -mu, np.where(np.arange(mesh.ncells) == 2, np.nan, mu),
                np.where(np.arange(mesh.ncells) == 0, np.inf, mu), mu[:-1]):
        with pytest.raises(wfx.WfxError):
            wfx.MassOperator(mesh, P, dtype, geometry=geo, cell_weight=bad)
    for bad in (np.zeros(len(fw)), np.where(np.arange(len(fw)) == 1, np.nan, fw), -fw, fw[:-1]):
        with pytest.raises(wfx.WfxError):
            wfx.BoundaryOperator(mesh, P, dtype, facet_weight=bad)


def _models(wfx, name, mesh, P, dtype, medium=None, **kw):
    if name == "linear":
        return wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, medium=medium, **kw)
    if name == "lossy":
        return wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, DELTA, dtype=dtype, medium=medium, **kw)
    return wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype, medium=medium, **kw)


def _run(eqn, u, v, t0, tf, dt):
    eqn.set_state(u, v)
    st = eqn.rk4(t0, tf, dt)
    return st, eqn.get_state()


def _random_state(n, seed, dtype):
    rng = np.random.default_rng(seed)
    u = (0.3 * P0 * rng.standard_normal(n)).astype(dtype).astype(np.float64)
    v = (0.3 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype).astype(np.float64)
    return u, v


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("model", ["linear", "lossy", "westervelt"])
def test_identity_medium_is_the_unweighted_model_bitwise(wfx, torch, model, dtype):
    P = 4
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.04, 0.02, 0.02), perturb=0.1)
    med = wfx.Medium(np.full(mesh.ncells, RHO_REF), np.full(mesh.ncells, C0), rho_ref=RHO_REF)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    u, v = _random_state(mesh.ndofs, 1, dtype)
    a = _run(_models(wfx, model, mesh, P, dtype), u, v, 1e-6, 1e-6 + 30.5 * dt, dt)
    eqn = _models(wfx, model, mesh, P, dtype, med)
    if model == "westervelt":
        assert eqn.kappa is not None and np.all(eqn.kappa == KAPPA)
    b = _run(eqn, u, v, 1e-6, 1e-6 + 30.5 * dt, dt)
    assert a[0] == b[0] and np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_identity_medium_ensemble_bitwise(wfx, torch, dtype):
    P = 4
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.04, 0.02, 0.02), perturb=0.1)
    med = wfx.Medium(RHO_REF, C0, rho_ref=RHO_REF)
    f0s, p0s = (0.5e6, 0.3e6, 0.8e6), (6e4, 1e4, 3e4)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, max(f0s))
    rng = np.random.default_rng(2)
    U, V = 1e-3 * rng.standard_normal((mesh.ndofs, 3)), rng.standard_normal((mesh.ndofs, 3))
    a = _run(wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s, p0s, dtype=dtype), U, V, 0.0, 20.5 * dt, dt)
    b = _run(wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s, p0s, dtype=dtype, medium=med), U, V, 0.0, 20.5 * dt, dt)
    assert a[0] == b[0] and np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("model", ["linear", "lossy", "westervelt"])
def test_power_of_two_medium_is_the_scaled_form_bitwise(wfx, torch, model, dtype):
    """rho = rho_ref (c0 / c)^2, c / c0 in {1/2, 1, 2}, the tagged cells (x = 0, x = L) in the reference medium: the
    same run as the model scaled with scale_cells((c / c0)^2)."""
    P = 3
    nx = 5
    mesh = wfx.create_box_hex((nx, 2, 2), P, (0.05, 0.02, 0.02), perturb=0.1)
    cx = np.arange(mesh.ncells) // 4
    ratio = np.random.default_rng(4).choice([0.5, 1.0, 2.0], mesh.ncells)
    ratio[(cx == 0) | (cx == nx - 1)] = 1.0
    med = wfx.Medium(RHO_REF / ratio ** 2, C0 * ratio, rho_ref=RHO_REF)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    u, v = _random_state(mesh.ndofs, 3, dtype)
    ref = _models(wfx, model, mesh, P, dtype)
    ref.geometry.scale_cells(ratio ** 2)
    a = _run(ref, u, v, 1e-6, 1e-6 + 25.5 * dt, dt)
    b = _run(_models(wfx, model, mesh, P, dtype, med), u, v, 1e-6, 1e-6 + 25.5 * dt, dt)
    assert a[0] == b[0] and np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])


PARITY = [  # (P, dtype, graph, stiffness mode)
    (2, np.float64, True, 0), (3, np.float64, False, 0), (4, np.float64, True, 0), (4, np.float64, False, 4),
    (5, np.float64, True, 0), (5, np.float64, False, 0), (4, np.float32, True, 0), (7, np.float32, True, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY, ids=[f"P{c[0]}-{np.dtype(c[1]).name}-graph{int(c[2])}-mode{c[3]}"
                                              for c in PARITY])
@pytest.mark.parametrize("model", ["linear", "lossy", "westervelt"])
def test_models_in_random_media_match_the_restatement(wfx, orc, mo, torch, monkeypatch, model, case):
    """RK4 with a shortened last step through the ramp's end, random per-cell rho, c (and beta for Westervelt), against
    the restatement with the weighted G, m, m1, m2 and the model's own kappa_i."""
    P, dtype, graph, mode = case
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 30 + P, beta=model == "westervelt")
    eqn = _models(wfx, model, mesh, P, dtype, med, stiffness_mode=mode)
    if P == 7:
        assert eqn.stiff_op.kernel_info()["variant"] == "cell-streamed"
    G, m, m1, m2 = weighted_inputs(orc, mo, mesh, P, med)
    delta = 0.0 if model == "linear" else DELTA
    kappa = eqn.kappa if model == "westervelt" else np.zeros(mesh.ndofs)
    if model == "westervelt":
        assert kappa.max() > 0
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    u, v = _random_state(mesh.ndofs, P, dtype)
    t0, steps = 7.5e-6, 12
    tf = t0 + (steps - 0.5) * dt
    uo, vo = u.copy(), v.copy()
    so, to = mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, kappa, C0, F0, P0, delta, t0, tf, dt, uo, vo,
                                      sumfact=True, nthreads=orc.max_threads())
    (s, t), (ug, vg) = _run(eqn, u, v, t0, tf, dt)
    assert (s, t) == (so, to) and s == steps
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    assert rel_l2(ug, uo) < tol and rel_l2(vg, vo) < tol, (rel_l2(ug, uo), rel_l2(vg, vo))
    # f1 against the restatement's f1
    fo = mo.f1_westervelt_medium(mesh, P, G, m, m1, m2, kappa, C0, F0, P0, delta, 3e-6, u, v)
    res = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64 if dtype == np.float64 else torch.float32,
                     device="cuda")
    tdev = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(dtype))).cuda()  # noqa: E731
    eqn.f1(3e-6, tdev(u), tdev(v), res)
    assert rel_l2(res.cpu().numpy(), fo) < (TOL64 if dtype == np.float64 else 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("delta", [0.0, DELTA])
def test_per_dof_kappa_path(wfx, torch, monkeypatch, dtype, delta):
    """kappa_i filled with the scalar: the scalar path bit for bit (with delta > 0 the Gamma2 kernel too); NULL
    restores the scalar path; a kappa changed between rk4 calls equals a fresh model (the captured graph is
    dropped); refusals."""
    P = 4
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.04, 0.02, 0.02), perturb=0.1)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    u, v = _random_state(mesh.ndofs, 9, dtype)
    mk = lambda: wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, delta, BETA, RHO0, dtype=dtype)  # noqa: E731
    t1 = 1e-6 + 20.5 * dt
    a = _run(mk(), u, v, 1e-6, t1, dt)
    eqn = mk()
    eqn.set_nonlinearity(np.full(mesh.ndofs, KAPPA))
    b = _run(eqn, u, v, 1e-6, t1, dt)
    assert a[0] == b[0] and np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])
    eqn.set_nonlinearity(None)
    b = _run(eqn, u, v, 1e-6, t1, dt)
    assert np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])
    # f1 with kappa_i = kappa
    tdev = lambda x: torch.from_numpy(np.ascontiguousarray(x.astype(dtype))).cuda()  # noqa: E731
    r1, r2 = torch.empty_like(tdev(u)), torch.empty_like(tdev(u))
    ref = mk()
    ref.f1(3e-6, tdev(u), tdev(v), r1)
    eqn.set_nonlinearity(np.full(mesh.ndofs, KAPPA))
    eqn.f1(3e-6, tdev(u), tdev(v), r2)
    assert torch.equal(r1, r2)
    # change kappa between rk4 calls: scalar -> per dof -> another per dof, against fresh models from the same state
    k1 = KAPPA * np.random.default_rng(1).uniform(0.0, 3.0, mesh.ndofs)
    k2 = KAPPA * np.random.default_rng(2).uniform(0.0, 3.0, mesh.ndofs)
    run = mk()
    run.set_state(u, v)
    s0, tA = run.rk4(1e-6, 1.0, dt, max_steps=10)
    sA = run.get_state()
    run.set_nonlinearity(k1)
    run.rk4(tA, 1.0, dt, max_steps=10)
    sB = run.get_state()
    run.set_nonlinearity(k2)
    _, tC = run.rk4(tA + 10 * dt, 1.0, dt, max_steps=10)
    sC = run.get_state()
    fresh = mk()
    fresh.set_nonlinearity(k1)
    fresh.set_state(*sA)
    fresh.rk4(tA, 1.0, dt, max_steps=10)
    assert all(np.array_equal(x, y) for x, y in zip(fresh.get_state(), sB))
    fresh2 = mk()
    fresh2.set_nonlinearity(k2)
    fresh2.set_state(*sB)
    fresh2.rk4(tA + 10 * dt, 1.0, dt, max_steps=10)
    assert all(np.array_equal(x, y) for x, y in zip(fresh2.get_state(), sC))
    assert not np.array_equal(sB[0], sC[0])
    # the configuration survives init: a run from rest after init equals a fresh model with the same kappa, and
    # differs from the scalar model's
    run.init()
    run.rk4(0.0, 1.0, dt, max_steps=40)
    fresh3 = mk()
    fresh3.set_nonlinearity(k2)
    fresh3.init()
    fresh3.rk4(0.0, 1.0, dt, max_steps=40)
    scalar = mk()
    scalar.init()
    scalar.rk4(0.0, 1.0, dt, max_steps=40)
    assert all(np.array_equal(x, y) for x, y in zip(run.get_state(), fresh3.get_state()))
    assert not np.array_equal(run.get_state()[0], scalar.get_state()[0])
    # refusals
    for bad in (np.full(mesh.ndofs, -1.0), np.where(np.arange(mesh.ndofs) == 3, np.nan, k1),
                np.where(np.arange(mesh.ndofs) == 0, np.inf, k1)):
        with pytest.raises(wfx.WfxError):
            run.set_nonlinearity(bad)
    with pytest.raises(wfx.WfxError):
        run.set_nonlinearity(k1[:-1])
    lin = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype)
    with pytest.raises(wfx.WfxError):
        wfx.capi.call("wfx_wave_set_nonlinearity", lin.handle, wfx.capi.f64p(k1))
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, (F0, F0), (P0, P0), dtype=dtype)
    with pytest.raises(wfx.WfxError):
        wfx.capi.call("wfx_wave_set_nonlinearity", ens.handle, wfx.capi.f64p(k1))
    with pytest.raises(wfx.WfxError):
        wfx.capi.call("wfx_wave_set_nonlinearity", None, wfx.capi.f64p(k1))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_westervelt_in_a_linear_medium_is_the_lossy_model(wfx, torch, dtype):
    """A Westervelt model (beta > 0) in a medium whose beta is zero everywhere steps kappa_i = 0, not its scalar
    kappa: the lossy model in the same medium, bit for bit."""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    m0 = random_medium(wfx, mesh.ncells, 81, beta=False)
    med = wfx.Medium(m0.rho, m0.c, 0.0, rho_ref=RHO_REF)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    u, v = _random_state(mesh.ndofs, 6, dtype)
    west = _models(wfx, "westervelt", mesh, P, dtype, med)
    assert west.kappa is not None and np.all(west.kappa == 0)
    a = _run(west, u, v, 1e-6, 1e-6 + 20.5 * dt, dt)
    b = _run(_models(wfx, "lossy", mesh, P, dtype, med), u, v, 1e-6, 1e-6 + 20.5 * dt, dt)
    c = _run(_models(wfx, "westervelt", mesh, P, dtype, wfx.Medium(m0.rho, m0.c, rho_ref=RHO_REF)), u, v, 1e-6,
             1e-6 + 20.5 * dt, dt)
    assert a[0] == b[0] and np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])
    assert not np.array_equal(a[1][0], c[1][0])      # the model's own beta (the medium has none) is nonlinear


@pytest.mark.gpu
def test_lossy_model_with_per_dof_kappa_steps_the_nonlinear_update(wfx, orc, mo, torch):
    """A model made with beta = 0 and given a per-dof kappa follows the Westervelt restatement with that kappa."""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    kap = KAPPA * np.random.default_rng(3).uniform(0.0, 3.0, mesh.ndofs)
    eqn = wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, DELTA)
    eqn.set_nonlinearity(kap)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    u, v = (0.01 * a for a in _random_state(mesh.ndofs, 4, np.float64))
    uo, vo = u.copy(), v.copy()
    mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, 2e-6, 2e-6 + 15.5 * dt, dt, uo, vo,
                             sumfact=True)
    _, (ug, vg) = _run(eqn, u, v, 2e-6, 2e-6 + 15.5 * dt, dt)
    assert rel_l2(ug, uo) < TOL64 and rel_l2(vg, vo) < TOL64


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_ensemble_in_a_medium(wfx, torch, dtype):
    """LinearGLLEnsemble with a random medium, nv = 1, 3, 8: every member equals a single-field model in the same
    medium."""
    P = 4
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 61, beta=False)
    f0s = np.array([0.5e6, 0.3e6, 0.8e6, 0.6e6, 0.4e6, 0.7e6, 0.55e6, 0.45e6])
    p0s = np.array([6e4, 1e4, 3e4, 2e4, 5e4, 4e4, 1.5e4, 2.5e4])
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, f0s.max())
    tf = 10.6 * dt
    rng = np.random.default_rng(8)
    U0, V0 = 1e-3 * rng.standard_normal((mesh.ndofs, 8)), rng.standard_normal((mesh.ndofs, 8))
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    for nv in (1, 3, 8):
        ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s[:nv], p0s[:nv], dtype=dtype, medium=med)
        (s, t), (U, V) = _run(ens, U0[:, :nv], V0[:, :nv], 0.0, tf, dt)
        assert s == 11
        for k in range(nv):
            one = wfx.LinearGLLOpt(mesh, None, P, C0, f0s[k], p0s[k], dtype=dtype, medium=med)
            (s1, t1), (u1, v1) = _run(one, U0[:, k], V0[:, k], 0.0, tf, dt)
            assert (s1, t1) == (s, t)
            assert rel_l2(U[:, k], u1.astype(np.float64)) < tol and rel_l2(V[:, k], v1.astype(np.float64)) < tol


@pytest.mark.gpu
def test_duct_transmission_on_the_device(wfx, torch):
    """The duct of the CPU known answer through the device's field statistics, with the bound measured there."""
    mesh, med, axis, exact, dt, t_start, nsteps = duct_case(wfx)
    eqn = wfx.LinearGLLOpt(mesh, None, DUCT_P, C0, F0, P0, medium=med)
    eqn.init()
    eqn.set_field_stats(t_start, 1)
    assert eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)[0] == nsteps
    fs = eqn.field_stats()
    assert fs.samples == int(round(DUCT_WINDOW / F0 / dt))
    err = duct_error(fs.harmonics[0][axis], exact)
    assert err < DUCT_BOUND, err


@pytest.mark.gpu
def test_two_layer_nonlinearity_on_the_device(wfx, torch):
    """The two-layer beta case through the Westervelt model in a Medium and the device's field statistics, with the
    bounds measured on the restatement."""
    mesh, P, med, dt, n0, n, line, x, a = beta2_case(wfx)
    eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, BETA2_P0, 0.0, BETA2, RHO_REF, medium=med)
    eqn.init()
    eqn.set_field_stats((n0 + 1) * dt, 2)
    assert eqn.rk4(0.0, 1.0, dt, max_steps=n0 + n)[0] == n0 + n
    fs = eqn.field_stats()
    assert fs.samples == n
    check_beta2(np.abs(fs.harmonics[0][line]), np.abs(fs.harmonics[1][line]), x, a)


@pytest.mark.gpu
def test_heating_in_a_medium(wfx, orc, torch):
    """heat_from_wave(..., medium=): Q_i = sum_h alpha0 (h f0 / 1 MHz)^y |p_h|^2 <1 / (rho c)>_i with the mass-weighted
    per-dof average, against numpy."""
    P = 3
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.012, 0.006, 0.006), perturb=0.1)
    med = random_medium(wfx, mesh.ncells, 71, beta=False)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, medium=med)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    eqn.init()
    eqn.set_field_stats(2.0 / F0, 3)
    eqn.rk4(0.0, 4.0 / F0, dt)
    fs = eqn.field_stats()
    th = wfx.PennesGLL(mesh, P, 0.5, 3.6e6)
    alpha0, y = 5.0, 1.1
    th.heat_from_wave(eqn, alpha0, y, RHO0, C0, medium=med)
    # <1 / (rho c)>_i = sum_c (detJ w)_{c,i} / (rho_c c_c) / sum_c (detJ w)_{c,i}, written out cell by cell
    _, detJ = orc.precompute_geometric_data(mesh, P)
    perm = wfx.capi.compute_permutations(P)
    num, den = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    for cell in range(mesh.ncells):
        for t in range(len(perm)):
            i = mesh.dofmap[cell, perm[t]]
            num[i] += detJ[cell, t] / (med.rho[cell] * med.c[cell])
            den[i] += detJ[cell, t]
    inv_z = num / den
    want = sum(alpha0 * (h * F0 / 1e6) ** y * np.abs(fs.harmonics[h - 1]) ** 2 for h in (1, 2, 3)) * inv_z
    assert want.max() > 0
    np.testing.assert_allclose(th.heat_source(), want, rtol=1e-13, atol=1e-13 * want.max())
    with pytest.raises(wfx.WfxError):
        wfx.PennesGLL.from_wave(eqn, 0.5, 3.6e6)


@pytest.mark.gpu
def test_medium_with_a_halo_is_refused(wfx, torch):
    mesh = wfx.create_box_hex((2, 2, 2), 2, (0.02, 0.02, 0.02))
    with pytest.raises(wfx.WfxError):
        wfx.LinearGLLOpt(mesh, None, 2, C0, F0, P0, halo=object(), medium=wfx.Medium(RHO_REF, C0))


# ---- C++ wrappers ------------------------------------------------------------------------------------------------
def _build_cpp(wfx, outdir):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_medium_hpp.cpp")
    exe = os.path.join(str(outdir), "test_wavefx_medium_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_medium_cpp_wrapper_compiles_and_links(wfx, tmp_path):
    assert os.path.exists(_build_cpp(wfx, tmp_path))


@pytest.mark.gpu
def test_medium_cpp_wrappers_reproduce_the_python_models(wfx, torch, tmp_path):
    """The C++ medium constructors (linear, lossy, Westervelt, ensemble) on the same mesh, weights and state as the
    Python models: the same final u bit for bit."""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 91)
    lin = wfx.Medium(med.rho, med.c, rho_ref=RHO_REF)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    t0, tf = 1e-6, 1e-6 + 14.5 * dt
    u, v = _random_state(mesh.ndofs, 5, np.float64)
    west = _models(wfx, "westervelt", mesh, P, np.float64, med)
    files = {"params.f64": np.array([P, C0, F0, P0, DELTA, BETA, RHO0, t0, tf, dt]),
             "x.f64": mesh.x, "xdofs.i32": mesh.xdofs, "dofmap.i32": mesh.dofmap,
             "fcell.i32": mesh.facet_cells, "flocal.i32": mesh.facet_local, "ftag.i32": mesh.facet_tags,
             "u.f64": u, "v.f64": v, "stiffness.f64": med.stiffness_weight(mesh.ncells),
             "mass.f64": med.mass_weight(mesh.ncells, C0), "facet.f64": med.facet_weight(mesh, C0),
             "kappa.f64": west.kappa}
    for name, a in files.items():
        np.ascontiguousarray(a, dtype=np.int32 if name.endswith("i32") else np.float64).tofile(str(tmp_path / name))
    r = subprocess.run([_build_cpp(wfx, tmp_path), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "medium hpp ok" in r.stdout, r.stdout + r.stderr
    got = lambda name: np.fromfile(str(tmp_path / name), dtype=np.float64)  # noqa: E731
    for name, eqn in (("linear", _models(wfx, "linear", mesh, P, np.float64, lin)),
                      ("lossy", _models(wfx, "lossy", mesh, P, np.float64, lin)), ("westervelt", west)):
        _, (ug, _) = _run(eqn, u, v, t0, tf, dt)
        assert np.array_equal(got(f"u_{name}.f64"), ug), name
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, (F0, 0.7 * F0), (P0, 0.5 * P0), medium=lin)
    _, (U, _) = _run(ens, np.stack([u, u], 1), np.stack([v, v], 1), t0, tf, dt)
    assert np.array_equal(got("u_ensemble.f64").reshape(-1, 2), U)


@pytest.mark.gpu
def test_demo_layer_option(wfx, torch):
    """demo/planar3d.py --layer with a bone slab, the Westervelt model, field statistics and heating: it runs, reports
    |p1| on both sides of the slab, and the slab (Z2 / Z1 = 3.55) transmits less than the source side carries."""
    r = subprocess.run(["python", os.path.join(ROOT, "demo", "planar3d.py"), "--nx", "16", "--nyz", "1",
                        "--length", "0.012", "--model", "westervelt", "--stats-periods", "2", "--layer", "0.0045",
                        "0.006", "--layer-rho", "1900", "--layer-c", "2800", "--heat-seconds", "0.5"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    out = r.stdout
    assert "layer: 2 cells" in out and "thermal: peak rise" in out, out
    vals = {}
    for side in ("before the layer", "after the layer"):
        line = [ln for ln in out.splitlines() if ln.startswith(side)][0]
        vals[side] = float(line.split("mean ")[1].split(",")[0])
    assert 0 < vals["after the layer"] < vals["before the layer"], vals
