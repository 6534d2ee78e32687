"""Relaxation absorption (DESIGN.md section 4.5f): power-law tissue absorption by M <= 3 relaxation processes with
per-dof memory variables on the mass side of the lossy and Westervelt models,

    (m~ (1 - kappa p) + q Gamma2) p_tt = b + m~ (kappa p_t^2 - sum_nu q_nu''),   tau_nu q_nu' + q_nu = eps_nu p.

CPU: the restatement (model_oracle wo_*_westervelt_relax) against a textbook RK4 of the augmented lumped system and,
without relaxation, against wo_rk4_westervelt_medium bit for bit; two known answers on the restatement -- the lowest
mode of a rigid box against the exact (M + 2)-dimensional ODE, and the attenuation and wavenumber of a plane wave in a
duct against the exact k(w); the fit of Medium.relaxation; eps_dofs; refusals on the host.
GPU: the models against the restatement, the model without relaxation bit for bit, checkpoints, field statistics and
heating, refusals, the demo and the C++ wrapper.
"""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL64 = 1e-12
TOL32_RUN = 1e-4
C0, F0, P0 = 1500.0, 0.5e6, 6e4
RHO_REF = 1000.0
DELTA, BETA, RHO0 = 1e-2, 900.0, 1000.0
KAPPA = 2.0 * BETA / (RHO0 * C0 * C0)       # the scalar of wfx_wave_create_westervelt, same rounding
DB_CM = np.log(10.0) / 20.0 * 100.0      # 1 dB/cm in Np/m


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


def random_medium(wfx, ncells, seed, beta=True):
    """rho in [900, 2000], c in [1400, 3000], beta in [0, 8] with some zeros, alpha0 in [0.3, 10] dB/cm/MHz, y 1.1"""
    rng = np.random.default_rng(seed)
    lu = lambda lo, hi: np.exp(rng.uniform(np.log(lo), np.log(hi), ncells))  # noqa: E731
    rho, c = lu(900.0, 2000.0), lu(1400.0, 3000.0)
    b = None
    if beta:
        b = lu(0.1, 8.0)
        b[rng.random(ncells) < 0.2] = 0.0
    return wfx.Medium(rho, c, b, rho_ref=RHO_REF, alpha0=lu(0.3, 10.0) * DB_CM, y=1.1)


def random_relaxation(wfx, ncells, M, seed):
    """M processes at 0.3 .. 3 MHz with random per-cell strengths (some cells without)"""
    rng = np.random.default_rng(seed)
    tau = 1.0 / (2 * np.pi * np.geomspace(0.3e6, 3e6, M))
    eps = rng.uniform(0.0, 0.05, (M, ncells))
    eps[:, rng.random(ncells) < 0.2] = 0.0
    return wfx.Relaxation(tau, eps, 1500.0)


def weighted_inputs(orc, mo, mesh, P, medium, c0=C0):
    """(G * sigma, m~, m1~, m2~, mu) of the restatement for a medium"""
    G, detJ = orc.precompute_geometric_data(mesh, P)
    Gs = np.ascontiguousarray(G * medium.stiffness_weight(mesh.ncells)[:, None, None, None])
    mu = medium.mass_weight(mesh.ncells, c0)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, np.ascontiguousarray(detJ * mu[:, None]), np.ones(mesh.ndofs), m)
    m1, m2 = mo.boundary_facet_mass_weighted(mesh, P, medium.facet_weight(mesh, c0))
    return Gs, m, m1, m2, mu, detJ


def dense_stiffness(orc, mesh, P, G):
    n = mesh.ndofs
    A = np.zeros((n, n))
    for j in range(n):
        e, col = np.zeros(n), np.zeros(n)
        e[j] = 1.0
        orc.stiffness_apply(mesh, P, G, e, col, dense=True)
        A[:, j] = col
    return A


# ---- CPU: the restatement ------------------------------------------------------------------------------------------
def test_restatement_matches_textbook_rk4(wfx, orc, mo):
    """wo_rk4_westervelt_relax against a textbook RK4 of the augmented lumped system (dense stiffness, per-dof kappa and
    eps, both tags, delta > 0), M = 2"""
    P = 2
    mesh = wfx.create_box_hex(2, P, (0.02, 0.02, 0.02), perturb=0.1)
    med = random_medium(wfx, mesh.ncells, 7)
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    kap = med.kappa(mesh, detJ, C0)
    rel = random_relaxation(wfx, mesh.ncells, 2, 3)
    eps = rel.eps_dofs(mesh, detJ, mu)
    tau = rel.tau
    A = dense_stiffness(orc, mesh, P, G)
    s = DELTA / 1500.0 ** 2

    def rhs(t, p, pd, q):
        kq = (eps * p - q) / tau[:, None]
        R = ((eps * pd - kq) / tau[:, None]).sum(0)
        g, gd = mo.source(t, F0, P0, C0)
        num = A @ p + s * (A @ pd) + kap * m * pd ** 2 + (C0 ** 2 * g + DELTA * gd) * m1 - C0 * m2 * pd - m * R
        return pd, num / (m * (1.0 - kap * p) + DELTA / C0 * m2), kq

    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), rel.max_dt())
    t0, nsteps = 1.0e-6, 8
    rng = np.random.default_rng(5)
    n = mesh.ndofs
    p, pd = 0.3 * P0 * rng.standard_normal(n), 0.3 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)
    q = eps * p * rng.uniform(0.5, 1.5, eps.shape)
    uo, vo, qo = p.copy(), pd.copy(), q.copy()
    steps, _ = mo.rk4_westervelt_relax(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, tau, eps, t0, 1.0, dt, uo, vo, qo,
                                       max_steps=nsteps)
    assert steps == nsteps
    t = t0
    for _ in range(nsteps):
        k1 = rhs(t, p, pd, q)
        k2 = rhs(t + dt / 2, p + dt / 2 * k1[0], pd + dt / 2 * k1[1], q + dt / 2 * k1[2])
        k3 = rhs(t + dt / 2, p + dt / 2 * k2[0], pd + dt / 2 * k2[1], q + dt / 2 * k2[2])
        k4 = rhs(t + dt, p + dt * k3[0], pd + dt * k3[1], q + dt * k3[2])
        p, pd, q = (x + dt / 6 * (a + 2 * b + 2 * c + d) for x, a, b, c, d in zip((p, pd, q), k1, k2, k3, k4))
        t += dt
    assert rel_l2(uo, p) < 1e-13 and rel_l2(vo, pd) < 1e-13 and rel_l2(qo, q) < 1e-13
    # f1 against the same right-hand side
    fo = mo.f1_westervelt_relax(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, tau, eps, 3e-6, p, pd, q)
    assert rel_l2(fo, rhs(3e-6, p, pd, q)[1]) < 1e-13


def test_restatement_without_relaxation_is_the_medium_restatement_bitwise(wfx, orc, mo):
    """M = 0, and eps = 0 with M = 2 (q stays 0): wo_rk4_westervelt_medium bit for bit"""
    P = 2
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 9)
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    kap = med.kappa(mesh, detJ, C0)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    rng = np.random.default_rng(2)
    u, v = 0.3 * P0 * rng.standard_normal(mesh.ndofs), 1e6 * rng.standard_normal(mesh.ndofs)
    u1, v1 = u.copy(), v.copy()
    r1 = mo.rk4_westervelt_medium(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, 1e-6, 1e-6 + 9.5 * dt, dt, u1, v1)
    for M in (0, 2):
        tau = 1.0 / (2 * np.pi * np.geomspace(0.5e6, 2e6, M)) if M else np.zeros(0)
        u2, v2, q2 = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
        r2 = mo.rk4_westervelt_relax(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, tau, np.zeros((M, mesh.ndofs)),
                                     1e-6, 1e-6 + 9.5 * dt, dt, u2, v2, q2)
        assert r1 == r2 and np.array_equal(u1, u2) and np.array_equal(v1, v2), M
        assert not np.any(q2)


# ---- CPU: known answers --------------------------------------------------------------------------------------------
# Mode: a rigid homogeneous box (no tags), P4, 4 x 1 x 1 cells, started from the lowest nonzero discrete eigenvector
# phi (-A phi = lam m phi) with p' = 0 and q = eps p.  The mode amplitude a(t) = phi^T m p / phi^T m phi follows
#   a'' = -lam a - sum_nu q_nu'',  q_nu' = (eps_nu a - q_nu) / tau_nu,
# exactly (the system is linear and eps is the same at every dof), so its state is expm(t B) x0.  B's oscillating
# eigenvalues are the damped roots of s^2 (1 + sum eps / (1 + s tau)) + lam = 0.
# Measured on the CPU restatement (fp64, 400 CFL steps, about 2.6 mode periods), before the bounds were set:
#   max_t |a_rk4(t) - a_exact(t)| = 3.0e-7 (M = 1), 2.4e-7 (2), 2.2e-7 (3); with dt / 2 it falls 16.0-16.1-fold (RK4's
#   fourth order: the difference is truncation); the mode decays to exp(Re s t_end) = 0.88, 0.78, 0.71
#   the root against B's eigenvalue: |s - s_B| / |s| < 1e-15
MODE_BOUNDS = dict(traj=1e-6, order=(13.0, 19.0), root=1e-12)
MODE_EPS = {1: [0.08], 2: [0.04, 0.06], 3: [0.03, 0.04, 0.05]}


def _mode_matrix(lam, tau, eps):
    """d/dt (a, a', q_1..q_M) = B (a, a', q)"""
    M = len(tau)
    B = np.zeros((M + 2, M + 2))
    B[0, 1] = 1.0
    B[1, 0] = -lam
    for j in range(M):
        # q_j' = (eps_j a - q_j) / tau_j;  q_j'' = (eps_j a' - q_j') / tau_j
        B[2 + j, 0], B[2 + j, 2 + j] = eps[j] / tau[j], -1.0 / tau[j]
        B[1, 1] -= eps[j] / tau[j]
        B[1, 0] += eps[j] / tau[j] ** 2
        B[1, 2 + j] -= 1.0 / tau[j] ** 2
    return B


@pytest.mark.parametrize("M", [1, 2, 3])
def test_rigid_box_mode_known_answer(wfx, orc, mo, M):
    from scipy.linalg import eigh, expm
    from scipy.optimize import fsolve
    P = 4
    mesh = wfx.create_box_hex((4, 1, 1), P, (0.012, 0.003, 0.003), tags=())
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    lams, vecs = eigh(-dense_stiffness(orc, mesh, P, G), np.diag(m))
    lam, phi = lams[1], vecs[:, 1]
    tau = 1.0 / (np.geomspace(0.2, 2.0, M) * np.sqrt(lam))    # relaxation frequencies around the mode's
    eps = np.array(MODE_EPS[M])
    rel = wfx.Relaxation(tau, eps, C0)
    dt = min(wfx.cfl_timestep(mesh.h_min, C0, P, F0), rel.max_dt())
    B = _mode_matrix(lam, tau, eps)
    x0 = np.r_[1.0, 0.0, eps]
    z = np.zeros(mesh.ndofs)
    errs = []
    for fac in (1, 2):
        u, v, q = phi.copy(), np.zeros(mesh.ndofs), eps[:, None] * phi[None, :]
        err, t = 0.0, 0.0
        for _ in range(20):
            _, t = mo.rk4_westervelt_relax(mesh, P, G, m, z, z, z, C0, F0, 0.0, 0.0, tau,
                                           np.repeat(eps[:, None], mesh.ndofs, 1), t, 1.0, dt / fac, u, v, q,
                                           max_steps=20 * fac, sumfact=True)
            a = phi @ (m * u) / (phi @ (m * phi))
            err = max(err, abs(a - (expm(t * B) @ x0)[0]))
        errs.append(err)
    assert errs[0] < MODE_BOUNDS["traj"], errs
    lo, hi = MODE_BOUNDS["order"]
    assert lo < errs[0] / errs[1] < hi, errs
    # the damped root of the dispersion relation is an eigenvalue of B, and it damps the mode measurably
    ev = np.linalg.eigvals(B)
    sB = ev[np.argmax(ev.imag)]
    disp = lambda s: s * s * (1 + sum(e / (1 + s * tt) for e, tt in zip(eps, tau))) + lam  # noqa: E731
    sol = fsolve(lambda x: [disp(x[0] + 1j * x[1]).real, disp(x[0] + 1j * x[1]).imag], [0.0, np.sqrt(lam)],
                 xtol=1e-15)
    s = sol[0] + 1j * sol[1]
    assert abs(s - sB) / abs(s) < MODE_BOUNDS["root"], abs(s - sB) / abs(s)
    assert 0.5 < np.exp(s.real * t) < 0.95, np.exp(s.real * t)


# Duct: a plane wave from the source (tag 1, x = 0) to the absorbing end (tag 2, x = L) in a homogeneous relaxing
# medium (c = 1500, alpha0 = 10 dB/cm/MHz, y = 1, fitted over 0.3 .. 1.2 MHz with three processes).  After the
# start-up, |p1| decays along the axis as exp(-alpha(f0) x) and arg p1 falls as -Re k(f0) x, with k(w) the exact
# wavenumber of the relaxing medium.  The first-order absorbing end reflects O(eps), a ripple the line fit averages.
# Measured on the CPU restatement (P4, 48 x 1 x 1 cells of 0.5 mm, 8.4 wavelengths, fp64, fit over the middle 80 %),
# before the bounds were set: the end reflects a 5 % ripple;
#   slope of log|p1| against -alpha(f0): rel. error 1.1e-4;  slope of the unwrapped phase against -Re k: 8.4e-6
# (with 24 cells and 12 settling periods the amplitude slope is off by 2.5 %: too few ripples to average)
DUCT_NX, DUCT_H, DUCT_P = 48, 0.5e-3, 4
DUCT_ALPHA0, DUCT_SETTLE, DUCT_WINDOW = 10.0 * DB_CM, 24, 2
DUCT_BOUNDS = dict(alpha=1e-3, k=1e-4)


def duct_case(wfx):
    mesh = wfx.create_box_hex((DUCT_NX, 1, 1), DUCT_P, (DUCT_NX * DUCT_H, DUCT_H, DUCT_H))
    med = wfx.Medium(RHO_REF, C0, rho_ref=RHO_REF, alpha0=DUCT_ALPHA0, y=1.0)
    rel = med.relaxation(0.6 * F0, 2.4 * F0)
    xyz = wfx.dof_coordinates(mesh)
    axis = np.nonzero((np.abs(xyz[:, 1]) < 1e-12) & (np.abs(xyz[:, 2]) < 1e-12))[0]
    axis = axis[np.argsort(xyz[axis, 0])]
    dt = min(wfx.cfl_timestep(mesh.h_min, C0, DUCT_P, F0), rel.max_dt())
    nper = int(np.ceil(1.0 / F0 / dt))
    dt = 1.0 / F0 / nper                     # whole steps per period
    return mesh, med, rel, axis, xyz[axis, 0], dt, nper


def duct_slopes(p1, x, rel):
    """(relative error of the amplitude slope against alpha(f0), of the phase slope against Re k(f0)), fitted over the
    middle of the duct (away from the source and the absorbing end)"""
    sel = (x > 0.1 * x[-1]) & (x < 0.9 * x[-1])
    sa = np.polyfit(x[sel], np.log(np.abs(p1[sel])), 1)[0]
    sp = np.polyfit(x[sel], np.unwrap(np.angle(p1[sel])), 1)[0]
    k = (2 * np.pi * F0 / C0) * np.sqrt(1 + sum(rel.eps[j, 0] / (1 + 1j * 2 * np.pi * F0 * rel.tau[j])
                                                for j in range(rel.M)))
    return abs(-sa / -k.imag - 1), abs(-sp / k.real - 1)


def test_duct_attenuation_known_answer(wfx, orc, mo):
    mesh, med, rel, axis, x, dt, nper = duct_case(wfx)
    P = DUCT_P
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    eps = rel.eps_dofs(mesh, detJ, mu)
    u, v, q = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs), np.zeros((rel.M, mesh.ndofs))
    z = np.zeros(mesh.ndofs)
    w = 2 * np.pi * F0
    acc = np.zeros(len(axis), dtype=complex)
    t = 0.0
    n0 = DUCT_SETTLE * nper
    for s in range((DUCT_SETTLE + DUCT_WINDOW) * nper):
        _, t = mo.rk4_westervelt_relax(mesh, P, G, m, m1, m2, z, C0, F0, P0, 0.0, rel.tau, eps, t, 1.0, dt, u, v, q,
                                       max_steps=1, sumfact=True)
        if s >= n0:
            acc += u[axis] * np.exp(-1j * w * t)
    ea, ek = duct_slopes(acc, x, rel)
    assert ea < DUCT_BOUNDS["alpha"] and ek < DUCT_BOUNDS["k"], (ea, ek)


def test_delta_model_has_the_wrong_frequency_law(wfx):
    """A strong absorber (10 dB/cm/MHz, y = 1): the delta model fitted to alpha(f0) gives alpha(2 f0) / alpha(f0) = 4;
    the relaxation fit keeps 2^y = 2 to within its fit error."""
    med = wfx.Medium(RHO_REF, C0, rho_ref=RHO_REF, alpha0=DUCT_ALPHA0, y=1.0)
    rel = med.relaxation(0.6 * F0, 2.4 * F0)
    w0 = 2 * np.pi * F0
    a0 = DUCT_ALPHA0 * F0 / 1e6
    delta = 2 * a0 * C0 ** 3 / w0 ** 2            # alpha_delta(w) = delta w^2 / (2 c^3), matched at f0
    ratio_delta = delta * (2 * w0) ** 2 / (2 * C0 ** 3) / a0
    ratio_relax = rel.alpha(2 * F0)[0] / rel.alpha(F0)[0]
    assert abs(ratio_delta - 4.0) < 1e-12
    assert abs(ratio_relax - 2.0) < 2 * 2 * rel.fit_error + 1e-12
    assert rel.fit_error < 5e-3


# ---- CPU: the fit and the per-dof strengths ------------------------------------------------------------------------
# Measured with Medium.relaxation (max relative error of the exact alpha over the band, 1024 log-spaced frequencies):
#   0.5 dB/cm/MHz^1.1 over 1-3 MHz: 2.9e-4, over 1-5 MHz: 9.5e-4;  0.6 dB/cm/MHz^1.3 over 1-4 MHz: 9.9e-4;
#   10 dB/cm/MHz (c = 3000) over 1-3 MHz: 2.3e-4;  two processes, 0.5 dB/cm/MHz^1.1 over 1-3 MHz: 2.4e-3
FIT_CASES = [  # (alpha0 dB/cm/MHz^y, y, c, f_lo, f_hi, M, bound on fit_error)
    (0.5, 1.1, 1540.0, 1e6, 3e6, 3, 1e-3), (0.5, 1.1, 1540.0, 1e6, 5e6, 3, 3e-3), (0.6, 1.3, 1540.0, 1e6, 4e6, 3, 3e-3),
    (10.0, 1.0, 3000.0, 1e6, 3e6, 3, 1e-3), (0.5, 1.1, 1540.0, 1e6, 3e6, 2, 5e-3),
]


@pytest.mark.parametrize("case", FIT_CASES, ids=[f"a{c[0]}-y{c[1]}-{c[3] / 1e6:g}-{c[4] / 1e6:g}MHz-M{c[5]}"
                                                 for c in FIT_CASES])
def test_fit_reproduces_the_power_law(wfx, case):
    a, y, c, lo, hi, M, bound = case
    med = wfx.Medium(np.full(3, 1000.0), c, rho_ref=RHO_REF, alpha0=np.array([a, 0.0, a]) * DB_CM, y=y)
    rel = med.relaxation(lo, hi, M)
    assert rel.M == M and rel.eps.shape == (M, 3)
    assert rel.fit_error < bound, rel.fit_error
    f = np.geomspace(lo, hi, 777)
    got = rel.alpha(f)
    want = a * DB_CM * (f / 1e6) ** y
    # fit_error is the maximum over 1024 frequencies; between them the error peaks within 0.1 % of it
    assert np.abs(got[:, 0] / want - 1).max() <= rel.fit_error * 1.001
    assert np.array_equal(rel.eps[:, 0], rel.eps[:, 2]) and not np.any(rel.eps[:, 1]) and not np.any(got[:, 1])
    # causal dispersion: the phase speed lies below c and rises with frequency
    cp = rel.phase_speed(f)[:, 0]
    assert np.all(cp < c) and np.all(np.diff(cp) > 0)
    assert rel.max_dt() < 2.5 * rel.tau.min() / (1 + rel.eps.max(axis=1).sum())


def test_eps_dofs_is_the_weighted_sum(wfx, orc):
    """eps_i against a direct loop over cells and points; a dof whose cells share one eps gets it exactly"""
    P = 2
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15, renumber=5)
    med = random_medium(wfx, mesh.ncells, 1)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    mu = med.mass_weight(mesh.ncells, C0)
    rel = random_relaxation(wfx, mesh.ncells, 3, 4)
    perm = wfx.capi.compute_permutations(P)
    num, den = np.zeros((3, mesh.ndofs)), np.zeros(mesh.ndofs)
    for cell in range(mesh.ncells):
        for t in range(len(perm)):
            i = mesh.dofmap[cell, perm[t]]
            num[:, i] += rel.eps[:, cell] * mu[cell] * detJ[cell, t]
            den[i] += mu[cell] * detJ[cell, t]
    got = rel.eps_dofs(mesh, detJ, mu)
    assert got.shape == (3, mesh.ndofs)
    assert np.abs(got - num / den).max() <= 1e-15 * rel.eps.max()
    shared = wfx.Relaxation(rel.tau, np.array([0.01, 0.0237, 0.031]), C0)
    assert np.all(shared.eps_dofs(mesh, detJ, mu) == np.array([0.01, 0.0237, 0.031])[:, None])


def test_refusals_on_the_host(wfx):
    tau = [1e-7, 2e-7]
    for args in (([0.0], [0.1], C0), ([-1e-7], [0.1], C0), ([np.nan], [0.1], C0), (tau, [0.1, -0.1], C0),
                 (tau, [0.1, np.inf], C0), ([1e-7] * 4, [0.1] * 4, C0), (tau, [0.1], C0), (tau, np.zeros((3, 5)), C0),
                 (tau, [0.1, 0.1], 0.0), (tau, np.zeros((2, 4)), np.full(5, C0)), ([], [], C0)):
        with pytest.raises(wfx.WfxError):
            wfx.Relaxation(*args)
    with pytest.raises(wfx.WfxError):
        wfx.Medium(RHO_REF, C0, alpha0=1.0)
    with pytest.raises(wfx.WfxError):
        wfx.Medium(RHO_REF, C0, alpha0=-1.0, y=1.0)
    with pytest.raises(wfx.WfxError):
        wfx.Medium(RHO_REF, C0, alpha0=1.0, y=0.0)
    with pytest.raises(wfx.WfxError):
        wfx.Medium(RHO_REF, C0).relaxation(1e6, 3e6)
    med = wfx.Medium(RHO_REF, C0, alpha0=5.0, y=1.1)
    for band, M in (((3e6, 1e6), 3), ((1e6, 3e6), 4), ((1e6, 3e6), 0), ((0.0, 3e6), 2)):
        with pytest.raises(wfx.WfxError):
            med.relaxation(*band, mechanisms=M)
    rel = med.relaxation(1e6, 3e6)
    with pytest.raises(wfx.WfxError):
        rel.eps_cells(7) if rel.eps.shape[1] == 7 else wfx.Relaxation(rel.tau, np.zeros((3, 5)), C0).eps_cells(7)
    mesh = wfx.create_box_hex((2, 1, 1), 2, (0.02, 0.01, 0.01))
    # linear and ensemble models refuse relaxation= before touching the device
    with pytest.raises(wfx.WfxError, match="LossyGLLOpt"):
        wfx.LinearGLLOpt(mesh, None, 2, C0, F0, P0, relaxation=rel)
    with pytest.raises(wfx.WfxError, match="LossyGLLOpt"):
        wfx.LinearGLLEnsemble(mesh, None, 2, C0, (F0,), (P0,), relaxation=rel)


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _model(wfx, name, mesh, P, dtype, medium, relaxation=None, **kw):
    if name.startswith("lossy"):
        delta = 0.0 if name == "lossy0" else DELTA
        return wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, delta, dtype=dtype, medium=medium, relaxation=relaxation,
                               **kw)
    return wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype, medium=medium,
                                relaxation=relaxation, **kw)


def _random_state(n, seed, dtype):
    rng = np.random.default_rng(seed)
    u = (0.3 * P0 * rng.standard_normal(n)).astype(dtype).astype(np.float64)
    v = (0.3 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype).astype(np.float64)
    return u, v


PARITY = [  # (P, dtype, graph, M, model); westervelt: scalar kappa (medium without beta), westervelt-kd: per-dof kappa
    (2, np.float64, True, 1, "lossy0"), (2, np.float64, False, 3, "westervelt-kd"), (3, np.float64, True, 2, "lossy"),
    (3, np.float64, False, 1, "westervelt"), (4, np.float64, True, 3, "lossy"), (4, np.float64, False, 2, "lossy0"),
    (4, np.float64, True, 1, "westervelt-kd"), (5, np.float64, True, 2, "westervelt"),
    (5, np.float64, False, 3, "lossy"), (4, np.float32, True, 3, "westervelt-kd"), (4, np.float32, False, 2, "lossy"),
    (7, np.float32, True, 2, "lossy"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY, ids=[f"P{c[0]}-{np.dtype(c[1]).name}-graph{int(c[2])}-M{c[3]}-{c[4]}"
                                              for c in PARITY])
def test_relaxing_models_match_the_restatement(wfx, orc, mo, torch, monkeypatch, case):
    """RK4 with a shortened last step through the ramp's end in a random medium with random per-cell eps (both tags, so
    the Gamma2 kernel runs), against the restatement; the memory variables too; f1 against wo_f1_westervelt_relax."""
    P, dtype, graph, M, name = case
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    rel = random_relaxation(wfx, mesh.ncells, M, 50 + P)
    if name == "westervelt":
        # the scalar kappa needs the model without a medium; the restatement takes the identity medium's weights (1)
        med = wfx.Medium(RHO_REF, C0, rho_ref=RHO_REF)
        eqn = _model(wfx, name, mesh, P, dtype, None, rel)
    else:
        med = random_medium(wfx, mesh.ncells, 40 + P, beta=name == "westervelt-kd")
        eqn = _model(wfx, name, mesh, P, dtype, med, rel)
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    eps = eqn.relaxation_eps                 # the model's own (from the device's detJ w), as the kappa below
    np.testing.assert_allclose(eps, rel.eps_dofs(mesh, detJ, mu), rtol=1e-14, atol=0)
    delta = 0.0 if name == "lossy0" else DELTA
    if name.startswith("westervelt"):
        kappa = eqn.kappa if eqn.kappa is not None else np.full(mesh.ndofs, KAPPA)
        assert (eqn.kappa is not None) == (name == "westervelt-kd")
    else:
        kappa = np.zeros(mesh.ndofs)
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), rel.max_dt())
    u, v = _random_state(mesh.ndofs, P, dtype)
    if name.startswith("westervelt"):
        u, v = 0.1 * u, 0.1 * v
    t0, steps = 7.5e-6, 12
    tf = t0 + (steps - 0.5) * dt
    uo, vo, qo = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
    so, to = mo.rk4_westervelt_relax(mesh, P, G, m, m1, m2, kappa, C0, F0, P0, delta, rel.tau, eps, t0, tf, dt, uo, vo,
                                     qo, sumfact=True, nthreads=orc.max_threads())
    eqn.set_state(u, v)
    s, t = eqn.rk4(t0, tf, dt)
    ug, vg = eqn.get_state()
    qg = eqn.relaxation_state()
    assert (s, t) == (so, to) and s == steps
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    errs = (rel_l2(ug, uo), rel_l2(vg, vo), rel_l2(qg, qo))
    assert max(errs) < tol, errs
    # f1 at the model's memory variables
    fo = mo.f1_westervelt_relax(mesh, P, G, m, m1, m2, kappa, C0, F0, P0, delta, rel.tau, eps, 3e-6, u, v,
                                np.ascontiguousarray(qg, dtype=np.float64))
    res = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64 if dtype == np.float64 else torch.float32,
                     device="cuda")
    tdev = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(dtype))).cuda()  # noqa: E731
    eqn.f1(3e-6, tdev(u), tdev(v), res)
    assert rel_l2(res.cpu().numpy(), fo) < (TOL64 if dtype == np.float64 else 2e-5)



def _run(eqn, u, v, t0, tf, dt):
    eqn.set_state(u, v)
    st = eqn.rk4(t0, tf, dt)
    return st, eqn.get_state()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", ["lossy", "westervelt-kd"])
def test_zero_strength_and_none_are_the_model_without_relaxation(wfx, torch, dtype, name):
    """eps = 0 (M = 3) and set_relaxation(None) give the model without relaxation bit for bit"""
    P = 4
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.04, 0.02, 0.02), perturb=0.1)
    med = random_medium(wfx, mesh.ncells, 3, beta=name == "westervelt-kd")
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    u, v = (0.1 * a for a in _random_state(mesh.ndofs, 1, dtype))
    tf = 1e-6 + 20.5 * dt
    a = _run(_model(wfx, name, mesh, P, dtype, med), u, v, 1e-6, tf, dt)
    # relaxation frequencies low enough for the CFL step to stay inside the relaxation's bound
    zero = wfx.Relaxation(1.0 / (2 * np.pi * np.array([0.1e6, 0.3e6, 0.6e6])), np.zeros((3, mesh.ncells)), C0)
    eqn = _model(wfx, name, mesh, P, dtype, med, zero)
    b = _run(eqn, u, v, 1e-6, tf, dt)
    assert a[0] == b[0] and np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])
    some = wfx.Relaxation(zero.tau[:2], np.random.default_rng(1).uniform(0.0, 0.05, (2, mesh.ncells)), C0)
    assert dt < some.max_dt()
    eqn.set_relaxation(some)
    c = _run(eqn, u, v, 1e-6, tf, dt)
    assert not np.array_equal(a[1][0], c[1][0])
    eqn.set_relaxation(None)
    d = _run(eqn, u, v, 1e-6, tf, dt)
    assert a[0] == d[0] and np.array_equal(a[1][0], d[1][0]) and np.array_equal(a[1][1], d[1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_checkpoint_restart_is_bitwise(wfx, torch, dtype):
    """get u, v and q after 15 steps, set_state + set_relaxation_state into a fresh model, continue: the same as one
    run of 30 steps; init zeroes q and keeps the configuration"""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 5)
    rel = random_relaxation(wfx, mesh.ncells, 3, 6)
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), rel.max_dt())
    u, v = (0.1 * a for a in _random_state(mesh.ndofs, 2, dtype))
    one = _model(wfx, "westervelt-kd", mesh, P, dtype, med, rel)
    one.set_state(u, v)
    _, t1 = one.rk4(0.0, 1.0, dt, max_steps=15)
    cu, cv = one.get_state()
    cq = one.relaxation_state()
    assert np.any(cq)
    one.rk4(t1, 1.0, dt, max_steps=15)
    two = _model(wfx, "westervelt-kd", mesh, P, dtype, med, rel)
    two.set_state(cu, cv)
    assert not np.any(two.relaxation_state())
    two.set_relaxation_state(cq)
    two.rk4(t1, 1.0, dt, max_steps=15)
    for x, y in zip(one.get_state() + (one.relaxation_state(),), two.get_state() + (two.relaxation_state(),)):
        assert np.array_equal(x, y)
    one.init()
    assert not np.any(one.relaxation_state()) and one.relaxation is rel
    with pytest.raises(wfx.WfxError):
        two.set_relaxation_state(cq[:2])


@pytest.mark.gpu
def test_refusals_on_the_device(wfx, torch):
    P = 2
    mesh = wfx.create_box_hex((2, 2, 2), P, (0.02, 0.02, 0.02))
    med = wfx.Medium(RHO_REF, C0)
    eqn = _model(wfx, "lossy", mesh, P, np.float64, med)
    h, n = eqn.handle, mesh.ndofs
    call = wfx.capi.call
    f = wfx.capi.f64p
    tau, eps = np.array([1e-7, 2e-7]), np.full(2 * n, 0.01)
    for bad_tau, bad_eps, M in ((np.array([0.0, 1e-7]), eps, 2), (np.array([-1e-7, 1e-7]), eps, 2),
                                (np.array([np.nan, 1e-7]), eps, 2), (tau, np.where(np.arange(2 * n) == 3, -0.1, eps), 2),
                                (tau, np.where(np.arange(2 * n) == 5, np.inf, eps), 2),
                                (np.full(4, 1e-7), np.full(4 * n, 0.01), 4), (tau, eps, -1)):
        with pytest.raises(wfx.WfxError):
            call("wfx_wave_set_relaxation", h, M, f(bad_tau), f(bad_eps))
    with pytest.raises(wfx.WfxError):
        eqn.relaxation_state()          # no relaxation yet
    with pytest.raises(wfx.WfxError):
        call("wfx_wave_get_relaxation_state", h, np.zeros(n).ctypes.data)
    lin = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, (F0, F0), (P0, P0))
    for other in (lin, ens):
        with pytest.raises(wfx.WfxError):
            call("wfx_wave_set_relaxation", other.handle, 2, f(tau), f(eps))
    # snapshots: refused with relaxation, and relaxation refused while snapshots are on
    rel = wfx.Relaxation(tau, [0.01, 0.02], C0)
    eqn.set_snapshot(5, lambda *a: None)
    with pytest.raises(wfx.WfxError):
        eqn.set_relaxation(rel)
    eqn.set_snapshot(0, None)
    eqn.set_relaxation(rel)
    with pytest.raises(wfx.WfxError):
        eqn.set_snapshot(5, lambda *a: None)
    # the step bound: dt (1 + sum max eps) / tau_min < 2.5
    bound = 2.5 * 1e-7 / 1.03 * (1 + 1e-12)
    eqn.init()
    eqn.rk4(0.0, 1.0, rel.max_dt(), max_steps=1)
    with pytest.raises(wfx.WfxError, match="2.5"):
        eqn.rk4(0.0, 1.0, bound, max_steps=1)
    with pytest.raises(wfx.WfxError):
        eqn.set_relaxation_state(np.zeros((3, n)))


@pytest.mark.gpu
def test_field_stats_and_heating_of_a_relaxing_model(wfx, orc, torch):
    """A relaxing Westervelt model's harmonic maps equal a reference accumulation of its probe series, and
    heat_from_wave(medium=) with alpha0 = None heats with the medium's per-dof mass-weighted alpha0"""
    P = 3
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.012, 0.006, 0.006), perturb=0.1)
    med = random_medium(wfx, mesh.ncells, 71, beta=False)
    rel = med.relaxation(0.5 * F0, 2 * F0)
    eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, 0.0, 3.5, RHO0, medium=med, relaxation=rel)
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), rel.max_dt())
    eqn.init()
    eqn.set_field_stats(2.0 / F0, 2)
    eqn.set_probes(np.arange(mesh.ndofs, dtype=np.int32), 4096)
    nsteps = int(np.ceil(4.0 / F0 / dt))
    eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)
    fs = eqn.field_stats()
    ts, vals = eqn.probe_series()
    sel = ts >= 2.0 / F0 - 0.5 * dt
    assert fs.samples == sel.sum() > 0
    for h in (1, 2):
        want = 2.0 / sel.sum() * (vals[sel] * np.exp(-1j * h * 2 * np.pi * F0 * ts[sel])[:, None]).sum(0)
        np.testing.assert_allclose(fs.harmonics[h - 1], want, rtol=0, atol=1e-10 * np.abs(want).max())
    assert np.array_equal(fs.pmax, vals[sel].max(0))
    th = wfx.PennesGLL(mesh, P, 0.5, 3.6e6)
    th.heat_from_wave(eqn, None, medium=med)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    a_i = wfx.cell_to_dof_average(mesh, detJ, med.alpha0)
    inv_z = wfx.cell_to_dof_average(mesh, detJ, 1.0 / (med.rho * med.c))
    want = sum((h * F0 / 1e6) ** 1.1 * np.abs(fs.harmonics[h - 1]) ** 2 for h in (1, 2)) * a_i * inv_z
    np.testing.assert_allclose(th.heat_source(), want, rtol=1e-13, atol=1e-13 * want.max())
    per_cell_y = wfx.Medium(med.rho, med.c, alpha0=med.alpha0, y=np.linspace(1.0, 1.2, mesh.ncells))
    with pytest.raises(wfx.WfxError):
        th.heat_from_wave(eqn, None, medium=per_cell_y)
    with pytest.raises(wfx.WfxError):
        th.heat_from_wave(eqn, None, medium=wfx.Medium(med.rho, med.c))


@pytest.mark.gpu
def test_demo_relaxation_option(wfx, torch):
    """demo/planar3d.py --relaxation 3 with a soft-tissue slab: it runs, reports the fit and the phase speed, and the
    wave loses amplitude across the absorbing slab"""
    r = subprocess.run(["python", os.path.join(ROOT, "demo", "planar3d.py"), "--nx", "16", "--nyz", "1",
                        "--length", "0.012", "--model", "lossy", "--delta", "0", "--stats-periods", "2",
                        "--layer", "0.0045", "0.0105", "--layer-rho", "1050", "--layer-c", "1540",
                        "--absorption", "60", "--absorption-power", "1.1", "--relaxation", "3",
                        "--heat-seconds", "0.5"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    out = r.stdout
    assert "relaxation: 3 processes" in out and "phase speed" in out and "thermal: peak rise" in out, out
    vals = {}
    for side in ("before the layer", "after the layer"):
        line = [ln for ln in out.splitlines() if ln.startswith(side)][0]
        vals[side] = float(line.split("mean ")[1].split(",")[0])
    assert 0 < vals["after the layer"] < vals["before the layer"], vals


# ---- C++ wrappers ------------------------------------------------------------------------------------------------
def _build_cpp(wfx, outdir):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_relaxation_hpp.cpp")
    exe = os.path.join(str(outdir), "test_wavefx_relaxation_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_relaxation_cpp_wrapper_compiles_and_links(wfx, tmp_path):
    assert os.path.exists(_build_cpp(wfx, tmp_path))


@pytest.mark.gpu
def test_relaxation_cpp_wrapper_reproduces_python(wfx, torch, tmp_path):
    """WesterveltGLLOpt with a medium and set_relaxation from C++, 15 steps, get / set of the memory variables through a
    restart, 15 more: the same u and q as the Python model bit for bit"""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 91)
    rel = random_relaxation(wfx, mesh.ncells, 2, 92)
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), rel.max_dt())
    u, v = (0.1 * a for a in _random_state(mesh.ndofs, 5, np.float64))
    west = _model(wfx, "westervelt-kd", mesh, P, np.float64, med, rel)
    files = {"params.f64": np.array([P, C0, F0, P0, DELTA, BETA, RHO0, dt, rel.M]),
             "x.f64": mesh.x, "xdofs.i32": mesh.xdofs, "dofmap.i32": mesh.dofmap,
             "fcell.i32": mesh.facet_cells, "flocal.i32": mesh.facet_local, "ftag.i32": mesh.facet_tags,
             "u.f64": u, "v.f64": v, "stiffness.f64": med.stiffness_weight(mesh.ncells),
             "mass.f64": med.mass_weight(mesh.ncells, C0), "facet.f64": med.facet_weight(mesh, C0),
             "kappa.f64": west.kappa, "tau.f64": rel.tau, "eps.f64": west.relaxation_eps}
    for name, a in files.items():
        np.ascontiguousarray(a, dtype=np.int32 if name.endswith("i32") else np.float64).tofile(str(tmp_path / name))
    r = subprocess.run([_build_cpp(wfx, tmp_path), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "relaxation hpp ok" in r.stdout, r.stdout + r.stderr
    west.set_state(u, v)
    _, t1 = west.rk4(0.0, 1.0, dt, max_steps=15)
    cu, cv = west.get_state()
    cq = west.relaxation_state()
    west.set_state(cu, cv)
    west.set_relaxation_state(cq)
    west.rk4(t1, 1.0, dt, max_steps=15)
    got = lambda name: np.fromfile(str(tmp_path / name), dtype=np.float64)  # noqa: E731
    assert np.array_equal(got("u.out.f64"), west.get_state()[0])
    assert np.array_equal(got("q.out.f64"), west.relaxation_state().reshape(-1))
