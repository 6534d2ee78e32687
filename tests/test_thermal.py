"""Thermal model (DESIGN.md section 4.5d): the Pennes bioheat equation on the GLL mesh, RK4 on the device, and the
CEM43 thermal dose, heated from the acoustic harmonic maps.

    rhoC theta_t = div(k grad theta) - wbCb theta + s Q,   -k d theta / dn = h_j (theta - (T_ext_j - T_art)) on tag j

CPU: the restatement (model_oracle.rk4_pennes) against a textbook numpy RK4 of the lumped system with a dense K,
known answers on the restatement, the mass-weighted conversion, and that the C++ wrapper compiles.  GPU: rhs and rk4
against the restatement, graph replay, split runs, the dose at constant temperatures, the stable step against
eigvalsh, the heat source from the wave model's harmonic maps, shared operators, the error paths and the C++ wrapper.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_ART = 37.0
K_T, RHOC, WBCB = 0.5, 3.6e6, 2.0e4      # soft-tissue-like conductivity, heat capacity and (raised) perfusion
H12, TEXT12 = (300.0, 40.0), (20.0, 45.0)  # a cooled face (tag 1) and a warm one (tag 2)
RK4_LIMIT = 2.785293563405282


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


def _inputs(orc, mesh, P):
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    return G, detJ, m, m1, m2


def _fields(mesh, seed):
    """non-uniform rhoC, perfusion and Q, and a start rise spanning 41..46 degC"""
    rng = np.random.default_rng(seed)
    n = mesh.ndofs
    rhoc = RHOC * (1 + 0.3 * rng.random(n))
    perf = WBCB * rng.random(n)
    Q = 5e6 * rng.random(n)
    theta = 4.0 + 5.0 * rng.random(n)
    return rhoc, perf, Q, theta


def dense_A(orc, mesh, P, G):
    """A = -1500^2 K assembled column by column from the oracle's stiffness apply"""
    n = mesh.ndofs
    A = np.empty((n, n))
    e = np.zeros(n)
    for j in range(n):
        e[:] = 0.0
        e[j] = 1.0
        y = np.zeros(n)
        orc.stiffness_apply(mesh, P, G, e, y, dense=True)
        A[:, j] = y
    return A


def lumped_system(A, m, m1, m2, k, rhoc, perf, h, T_ext, Q, s):
    """theta' = L theta + F of the lumped system"""
    cap = rhoc * m
    Lm = (k / 1500.0 ** 2) * A - np.diag(perf * m + h[0] * m1 + h[1] * m2)
    F = h[0] * m1 * (T_ext[0] - T_ART) + h[1] * m2 * (T_ext[1] - T_ART) + s * Q * m
    return Lm / cap[:, None], F / cap


def dose_rate(theta):
    T = T_ART + theta
    return np.where(T >= 43.0, 0.5, 0.25) ** (43.0 - T)


# ---- CPU ------------------------------------------------------------------------------------------------------
def test_restatement_matches_textbook_numpy_rk4(wfx, orc, mo):
    """wo_rk4_pennes against classical RK4 of theta' = L theta + F, L from a dense K, with the dose and peak rise
    summed after every step (2^3 cells, P2, both Robin tags, non-uniform rhoC and perfusion, a shortened last step)."""
    P = 2
    mesh = wfx.create_box_hex(2, P, (0.01, 0.01, 0.01), perturb=0.1)
    G, _, m, m1, m2 = _inputs(orc, mesh, P)
    rhoc, perf, Q, theta0 = _fields(mesh, 1)
    s = 0.7
    L, F = lumped_system(dense_A(orc, mesh, P, G), m, m1, m2, K_T, rhoc, perf, H12, TEXT12, Q, s)
    dt = 0.5 * RK4_LIMIT / np.abs(np.linalg.eigvals(L)).max()
    tf = 12.3 * dt
    th, cem, thmax, t, steps = theta0.copy(), np.zeros(mesh.ndofs), np.full(mesh.ndofs, -np.inf), 0.0, 0
    f = lambda x: L @ x + F
    while t < tf:
        h = min(dt, tf - t)
        k1 = f(th)
        k2 = f(th + 0.5 * h * k1)
        k3 = f(th + 0.5 * h * k2)
        k4 = f(th + h * k3)
        th = th + h / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
        cem += h / 60 * dose_rate(th)
        thmax = np.maximum(thmax, th)
        t += h
        steps += 1
    u, c, mx = theta0.copy(), np.zeros(mesh.ndofs), np.full(mesh.ndofs, -np.inf)
    n, t_end = mo.rk4_pennes(mesh, P, G, m, m1, m2, K_T, rhoc, perf, T_ART, H12, TEXT12, Q, s, 0.0, tf, dt, u, c, mx)
    assert (n, t_end) == (steps, t) and steps == 13
    rel = lambda a, b: np.abs(a - b).max() / np.abs(b).max()
    assert rel(u, th) <= 1e-13 and rel(c, cem) <= 1e-13 and rel(mx, thmax) <= 1e-13
    assert (T_ART + th).min() < 43 < (T_ART + th).max()             # both branches of R
    r = mo.rhs_pennes(mesh, P, G, m, m1, m2, K_T, rhoc, perf, T_ART, H12, TEXT12, Q, s, theta0)
    assert rel(r, f(theta0)) <= 1e-13


# Known answers on the restatement.  Bounds set from these runs (fp64), where they measured:
#   uniform relaxation  max |theta / exact - 1| = 1.6e-8, the RK4 truncation (r dt = 0.05, 40 steps); against
#                       RK4's own amplification factor R(-r dt)^n in place of e^{-rt}: 4.4e-16
#   cos mode            |decay / exp(-(k / rhoC)(pi / L)^2 t) - 1| = 3.9e-10   (4 cells of P4 along x, t = 20 s)
#   Robin slab          max |rhs(theta_ss)| / (Q / rhoC) = 3.5e-15 (P2), 6.8e-13 (P4)
KNOWN_BOUNDS = dict(uniform=5e-8, uniform_discrete=1e-13, cos_mode=2e-9, slab=1e-11)


def test_uniform_relaxation_known_answer(wfx, orc, mo):
    """uniform theta, perfusion and Q, insulated: theta(t) = theta_inf + (theta0 - theta_inf) e^{-rt}"""
    P = 3
    mesh = wfx.create_box_hex((2, 2, 1), P, (0.02, 0.02, 0.01), perturb=0.1, tags=())
    G, _, m, m1, m2 = _inputs(orc, mesh, P)
    n = mesh.ndofs
    wb, Q = 2e6, 4e7                         # strong perfusion: r dt = 0.05 lies well inside the diffusion's limit
    r, theta_inf = wb / RHOC, Q / wb
    dt = 0.05 / r
    u, c, mx = np.full(n, 1.0), np.zeros(n), np.full(n, -np.inf)
    steps, t = mo.rk4_pennes(mesh, P, G, m, m1, m2, K_T, np.full(n, RHOC), np.full(n, wb), T_ART, (0, 0), (0, 0),
                             np.full(n, Q), 1.0, 0.0, 1e9, dt, u, c, mx, max_steps=40)
    exact = theta_inf + (1.0 - theta_inf) * np.exp(-r * t)
    assert steps == 40 and np.abs(u / exact - 1).max() < KNOWN_BOUNDS["uniform"]
    z = -r * dt
    discrete = theta_inf + (1.0 - theta_inf) * (1 + z + z ** 2 / 2 + z ** 3 / 6 + z ** 4 / 24) ** 40
    assert np.abs(u / discrete - 1).max() < KNOWN_BOUNDS["uniform_discrete"], np.abs(u / discrete - 1).max()


def test_cosine_mode_decay_known_answer(wfx, orc, mo):
    """cos(pi x / L) on an insulated box decays as exp(-(k / rhoC)(pi / L)^2 t)"""
    P, L = 4, 0.01
    mesh = wfx.create_box_hex((4, 1, 1), P, (L, L / 4, L / 4), tags=())
    G, _, m, m1, m2 = _inputs(orc, mesh, P)
    x = wfx.dof_coordinates(mesh)[:, 0]
    u = np.cos(np.pi * x / L)
    n = mesh.ndofs
    c, mx = np.zeros(n), np.full(n, -np.inf)
    steps, t = mo.rk4_pennes(mesh, P, G, m, m1, m2, K_T, np.full(n, RHOC), None, T_ART, (0, 0), (0, 0), None, 1.0,
                             0.0, 1e9, 0.02, u, c, mx, max_steps=1000)
    decay = (u @ (m * np.cos(np.pi * x / L))) / ((m * np.cos(np.pi * x / L)) @ np.cos(np.pi * x / L))
    exact = np.exp(-(K_T / RHOC) * (np.pi / L) ** 2 * t)
    assert steps == 1000 and abs(decay / exact - 1) < KNOWN_BOUNDS["cos_mode"], decay / exact - 1


def slab_steady_state(x, L, h, T_ext, Q):
    """k theta'' + Q = 0, -k theta'(0)(-1) = h (theta(0) - (T_ext - T_art)), theta'(L) = 0"""
    return (T_ext - T_ART) + Q * L / h + Q / K_T * (L * x - x * x / 2)


@pytest.mark.parametrize("P", [2, 4])
def test_robin_slab_steady_state_has_rounding_level_residual(wfx, orc, mo, P):
    L, h, T_ext, Q = 0.02, 500.0, 30.0, 2e5
    mesh = wfx.create_box_hex((3, 2, 1), P, (L, 0.01, 0.005), tags=((0, 0, 1),))
    G, _, m, m1, m2 = _inputs(orc, mesh, P)
    x = wfx.dof_coordinates(mesh)[:, 0]
    n = mesh.ndofs
    theta = slab_steady_state(x, L, h, T_ext, Q)
    r = mo.rhs_pennes(mesh, P, G, m, m1, m2, K_T, np.full(n, RHOC), None, T_ART, (h, 0.0), (T_ext, T_ART),
                      np.full(n, Q), 1.0, theta)
    assert np.abs(r).max() / (Q / RHOC) < KNOWN_BOUNDS["slab"]


def test_mass_weighted_conversion_conserves_heat_capacity(wfx, orc):
    """sum_i rhoC_i m_i = sum_c rhoC_c vol_c for the per-dof average of a per-cell rhoC"""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15, renumber=5)
    _, detJ, m, _, _ = _inputs(orc, mesh, P)
    rhoc_c = RHOC * (1 + np.random.default_rng(2).random(mesh.ncells))
    rhoc = wfx.cell_to_dof_average(mesh, detJ, rhoc_c)
    want = (rhoc_c * detJ.sum(axis=1)).sum()
    assert abs((rhoc * m).sum() / want - 1) < 1e-13
    assert rhoc.min() >= rhoc_c.min() * (1 - 1e-15) and rhoc.max() <= rhoc_c.max() * (1 + 1e-15)
    assert np.allclose(wfx.cell_to_dof_average(mesh, detJ, np.full(mesh.ncells, 7.0)), 7.0, rtol=1e-15, atol=0)


def _build_cpp(wfx, outdir):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_thermal_hpp.cpp")
    exe = os.path.join(str(outdir), "test_wavefx_thermal_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_thermal_cpp_wrapper_compiles_and_links(wfx, tmp_path):
    assert os.path.exists(_build_cpp(wfx, tmp_path))


# planar linear wave (the case of tests/test_field_stats.py): Q = alpha0 (f0 / 1 MHz)^y p0^2 / (rho0 c0) away from
# both ends.  On the CPU restatement (oracle.rk4, two whole periods sampled from 9 periods on) the heat source built
# from the DFT of the records measured max |Q / Q_plane - 1| = 2.5e-7 over the line; bound 1e-5.
C0, F0, P0, RHO0 = 1500.0, 0.5e6, 6e4, 1000.0
ALPHA0, ALPHA_Y = 5.0, 1.1
PLANAR_L, PLANAR_NX, PLANAR_Q_BOUND = 0.01, 33, 1e-5


def _planar_case(wfx):
    P = 4
    side = PLANAR_L / PLANAR_NX
    mesh = wfx.create_box_hex((PLANAR_NX, 2, 2), P, (PLANAR_L, 2 * side, 2 * side))
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    k = int(round(1.0 / F0 / dt))
    n0, n = 9 * k, 2 * k
    X = wfx.dof_coordinates(mesh)
    line = np.where((np.abs(X[:, 1]) < 1e-12) & (np.abs(X[:, 2]) < 1e-12))[0]
    return mesh, P, dt, n0, n, line[np.argsort(X[line, 0])]


def heat_from_harmonics(harm, f0, alpha0, y):
    """numpy statement of Q from amplitudes harm [H, ...] (already scaled by 2 / N)"""
    Q = np.zeros(harm.shape[1:])
    for h in range(1, harm.shape[0] + 1):
        Q += alpha0 * (h * f0 / 1e6) ** y * np.abs(harm[h - 1]) ** 2 / (RHO0 * C0)
    return Q


def plane_wave_heat():
    return ALPHA0 * (F0 / 1e6) ** ALPHA_Y * P0 ** 2 / (RHO0 * C0)


def test_planar_heat_source_known_answer_on_the_cpu_restatement(wfx, orc):
    mesh, P, dt, n0, n, line = _planar_case(wfx)
    G, _, m, m1, m2 = _inputs(orc, mesh, P)
    u, v = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    kw = dict(sumfact=True, nthreads=orc.max_threads())
    _, t = orc.rk4(mesh, P, G, m, m1, m2, C0, F0, P0, 0.0, 1.0, dt, u, v, max_steps=n0, **kw)
    rec, times = [], []
    for _ in range(n):
        _, t = orc.rk4(mesh, P, G, m, m1, m2, C0, F0, P0, t, 1.0, dt, u, v, max_steps=1, **kw)
        rec.append(u[line].copy())
        times.append(t)
    rec, times = np.array(rec), np.array(times)
    harm = np.array([(2.0 / n) * (rec * np.exp(-1j * h * 2 * np.pi * F0 * times)[:, None]).sum(axis=0)
                     for h in (1, 2, 3)])
    Q = heat_from_harmonics(harm, F0, ALPHA0, ALPHA_Y)
    assert np.abs(Q / plane_wave_heat() - 1).max() < PLANAR_Q_BOUND


# ---- GPU ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


TOL = {np.float64: 1e-12, np.float32: 2e-5}


def rel(a, b):
    return np.abs(np.asarray(a, dtype=np.float64) - b).max() / np.abs(b).max()


def _case(wfx, orc, P, renumber=None, dtype=np.float64, boundary=True, per_cell_k=False, seed=0):
    """a perturbed box with both Robin tags, non-uniform rhoC / perfusion (per cell), a heat source, and the
    restatement's inputs for the same model"""
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.015, 0.01, 0.01), perturb=0.15, renumber=renumber)
    rng = np.random.default_rng(seed)
    rhoc_c = RHOC * (1 + 0.4 * rng.random(mesh.ncells))
    perf_c = WBCB * rng.random(mesh.ncells)
    k = K_T * (1 + rng.random(mesh.ncells)) if per_cell_k else K_T
    h = H12 if boundary else (0.0, 0.0)
    th = wfx.PennesGLL(mesh, P, k, rhoc_c, perf_c, T_ART, h, TEXT12, dtype=dtype, boundary=boundary)
    G, _, m, m1, m2 = _inputs(orc, mesh, P)
    if per_cell_k:
        G = G * (np.asarray(k) / th.k)[:, None, None, None]
    Q = 3e6 * rng.random(mesh.ndofs)
    th.set_heat_source(Q)
    theta0 = 4.0 + 5.0 * rng.random(mesh.ndofs)
    args = (mesh, P, G, m, m1, m2, th.k, th.rhoc, th.perf, T_ART, h, TEXT12)
    return mesh, th, args, Q, theta0


def _dt(th):
    return 0.5 * th.max_eigenvalue(300)[1]


def _oracle_run(mo, orc, args, Q, s, theta, cem, mx, t0, tf, dt, max_steps=0):
    return mo.rk4_pennes(*args, Q, s, t0, tf, dt, theta, cem, mx, max_steps=max_steps, sumfact=True,
                         nthreads=orc.max_threads())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("P,renumber,boundary,per_cell_k", [(2, None, True, False), (3, 11, True, True),
                                                            (4, None, False, False), (5, 7, True, False),
                                                            (4, 3, False, True)])
def test_rhs_and_rk4_match_restatement(wfx, orc, mo, torch, P, renumber, boundary, per_cell_k, dtype):
    mesh, th, args, Q, theta0 = _case(wfx, orc, P, renumber, dtype, boundary, per_cell_k)
    tol = TOL[dtype]
    # rhs at a random state
    x = theta0.astype(dtype)
    want = mo.rhs_pennes(*args, Q, 1.0, x.astype(np.float64))
    out = torch.empty(mesh.ndofs, dtype=torch.float64 if dtype == np.float64 else torch.float32, device="cuda")
    th.rhs(torch.from_numpy(x).cuda(), out)
    assert rel(out.cpu().numpy(), want) <= tol
    # rk4 with a shortened last step
    dt = _dt(th)
    tf = 20.4 * dt
    th.set_state(T_ART + x.astype(np.float64))
    steps, t_end = th.rk4(0.0, tf, dt)
    u, cem, mx = x.astype(np.float64), np.zeros(mesh.ndofs), np.full(mesh.ndofs, -np.inf)
    s_o, t_o = _oracle_run(mo, orc, args, Q, 1.0, u, cem, mx, 0.0, tf, dt)
    assert (steps, t_end) == (s_o, t_o) == (21, t_o)
    d = th.dose()
    assert d.steps == 21
    assert rel(th.rise(), u) <= tol and rel(d.cem43, cem) <= tol and rel(d.T_max - T_ART, mx) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_graph_replay_split_runs_and_heat_scale(wfx, orc, mo, torch, monkeypatch, dtype):
    """graph replay on / off bitwise equal (with a shortened last step); several rk4 calls bitwise one call; a heat
    scale change between calls (heating, then cooling) against the restatement"""
    def run(graph, chunks, scales=None):
        monkeypatch.setenv("WFX_WAVE_GRAPH", "1" if graph else "0")
        mesh, th, args, Q, theta0 = _case(wfx, orc, 4, 5, dtype)
        dt = 0.5 * th.max_eigenvalue(300)[1]
        th.set_state(T_ART + theta0.astype(dtype).astype(np.float64))
        t = 0.0
        for i, c in enumerate(chunks):
            if scales:
                th.set_heat_scale(scales[i])
            t = th.rk4(t, 30.5 * dt, dt, max_steps=c)[1]
        d = th.dose()
        return th.rise(), d, (mesh, args, Q, theta0, dt)

    a, da, _ = run(True, [0])
    b, db, _ = run(False, [0])
    c, dc, _ = run(True, [7, 1, 12, 0])
    assert da.steps == db.steps == dc.steps == 31
    for x, y in ((a, b), (a, c), (da.cem43, db.cem43), (da.cem43, dc.cem43), (da.T_max, db.T_max), (da.T_max, dc.T_max)):
        assert np.array_equal(x, y)
    u, d, (mesh, args, Q, theta0, dt) = run(True, [10, 0], scales=[1.0, 0.0])
    w = theta0.astype(dtype).astype(np.float64)
    cem, mx = np.zeros(mesh.ndofs), np.full(mesh.ndofs, -np.inf)
    _, t = _oracle_run(mo, orc, args, Q, 1.0, w, cem, mx, 0.0, 30.5 * dt, dt, max_steps=10)
    _oracle_run(mo, orc, args, Q, 0.0, w, cem, mx, t, 30.5 * dt, dt)
    assert rel(u, w) <= TOL[dtype] and rel(d.cem43, cem) <= TOL[dtype] and rel(d.T_max - T_ART, mx) <= TOL[dtype]


@pytest.mark.gpu
@pytest.mark.parametrize("T", [41.0, 43.0, 45.0])
def test_cem43_at_constant_temperature(wfx, torch, T):
    P = 3
    mesh = wfx.create_box_hex((2, 2, 2), P, (0.01, 0.01, 0.01), perturb=0.1)
    th = wfx.PennesGLL(mesh, P, K_T, RHOC, 0.0, T_ART)
    th.set_state(np.full(mesh.ndofs, T))
    dt, N = 0.25, 37
    assert th.rk4(0.0, 100.0, dt, max_steps=N) == (N, N * dt)
    d = th.dose()
    want = N * dt / 60 * (0.5 if T >= 43 else 0.25) ** (43 - T)
    assert d.steps == N and np.abs(d.cem43 / want - 1).max() <= 1e-14
    assert np.abs(d.T_max - T).max() <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("P,boundary", [(2, True), (3, False), (4, True)])
def test_stable_dt_against_eigvalsh(wfx, orc, torch, P, boundary):
    """lambda of the power iteration never above the largest eigenvalue of the symmetrised dense operator and
    within 2 % below it"""
    mesh, th, args, Q, _ = _case(wfx, orc, P, boundary=boundary)
    mesh_, P_, G, m, m1, m2, k, rhoc, perf, _, h, _ = args
    A = dense_A(orc, mesh, P, G)
    cap = rhoc * m
    S = -(k / 1500.0 ** 2) * A + np.diag(perf * m + h[0] * m1 + h[1] * m2)
    S = 0.5 * (S + S.T)
    lam_max = np.linalg.eigvalsh(S / np.sqrt(cap)[:, None] / np.sqrt(cap)[None, :]).max()
    lam, dt_max = th.max_eigenvalue(200)
    assert lam <= lam_max * (1 + 1e-12) and lam >= 0.98 * lam_max, (lam, lam_max)
    assert dt_max == RK4_LIMIT / lam and th.stable_dt() == 0.8 * (RK4_LIMIT / lam)
    assert th.max_eigenvalue(200) == (lam, dt_max)                  # deterministic


def _wave_with_stats(wfx, mesh, P, nsteps=40, k0=10, nharm=3):
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    eqn.init()
    t = 0.0
    for _ in range(k0):
        t += dt
    eqn.set_field_stats(t, harmonics=nharm)
    eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)
    return eqn


@pytest.mark.gpu
def test_heat_from_wave_matches_numpy_on_field_stats(wfx, torch):
    P = 4
    mesh = wfx.create_box_hex((4, 3, 3), P, (0.04, 0.03, 0.03), perturb=0.15)
    eqn = _wave_with_stats(wfx, mesh, P)
    fs = eqn.field_stats()
    th = wfx.PennesGLL.from_wave(eqn, K_T, RHOC)
    alpha = ALPHA0 * (1 + np.random.default_rng(4).random(mesh.ndofs))
    for a0 in (ALPHA0, alpha):
        th.heat_from_wave(eqn, a0, ALPHA_Y, RHO0, C0)
        want = heat_from_harmonics(fs.harmonics, F0, a0, ALPHA_Y)
        assert want.max() > 0 and rel(th.heat_source(), want) <= 1e-13


@pytest.mark.gpu
def test_heat_from_wave_selects_the_ensemble_member(wfx, torch):
    P = 3
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.1)
    f0s, p0s = F0 * np.array([1.0, 1.13, 1.26]), P0 * np.array([1.0, 1.5, 2.0])
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, f0s.max())
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s, p0s)
    ens.init()
    ens.set_field_stats(10 * dt, harmonics=2)
    ens.rk4(0.0, 1.0, dt, max_steps=40)
    fs = ens.field_stats()
    th = wfx.PennesGLL(mesh, P, K_T, RHOC)
    qs = []
    for mbr in range(3):
        th.heat_from_wave(ens, ALPHA0, ALPHA_Y, RHO0, C0, member=mbr)
        want = heat_from_harmonics(fs.harmonics[..., mbr], f0s[mbr], ALPHA0, ALPHA_Y)
        qs.append(th.heat_source())
        assert rel(qs[-1], want) <= 1e-13
    assert rel(qs[1], qs[0]) > 1e-2 and rel(qs[2], qs[1]) > 1e-2


@pytest.mark.gpu
def test_planar_heat_source_known_answer_on_the_gpu(wfx, torch):
    mesh, P, dt, n0, n, line = _planar_case(wfx)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    eqn.init()
    t = 0.0
    for _ in range(n0 + 1):
        t += dt
    eqn.set_field_stats(t, harmonics=3)
    eqn.rk4(0.0, 1.0, dt, max_steps=n0 + n)
    th = wfx.PennesGLL.from_wave(eqn, K_T, RHOC)
    th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0)
    Q = th.heat_source()[line]
    assert np.abs(Q / plane_wave_heat() - 1).max() < PLANAR_Q_BOUND


@pytest.mark.gpu
def test_shared_operators_give_the_same_run_bitwise(wfx, torch):
    P = 4
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.015, 0.01, 0.01), perturb=0.15)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    rhoc_c = RHOC * (1 + 0.4 * np.random.default_rng(1).random(mesh.ncells))
    own = wfx.PennesGLL(mesh, P, K_T, rhoc_c, WBCB, T_ART, H12, TEXT12)
    shared = wfx.PennesGLL.from_wave(eqn, K_T, rhoc_c, WBCB, T_ART, H12, TEXT12)
    assert shared.stiff_op is eqn.stiff_op and shared.bnd_op is eqn.bnd_op
    theta0 = T_ART + 5 * np.random.default_rng(2).random(mesh.ndofs)
    Q = 1e6 * np.random.default_rng(3).random(mesh.ndofs)
    dt = own.stable_dt()
    assert shared.stable_dt() == dt
    outs = []
    for th in (own, shared):
        th.set_heat_source(Q)
        th.set_state(theta0)
        th.rk4(0.0, 1.0, dt, max_steps=25)
        outs.append((th.rise(), *th.dose()[1:]))
    for x, y in zip(*outs):
        assert np.array_equal(x, y)
    # a scaled acoustic geometry is refused: the diffusion term would carry the acoustic coefficient
    eqn.geometry.scale_cells(np.full(mesh.ncells, 1.0))
    with pytest.raises(wfx.WfxError, match="scaled"):
        wfx.PennesGLL.from_wave(eqn, K_T, RHOC)


@pytest.mark.gpu
def test_thermal_error_paths(wfx, torch):
    capi = wfx.capi
    P = 2
    mesh = wfx.create_box_hex((2, 2, 2), P, (0.01, 0.01, 0.01))
    n = mesh.ndofs
    geo = wfx.Geometry(mesh, P)
    stiff, mass = wfx.StiffnessOperator(mesh, P, geometry=geo), wfx.MassOperator(mesh, P, geometry=geo)
    bnd = wfx.BoundaryOperator(mesh, P)
    rhoc = np.full(n, RHOC)
    h = C.c_void_p()
    f = capi.f64p

    def create(stiff=stiff, mass=mass, bnd=bnd, k=K_T, rhoc=rhoc, perf=None, T_art=T_ART, hh=None, te=None):
        capi.call("wfx_thermal_create", wfx.Context.get().handle, stiff and stiff.handle, mass and mass.handle,
                  bnd and bnd.handle, k, f(rhoc), f(perf), T_art, f(hh), f(te), C.byref(h))
        capi.call("wfx_thermal_destroy", h)

    create()
    for kw, msg in ((dict(stiff=None), "NULL"), (dict(rhoc=None), "NULL"), (dict(k=0.0), "positive"),
                    (dict(k=float("nan")), "non-finite"), (dict(T_art=float("inf")), "non-finite"),
                    (dict(rhoc=np.where(np.arange(n) == 3, 0.0, RHOC)), "positive"),
                    (dict(rhoc=np.where(np.arange(n) == 3, np.nan, RHOC)), "non-finite"),
                    (dict(perf=np.where(np.arange(n) == 2, -1.0, 0.0)), "negative"),
                    (dict(hh=np.array([-1.0, 0.0])), "negative"), (dict(hh=np.array([np.inf, 0.0])), "non-finite"),
                    (dict(te=np.array([np.nan, 0.0])), "non-finite"),
                    (dict(bnd=None, hh=np.array([0.0, 10.0])), "boundary operator")):
        with pytest.raises(capi.WfxError, match=msg):
            create(**kw)
    # dtype mismatch
    geo32 = wfx.Geometry(mesh, P, np.float32)
    mass32 = wfx.MassOperator(mesh, P, np.float32, geometry=geo32)
    with pytest.raises(capi.WfxError, match="dtype"):
        create(mass=mass32)
    # operators of another mesh (other ndofs)
    mesh3 = wfx.create_box_hex((3, 2, 2), P, (0.015, 0.01, 0.01))
    mass3 = wfx.MassOperator(mesh3, P)
    with pytest.raises(capi.WfxError, match="mass operator has"):
        create(mass=mass3)
    with pytest.raises(capi.WfxError, match="boundary operator has"):
        create(bnd=wfx.BoundaryOperator(mesh3, P))
    # rank-shared dofs
    shared = wfx.StiffnessOperator.__new__(wfx.StiffnessOperator)
    shared.handle = C.c_void_p()
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    sh = np.array([0, 1], dtype=np.int32)
    capi.call("wfx_stiffness_create_partitioned", wfx.Context.get().handle, geo.handle, n, capi.i32p(dm.reshape(-1)),
              1500.0, 0, 2, capi.i32p(sh), C.byref(shared.handle))
    with pytest.raises(capi.WfxError, match="one rank"):
        create(stiff=shared)
    th = wfx.PennesGLL(mesh, P, K_T, RHOC)
    for s in (-1.0, float("nan")):
        with pytest.raises(capi.WfxError, match="heat scale"):
            th.set_heat_scale(s)
    with pytest.raises(capi.WfxError, match="non-finite"):
        th.set_heat_source(np.where(np.arange(n) == 1, np.inf, 0.0))
    for name, args in (("wfx_thermal_init", ()), ("wfx_thermal_set_heat_scale", (1.0,)),
                       ("wfx_thermal_rk4", (0.0, 1.0, 0.1, 0, None, None, None)),
                       ("wfx_thermal_get_dose", (None, None, None)), ("wfx_thermal_stable_dt", (10, None, None)),
                       ("wfx_thermal_heat_from_wave", (None, 0, 1.0, None, 1.0, RHO0, C0))):
        with pytest.raises(capi.WfxError, match="NULL"):
            capi.call(name, None, *args)
    # heat_from_wave
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    with pytest.raises(capi.WfxError, match="off"):
        th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0)
    eqn.set_field_stats(0.0, harmonics=0)
    eqn.rk4(0.0, 1.0, 1e-8, max_steps=2)
    with pytest.raises(capi.WfxError, match="nharm = 0"):
        th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0)
    eqn.set_field_stats(0.0, harmonics=2)
    with pytest.raises(capi.WfxError, match="N = 0"):
        th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0)
    eqn.rk4(0.0, 1.0, 1e-8, max_steps=2)
    th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0)
    for mbr in (-1, 1):
        with pytest.raises(capi.WfxError, match="member"):
            th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0, member=mbr)
    for a0, y, rho0, c0, msg in ((-1.0, 1.0, RHO0, C0, "negative"), (1.0, np.nan, RHO0, C0, "non-finite"),
                                 (1.0, 1.0, 0.0, C0, "positive"), (1.0, 1.0, RHO0, -C0, "positive")):
        with pytest.raises(capi.WfxError, match=msg):
            th.heat_from_wave(eqn, a0, y, rho0, c0)
    other_mesh = wfx.create_box_hex((3, 2, 2), P, (0.015, 0.01, 0.01))
    other = wfx.LinearGLLOpt(other_mesh, None, P, C0, F0, P0)
    other.set_field_stats(0.0, harmonics=1)
    other.rk4(0.0, 1.0, 1e-8, max_steps=1)
    with pytest.raises(capi.WfxError, match="dofs"):
        th.heat_from_wave(other, ALPHA0, ALPHA_Y, RHO0, C0)
    if torch.cuda.device_count() > 1:
        ctx1 = wfx.Context.get(1)
        other1 = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, ctx=ctx1)
        other1.set_field_stats(0.0, harmonics=1)
        other1.rk4(0.0, 1.0, 1e-8, max_steps=1)
        with pytest.raises(capi.WfxError, match="context"):
            th.heat_from_wave(other1, ALPHA0, ALPHA_Y, RHO0, C0)
    with pytest.raises(capi.WfxError, match="iters"):
        th.max_eigenvalue(0)
    x = torch.zeros(n, dtype=torch.float64, device="cuda")
    with pytest.raises(capi.WfxError, match="alias"):
        th.rhs(x, x)
    with pytest.raises(capi.WfxError, match="dt"):
        th.rk4(0.0, 1.0, 0.0)


@pytest.mark.gpu
def test_heat_from_wave_refuses_another_context(wfx, torch):
    """a wave on another context (a second context on the same device is another context)"""
    P = 2
    mesh = wfx.create_box_hex((2, 2, 2), P, (0.01, 0.01, 0.01))
    ctx2 = wfx.Context(0)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, ctx=ctx2)
    eqn.set_field_stats(0.0, harmonics=1)
    eqn.rk4(0.0, 1.0, 1e-8, max_steps=1)
    th = wfx.PennesGLL(mesh, P, K_T, RHOC)
    with pytest.raises(wfx.WfxError, match="context"):
        th.heat_from_wave(eqn, ALPHA0, ALPHA_Y, RHO0, C0)


@pytest.mark.gpu
def test_demo_reports_heating_and_dose(wfx, torch):
    r = subprocess.run(["python", os.path.join(ROOT, "demo", "planar3d.py"), "--nx", "8", "--nyz", "1",
                        "--stats-periods", "2", "--heat-seconds", "2", "--cool-seconds", "1", "--absorption", "50"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "peak rise" in r.stdout and "max CEM43" in r.stdout and ">= 240 min" in r.stdout, r.stdout


@pytest.mark.gpu
def test_thermal_cpp_wrapper_runs(wfx, torch, tmp_path):
    r = subprocess.run([_build_cpp(wfx, tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "thermal hpp ok" in r.stdout, r.stdout + r.stderr
