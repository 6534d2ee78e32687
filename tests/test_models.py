"""Lossy and Westervelt wave models (DESIGN.md section 4.5a):

    (1 - kappa p) p_tt - c0^2 lap p - delta lap p_t = kappa p_t^2,   kappa = 2 beta / (rho0 c0^2)

CPU: the CPU restatement (model_oracle) reduces to oracle/wave_oracle.c's wo_rk4 bit for bit at delta = beta = 0,
equals a textbook numpy RK4 of the lumped system, and its analytic g' agrees with central differences of g; the
C++ wrappers compile and link.  GPU: f1 and RK4 trajectories against the restatement, delta = beta = 0 against
LinearGLLOpt bit for bit, two known answers independent of any oracle (a uniform nonlinear state, a damped
lowest mode), probes and snapshot restarts, the error paths and the C++ wrappers.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C0, F0, P0 = 1500.0, 0.5e6, 6e4
TOL64 = 1e-12
TOL32 = 2e-5   # as test_stiffness_fp32
# exaggerated parameters: the delta term is visible within tens of steps, kappa p ~ 0.05 at |p| ~ P0
DELTA, BETA, RHO0 = 1e-2, 900.0, 1000.0
MODELS = {"lossy": (DELTA, 0.0, 1.0), "westervelt": (DELTA, BETA, RHO0)}


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


def _inputs(orc, mesh, P):
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    return G, m, m1, m2


def _random_state(n, seed, scale=P0):
    rng = np.random.default_rng(seed)
    return scale * rng.standard_normal(n), scale * 2 * np.pi * F0 * rng.standard_normal(n)


# ---- CPU ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [2, 3, 4])
@pytest.mark.parametrize("start", ["rest", "random"])
def test_oracle_linear_limit_is_wo_rk4_bitwise(wfx, orc, mo, P, start):
    """delta = beta = 0: wo_rk4_westervelt is wo_rk4 bit for bit (through the Hann ramp, last step shortened)."""
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    if start == "rest":
        t0, u, v = 0.0, np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    else:
        t0, (u, v) = 3e-6, _random_state(mesh.ndofs, P)
    tf = 4.0 / F0 + 2.5 * dt
    uo, vo, uw, vw = u.copy(), v.copy(), u.copy(), v.copy()
    so, to = orc.rk4(mesh, P, G, m, m1, m2, C0, F0, P0, t0, tf, dt, uo, vo, sumfact=True)
    sw, tw = mo.rk4_westervelt(mesh, P, G, m, m1, m2, C0, F0, P0, 0.0, 0.0, 1.0, t0, tf, dt, uw, vw, sumfact=True)
    assert (sw, tw) == (so, to) and so > 3
    assert np.abs(uo).max() > 0
    assert np.array_equal(uw, uo) and np.array_equal(vw, vo)


def test_oracle_matches_textbook_numpy_rk4(wfx, orc, mo):
    """The restatement's Westervelt RK4 against a textbook RK4 of the lumped system written with a dense
    stiffness matrix assembled column by column through oracle applies (2^3 cells, P2, both boundary tags)."""
    P = 2
    mesh = wfx.create_box_hex(2, P, (0.02, 0.02, 0.02), perturb=0.1)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    n = mesh.ndofs
    A = np.zeros((n, n))
    for j in range(n):
        e, col = np.zeros(n), np.zeros(n)
        e[j] = 1.0
        orc.stiffness_apply(mesh, P, G, e, col, dense=True)
        A[:, j] = col                                   # A = -1500^2 K
    delta, beta, rho0 = MODELS["westervelt"]
    kappa, s = 2 * beta / (rho0 * C0 ** 2), delta / 1500.0 ** 2

    def acc(t, p, pd):
        g, gd = mo.source(t, F0, P0, C0)
        num = A @ p + s * (A @ pd) + kappa * m * pd ** 2 + (C0 ** 2 * g + delta * gd) * m1 - C0 * m2 * pd
        return num / (m * (1.0 - kappa * p) + delta / C0 * m2)

    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    t0, nsteps = 1.0e-6, 8
    p, pd = _random_state(n, 5, scale=0.3 * P0)
    uo, vo = p.copy(), pd.copy()
    steps, _ = mo.rk4_westervelt(mesh, P, G, m, m1, m2, C0, F0, P0, delta, beta, rho0, t0, 1.0, dt, uo, vo,
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


@pytest.mark.parametrize("t", [1.3e-6, 4.0 / F0, 2.1e-5])
def test_source_rate_is_the_derivative_of_the_source(mo, t):
    """g' (analytic) against central differences of g inside the ramp, at its end and after it.  At the end
    of the ramp g' is continuous and g'' jumps: the difference quotient is then first-order accurate."""
    h = 3e-12
    g, gd = mo.source(t, F0, P0, C0)
    gp, _ = mo.source(t + h, F0, P0, C0)
    gm, _ = mo.source(t - h, F0, P0, C0)
    w0 = 2 * np.pi * F0
    scale = P0 * w0 / C0 * w0                           # |g'| <= ~ A w0
    assert abs((gp - gm) / (2 * h) - gd) < 1e-6 * scale
    assert abs(g - mo.source(t, F0, P0, C0)[0]) == 0


def _build_cpp(wfx):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_models_hpp.cpp")
    exe = os.path.join(ROOT, "tests", "cpp", "test_wavefx_models_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_models_cpp_wrappers_compile_and_link(wfx):
    assert os.path.exists(_build_cpp(wfx))


# ---- GPU ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("P,renumber", [(2, None), (3, 11), (4, None), (5, 7)])
def test_f1_matches_oracle(wfx, orc, mo, torch, P, renumber, dtype):
    """f1 of both models on perturbed (and renumbered) meshes, random u, v, t inside / at the end of / after
    the ramp, against the restatement's f1 with the dense (reference) stiffness kernel."""
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.15, renumber=renumber)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    u, v = _random_state(mesh.ndofs, P)
    u, v = u.astype(dtype), v.astype(dtype)
    ud, vd = dev(torch, u), dev(torch, v)
    res = torch.full_like(ud, float("nan"))
    for name, (delta, beta, rho0) in MODELS.items():
        if beta:
            eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, delta, beta, rho0, dtype=dtype)
        else:
            eqn = wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, delta, dtype=dtype)
        for t in (1.3e-6, 4.0 / F0, 2.1e-5):
            want = mo.f1_westervelt(mesh, P, G, m, m1, m2, C0, F0, P0, delta, beta, rho0, t,
                                    u.astype(np.float64), v.astype(np.float64))
            eqn.f1(t, ud, vd, res)
            err = rel_l2(res.cpu().numpy(), want)
            assert err < (TOL64 if dtype == np.float64 else TOL32), (name, t, err)
        with pytest.raises(RuntimeError):
            eqn.f1(0.0, ud, vd, vd)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("model", ["lossy", "westervelt"])
@pytest.mark.parametrize("start,steps", [("rest", 60), ("random", 6)])
def test_rk4_matches_oracle(wfx, orc, mo, torch, monkeypatch, graph, model, start, steps):
    """RK4 trajectories with a shortened last step, from rest (through the ramp) and from a random state, with
    CUDA-graph replay on and off."""
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    P = 4
    mesh = wfx.create_box_hex((4, 3, 3), P, (0.04, 0.03, 0.03), perturb=0.15)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    delta, beta, rho0 = MODELS[model]
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    if start == "rest":
        t0, u, v = 0.0, np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    else:
        t0, (u, v) = 5e-6, _random_state(mesh.ndofs, 3)
    tf = t0 + (steps - 0.5) * dt
    uo, vo = u.copy(), v.copy()
    so, to = mo.rk4_westervelt(mesh, P, G, m, m1, m2, C0, F0, P0, delta, beta, rho0, t0, tf, dt, uo, vo,
                               sumfact=True, nthreads=orc.max_threads())
    eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, delta, beta, rho0)
    eqn.set_state(u, v)
    s, t = eqn.rk4(t0, tf, dt)
    ug, vg = eqn.get_state()
    assert (s, t) == (so, to) and s == steps
    assert np.abs(uo).max() > 0
    assert rel_l2(ug, uo) < TOL64 and rel_l2(vg, vo) < TOL64


@pytest.mark.gpu
def test_zero_delta_beta_is_the_linear_model_bitwise(wfx, torch):
    """wfx_wave_create_westervelt(..., 0, 0, 1) and wfx_wave_create: identical states over 50 steps through
    the ramp, source and absorbing tags present."""
    P = 4
    mesh = wfx.create_box_hex((6, 3, 3), P, (0.075, 0.0375, 0.0375), perturb=0.1)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    assert 50 * dt > 4.0 / F0
    lin = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    wv = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, 0.0, 0.0, 1.0)
    states = []
    for eqn in (lin, wv):
        eqn.init()
        assert eqn.rk4(0.0, 1.0, dt, max_steps=50)[0] == 50
        states.append(eqn.get_state())
    (ul, vl), (uw, vw) = states
    assert np.abs(ul).max() > 0
    assert np.array_equal(uw, ul) and np.array_equal(vw, vl)


@pytest.mark.gpu
def test_uniform_nonlinear_state_known_answer(wfx, torch):
    """Box without boundary tags, spatially uniform state: K 1 = 0, so every dof follows
    (1 - kappa p) p'' = kappa p'^2, whose first integral (1 - kappa p) p' = C gives p - kappa p^2 / 2 = C t + D.
    kappa is exaggerated (kappa p ~ 0.1-0.14 over the run)."""
    P, U0, V0 = 2, 1e4, 2e8
    kappa = 1e-5
    beta = kappa * RHO0 * C0 ** 2 / 2
    mesh = wfx.create_box_hex((4, 2, 2), P, (0.04, 0.02, 0.02), tags=())
    eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, 1e-3, beta, RHO0)
    n, dt, nsteps = mesh.ndofs, 1e-6, 20
    eqn.set_state(np.full(n, U0), np.full(n, V0))
    assert eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)[0] == nsteps
    u, v = eqn.get_state()
    assert np.ptp(u) <= 1e-13 * U0 and np.ptp(v) <= 1e-13 * V0    # stays uniform
    T = nsteps * dt
    Cc, D = (1 - kappa * U0) * V0, U0 - kappa * U0 ** 2 / 2
    p_exact = (1 - np.sqrt(1 - 2 * kappa * (Cc * T + D))) / kappa
    v_exact = Cc / (1 - kappa * p_exact)
    assert 0.09 < kappa * U0 and kappa * p_exact < 0.2

    def rk4(h, k):
        f = lambda p, q: kappa * q * q / (1 - kappa * p)  # noqa: E731
        p, q = U0, V0
        for _ in range(k):
            k1p, k1v = q, f(p, q)
            k2p, k2v = q + h / 2 * k1v, f(p + h / 2 * k1p, q + h / 2 * k1v)
            k3p, k3v = q + h / 2 * k2v, f(p + h / 2 * k2p, q + h / 2 * k2v)
            k4p, k4v = q + h * k3v, f(p + h * k3p, q + h * k3v)
            p, q = p + h / 6 * (k1p + 2 * k2p + 2 * k3p + k4p), q + h / 6 * (k1v + 2 * k2v + 2 * k3v + k4v)
        return p, q

    p1, q1 = rk4(dt, nsteps)
    assert abs(u[0] - p1) < 1e-10 * abs(p1) and abs(v[0] - q1) < 1e-10 * abs(q1)
    # against the closed form: the GPU is off by RK4's truncation error, which is fourth order in dt
    p2, q2 = rk4(dt / 2, 2 * nsteps)
    e1, e2 = abs(p1 - p_exact), abs(p2 - p_exact)
    assert 8 < e1 / e2 < 24
    assert abs(u[0] - p_exact) < 1.1 * e1 + 1e-13 * p_exact
    assert abs(v[0] - v_exact) < 1.1 * abs(q1 - v_exact) + 1e-13 * v_exact


@pytest.mark.gpu
def test_lowest_mode_decays_like_a_damped_oscillator(wfx, torch):
    """Unperturbed box, no tags, v = 0, u the interpolant of cos(pi x / Lx).  Projected on u0 (M inner product)
    the amplitude a(t) follows a'' + delta lam a' + c0^2 lam a = 0, lam = u0^T K u0 / u0^T M u0 (GPU operators):
    a = e^(-g t) (cos(w t) + g / w sin(w t)), g = delta lam / 2, w = sqrt(c0^2 lam - g^2).  Its envelope
    a^2 + ((a' + g a) / w)^2 = (1 + g^2 / w^2) e^(-2 g t) gives the measured decay exponent.

    Why 1e-4 relative holds: components of u0 outside the lowest discrete mode are O(1e-5) and enter the
    projection squared (~1e-10); RK4's error on the exponent at |mu| dt ~ 0.03 is O((|mu| dt)^4) ~ 1e-6 of it;
    fp64 rounding is ~1e-13.  A wrong delta term (missing or doubled, wrong scaling) moves g by O(1)."""
    P, Lx = 4, 0.1
    mesh = wfx.create_box_hex((4, 1, 1), P, (Lx, 0.025, 0.025), tags=())
    dt, nsteps = wfx.cfl_timestep(mesh.h_min, C0, P, F0), 1500
    delta = 0.72
    eqn = wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, delta)
    x = wfx.dof_coordinates(mesh)[:, 0]
    u0 = np.cos(np.pi * x / Lx)
    mdiag = eqn.mass_op.diagonal()
    y = torch.zeros(mesh.ndofs, dtype=torch.float64, device="cuda")
    eqn.stiff_op.apply(dev(torch, u0), y, beta=0)       # y = -1500^2 K u0
    lam = -(u0 @ y.cpu().numpy()) / 1500.0 ** 2 / (u0 @ (mdiag * u0))
    assert abs(lam / (np.pi / Lx) ** 2 - 1) < 1e-6
    g = delta * lam / 2
    w = np.sqrt(C0 ** 2 * lam - g ** 2)
    eqn.set_state(u0, np.zeros(mesh.ndofs))
    assert eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)[0] == nsteps
    u, v = eqn.get_state()
    T = nsteps * dt
    nrm = u0 @ (mdiag * u0)
    a, ad = (u @ (mdiag * u0)) / nrm, (v @ (mdiag * u0)) / nrm
    env = lambda a, ad: a * a + ((ad + g * a) / w) ** 2  # noqa: E731
    g_meas = -np.log(env(a, ad) / env(1.0, 0.0)) / (2 * T)
    assert np.exp(-g * T) < 0.8                         # a visible loss of amplitude
    assert delta * 9e5 * dt < 2.0                       # delta lam_max dt inside RK4's real stability interval
    assert abs(g_meas / g - 1) < 1e-4, (g_meas, g)
    # and the phase: a(T) itself
    a_exact = np.exp(-g * T) * (np.cos(w * T) + g / w * np.sin(w * T))
    assert abs(a - a_exact) < 1e-4 * np.exp(-g * T)


@pytest.mark.gpu
def test_probes_and_snapshot_restart_bitwise(wfx, torch):
    """Probe series of a Westervelt run, and a snapshot fed back through set_state of the SAME model resumes
    the run bit for bit: the stiffness input w is rebuilt from the new state (a stale w would not be)."""
    P = 4
    mesh = wfx.create_box_hex((6, 3, 3), P, (0.075, 0.0375, 0.0375), perturb=0.1)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    nsteps, every = 24, 8
    probes = np.array([0, 17, mesh.ndofs // 2, mesh.ndofs - 1], dtype=np.int32)
    eqn = wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, *MODELS["westervelt"])
    eqn.init()
    eqn.set_probes(probes, max_records=nsteps + 5)
    snaps = {}
    eqn.set_snapshot(every, lambda step, tt, u, v: snaps.__setitem__(step, (tt, u.copy(), v.copy())))
    s, t_end = eqn.rk4(0.0, 1.0, dt, max_steps=10)
    s2, t_end = eqn.rk4(t_end, 1.0, dt, max_steps=nsteps - 10)
    assert s + s2 == nsteps and sorted(snaps) == [8, 16, 24]
    u_end, v_end = eqn.get_state()
    tt, vals = eqn.probe_series()
    assert vals.shape == (nsteps, len(probes)) and tt[-1] == t_end
    assert np.array_equal(vals[-1], u_end[probes]) and np.array_equal(snaps[24][1], u_end)
    assert np.abs(u_end).max() > 0
    eqn.set_snapshot(0, None)
    eqn.set_state(snaps[16][1], snaps[16][2])
    eqn.rk4(snaps[16][0], 1.0, dt, max_steps=nsteps - 16)
    u2, v2 = eqn.get_state()
    assert np.array_equal(u2, u_end) and np.array_equal(v2, v_end)
    # writing the state through the device pointers works the same way
    up, vp = C.c_void_p(), C.c_void_p()
    wfx.capi.call("wfx_wave_state_ptrs", eqn.handle, C.byref(up), C.byref(vp))
    for ptr, a in ((up, snaps[16][1]), (vp, snaps[16][2])):
        a = np.ascontiguousarray(a)
        wfx.capi.call("wfx_memcpy_h2d", eqn.ctx.handle, ptr, C.c_void_p(a.ctypes.data), a.nbytes)
    eqn.rk4(snaps[16][0], 1.0, dt, max_steps=nsteps - 16)
    u3, v3 = eqn.get_state()
    assert np.array_equal(u3, u_end) and np.array_equal(v3, v_end)


@pytest.mark.gpu
def test_create_westervelt_error_paths(wfx, torch):
    capi = wfx.capi
    P = 2
    mesh = wfx.create_box_hex(2, P, (0.02, 0.02, 0.02))
    ctx = wfx.Context.get()
    geo = wfx.Geometry(mesh, P)
    stiff = wfx.StiffnessOperator(mesh, P, geometry=geo)
    mass = wfx.MassOperator(mesh, P, geometry=geo)
    bnd = wfx.BoundaryOperator(mesh, P)
    nan, inf = float("nan"), float("inf")

    def create(c0=C0, f0=F0, p0=P0, delta=DELTA, beta=BETA, rho0=RHO0, stiff_h=stiff.handle, mass_h=mass.handle,
               bnd_h=bnd.handle):
        h = C.c_void_p()
        capi.call("wfx_wave_create_westervelt", ctx.handle, stiff_h, mass_h, bnd_h, mesh.size_local, c0, f0, p0,
                  delta, beta, rho0, C.byref(h))
        capi.lib.wfx_wave_destroy(h)

    create()
    create(beta=0.0, rho0=0.0)                          # rho0 is not used by the lossy model
    bad = [dict(delta=-1e-6), dict(beta=-1.0), dict(rho0=0.0), dict(rho0=-1.0), dict(f0=0.0), dict(f0=-1.0),
           dict(delta=nan), dict(beta=inf), dict(c0=nan), dict(p0=inf), dict(rho0=nan, beta=0.0), dict(c0=0.0)]
    for kw in bad:
        with pytest.raises(capi.WfxError):
            create(**kw)
    # scalar types must agree
    geo32 = wfx.Geometry(mesh, P, dtype=np.float32)
    mass32 = wfx.MassOperator(mesh, P, dtype=np.float32, geometry=geo32)
    with pytest.raises(capi.WfxError, match="dtype"):
        create(mass_h=mass32.handle)
    # one rank only: an operator with rank-shared dofs is refused
    shared = np.array([0, 1], dtype=np.int32)
    h = C.c_void_p()
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    capi.call("wfx_stiffness_create_partitioned", ctx.handle, geo.handle, mesh.ndofs, capi.i32p(dm.reshape(-1)),
              C0, capi.STIFF_AUTO, len(shared), capi.i32p(shared), C.byref(h))
    try:
        with pytest.raises(capi.WfxError, match="rank-shared"):
            create(stiff_h=h)
    finally:
        capi.lib.wfx_stiffness_destroy(h)


@pytest.mark.gpu
def test_models_cpp_wrappers_run(wfx, torch):
    r = subprocess.run([_build_cpp(wfx)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "models hpp ok" in r.stdout, r.stdout + r.stderr
