"""Source profiles (DESIGN.md section 4.5c): phased-array sources on the tag-1 facets.  With a profile the boundary
term of every model uses, per entry i,

    g_i(t) = a_i g(t - tau_i),   g(s) = g'(s) = 0 for s < 0

in place of g(t), evaluated on the device at every stage time.

CPU: the profiled CPU restatement with a = 1, tau = 0 is wo_rk4_westervelt bit for bit; a numpy statement of g_i
matches the C one; focus_delays; a duct-mode known answer that checks apodisation against physics.  GPU: every
model against the restatement, ensembles against single-field runs, identity / time-shift / superposition
properties, graph invalidation, probes / statistics / snapshot restarts, the error paths, the C++ wrappers and a
focused field against a discrete Rayleigh integral.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C0, F0, P0 = 1500.0, 0.5e6, 6e4
TOL64, TOL32 = 1e-12, 2e-5
# exaggerated loss and nonlinearity, as tests/test_models.py: both terms are visible within tens of steps
DELTA, BETA, RHO0 = 1e-2, 900.0, 1000.0
MODELS = {"linear": (0.0, 0.0, 1.0), "lossy": (DELTA, 0.0, 1.0), "westervelt": (DELTA, BETA, RHO0)}


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


def g_profile_numpy(t, amp, delay, f0, p0, c0, delta=0.0):
    """amp (g + (delta / c0^2) g')(t - delay), zero before the delay, written out independently of the C code."""
    s = t - np.asarray(delay, dtype=np.float64)
    on = s >= 0
    s = np.where(on, s, 0.0)
    w0, ramp_end = 2 * np.pi * f0, 4.0 / f0
    ramp = s < ramp_end
    W = np.where(ramp, 0.5 * (1 - np.cos(np.pi * f0 * s / 4)), 1.0)
    Wd = np.where(ramp, 0.5 * np.sin(np.pi * f0 * s / 4) * np.pi * f0 / 4, 0.0)
    A = p0 * w0 / c0
    g = A * W * np.cos(w0 * s)
    gd = A * (Wd * np.cos(w0 * s) - W * w0 * np.sin(w0 * s))
    return np.where(on, amp * (g + delta / c0 ** 2 * gd), 0.0)


def _small_mesh(wfx, P=4):
    mesh = wfx.create_box_hex((4, 3, 3), P, (0.04, 0.03, 0.03), perturb=0.15)
    return mesh, P, wfx.cfl_timestep(mesh.h_min, C0, P, F0)


def _random_profile(mesh, seed, nv=None, periods=3.0, model="linear"):
    """random amplitudes in [0.2, 1.5) and delays spanning `periods` source periods.  Independent random delays
    make a source that is rough on the scale of the mesh, and at P4 / P5 its field grows to ~1e6 Pa within the
    60 steps of these tests: for the exaggerated Westervelt model (1 - kappa p vanishes at 1.25 MPa) the
    amplitudes are scaled by 1/4, which keeps kappa p below 0.4 in the CPU restatement."""
    rng = np.random.default_rng(seed)
    shape = (mesh.ndofs,) if nv is None else (mesh.ndofs, nv)
    scale = 0.25 if model == "westervelt" else 1.0
    return scale * (0.2 + 1.3 * rng.random(shape)), periods / F0 * rng.random(shape)


# ---- CPU ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["linear", "westervelt"])
def test_restatement_identity_profile_is_bitwise_the_unprofiled_restatement(wfx, orc, mo, model):
    mesh, P, dt = _small_mesh(wfx, 3)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    args = (mesh, P, G, m, m1, m2, C0, F0, P0, *MODELS[model])
    u0, v0 = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    u1, v1 = u0.copy(), v0.copy()
    s0 = mo.rk4_westervelt(*args, 0.0, 1.0, dt, u0, v0, max_steps=40)
    s1 = mo.rk4_westervelt_profile(*args, np.ones(mesh.ndofs), np.zeros(mesh.ndofs), 0.0, 1.0, dt, u1, v1,
                                   max_steps=40)
    assert s0 == s1 and np.abs(u0).max() > 0
    assert np.array_equal(u0, u1) and np.array_equal(v0, v1)
    rng = np.random.default_rng(5)
    u, v = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    f_a = mo.f1_westervelt(*args, 7 * dt, u, v)
    f_b = mo.f1_westervelt_profile(*args, None, None, 7 * dt, u, v)
    assert np.array_equal(f_a, f_b)


@pytest.mark.parametrize("delta", [0.0, DELTA])
def test_numpy_statement_of_the_delayed_source_matches_the_restatement(wfx, orc, mo, delta):
    """f1 of the restatement with u = v = 0 and no stiffness contribution is M^-1 c0^2 g_i m1: read g_i off it on
    the tag-1 dofs and compare with the numpy statement, through the ramp, past it and before the delays."""
    mesh, P, dt = _small_mesh(wfx, 2)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    amp, delay = _random_profile(mesh, 11, periods=6.0)
    src = m1 > 0
    z = np.zeros(mesh.ndofs)
    for t in (0.0, 0.3 / F0, 2.7 / F0, 3.9 / F0, 4.0 / F0, 5.3 / F0, 9.1 / F0):
        kv = mo.f1_westervelt_profile(mesh, P, G, m, m1, m2, C0, F0, P0, delta, 0.0, 1.0, amp, delay, t, z, z)
        g = kv[src] * (m[src] + delta / C0 * m2[src]) / (C0 ** 2 * m1[src])
        want = g_profile_numpy(t, amp[src], delay[src], F0, P0, C0, delta)
        assert np.all(g[delay[src] > t] == 0.0)
        scale = P0 * 2 * np.pi * F0 / C0
        assert np.abs(g - want).max() <= 1e-12 * scale, (t, np.abs(g - want).max())
        assert np.all(kv[~src] == 0.0)


def test_focus_delays(wfx):
    rng = np.random.default_rng(2)
    pts = rng.random((200, 3)) * [0.0, 0.01, 0.01]
    focus = np.array([0.02, 0.004, 0.006])
    tau = wfx.focus_delays(pts, focus, C0)
    d = np.linalg.norm(pts - focus, axis=1)
    assert tau.shape == (200,) and np.all(tau >= 0)
    assert tau[d.argmax()] == 0.0 and tau.min() == 0.0
    # every source arrives at the focus at the same time
    arrival = tau + d / C0
    assert np.ptp(arrival) < 1e-15
    assert wfx.focus_delays(np.zeros((0, 3)), focus, C0).shape == (0,)


# ---- the duct-mode known answer -------------------------------------------------------------------------------
# A box of Lx = 2 lambda along x, Ly = lambda across and two cells thick, lateral faces rigid (untagged), source
# (tag 1) at x = 0 with a(y) = cos(pi y / Ly) and no delay, first-order absorbing end (tag 2) at x = Lx.  Only the
# first duct mode is excited: k_x = sqrt(k^2 - (pi / Ly)^2), and the absorbing end reflects it with
# R = (k_x - k) / (k_x + k) = -0.072.  Steady state:
#   |p_1(x, y)| = p0 (k / k_x) |cos(pi y / Ly)| |e^{-i k_x x} + R e^{-i k_x (2L - x)}| / |1 - R e^{-2 i k_x L}|
# Two whole periods are sampled from 24 periods on.  The ramp (4 periods) and three transits at the group velocity
# c0 k_x / k (2.3 periods each, |R|^3 = 4e-4) are not enough: the ramp's spectrum reaches down towards the mode's
# cut-off, where the group velocity vanishes, and that tail decays slowly.  P4, four cells per wavelength.
DUCT_CELLS, DUCT_N0, DUCT_PERIODS = (8, 4, 2), 24, 2
# Bound set from the CPU restatement (fp64) on this case.  max | |p_1| - exact | / max exact measured 4.9e-3 when
# sampled from 11 periods on, 8.8e-4 from 16, 4.7e-4 from 20 and 2.2e-4 from 24 (the transient, not the mesh:
# six cells per wavelength measured the same 4.9e-3 from 11 periods on).
DUCT_BOUND = 5e-4


def _duct_case(wfx):
    P, lam = 4, C0 / F0
    L, Ly = 2 * lam, lam
    nx, ny, nz = DUCT_CELLS
    mesh = wfx.create_box_hex((nx, ny, nz), P, (L, Ly, nz * Ly / ny))
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    k = int(round(1.0 / F0 / dt))
    assert abs(k * dt * F0 - 1) < 1e-12
    X = wfx.dof_coordinates(mesh)
    amp = np.cos(np.pi * X[:, 1] / Ly)
    kk = 2 * np.pi / lam
    kx = np.sqrt(kk ** 2 - (np.pi / Ly) ** 2)
    R = (kx - kk) / (kx + kk)
    x, y = X[:, 0], X[:, 1]
    exact = (P0 * kk / kx * np.abs(np.cos(np.pi * y / Ly))
             * np.abs(np.exp(-1j * kx * x) + R * np.exp(-1j * kx * (2 * L - x))) / np.abs(1 - R * np.exp(-2j * kx * L)))
    return mesh, P, dt, k, amp, exact


def _duct_error(p1, exact):
    return np.abs(np.abs(p1) - exact).max() / exact.max()


def test_duct_mode_known_answer_on_the_cpu_restatement(wfx, orc, mo):
    mesh, P, dt, k, amp, exact = _duct_case(wfx)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    u, v = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    args = (mesh, P, G, m, m1, m2, C0, F0, P0, 0.0, 0.0, 1.0, amp, None)
    kw = dict(sumfact=True, nthreads=orc.max_threads())
    _, t = mo.rk4_westervelt_profile(*args, 0.0, 1.0, dt, u, v, max_steps=DUCT_N0 * k, **kw)
    acc = np.zeros(mesh.ndofs, dtype=np.complex128)
    n = DUCT_PERIODS * k
    for _ in range(n):
        _, t = mo.rk4_westervelt_profile(*args, t, 1.0, dt, u, v, max_steps=1, **kw)
        acc += u * np.exp(-2j * np.pi * F0 * t)
    err = _duct_error(acc * 2 / n, exact)
    assert err < DUCT_BOUND, err


# ---- GPU ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _model(wfx, name, mesh, P, dtype=np.float64, **kw):
    if name == "linear":
        return wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, **kw)
    if name == "lossy":
        return wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, DELTA, dtype=dtype, **kw)
    return wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype, **kw)


NSTEPS = 60          # five periods of the small mesh's step: the random delays (up to three periods) all start


def _oracle_run(orc, mo, mesh, P, model, amp, delay, nsteps, dt):
    """the restatement stepped one step at a time"""
    G, m, m1, m2 = _inputs(orc, mesh, P)
    u, v = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    t = 0.0
    for _ in range(nsteps):
        _, t = mo.rk4_westervelt_profile(mesh, P, G, m, m1, m2, C0, F0, P0, *MODELS[model], amp, delay, t, 1.0, dt,
                                         u, v, max_steps=1, sumfact=True, nthreads=orc.max_threads())
    return u, v


def _run(eqn, nsteps, dt, t0=0.0):
    eqn.init()
    eqn.rk4(t0, 1.0, dt, max_steps=nsteps)
    return eqn.get_state()


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("P", [2, 3, 4, 5])
@pytest.mark.parametrize("model", ["linear", "lossy", "westervelt"])
def test_profiled_run_matches_restatement(wfx, orc, mo, torch, monkeypatch, model, P, graph):
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh, P, dt = _small_mesh(wfx, P)
    amp, delay = _random_profile(mesh, P, model=model)
    uo, vo = _oracle_run(orc, mo, mesh, P, model, amp, delay, NSTEPS, dt)
    assert np.isfinite(uo).all()
    eqn = _model(wfx, model, mesh, P)
    eqn.set_source_profile(amp, delay)
    u, v = _run(eqn, NSTEPS, dt)
    assert np.abs(uo).max() > 0
    assert rel_l2(u, uo) < TOL64 and rel_l2(v, vo) < TOL64, (rel_l2(u, uo), rel_l2(v, vo))


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("model", ["linear", "westervelt"])
def test_profiled_run_fp32(wfx, orc, mo, torch, monkeypatch, model, graph):
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh, P, dt = _small_mesh(wfx)
    amp, delay = _random_profile(mesh, 7, model=model)
    uo, vo = _oracle_run(orc, mo, mesh, P, model, amp, delay, NSTEPS, dt)
    eqn = _model(wfx, model, mesh, P, np.float32)
    eqn.set_source_profile(amp, delay)
    u, v = _run(eqn, NSTEPS, dt)
    assert u.dtype == np.float32
    assert rel_l2(u, uo) < TOL32 and rel_l2(v, vo) < TOL32, (rel_l2(u, uo), rel_l2(v, vo))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["linear", "lossy", "westervelt"])
def test_f1_with_profile_matches_restatement(wfx, orc, mo, torch, model):
    mesh, P, dt = _small_mesh(wfx)
    G, m, m1, m2 = _inputs(orc, mesh, P)
    amp, delay = _random_profile(mesh, 3, model=model)
    rng = np.random.default_rng(4)
    u, v = 1e3 * rng.standard_normal(mesh.ndofs), 1e9 * rng.standard_normal(mesh.ndofs)
    eqn = _model(wfx, model, mesh, P)
    eqn.set_source_profile(amp, delay)
    dev = torch.device("cuda")
    ud, vd = torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev)
    out = torch.empty_like(ud)
    for t in (0.5 / F0, 2.2 / F0, 6.0 / F0):
        eqn.f1(t, ud, vd, out)
        torch.cuda.synchronize()
        want = mo.f1_westervelt_profile(mesh, P, G, m, m1, m2, C0, F0, P0, *MODELS[model], amp, delay, t, u, v,
                                        sumfact=True, nthreads=orc.max_threads())
        assert rel_l2(out.cpu().numpy(), want) < TOL64


@pytest.mark.gpu
@pytest.mark.parametrize("nv", [1, 3, 8])
def test_ensemble_members_use_their_own_profile(wfx, torch, nv):
    P = 4
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.1)
    f0s = F0 * (1 + 0.13 * np.arange(nv))
    p0s = P0 * (1 + 0.5 * np.arange(nv))
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, f0s.max())
    amp, delay = _random_profile(mesh, 20 + nv, nv=nv)
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s, p0s)
    ens.set_source_profile(amp, delay)
    u, v = _run(ens, NSTEPS, dt)
    for mbr in range(nv):
        one = wfx.LinearGLLOpt(mesh, None, P, C0, f0s[mbr], p0s[mbr])
        one.set_source_profile(amp[:, mbr], delay[:, mbr])
        uo, vo = _run(one, NSTEPS, dt)
        assert np.abs(uo).max() > 0
        assert rel_l2(u[:, mbr], uo) < TOL64 and rel_l2(v[:, mbr], vo) < TOL64
    with pytest.raises(wfx.WfxError, match="shape"):
        ens.set_source_profile(amp[:, 0], None)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["linear", "lossy", "westervelt"])
def test_identity_profile_and_clearing(wfx, torch, model):
    """a = 1, tau = 0 is the unprofiled run up to device cos against host cos; clearing the profile restores the
    unprofiled run bit for bit (both on the graph path, which set_source_profile re-captures)."""
    mesh, P, dt = _small_mesh(wfx)
    eqn = _model(wfx, model, mesh, P)
    u_ref, v_ref = _run(eqn, NSTEPS, dt)
    eqn.set_source_profile(np.ones(mesh.ndofs), np.zeros(mesh.ndofs))
    u1, v1 = _run(eqn, NSTEPS, dt)
    assert rel_l2(u1, u_ref) < 1e-13 and rel_l2(v1, v_ref) < 1e-13, (rel_l2(u1, u_ref), rel_l2(v1, v_ref))
    eqn.set_source_profile(None, np.zeros(mesh.ndofs))        # a NULL array: a = 1
    u2, _ = _run(eqn, NSTEPS, dt)
    assert np.array_equal(u2, u1)
    eqn.set_source_profile()
    u3, v3 = _run(eqn, NSTEPS, dt)
    assert np.array_equal(u3, u_ref) and np.array_equal(v3, v_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_uniform_delay_is_a_time_shift(wfx, torch, monkeypatch, graph):
    """The equations do not depend on time: a uniform delay of k steps, run for N + k steps, is the unprofiled run
    after N steps; the first k steps leave the (linear) state at exactly zero."""
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh, P, dt = _small_mesh(wfx)
    k = 17
    eqn = _model(wfx, "linear", mesh, P)
    u_ref, v_ref = _run(eqn, NSTEPS, dt)
    eqn.set_source_profile(None, np.full(mesh.ndofs, k * dt))
    u0, v0 = _run(eqn, k, dt)
    assert not u0.any() and not v0.any()
    u, v = _run(eqn, NSTEPS + k, dt)
    assert rel_l2(u, u_ref) < TOL64 and rel_l2(v, v_ref) < TOL64, (rel_l2(u, u_ref), rel_l2(v, v_ref))


@pytest.mark.gpu
def test_superposition_of_disjoint_profiles(wfx, torch):
    mesh, P, dt = _small_mesh(wfx)
    amp, delay = _random_profile(mesh, 9)
    half = np.random.default_rng(10).random(mesh.ndofs) < 0.5
    eqn = _model(wfx, "linear", mesh, P)
    runs = []
    for a in (np.where(half, amp, 0.0), np.where(half, 0.0, amp), amp):
        eqn.set_source_profile(a, delay)
        runs.append(_run(eqn, NSTEPS, dt))
    (ua, va), (ub, vb), (u, v) = runs
    assert np.abs(ua).max() > 0 and np.abs(ub).max() > 0
    assert rel_l2(ua + ub, u) < 1e-13 and rel_l2(va + vb, v) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["linear", "westervelt"])
def test_setting_or_clearing_a_profile_drops_the_step_graph(wfx, torch, monkeypatch, model):
    """A graph captured with the unprofiled boundary kernel must not be replayed after a profile is set, nor one
    captured with the profiled kernel after it is cleared: each run equals the same run without graph replay."""
    mesh, P, dt = _small_mesh(wfx)
    amp, delay = _random_profile(mesh, 12, model=model)
    g = _model(wfx, model, mesh, P)
    monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    ng = _model(wfx, model, mesh, P)
    monkeypatch.delenv("WFX_WAVE_GRAPH")
    want_plain = _run(ng, NSTEPS, dt)
    ng.set_source_profile(amp, delay)
    want_prof = _run(ng, NSTEPS, dt)
    assert rel_l2(want_prof[0], want_plain[0]) > 1e-2
    for prof, want in ((False, want_plain), (True, want_prof), (False, want_plain), (True, want_prof)):
        if prof:
            g.set_source_profile(amp, delay)
        else:
            g.set_source_profile()
        got = _run(g, NSTEPS, dt)
        assert rel_l2(got[0], want[0]) < 1e-14 and rel_l2(got[1], want[1]) < 1e-14, prof
    # a profile changed between rk4 calls of one run: re-steering between pulses
    g.set_source_profile(amp, delay)
    g.init()
    t = g.rk4(0.0, 1.0, dt, max_steps=20)[1]
    g.set_source_profile(amp[::-1].copy(), delay)
    g.rk4(t, 1.0, dt, max_steps=20)
    ng.set_source_profile(amp, delay)
    ng.init()
    t = ng.rk4(0.0, 1.0, dt, max_steps=20)[1]
    ng.set_source_profile(amp[::-1].copy(), delay)
    ng.rk4(t, 1.0, dt, max_steps=20)
    assert rel_l2(g.get_state()[0], ng.get_state()[0]) < 1e-14


@pytest.mark.gpu
def test_profile_with_probes_stats_and_snapshot_restart(wfx, torch):
    """The profile is model configuration: it survives init and set_state, so a restart from a snapshot continues
    the profiled run bit for bit; probes and field statistics see the profiled state."""
    mesh, P, dt = _small_mesh(wfx)
    amp, delay = _random_profile(mesh, 13, model="westervelt")
    eqn = _model(wfx, "westervelt", mesh, P)
    eqn.set_source_profile(amp, delay)
    eqn.init()
    probes = np.arange(mesh.ndofs, dtype=np.int32)
    eqn.set_probes(probes, max_records=NSTEPS)
    eqn.set_field_stats(0.0, harmonics=1)
    snaps = {}
    eqn.set_snapshot(20, lambda step, t, u, v: snaps.__setitem__(step, (t, u.copy(), v.copy())))
    eqn.rk4(0.0, 1.0, dt, max_steps=NSTEPS)
    eqn.set_snapshot(0, None)
    u_end, v_end = eqn.get_state()
    tp, rec = eqn.probe_series()
    fs = eqn.field_stats()
    assert np.array_equal(rec[-1], u_end) and np.array_equal(fs.pmax, rec.max(axis=0))
    t20, u20, v20 = snaps[20]
    eqn.set_state(u20, v20)
    eqn.rk4(t20, 1.0, dt, max_steps=NSTEPS - 20)
    u, v = eqn.get_state()
    assert np.array_equal(u, u_end) and np.array_equal(v, v_end)
    _, rec2 = eqn.probe_series()
    assert np.array_equal(rec2, rec[20:])


def _single_rank_halo(wfx, ctx, ndofs):
    capi = wfx.capi
    buf = C.create_string_buffer(128)
    capi.call("wfx_comm_unique_id", buf)
    comm = C.c_void_p()
    capi.call("wfx_comm_create", ctx.handle, buf.raw, 1, 0, C.byref(comm))
    halo = C.c_void_p()
    z = np.zeros(1, dtype=np.int32)
    capi.call("wfx_halo_create", ctx.handle, comm, capi.F64, ndofs, 0, 0, None, capi.i32p(z), None, 0, None,
              capi.i32p(z), None, C.byref(halo))
    return comm, halo


@pytest.mark.gpu
def test_source_profile_error_paths(wfx, torch):
    capi = wfx.capi
    mesh, P, dt = _small_mesh(wfx)
    eqn = _model(wfx, "linear", mesh, P)
    n = mesh.ndofs
    ones, zeros = np.ones(n), np.zeros(n)
    for bad in (np.nan, np.inf, -np.inf):
        a = ones.copy()
        a[5] = bad
        with pytest.raises(capi.WfxError, match="non-finite amplitude"):
            eqn.set_source_profile(a, None)
        d = zeros.copy()
        d[5] = bad
        with pytest.raises(capi.WfxError, match="non-finite delay"):
            eqn.set_source_profile(None, d)
    d = zeros.copy()
    d[7] = -1e-12
    with pytest.raises(capi.WfxError, match="negative delay"):
        eqn.set_source_profile(ones, d)
    with pytest.raises(capi.WfxError, match="shape"):
        eqn.set_source_profile(ones[:-1], None)
    with pytest.raises(capi.WfxError, match="NULL"):
        capi.call("wfx_wave_set_source_profile", None, capi.f64p(ones), None)
    # a refused profile leaves the model as it was: unprofiled
    u_ref, _ = _run(_model(wfx, "linear", mesh, P), 10, dt)
    assert np.array_equal(_run(eqn, 10, dt)[0], u_ref)
    # a model without a boundary operator
    h = C.c_void_p()
    capi.call("wfx_wave_create", eqn.ctx.handle, eqn.stiff_op.handle, eqn.mass_op.handle, None, None, n, C0, F0, P0,
              C.byref(h))
    try:
        with pytest.raises(capi.WfxError, match="no boundary operator"):
            capi.call("wfx_wave_set_source_profile", h, capi.f64p(ones), None)
    finally:
        capi.lib.wfx_wave_destroy(h)
    # a distributed model (a halo, here over one rank)
    comm, halo = _single_rank_halo(wfx, eqn.ctx, n)
    hd = C.c_void_p()
    try:
        capi.call("wfx_wave_create", eqn.ctx.handle, eqn.stiff_op.handle, eqn.mass_op.handle, eqn.bnd_op.handle,
                  halo, n, C0, F0, P0, C.byref(hd))
        with pytest.raises(capi.WfxError, match="one rank only"):
            capi.call("wfx_wave_set_source_profile", hd, capi.f64p(ones), None)
    finally:
        if hd:
            capi.lib.wfx_wave_destroy(hd)
        capi.lib.wfx_halo_destroy(halo)
        capi.lib.wfx_comm_destroy(comm)


def _build_cpp(wfx, outdir):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_source_profile_hpp.cpp")
    exe = os.path.join(str(outdir), "test_wavefx_source_profile_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_source_profile_cpp_wrappers_compile_and_link(wfx, tmp_path):
    assert os.path.exists(_build_cpp(wfx, tmp_path))


@pytest.mark.gpu
def test_source_profile_cpp_wrappers_run(wfx, torch, tmp_path):
    r = subprocess.run([_build_cpp(wfx, tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "source profile hpp ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_duct_mode_known_answer_on_the_gpu(wfx, torch):
    mesh, P, dt, k, amp, exact = _duct_case(wfx)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    eqn.set_source_profile(amp, None)
    eqn.init()
    t = 0.0
    for _ in range(DUCT_N0 * k):
        t += dt
    eqn.set_field_stats(t + dt, harmonics=1)
    assert eqn.rk4(0.0, 1.0, dt, max_steps=(DUCT_N0 + DUCT_PERIODS) * k)[0] == (DUCT_N0 + DUCT_PERIODS) * k
    fs = eqn.field_stats()
    assert fs.samples == DUCT_PERIODS * k
    assert _duct_error(fs.harmonics[0], exact) < DUCT_BOUND


# ---- focusing: a discrete Rayleigh integral --------------------------------------------------------------------
# A box of 4 lambda per side at 8 cells per lambda, P4, source on x = 0 with delays focusing at 3 lambda depth on
# the axis through the centre of the face, the other five faces absorbing.  Steady state against the Rayleigh
# integral of the same discrete source over a rigid baffle,
#   p_1(r) = (p0 k / 2 pi) sum_i m1_i a_i e^{-i w tau_i} e^{-i k R_i} / R_i,   R_i = |r - x_i|,
# which gives |p_1| = p0 for a uniform infinite plane.  Required (set before any run): the on-axis peak within
# lambda / 4 of the Rayleigh peak and its amplitude within 10 %.  Measured on a B200: 3.397e5 Pa at 2.022 lambda
# against the Rayleigh 3.349e5 Pa at 2.000 lambda (+1.4 %).  Both lie short of the geometric focus at 3 lambda
# (the focal shift of a source of Fresnel number 4 / 3).
FOCUS_SIDE, FOCUS_CELLS, FOCUS_DEPTH = 4, 32, 3


def focus_case(wfx):
    P, lam = 4, C0 / F0
    L = FOCUS_SIDE * lam
    n = FOCUS_CELLS
    tags = ((0, 0, 1), (0, 1, 2), (1, 0, 2), (1, 1, 2), (2, 0, 2), (2, 1, 2))
    mesh = wfx.create_box_hex((n, n, n), P, (L, L, L), tags=tags)
    X = wfx.dof_coordinates(mesh)
    focus = np.array([FOCUS_DEPTH * lam, L / 2, L / 2])
    face = np.abs(X[:, 0]) < 1e-12
    delay = np.zeros(mesh.ndofs)
    delay[face] = wfx.focus_delays(X[face], focus, C0)
    axis = np.where((np.abs(X[:, 1] - L / 2) < 1e-9) & (np.abs(X[:, 2] - L / 2) < 1e-9))[0]
    axis = axis[np.argsort(X[axis, 0])]
    return mesh, P, X, delay, axis, focus


def rayleigh_on_axis(X, m1, amp, delay, xs, yz, f0=F0, c0=C0, p0=P0):
    k = 2 * np.pi * f0 / c0
    src = m1 > 0
    xi, w = X[src], m1[src] * amp[src] * np.exp(-2j * np.pi * f0 * delay[src])
    out = np.empty(len(xs), dtype=np.complex128)
    for j, x in enumerate(xs):
        R = np.linalg.norm(xi - np.array([x, yz, yz]), axis=1)
        out[j] = (w * np.exp(-1j * k * R) / R).sum()
    return p0 * k / (2 * np.pi) * out


@pytest.mark.gpu
def test_focus_against_rayleigh_integral(wfx, torch):
    mesh, P, X, delay, axis, focus = focus_case(wfx)
    lam = C0 / F0
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0)
    eqn.set_source_profile(None, delay)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    k = int(round(1.0 / F0 / dt))
    n0 = 12 * k                        # ramp (4), longest delay (~1.1), transit (~4.5) and settling, in periods
    t = 0.0
    for _ in range(n0):
        t += dt
    eqn.init()
    eqn.set_field_stats(t + dt, harmonics=1)
    eqn.rk4(0.0, 1.0, dt, max_steps=n0 + 2 * k)
    fs = eqn.field_stats()
    assert fs.samples == 2 * k
    p1 = np.abs(fs.harmonics[0, axis])
    xs = X[axis, 0]
    m1, _ = eqn.bnd_op.facet_masses()
    sel = xs > lam                     # the near field next to the source face is not the focal region
    ray = np.zeros(len(xs))
    ray[sel] = np.abs(rayleigh_on_axis(X, m1, np.ones(mesh.ndofs), delay, xs[sel], focus[1]))
    jg, jr = np.argmax(np.where(sel, p1, 0)), np.argmax(np.where(sel, ray, 0))
    print(f"focus: simulated peak {p1[jg]:.4e} Pa at x = {xs[jg] / lam:.3f} lambda, "
          f"Rayleigh {ray[jr]:.4e} Pa at x = {xs[jr] / lam:.3f} lambda")
    assert abs(xs[jg] - xs[jr]) <= lam / 4, (xs[jg] / lam, xs[jr] / lam)
    assert abs(p1[jg] / ray[jr] - 1) <= 0.10, (p1[jg], ray[jr])


@pytest.mark.gpu
def test_demo_reports_the_focal_maximum(wfx, torch):
    """The demo's focused box is the case of test_focus_against_rayleigh_integral.  At this Fresnel number
    (aperture radius^2 / (lambda depth) = 4 / 3) the on-axis maximum lies well short of the geometric focus, at
    ~2 lambda for a focus requested at 3 lambda (the focal shift; the Rayleigh integral puts it there too): the
    reported maximum is held to the Rayleigh peak, and to lie between lambda and the requested depth."""
    lam = C0 / F0
    r = subprocess.run(["python", os.path.join(ROOT, "demo", "planar3d.py"), "--length", str(FOCUS_SIDE * lam),
                        "--nx", str(FOCUS_CELLS), "--nyz", str(FOCUS_CELLS), "--focus", str(FOCUS_DEPTH * lam),
                        "--stats-periods", "2"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    print(r.stdout)
    line = r.stdout.split("on-axis maximum: |p1| = ")[1]
    p_max, x_max = float(line.split(" at x = ")[0]), float(line.split(" at x = ")[1].split(",")[0])
    mesh, P, X, delay, axis, focus = focus_case(wfx)
    m1, _ = wfx.BoundaryOperator(mesh, P).facet_masses()
    xs = X[axis, 0]
    xs = xs[xs > lam]
    ray = np.abs(rayleigh_on_axis(X, m1, np.ones(mesh.ndofs), delay, xs, focus[1]))
    assert abs(x_max - xs[ray.argmax()]) <= lam / 4, (x_max / lam, xs[ray.argmax()] / lam)
    assert abs(p_max / ray.max() - 1) <= 0.10, (p_max, ray.max())
    assert lam < x_max <= FOCUS_DEPTH * lam
