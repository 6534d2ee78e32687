"""Ensembles: nv fields on one mesh, operator and c0, stored member-interleaved (entry (dof i, member m) at
i*nv + m, DOLFINx's blocked layout with bs = nv).  The ensemble stiffness apply reads the geometric factors
and the dofmap once for all members; the ensemble wave model steps nv LinearGLLOpt models together.

CPU: the ensemble plan passes the plan verifier, the C++ wrappers compile and link.  GPU: the apply against
the reference's dense skernel per member, member independence and determinism, ensemble RK4 against the
reference time stepper and single-field runs, and the error paths.
"""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = 0.1
TOL64 = 1e-12
TOL32 = 2e-5   # as test_stiffness_fp32
NVS = (1, 2, 3, 4, 8)


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


# ---- CPU ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P,shape", [(2, (5, 4, 3)), (4, (5, 6, 9)), (7, (2, 3, 1))])
def test_ensemble_plan_verified_on_ragged_meshes(wfx, P, shape):
    """The ensemble path's plan is the streamed-cell plan in colour order with the mesh's own axes (G is read
    as stored): the verifier replays it (no two cells of a colour share a dof, FIRST / LAST exactly once)."""
    capi = wfx.capi
    mesh = wfx.create_box_hex(shape, P, (1.0, 0.7, 1.3), perturb=0.1)
    s = capi.debug_stream_plan_check(P, mesh.dofmap, mesh.ndofs + 2, None, False, (1, 1, 1), 1, relabel_axes=False)
    assert s["axis_perm"] == [0, 1, 2] and s["untouched"] == 2 and s["colours"] == (8 if min(shape) > 1 else 4)
    ren = wfx.create_box_hex(shape, P, (1.0, 0.7, 1.3), perturb=0.1, renumber=5)
    capi.debug_stream_plan_check(P, ren.dofmap, ren.ndofs, None, False, (1, 1, 1), 1, relabel_axes=False)


@pytest.mark.parametrize("grid,rank", [((2, 1, 1), 1), ((2, 2, 1), 3), ((1, 2, 2), 0)])
def test_ensemble_plan_verified_on_partition_shaped_meshes(wfx, grid, rank):
    """A rank's part of a partitioned box (owned and ghost dofs numbered DOLFINx-style) as a mesh of its own."""
    from wave_fenics_b200.partition import create_box_hex_partition
    P = 3
    mesh = create_box_hex_partition((5, 4, 3), P, (1.0, 1.0, 1.0), grid, rank, perturb=0.1)
    wfx.capi.debug_stream_plan_check(P, mesh.dofmap, mesh.ndofs, None, False, (1, 1, 1), 1, relabel_axes=False)


def _build_cpp(wfx):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_ensemble_hpp.cpp")
    exe = os.path.join(ROOT, "tests", "cpp", "test_wavefx_ensemble_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_ensemble_cpp_wrappers_compile_and_link(wfx):
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
def test_ensemble_cpp_wrappers_run(wfx, torch):
    r = subprocess.run([_build_cpp(wfx)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ensemble hpp ok" in r.stdout, r.stdout + r.stderr


def _single_cell(wfx, P):
    mesh = wfx.create_box_hex((1, 1, 1), P, (L, 0.8 * L, 1.1 * L), perturb=0.0)
    mesh.x = mesh.x + 0.05 * L * np.random.default_rng(P).uniform(-1, 1, mesh.x.shape)
    return mesh


MESHES = {
    "perturbed": lambda wfx, P: wfx.create_box_hex(4 if P < 5 else (3 if P == 5 else 2), P, (L, L, L), perturb=0.15),
    "renumbered": lambda wfx, P: wfx.create_box_hex(3 if P < 6 else 2, P, (L, L, L), perturb=0.15, renumber=17),
    "ragged": lambda wfx, P: wfx.create_box_hex((3, 2, 4) if P < 6 else (2, 1, 3), P, (L, L, L), perturb=0.15),
    "single_cell": _single_cell,
}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(MESHES))
@pytest.mark.parametrize("P", [2, 3, 4, 5, 6, 7])
def test_apply_ensemble_matches_dense_reference_kernel(wfx, orc, torch, monkeypatch, P, kind):
    """Every member against the reference's dense skernel, for nv in NVS, beta 0 / 1, with and without a
    per-dof scale; the ensemble plan runs through the verifier (WFX_VERIFY_PLAN)."""
    monkeypatch.setenv("WFX_VERIFY_PLAN", "1")
    mesh = MESHES[kind](wfx, P)
    n = mesh.ndofs
    op = wfx.StiffnessOperator(mesh, P, {"c0": 1500.0}, ensemble=True)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    rng = np.random.default_rng(P)
    X = rng.standard_normal((n, max(NVS)))
    KX = np.zeros_like(X)
    for m in range(X.shape[1]):
        km = np.zeros(n)
        orc.stiffness_apply(mesh, P, Go, np.ascontiguousarray(X[:, m]), km, dense=True)
        KX[:, m] = km
    sc = rng.uniform(0.5, 2.0, n)
    scd = dev(torch, sc)
    for nv in NVS:
        Xd = dev(torch, X[:, :nv])
        Y0 = rng.standard_normal((n, nv))
        Y = torch.full((n, nv), float("nan"), dtype=torch.float64, device="cuda")
        op.apply_ensemble(Xd, Y, beta=0)
        assert rel_l2(Y.cpu().numpy(), KX[:, :nv]) < TOL64, nv
        Y = dev(torch, Y0)
        op.apply_ensemble(Xd, Y, beta=1)
        assert rel_l2(Y.cpu().numpy() - Y0, KX[:, :nv]) < TOL64, nv
        Y = torch.full((n, nv), float("nan"), dtype=torch.float64, device="cuda")
        op.apply_ensemble(Xd, Y, beta=0, scale_ptr=scd.data_ptr())
        assert rel_l2(Y.cpu().numpy(), KX[:, :nv] * sc[:, None]) < TOL64, nv


@pytest.mark.gpu
@pytest.mark.parametrize("P", [4, 7])
def test_apply_ensemble_fp32(wfx, orc, torch, P):
    """fp32 at the two measured configurations (P7 fp32 shares the operator's own streamed-cell plan)."""
    mesh = wfx.create_box_hex(4 if P == 4 else 3, P, (L, L, L), perturb=0.15)
    op = wfx.StiffnessOperator(mesh, P, dtype=np.float32, ensemble=True)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    X = np.random.default_rng(1).standard_normal((mesh.ndofs, 4)).astype(np.float32)
    Y = torch.full(X.shape, float("nan"), dtype=torch.float32, device="cuda")
    op.apply_ensemble(dev(torch, X), Y)
    for m in range(4):
        yo = np.zeros(mesh.ndofs)
        orc.stiffness_apply(mesh, P, Go, X[:, m].astype(np.float64), yo, dense=False)
        assert rel_l2(Y[:, m].cpu().numpy(), yo) < TOL32


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["cell_colour", "cell_stream"])
def test_apply_ensemble_next_to_other_kernels(wfx, orc, torch, mode):
    """The flag adds the ensemble path to whichever kernel the operator runs; both give the same result."""
    P = 4
    mesh = wfx.create_box_hex(3, P, (L, L, L), perturb=0.15, renumber=3)
    flag = {"cell_colour": wfx.capi.STIFF_CELL_COLOUR, "cell_stream": wfx.capi.STIFF_CELL_STREAM}[mode]
    op = wfx.StiffnessOperator(mesh, P, mode=flag, ensemble=True)
    X = np.random.default_rng(5).standard_normal((mesh.ndofs, 3))
    Y = torch.full(X.shape, float("nan"), dtype=torch.float64, device="cuda")
    op.apply_ensemble(dev(torch, X), Y)
    for m in range(3):
        y = torch.zeros(mesh.ndofs, dtype=torch.float64, device="cuda")
        op.apply(dev(torch, X[:, m]), y, beta=0)
        assert rel_l2(Y[:, m].cpu().numpy(), y.cpu().numpy()) < TOL64


@pytest.mark.gpu
@pytest.mark.parametrize("P,dtype", [(4, np.float64), (7, np.float32), (3, np.float64)])
def test_members_independent_and_deterministic(wfx, torch, P, dtype):
    """Permuting the members permutes the result bit for bit, two applies give identical bits, and a zero
    member gives exactly zero."""
    mesh = wfx.create_box_hex(3, P, (L, L, L), perturb=0.15)
    op = wfx.StiffnessOperator(mesh, P, dtype=dtype, ensemble=True)
    mass = wfx.MassOperator(mesh, P, dtype=dtype, geometry=op.geometry)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    X = np.random.default_rng(2).standard_normal((mesh.ndofs, 8)).astype(dtype)
    X[:, 5] = 0
    Xd = dev(torch, X)
    Y = torch.full(X.shape, float("nan"), dtype=tdt, device="cuda")
    op.apply_ensemble(Xd, Y, scale_ptr=mass.inverse_diagonal_ptr())
    Y2 = torch.full_like(Y, float("nan"))
    op.apply_ensemble(Xd, Y2, scale_ptr=mass.inverse_diagonal_ptr())
    assert torch.equal(Y, Y2)
    assert (Y[:, 5] == 0).all() and (Y[:, 4] != 0).any()
    perm = torch.tensor([3, 7, 0, 5, 1, 6, 2, 4], device="cuda")
    Yp = torch.full_like(Y, float("nan"))
    op.apply_ensemble(Xd[:, perm].contiguous(), Yp, scale_ptr=mass.inverse_diagonal_ptr())
    assert torch.equal(Yp, Y[:, perm])
    # a member's bits do not depend on nv either
    Y1 = torch.full((mesh.ndofs, 1), float("nan"), dtype=tdt, device="cuda")
    op.apply_ensemble(Xd[:, 4:5].contiguous(), Y1, scale_ptr=mass.inverse_diagonal_ptr())
    assert torch.equal(Y1[:, 0], Y[:, 4])


def _model_inputs(wfx, orc, mesh, P):
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    return Go, m, m1, m2


F0S = (0.5e6, 0.3e6, 0.8e6)
P0S = (6e4, 1e4, 3e4)


@pytest.mark.gpu
def test_ensemble_rk4_matches_single_runs_and_reference(wfx, orc, torch):
    """Three members that differ in (f0, p0) and in their random initial states, over a run whose last step is
    shortened: each member equals the reference's own time stepper (when built) and a single-field
    LinearGLLOpt run with its parameters; the probe series hold the per-member states."""
    P, c0 = 4, 1500.0
    mesh = wfx.create_box_hex((4, 3, 3), P, (L, 0.75 * L, 0.75 * L), perturb=0.15)
    n, nv = mesh.ndofs, len(F0S)
    Go, m, m1, m2 = _model_inputs(wfx, orc, mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, max(F0S))
    tf = 12.6 * dt
    rng = np.random.default_rng(11)
    U0, V0 = 1e-3 * rng.standard_normal((n, nv)), rng.standard_normal((n, nv))
    ens = wfx.LinearGLLEnsemble(mesh, None, P, c0, F0S, P0S)
    ens.set_state(U0, V0)
    probes = np.array([0, n // 3, n - 1], dtype=np.int32)
    ens.set_probes(probes, 100)
    s, t = ens.rk4(0.0, tf, dt)
    U, V = ens.get_state()
    tt, vals = ens.probe_series()
    assert s == 13 and len(tt) == s and vals.shape == (s, len(probes), nv)
    assert np.array_equal(vals[-1], U[probes])
    for k in range(nv):
        one = wfx.LinearGLLOpt(mesh, None, P, c0, F0S[k], P0S[k])
        one.set_state(U0[:, k], V0[:, k])
        one.set_probes(probes, 100)
        s1, t1 = one.rk4(0.0, tf, dt)
        u1, v1 = one.get_state()
        assert (s1, t1) == (s, t)
        assert rel_l2(U[:, k], u1) < TOL64 and rel_l2(V[:, k], v1) < TOL64
        t1s, vals1 = one.probe_series()
        assert np.array_equal(t1s, tt)
        assert rel_l2(vals[:, :, k], vals1) < TOL64
        uo, vo = U0[:, k].copy(), V0[:, k].copy()
        orc.rk4(mesh, P, Go, m, m1, m2, c0, F0S[k], P0S[k], 0.0, tf, dt, uo, vo, sumfact=True)
        assert rel_l2(U[:, k], uo) < TOL64 and rel_l2(V[:, k], vo) < TOL64
        if orc.ref_cpu() is not None:
            ur, vr = U0[:, k].copy(), V0[:, k].copy()
            orc.reference_rk4(mesh, P, Go, m, m1, m2, c0, F0S[k], P0S[k], 0.0, tf, dt, ur, vr)
            assert rel_l2(U[:, k], ur) < TOL64 and rel_l2(V[:, k], vr) < TOL64


@pytest.mark.gpu
def test_ensemble_rk4_from_rest_and_right_hand_sides(wfx, orc, torch):
    """From rest the members differ through their sources only; f0 / f1 of the ensemble equal the single
    models' per member."""
    P, c0 = 3, 1500.0
    mesh = wfx.create_box_hex(4, P, (L, L, L), perturb=0.1)
    n, nv = mesh.ndofs, 2
    f0s, p0s = F0S[:nv], P0S[:nv]
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, max(f0s))
    ens = wfx.LinearGLLEnsemble(mesh, None, P, c0, f0s, p0s)
    ens.init()
    s, t = ens.rk4(0.0, 1.0, dt, max_steps=30)
    U, V = ens.get_state()
    rng = np.random.default_rng(4)
    u, v = dev(torch, rng.standard_normal((n, nv))), dev(torch, rng.standard_normal((n, nv)))
    r0, r1 = torch.empty_like(u), torch.empty_like(u)
    tq = 0.7 * 4 / max(f0s)
    ens.f0(tq, u, v, r0)
    ens.f1(tq, u, v, r1)
    for k in range(nv):
        one = wfx.LinearGLLOpt(mesh, None, P, c0, f0s[k], p0s[k])
        one.init()
        assert one.rk4(0.0, 1.0, dt, max_steps=30) == (s, t)
        u1, v1 = one.get_state()
        assert np.abs(u1).max() > 0
        assert rel_l2(U[:, k], u1) < TOL64 and rel_l2(V[:, k], v1) < TOL64
        q = torch.empty(n, dtype=torch.float64, device="cuda")
        one.f1(tq, u[:, k].contiguous(), v[:, k].contiguous(), q)
        assert rel_l2(r1[:, k].cpu().numpy(), q.cpu().numpy()) < TOL64
        assert torch.equal(r0[:, k], v[:, k])


@pytest.mark.gpu
def test_ensemble_rk4_fp32(wfx, torch):
    P, c0 = 4, 1500.0
    mesh = wfx.create_box_hex(3, P, (L, L, L), perturb=0.15)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, max(F0S))
    ens = wfx.LinearGLLEnsemble(mesh, None, P, c0, F0S, P0S, dtype=np.float32)
    ens.init()
    ens.rk4(0.0, 1.0, dt, max_steps=40)
    U, V = ens.get_state()
    assert U.dtype == np.float32
    for k in range(len(F0S)):
        one = wfx.LinearGLLOpt(mesh, None, P, c0, F0S[k], P0S[k], dtype=np.float32)
        one.init()
        one.rk4(0.0, 1.0, dt, max_steps=40)
        u1, v1 = one.get_state()
        assert rel_l2(U[:, k], u1.astype(np.float64)) < 1e-4 and rel_l2(V[:, k], v1.astype(np.float64)) < 1e-4


@pytest.mark.gpu
def test_ensemble_error_paths(wfx, torch):
    P = 2
    mesh = wfx.create_box_hex(3, P, (L, L, L))
    n = mesh.ndofs
    X = torch.ones((n, 2), dtype=torch.float64, device="cuda")
    Y = torch.zeros_like(X)
    plain = wfx.StiffnessOperator(mesh, P)
    with pytest.raises(wfx.WfxError, match="WFX_STIFF_ENSEMBLE"):
        plain.apply_ensemble(X, Y)
    op = wfx.StiffnessOperator(mesh, P, ensemble=True)
    for nv in (0, 9):
        Xn = torch.ones((n, nv), dtype=torch.float64, device="cuda")
        with pytest.raises(wfx.WfxError, match="nv = %d" % nv):
            op.apply_ensemble(Xn, torch.zeros_like(Xn))
    mass = wfx.MassOperator(mesh, P, geometry=op.geometry)
    with pytest.raises(wfx.WfxError, match="beta == 0"):
        op.apply_ensemble(X, Y, beta=1, scale_ptr=mass.inverse_diagonal_ptr())
    with pytest.raises(wfx.WfxError, match="shape|dtype"):
        op.apply_ensemble(X, torch.zeros((n, 3), dtype=torch.float64, device="cuda"))
    with pytest.raises(wfx.WfxError, match="alias"):
        op.apply_ensemble(X, X)
    # a partitioned operator: rank-shared dofs
    from wave_fenics_b200.partition import create_box_hex_partition
    part = create_box_hex_partition((4, 3, 3), P, (L, L, L), (2, 1, 1), 1)
    assert len(part.halo["send_indices"]) + len(part.halo["recv_indices"]) > 0
    pop = wfx.StiffnessOperator(part, P, ensemble=True)
    Xp = torch.ones((part.ndofs, 2), dtype=torch.float64, device="cuda")
    with pytest.raises(wfx.WfxError, match="rank-shared"):
        pop.apply_ensemble(Xp, torch.zeros_like(Xp))
    # the model: snapshots refused, a stiffness operator without the flag refused
    ens = wfx.LinearGLLEnsemble(mesh, None, P, 1500.0, (0.5e6, 0.2e6), (6e4, 6e4))
    with pytest.raises(wfx.WfxError, match="snapshot"):
        ens.set_snapshot(5, lambda *a: None)
    import ctypes as C
    h = C.c_void_p()
    f = np.array([0.5e6]), np.array([6e4])
    with pytest.raises(wfx.WfxError, match="WFX_STIFF_ENSEMBLE"):
        wfx.capi.call("wfx_wave_create_ensemble", ens.ctx.handle, plain.handle, mass.handle, None, 1, n, 1500.0,
                      wfx.capi.f64p(f[0]), wfx.capi.f64p(f[1]), C.byref(h))
