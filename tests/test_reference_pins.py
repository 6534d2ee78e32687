"""The oracle pinned to REFERENCE CODE where the reference compiles.  Cut out of the headers of the reference sources
(WFX_REFERENCE at build time) and compiled into oracle/_ref/libwfref_cpu.so (oracle/build_ref.py) against the small
container stand-ins of oracle/ref_cpu_shim.cpp: the cell kernels `skernel` / `mkernel`, the call loops
StiffnessOperator::operator() / MassOperatorCPU::operator() (common/operators.hpp), kernels::copy / axpy and
LinearGLLOpt::init / f0 / f1 / rk4 (common/LinearGLL.hpp).  The oracle's restatements must reproduce them BIT
FOR BIT (same flags: -O2 -ffp-contract=off) -- operators, right-hand side and whole RK4 trajectories.  What
stays restated (third-party arithmetic, absent here): Basix tables, DOLFINx geometry, the FFCx facet kernel.
Without the reference sources the library is not built and the tests that call it skip; the reference outputs
stored in tests/golden/reference_*.npz are compared in every checkout (test_oracle_reproduces_the_reference_golden_vectors,
test_cuda_path_matches_the_reference_golden_vectors)."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import refmesh

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_reference_golden",
                                               os.path.join(HERE, "golden", "make_reference_golden.py"))
mrg = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mrg)

CASES = [(2, (3, 2, 2), 0.15), (3, (2, 2, 3), 0.15), (4, (2, 2, 2), 0.15), (4, (3, 1, 2), 0.0), (5, (1, 2, 1), 0.2)]


@pytest.fixture(scope="module")
def ref(orc):
    L = orc.ref_cpu()
    if L is None:
        pytest.skip("oracle/_ref/libwfref_cpu.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    return L


@pytest.mark.parametrize("P,shape,perturb", CASES)
def test_oracle_stiffness_is_the_reference_skernel(orc, ref, P, shape, perturb):
    mesh = refmesh.box(shape, P, (0.1, 0.07, 0.13), perturb=perturb)
    G, _ = orc.precompute_geometric_data(mesh, P)
    rng = np.random.default_rng(P)
    x, y0 = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    yo, yr = y0.copy(), y0.copy()
    orc.stiffness_apply(mesh, P, G, x, yo, dense=True)       # the oracle's restatement
    orc.reference_stiffness_apply(mesh, P, G, x, yr)         # the reference's own skernel
    assert np.abs(yr - y0).max() > 0
    assert np.array_equal(yo, yr)
    # the sum-factorised form of the oracle (what the large GPU comparisons use) agrees to rounding
    ys = y0.copy()
    orc.stiffness_apply(mesh, P, G, x, ys, dense=False)
    assert np.linalg.norm(ys - yr) <= 1e-13 * np.linalg.norm(yr - y0)


@pytest.mark.parametrize("P,shape,perturb", CASES)
def test_oracle_mass_is_the_reference_mkernel(orc, ref, P, shape, perturb):
    mesh = refmesh.box(shape, P, (0.1, 0.07, 0.13), perturb=perturb)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    rng = np.random.default_rng(10 + P)
    x, y0 = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    yo, yr = y0.copy(), y0.copy()
    orc.mass_apply(mesh, P, detJ, x, yo)
    orc.reference_mass_apply(mesh, P, detJ, x, yr)
    assert np.array_equal(yo, yr)


def test_reference_skernel_ignores_params_and_accumulates(orc, ref):
    """Quirks the restatement keeps (SURVEY App. B): c0 = 1500 hard-coded, A is accumulated into."""
    P, nd = 2, 27
    dphi = np.ascontiguousarray(orc.tabulate_dphi(P))
    rng = np.random.default_rng(0)
    w, G = rng.standard_normal(nd), rng.standard_normal((nd, 3, 3))
    A = np.ones(nd)
    ref.wfref_skernel(orc._f(A), orc._f(w), orc._f(G.reshape(-1)), orc._f(dphi.reshape(-1)), nd, nd)
    B = np.zeros(nd)
    ref.wfref_skernel(orc._f(B), orc._f(w), orc._f(G.reshape(-1)), orc._f(dphi.reshape(-1)), nd, nd)
    assert np.allclose(A - 1.0, B, rtol=0, atol=1e-9 * np.abs(B).max())
    # -c0^2 with c0 = 1500: against the formula evaluated in numpy
    wq = np.einsum("aqi,i->qa", dphi, w)
    f = -1500.0 ** 2 * np.einsum("qab,qb->qa", G, wq)
    want = np.einsum("qa,aqi->i", f, dphi)
    assert np.linalg.norm(B - want) <= 1e-13 * np.linalg.norm(want)


def _wave_setup(wfx, orc, P, shape, perturb):
    Lx = 0.1
    mesh = wfx.create_box_hex(shape, P, (Lx * shape[0] / 8, Lx * shape[1] / 8, Lx * shape[2] / 8), perturb=perturb)
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.reference_mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)      # m = M 1 (LinearGLL.hpp:102-110)
    mo = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), mo)
    assert np.array_equal(m, mo)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    return mesh, G, m, m1, m2


@pytest.mark.parametrize("P,shape,perturb", [(2, (4, 3, 2), 0.15), (4, (2, 2, 2), 0.15), (3, (3, 2, 2), 0.0)])
def test_oracle_f1_is_the_reference_f1(wfx, orc, ref, P, shape, perturb):
    c0, f0, p0 = 1500.0, 0.5e6, 6e4
    mesh, G, m, m1, m2 = _wave_setup(wfx, orc, P, shape, perturb)
    rng = np.random.default_rng(3)
    u, v = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    for t in (0.0, 0.3e-6, 7.9e-6, 2.0e-5):              # inside, at the end of and after the Hann ramp
        got = orc.reference_f1(mesh, P, G, m, m1, m2, c0, f0, p0, t, u, v)
        # one Euler-free way to reach the oracle's f1: a single RK4 stage is not exposed, so compose it from
        # the oracle's operator (bit-identical to the reference's, above) and the formulas of :155-191
        w0, T, alpha = 2.0 * np.pi * f0, 1.0 / f0, 4.0
        window = 0.5 * (1.0 - np.cos(f0 * np.pi * t / alpha)) if t < T * alpha else 1.0
        g = window * p0 * w0 / c0 * np.cos(w0 * t)
        b = np.zeros(mesh.ndofs)
        orc.stiffness_apply(mesh, P, G, u, b, dense=True)
        want = (b + (c0 * c0 * g * m1 - c0 * v * m2)) / m
        assert np.linalg.norm(got - want) <= 1e-15 * np.linalg.norm(want)


@pytest.mark.parametrize("P,shape,perturb,nsteps,frac", [(2, (4, 3, 2), 0.15, 12, 0.0), (4, (2, 2, 2), 0.15, 6, 0.0),
                                                         (3, (3, 2, 2), 0.0, 9, 0.37), (4, (3, 2, 1), 0.1, 60, 0.5)])
def test_oracle_rk4_is_the_reference_rk4(wfx, orc, ref, capfd, P, shape, perturb, nsteps, frac):
    """Whole trajectories: the reference's rk4 loop (tableau, stage algebra, axpy on owned entries, dt clipped
    at the final time, final copies), its f0 / f1 and its stiffness operator, against the oracle's restatement
    -- bit for bit, from rest through the source ramp and from a random state."""
    c0, f0, p0 = 1500.0, 0.5e6, 6e4
    mesh, G, m, m1, m2 = _wave_setup(wfx, orc, P, shape, perturb)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, f0)
    tf = (nsteps + frac) * dt                            # frac > 0: a last, shorter step (:241)
    rng = np.random.default_rng(5)
    for u0, v0 in ((np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)),
                   (rng.standard_normal(mesh.ndofs), 1e3 * rng.standard_normal(mesh.ndofs))):
        uo, vo = u0.copy(), v0.copy()
        steps, t_end = orc.rk4(mesh, P, G, m, m1, m2, c0, f0, p0, 0.0, tf, dt, uo, vo, sumfact=False)
        ur, vr = u0.copy(), v0.copy()
        orc.reference_rk4(mesh, P, G, m, m1, m2, c0, f0, p0, 0.0, tf, dt, ur, vr)
        assert steps >= nsteps + (1 if frac else 0)  # (+1 when the accumulated t rounds below tf)
        assert np.abs(ur).max() > 0
        assert np.array_equal(uo, ur) and np.array_equal(vo, vr)
    capfd.readouterr()                                   # (the reference prints its progress every 50 steps)


# ---- golden vectors generated by the reference's own code (tests/golden/reference_*.npz) --------------------
def _golden(name):
    return dict(np.load(os.path.join(HERE, "golden", name + ".npz")))


@pytest.mark.parametrize("name", list(mrg.CASES))
def test_reference_code_regenerates_its_golden_vectors(wfx, orc, ref, capfd, name):
    want, got = _golden(name), mrg.compute_reference(wfx, orc, name)
    capfd.readouterr()
    assert sorted(got) == sorted(want)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), want[k]), k


@pytest.mark.parametrize("name", list(mrg.CASES))
def test_oracle_reproduces_the_reference_golden_vectors(wfx, orc, name):
    """Runs wherever the fixtures are, with or without the reference library: bit for bit."""
    want, got = _golden(name), mrg.compute_oracle(wfx, orc, name)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), want[k]), k
    assert np.abs(want["rk4_from_rest_u"]).max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(mrg.CASES))
def test_cuda_path_matches_the_reference_golden_vectors(wfx, orc, name):
    """The CUDA path through the C ABI against the stored outputs of the reference's own code (1e-12)."""
    import torch
    want = _golden(name)
    P, mesh, G, detJ, m1, m2, x, u0, v0, dt, tf = mrg.setup(wfx, orc, name)
    rel = lambda a, b: np.linalg.norm(np.asarray(a) - b) / np.linalg.norm(b)
    geo = wfx.Geometry(mesh, P)
    for mode in (wfx.capi.STIFF_AUTO, wfx.capi.STIFF_CELL_STREAM):
        op = wfx.StiffnessOperator(mesh, P, geometry=geo, mode=mode)
        y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
        op.apply(torch.from_numpy(x).cuda(), y, beta=0)
        assert rel(y.cpu().numpy(), want["stiffness_of_x"]) < 1e-12
    assert np.array_equal(wfx.MassOperator(mesh, P, geometry=geo).diagonal(), want["lumped_mass"])
    for key, (ua, va) in (("rest", (np.zeros(mesh.ndofs), np.zeros(mesh.ndofs))), ("state", (u0, v0))):
        eqn = wfx.LinearGLLOpt(mesh, None, P, mrg.C0, mrg.F0, mrg.P0)
        eqn.init()
        eqn.set_state(ua, va)
        eqn.rk4(0.0, float(want["rk4_tf"]), float(want["rk4_dt"]))
        u, v = eqn.get_state()
        assert rel(u, want[f"rk4_from_{key}_u"]) < 1e-12 and rel(v, want[f"rk4_from_{key}_v"]) < 1e-12


# ---- the reference's partition arithmetic (demo/gpu_cg/mesh.hpp:37-62) ------------------------------------
def test_rank_grid_is_the_reference_decompose3d(wfx, orc):
    import ctypes as C
    L = orc.ref_mesh()
    if L is None:
        pytest.skip("oracle/_ref/libwfref_mesh.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    from wave_fenics_b200 import partition
    for x in range(0, 10):                                # 1 .. 512 ranks (powers of two: all the reference handles)
        out = (C.c_int * 3)()
        L.wfref_decompose3d(x, out)
        grid = partition.rank_grid(2 ** x)
        assert tuple(out) == tuple(grid)
        idx = (C.c_longlong * (3 * 2 ** x))()
        L.wfref_cartesian_indices((C.c_int * 3)(*grid), idx)
        want = np.array(list(idx)).reshape(-1, 3)
        got = np.array([partition.rank_coords(grid, r) for r in range(2 ** x)])
        assert np.array_equal(got, want)


@pytest.mark.parametrize("P", [1, 2, 4, 7])
def test_reorder_dofmap_is_the_reference_loop(wfx, orc, P):
    """reorder_dofmap (common/permute.hpp:10-28) with the tensor-product permutation supplied (Basix's part):
    the oracle's and the product's host function equal the reference's own loop."""
    L = orc.ref_mesh()
    if L is None:
        pytest.skip("oracle/_ref/libwfref_mesh.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    nd = (P + 1) ** 3
    rng = np.random.default_rng(P)
    dm = rng.integers(0, 10 ** 6, size=(11, nd)).astype(np.int32)
    pm = np.ascontiguousarray(orc.perm(P), dtype=np.int32)
    out = np.empty_like(dm)
    L.wfref_reorder_dofmap(P, nd, dm.shape[0], orc._i(pm), orc._i(dm.reshape(-1)), orc._i(out.reshape(-1)))
    assert np.array_equal(orc.reorder_dofmap(dm, P), out)
    assert np.array_equal(wfx.capi.reorder_dofmap(dm, P), out)


def test_time_step_is_the_reference_demos(wfx, orc):
    """cfl_timestep and the final time of the planar-wave runs against the demo's own statements
    (demo/cpu_planar3d/main.cpp:59-66), bit for bit."""
    import ctypes as C
    L = orc.ref_mesh()
    if L is None:
        pytest.skip("oracle/_ref/libwfref_mesh.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    rng = np.random.default_rng(2)
    for P in (2, 3, 4, 5, 7):
        for h in list(rng.uniform(1e-4, 5e-2, 6)) + [np.sqrt(3.0) * 0.1 / 16]:
            dt, tf, spp = C.c_double(), C.c_double(), C.c_int()
            L.wfref_demo_time_parameters(float(h), 1500.0, 0.5e6, 0.1, P, C.byref(dt), C.byref(tf), C.byref(spp))
            assert wfx.cfl_timestep(float(h), 1500.0, P, 0.5e6) == dt.value
            assert 0.1 / 1500.0 + 8.0 / 0.5e6 == tf.value


def test_general_point_jacobian_and_factor_use_the_reference_dot(wfx, orc):
    """compute_jacobian and compute_geometrical_factor (common/precompute.hpp:49-96, 148-176) are the reference's
    small matrix product `dot` (:17-41) around DOLFINx's det / inv: with the oracle's inverse supplied, its J and G
    equal the reference's own `dot` bit for bit (row a9)."""
    L = orc.ref_mesh()
    if L is None:
        pytest.skip("oracle/_ref/libwfref_mesh.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    mesh = wfx.create_box_hex((2, 2, 1), 2, (1.0, 0.7, 1.3), perturb=0.2)
    pts = np.random.default_rng(4).uniform(0, 1, size=(5, 3))
    wts = np.random.default_rng(5).uniform(0.1, 1, size=5)
    d = orc.jacobian_data(mesh, pts, wts)
    for c in range(mesh.ncells):
        for q in range(5):
            K = np.ascontiguousarray(d["K"][c, q])
            KT = np.ascontiguousarray(K.T)
            G = np.zeros((3, 3))
            L.wfref_dot(orc._f(K.reshape(-1)), 3, 3, orc._f(KT.reshape(-1)), 3, 3, orc._f(G.reshape(-1)), 0)
            assert np.array_equal(G * (d["detJ"][c, q] * wts[q]), d["G"][c, q])
    # the Jacobian: dot(coords [8][3], dphi [3][8], J, transpose = true); dphi from J itself is not available, so
    # check the transpose branch on random operands against the same sum written out in the oracle's order
    rng = np.random.default_rng(6)
    A, B = rng.standard_normal((8, 3)), rng.standard_normal((3, 8))
    Cm = np.zeros((3, 3))
    L.wfref_dot(orc._f(np.ascontiguousarray(A).reshape(-1)), 8, 3, orc._f(np.ascontiguousarray(B).reshape(-1)), 3, 8,
                orc._f(Cm.reshape(-1)), 1)
    want = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            s_ = 0.0
            for k in range(8):
                s_ += A[k, i] * B[j, k]
            want[i, j] = s_
    assert np.array_equal(Cm, want)
