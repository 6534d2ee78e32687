"""Parity of the CUDA path (through the C ABI) against the CPU oracle, on a B200.

Tolerances: fp64 operator and RK4 results within 1e-12 relative L2 of the oracle
(BASELINE.json north_star); geometry factors and the lumped mass are bit-exact because
the GPU precompute follows the oracle's operation order with explicit rounding; fp32
within 2e-5 relative L2.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L = 0.1
TOL64 = 1e-12
TOL32 = 2e-5


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _mesh(wfx, N, P, perturb=0.15, **kw):
    return wfx.create_box_hex(N, P, (L, L, L), perturb=perturb, **kw)


# ---- a1: geometry ---------------------------------------------------------------------------
@pytest.mark.parametrize("P,perturb", [(2, 0.0), (4, 0.0), (4, 0.15), (3, 0.15), (7, 0.15)])
def test_geometry_bit_exact(wfx, orc, torch, P, perturb):
    mesh = _mesh(wfx, 3 if P < 7 else 2, P, perturb)
    G, detJ = wfx.Geometry(mesh, P).get()
    Go, detJo = orc.precompute_geometric_data(mesh, P)
    assert np.array_equal(detJ, detJo)
    iu = np.triu_indices(3)
    assert np.array_equal(G[:, :, iu[0], iu[1]], Go[:, :, iu[0], iu[1]])  # stored entries: bit-exact
    assert np.array_equal(G, np.swapaxes(G, 2, 3))                        # symmetric storage
    assert rel_l2(G, Go) < 1e-15                                          # mirrored entries: roundoff


def test_geometry_clamp_triggers_like_reference(wfx, orc, torch):
    # tiny cells: legitimate G entries below 1e-8 are zeroed (SURVEY.md App. B #1)
    mesh = wfx.create_box_hex(2, 4, (1e-4,) * 3)
    G, _ = wfx.Geometry(mesh, 4).get()
    Go, _ = orc.precompute_geometric_data(mesh, 4)
    assert np.array_equal(G, Go) and (np.diagonal(G, axis1=2, axis2=3) == 0).any()


def test_general_point_jacobian_data(wfx, orc, torch):
    mesh = _mesh(wfx, 3, 2)
    pts, wts = orc.gauss_legendre(3)
    P3 = np.array([[a, b, c] for a in pts for b in pts for c in pts])
    W3 = np.array([a * b * c for a in wts for b in wts for c in wts])
    got = wfx.compute_jacobian_data(mesh, P3, W3)
    want = orc.jacobian_data(mesh, P3, W3)
    for k in ("J", "detJ", "K", "G"):
        assert np.array_equal(got[k], want[k]), k


# ---- a3: mass ---------------------------------------------------------------------------------
@pytest.mark.parametrize("P,renumber", [(2, None), (4, None), (4, 5), (5, 9)])
def test_lumped_mass_bit_exact_and_apply(wfx, orc, torch, P, renumber):
    mesh = _mesh(wfx, 3, P, renumber=renumber)
    op = wfx.MassOperator(mesh, P)
    _, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)  # m = M.1 (LinearGLL.hpp:102-110)
    assert np.array_equal(op.diagonal(), m)
    assert np.array_equal(op.inverse_diagonal(), 1.0 / m)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    y0 = np.random.default_rng(43).standard_normal(mesh.ndofs)
    yo = y0.copy()
    orc.mass_apply(mesh, P, detJ, x, yo)
    yd = dev(torch, y0)
    op(dev(torch, x), yd)  # y += M x
    assert rel_l2(yd.cpu().numpy(), yo) < 1e-15
    yh = y0.copy()
    op(x, yh)              # host path
    assert np.array_equal(yh, yd.cpu().numpy())


# ---- a4: stiffness ------------------------------------------------------------------------------
CASES = [(2, 4, 0.15, None), (2, 9, 0.15, 3), (3, 5, 0.15, None), (4, 4, 0.0, None), (4, 4, 0.15, None),
         (4, 6, 0.15, 17), (5, 3, 0.15, None), (6, 2, 0.15, 1), (7, 2, 0.15, None)]


@pytest.mark.parametrize("mode", ["brick", "cell_colour", "brick_stream", "colour_stream"])
@pytest.mark.parametrize("P,N,perturb,renumber", CASES)
def test_stiffness_matches_dense_reference_kernel(wfx, orc, torch, monkeypatch, mode, P, N, perturb, renumber):
    mesh = _mesh(wfx, N, P, perturb, renumber=renumber)
    flag = {"brick": wfx.capi.STIFF_AUTO, "cell_colour": wfx.capi.STIFF_CELL_COLOUR,
            "brick_stream": wfx.capi.STIFF_CELL_STREAM, "colour_stream": wfx.capi.STIFF_CELL_STREAM}[mode]
    if mode == "colour_stream":
        monkeypatch.setenv("WFX_STREAM_ORDER", "colour")
    op = wfx.StiffnessOperator(mesh, P, {"c0": 1500.0}, mode=flag)
    assert op.kernel_info()["variant"] == {"brick": op.kernel_info()["variant"], "cell_colour": "cell",
                                           "brick_stream": "brick-streamed", "colour_stream": "cell-streamed"}[mode]
    Go, _ = orc.precompute_geometric_data(mesh, P)
    rng = np.random.default_rng(42)
    x, y0 = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    yo = y0.copy()
    orc.stiffness_apply(mesh, P, Go, x, yo, dense=True)   # the reference's skernel
    kx = yo - y0
    yd = dev(torch, y0)
    op(dev(torch, x), yd)                                  # y += A x
    assert rel_l2(yd.cpu().numpy() - y0, kx) < TOL64
    yd2 = dev(torch, y0)
    op.apply(dev(torch, x), yd2, beta=0)                   # y = A x, old y never read
    assert rel_l2(yd2.cpu().numpy(), kx) < TOL64
    # deterministic: bitwise repeatable
    yd3 = torch.full_like(yd2, float("nan"))
    op.apply(dev(torch, x), yd3, beta=0)
    assert torch.equal(yd2, yd3)


def test_stiffness_host_call_shape(wfx, orc, torch):
    mesh = _mesh(wfx, 4, 4)
    op = wfx.StiffnessOperator(mesh, 4, {"c0": 1.0})       # params ignored like the reference: c0 = 1500
    Go, _ = orc.precompute_geometric_data(mesh, 4)
    x = np.random.default_rng(0).standard_normal(mesh.ndofs)
    y, yo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    op(x, y)
    orc.stiffness_apply(mesh, 4, Go, x, yo)
    assert rel_l2(y, yo) < TOL64
    with pytest.raises(wfx.WfxError):
        op(x[:-1].copy(), y)
    with pytest.raises(wfx.WfxError):
        op(x.astype(np.float32), y)


def test_stiffness_fused_mass_inverse(wfx, orc, torch):
    P = 4
    mesh = _mesh(wfx, 5, P, renumber=2)
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    mass = wfx.MassOperator(mesh, P, geometry=geo)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(3).standard_normal(mesh.ndofs)
    b = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, b)
    want = b / mass.diagonal()                              # LinearGLL.hpp:188-191
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply_scaled(dev(torch, x), mass.inverse_diagonal_ptr(), y)
    assert rel_l2(y.cpu().numpy(), want) < TOL64


@pytest.mark.parametrize("order,renumber", [("brick", None), ("brick", 11), ("colour", None), ("colour", 11)])
@pytest.mark.parametrize("P,N,dtype,cps", [(7, 3, np.float64, 1), (7, 5, np.float64, 4), (6, 3, np.float64, 3),
                                           (5, 4, np.float64, 2), (4, 5, np.float64, 4), (4, 9, np.float64, 4),
                                           (7, 3, np.float32, 4), (6, 3, np.float32, 2), (2, 7, np.float64, 5),
                                           (3, 9, np.float32, 3)])
def test_streamed_cell_kernel_fused_apply(wfx, orc, torch, monkeypatch, P, N, dtype, cps, order, renumber):
    """The streamed-cell kernel (stiff_cell2_kernel) through the fused stiffness + mass call, in both cell
    orders (batches of a brick plan with a round barrier; global colours): FIRST flags (NaN-filled output is
    never read), LAST flags (1/m applied exactly once per dof), every pipeline depth, ragged meshes (partial
    bricks, ragged colours), lexicographic dofs (relabelled tensor axes, private G copy) and renumbered dofs
    (identity axes), a vector with unreferenced entries."""
    import copy
    monkeypatch.setenv("WFX_CELL2_CPS", str(cps))
    monkeypatch.setenv("WFX_STREAM_ORDER", order)
    mesh = copy.copy(_mesh(wfx, (N, N + 1, N), P, renumber=renumber))
    mesh.ndofs += 5                                          # entries no cell references
    geo = wfx.Geometry(mesh, P, dtype)
    op = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo, mode=wfx.capi.STIFF_CELL_STREAM)
    assert op.kernel_info()["variant"] == ("brick-streamed" if order == "brick" else "cell-streamed")
    Go, _ = orc.precompute_geometric_data(mesh, P)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    tol = TOL64 if dtype == np.float64 else TOL32
    x = np.random.default_rng(8).standard_normal(mesh.ndofs).astype(dtype)
    b = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x.astype(np.float64), b, dense=False)
    sc = np.random.default_rng(9).uniform(0.5, 2.0, mesh.ndofs).astype(dtype)
    y = torch.full((mesh.ndofs,), float("nan"), dtype=tdt, device="cuda")
    scd = dev(torch, sc)
    op.apply_scaled(dev(torch, x), scd.data_ptr(), y)
    yh = y.cpu().numpy()
    assert np.isfinite(yh).all() and (yh[-5:] == 0).all()
    assert rel_l2(yh, b * sc.astype(np.float64)) < tol
    y2 = dev(torch, np.ones(mesh.ndofs, dtype=dtype))
    op(dev(torch, x), y2)                                    # y += A x
    assert rel_l2(y2.cpu().numpy() - 1.0, b) < (tol if dtype == np.float64 else 1e-3)
    y3 = torch.full_like(y, float("nan"))
    op.apply_scaled(dev(torch, x), scd.data_ptr(), y3)       # bitwise repeatable
    assert torch.equal(y, y3)
    # against the brick kernel on the same inputs
    ob = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo)
    y4 = torch.full_like(y, float("nan"))
    ob.apply_scaled(dev(torch, x), scd.data_ptr(), y4)
    assert rel_l2(yh, y4.cpu().numpy().astype(np.float64)) < tol


def test_stiffness_ghost_only_entries_and_errors(wfx, orc, torch):
    # vector longer than the dofs the cells reference (ghost-only slots): y = A x zeroes them
    import copy
    mesh = copy.copy(_mesh(wfx, 3, 2))
    mesh.ndofs += 7
    op = wfx.StiffnessOperator(mesh, 2)
    x = torch.ones(mesh.ndofs, dtype=torch.float64, device="cuda")
    y = torch.full_like(x, float("nan"))
    op.apply(x, y, beta=0)
    assert torch.isfinite(y).all() and (y[-7:] == 0).all()
    with pytest.raises(wfx.WfxError, match="alias"):
        op.apply(x, x, beta=0)


@pytest.mark.parametrize("P", [2, 4, 6, 7])
def test_stiffness_fp32(wfx, orc, torch, P):
    mesh = _mesh(wfx, 4 if P < 6 else (2 if P == 6 else 3), P)
    op = wfx.StiffnessOperator(mesh, P, dtype=np.float32)
    # WFX_STIFF_AUTO: the streamed-cell kernel where it measured faster (P7 fp32), else a brick kernel
    assert (op.kernel_info()["variant"] == "cell-streamed") == (P == 7)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(1).standard_normal(mesh.ndofs)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x.astype(np.float32).astype(np.float64), yo, dense=False)
    y = torch.zeros(mesh.ndofs, dtype=torch.float32, device="cuda")
    op(dev(torch, x.astype(np.float32)), y)
    assert rel_l2(y.cpu().numpy(), yo) < TOL32


def test_stiffness_medium_mesh_vs_sumfact_oracle(wfx, orc, torch):
    P, N = 4, 16
    mesh = _mesh(wfx, N, P)
    op = wfx.StiffnessOperator(mesh, P)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, yo, dense=False, nthreads=orc.max_threads())
    y = torch.zeros(mesh.ndofs, dtype=torch.float64, device="cuda")
    op(dev(torch, x), y)
    assert rel_l2(y.cpu().numpy(), yo) < TOL64


def test_config2_full_size_properties(wfx, torch):
    """BASELINE config 2 (64^3 cells, P4, 16 974 593 dofs): size-independent properties --
    the two kernels agree, constants are annihilated, K is symmetric, and the energy of a
    linear field is exact."""
    P, N = 4, 64
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.0)
    assert mesh.ndofs == 16974593
    geo = wfx.Geometry(mesh, P)
    brick = wfx.StiffnessOperator(mesh, P, geometry=geo)
    simple = wfx.StiffnessOperator(mesh, P, geometry=geo, mode=wfx.capi.STIFF_CELL_COLOUR)
    g = torch.Generator(device="cuda").manual_seed(42)
    x1 = torch.randn(mesh.ndofs, dtype=torch.float64, device="cuda", generator=g)
    x2 = torch.randn(mesh.ndofs, dtype=torch.float64, device="cuda", generator=g)
    y1, y1s, y2 = torch.empty_like(x1), torch.empty_like(x1), torch.empty_like(x1)
    brick.apply(x1, y1, beta=0)
    simple.apply(x1, y1s, beta=0)
    assert float((y1 - y1s).norm() / y1.norm()) < 1e-14
    brick.apply(x2, y2, beta=0)
    a, b = float(x2 @ y1), float(x1 @ y2)
    assert abs(a - b) < 1e-11 * abs(a)
    ones = torch.ones_like(x1)
    brick.apply(ones, y2, beta=0)
    assert float(y2.abs().max()) < 1e-9 * 1500.0 ** 2 * (L / N)
    X = torch.from_numpy(wfx.dof_coordinates(mesh)).cuda()
    av = torch.tensor([1.0, -2.0, 0.5], dtype=torch.float64, device="cuda")
    xl = X @ av
    brick.apply(xl, y2, beta=0)
    want = -1500.0 ** 2 * float(av @ av) * L ** 3
    assert abs(float(xl @ y2) - want) < 1e-11 * abs(want)


def _host_threads():
    import os
    return max(1, min(len(os.sched_getaffinity(0)), 32))


def test_config2_as_benchmarked_vs_oracle(wfx, orc, torch):
    """BASELINE config 2 exactly as bench.py times it -- 64^3 cells, P4, fp64, perturb = 0.15 (non-affine,
    full 3x3 G), the regular-brick kernel with the fused mass inverse -- against the reference's dense
    skernel applied to EVERY cell (OpenMP over cells) and against the sum-factorised oracle."""
    P, N = 4, 64
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    assert mesh.ndofs == 16974593
    nt = _host_threads()
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    kd = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, kd, dense=True, nthreads=nt)      # common/operators.hpp:113-133,183-200
    ks = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, ks, dense=False, nthreads=nt)
    assert rel_l2(ks, kd) < 1e-13
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    mass = wfx.MassOperator(mesh, P, geometry=geo)
    assert np.array_equal(mass.diagonal(), m)
    xd = dev(torch, x)
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply_scaled(xd, mass.inverse_diagonal_ptr(), y)                    # the timed call of bench.py
    assert rel_l2(y.cpu().numpy(), kd / m) < TOL64                         # LinearGLL.hpp:188-191
    y0 = np.random.default_rng(43).standard_normal(mesh.ndofs)
    yd = dev(torch, y0)
    op(xd, yd)                                                             # y += A x
    assert rel_l2(yd.cpu().numpy() - y0, kd) < TOL64
    # the end-to-end host entry point of bench.py's e2e leg gives the same bits as the device path
    import ctypes as C
    yh = np.empty(mesh.ndofs)
    wfx.capi.call("wfx_stiffness_mass_apply_host", op.handle, mass.handle, C.c_void_p(x.ctypes.data),
                  C.c_void_p(yh.ctypes.data))
    assert np.array_equal(yh, y.cpu().numpy())
    # a random 512-cell subset of the same mesh as a mesh of its own (irregular batches: the generic
    # staged-dofmap kernel) against the dense skernel on those cells
    import copy
    sel = np.sort(np.random.default_rng(1).choice(mesh.ncells, 512, replace=False))
    sub = copy.copy(mesh)
    sub.xdofs = np.ascontiguousarray(mesh.xdofs[sel])
    sub.dofmap = np.ascontiguousarray(mesh.dofmap[sel])
    sop = wfx.StiffnessOperator(sub, P)
    ys = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    sop.apply(xd, ys, beta=0)
    kss = np.zeros(mesh.ndofs)
    orc.stiffness_apply(sub, P, np.ascontiguousarray(Go[sel]), x, kss, dense=True)
    assert rel_l2(ys.cpu().numpy(), kss) < TOL64


@pytest.mark.parametrize("N", [9, 13])
def test_ragged_mesh_mixed_plan_vs_oracle(wfx, orc, torch, N):
    """Cells per axis not a multiple of the 4-cell brick (config 5's 133 = 33*4 + 1): full bricks run
    the regular-brick kernel, the ragged rim the generic one, in the same apply."""
    P = 4
    mesh = _mesh(wfx, N, P, 0.15)
    op = wfx.StiffnessOperator(mesh, P)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, yo, dense=True, nthreads=_host_threads())
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply(dev(torch, x), y, beta=0)
    assert rel_l2(y.cpu().numpy(), yo) < TOL64
    y2 = torch.full_like(y, float("nan"))
    op.apply(dev(torch, x), y2, beta=0)
    assert torch.equal(y, y2)


def test_config5_size_ragged_rim_vs_oracle(wfx, orc, torch):
    """BASELINE config 5's per-GPU size, 133^3 cells (151 M dofs; 133 = 33 * 4 + 1: full bricks plus a
    one-cell ragged rim per axis), at full size.  The whole mesh does not fit the CPU oracle's memory, so
    the comparison is exact where it can be: the reference's dense skernel is applied to the slab of the
    last five cell layers in x (which contains the ragged rim and full bricks), and every dof strictly
    inside that slab -- touched by no cell outside it -- must agree with the GPU apply of the whole mesh."""
    import copy
    P, N = 4, 133
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    assert mesh.ndofs == 151419437
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    ki = op.kernel_info()
    assert ki["variant"] == "brick-regular" and ki["regular_batches"] == ki["batches"] == 34 ** 3
    g = torch.Generator(device="cuda").manual_seed(42)
    xd = torch.randn(mesh.ndofs, dtype=torch.float64, device="cuda", generator=g)
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply(xd, y, beta=0)
    del geo
    x = xd.cpu().numpy()
    yg = y.cpu().numpy()
    del xd, y, op
    torch.cuda.empty_cache()
    cx0 = 128
    sel = np.arange(cx0 * N * N, N * N * N)                    # cells c = (cx*N + cy)*N + cz with cx >= 128
    sub = copy.copy(mesh)
    sub.xdofs = np.ascontiguousarray(mesh.xdofs[sel])
    sub.dofmap = np.ascontiguousarray(mesh.dofmap[sel])
    Go, _ = orc.precompute_geometric_data(sub, P)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(sub, P, Go, x, yo, dense=True, nthreads=_host_threads())
    M = P * N + 1
    inside = np.arange((cx0 * P + 1) * M * M, mesh.ndofs)      # lattice planes X > 4 * 128 (lexicographic dofs)
    assert np.isfinite(yg).all()
    assert rel_l2(yg[inside], yo[inside]) < TOL64


# ---- f2: affine / structured fast path -------------------------------------------------------------
@pytest.mark.parametrize("P,N,dtype", [(4, 8, np.float64), (2, 16, np.float64), (3, 8, np.float64), (5, 4, np.float64),
                                       (4, 8, np.float32)])
def test_affine_fast_path_matches_reference(wfx, orc, torch, monkeypatch, P, N, dtype):
    """Parallelepiped cells (sheared box: full symmetric A, not just a diagonal): every cell is
    detected as affine, the operator takes the kernels that read 6 scalars of G per CELL, and the
    result still matches the reference's per-point G through the dense skernel."""
    mesh = wfx.create_box_hex(N, P, (L, 0.8 * L, 1.3 * L))
    shear = np.array([[1.0, 0.2, 0.1], [0.0, 1.0, 0.3], [0.0, 0.0, 1.0]])
    mesh.x = mesh.x @ shear.T                                   # affine map of the whole mesh
    geo = wfx.Geometry(mesh, P, dtype=dtype)
    assert geo.info()["n_affine"] == mesh.ncells
    op = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo)
    assert op.kernel_info()["affine"] and op.kernel_info()["variant"] == "brick-regular"
    assert op.info()["bytes"] == mesh.ncells * 6 * np.dtype(dtype).itemsize + 3 * mesh.ndofs * np.dtype(dtype).itemsize
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs).astype(dtype)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x.astype(np.float64), yo, dense=True, nthreads=_host_threads())
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    y = torch.full((mesh.ndofs,), float("nan"), dtype=tdt, device="cuda")
    op.apply(dev(torch, x), y, beta=0)
    assert rel_l2(y.cpu().numpy(), yo) < (TOL64 if dtype == np.float64 else TOL32)
    # the general kernel on the same geometry (per-point G) agrees to rounding
    monkeypatch.setenv("WFX_AFFINE", "0")
    op2 = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo)
    assert not op2.kernel_info()["affine"]
    y2 = torch.full_like(y, float("nan"))
    op2.apply(dev(torch, x), y2, beta=0)
    assert rel_l2(y2.cpu().numpy(), y.cpu().numpy().astype(np.float64)) < (1e-14 if dtype == np.float64 else 1e-6)


def test_affine_detection_is_per_cell(wfx, torch):
    """One moved vertex makes exactly the cells around it non-affine; the operator then stays on
    the general path."""
    P, N = 4, 6
    mesh = wfx.create_box_hex(N, P, (L, L, L))
    v = (3 * (N + 1) + 3) * (N + 1) + 3                       # an interior vertex
    mesh.x[v] += 0.1 * L / N
    geo = wfx.Geometry(mesh, P)
    assert geo.info()["n_affine"] == mesh.ncells - 8
    assert not wfx.StiffnessOperator(mesh, P, geometry=geo).kernel_info()["affine"]


# ---- f4: heterogeneous speed of sound folded into G ---------------------------------------------------
@pytest.mark.parametrize("perturb", [0.0, 0.15])
def test_piecewise_constant_speed_of_sound(wfx, orc, torch, perturb):
    """c0(x) constant per cell (the reference's `// TODO: Compute coefficients`, LinearGLL.hpp:170):
    scaling the stored G of cell c by (c0[c]/c0_ref)^2 makes the unchanged kernels apply -c0(x)^2 K."""
    P, N = 4, 6
    mesh = _mesh(wfx, N, P, perturb)
    c0 = 1500.0 * (1.0 + 0.3 * np.random.default_rng(5).uniform(-1, 1, mesh.ncells))
    geo = wfx.Geometry(mesh, P)
    geo.scale_cells((c0 / 1500.0) ** 2)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    Go = Go * ((c0 / 1500.0) ** 2)[:, None, None, None]
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, np.ascontiguousarray(Go), x, yo, dense=True, nthreads=_host_threads())
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply(dev(torch, x), y, beta=0)
    assert rel_l2(y.cpu().numpy(), yo) < TOL64
    with pytest.raises(wfx.WfxError):
        geo.scale_cells(np.zeros(mesh.ncells))


# ---- mixed plans: lattice bricks and irregular batches in one apply ------------------------------------
def test_mixed_plan_regular_and_irregular_batches(wfx, orc, torch):
    """A structured mesh with some cells duplicated in place (overlapping cells with fresh dofs): the
    bricks holding a duplicate are no lattice bricks any more.  Those batches run the generic
    (staged-dofmap) kernel, all others the regular-brick kernel, two launches per colour."""
    import copy
    P, N = 4, 8
    base = _mesh(wfx, N, P, 0.15)
    dup = np.array([3, 77, 200, 201, 450], dtype=np.int64)
    mesh = copy.copy(base)
    nd = (P + 1) ** 3
    extra = base.ndofs + np.arange(len(dup) * nd, dtype=np.int32).reshape(len(dup), nd)
    mesh.xdofs = np.concatenate([base.xdofs, base.xdofs[dup]])
    mesh.dofmap = np.concatenate([base.dofmap, extra])
    mesh.ndofs = base.ndofs + len(dup) * nd
    op = wfx.StiffnessOperator(mesh, P)
    ki = op.kernel_info()
    assert ki["mixed"] and 0 < ki["regular_batches"] < ki["batches"]
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(42).standard_normal(mesh.ndofs)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, yo, dense=True, nthreads=_host_threads())
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply(dev(torch, x), y, beta=0)
    assert rel_l2(y.cpu().numpy(), yo) < TOL64
    y0 = np.random.default_rng(1).standard_normal(mesh.ndofs)
    yd = dev(torch, y0)
    op(dev(torch, x), yd)
    assert rel_l2(yd.cpu().numpy() - y0, yo) < TOL64


# ---- a5: boundary form -------------------------------------------------------------------------
def test_boundary_operator(wfx, orc, torch):
    P = 4
    mesh = _mesh(wfx, 3, P)
    op = wfx.BoundaryOperator(mesh, P)
    m1o, m2o = orc.boundary_facet_mass(mesh, P)
    m1, m2 = op.facet_masses()
    np.testing.assert_allclose(m1, m1o, rtol=1e-14, atol=0)
    np.testing.assert_allclose(m2, m2o, rtol=1e-14, atol=0)
    rng = np.random.default_rng(8)
    vn, b0 = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    c0, g = 1500.0, 123.456
    want = b0 + c0 * c0 * g * m1o - c0 * m2o * vn
    b = dev(torch, b0)
    op.apply(c0, g, dev(torch, vn), b)
    got = b.cpu().numpy()
    assert rel_l2(got - b0, want - b0) < 1e-14
    assert np.array_equal(got[(m1o == 0) & (m2o == 0)], b0[(m1o == 0) & (m2o == 0)])


# ---- a6/a7: f1 + RK4 (cpu_planar3d in miniature, config 1) ----------------------------------------
@pytest.mark.parametrize("shape,perturb,steps", [((8, 8, 8), 0.0, 60), ((6, 5, 4), 0.15, 40)])
def test_rk4_matches_reference_time_stepper(wfx, orc, torch, shape, perturb, steps):
    P, c0, f0, p0 = 4, 1500.0, 0.5e6, 6e4
    mesh = wfx.create_box_hex(shape, P, (L * shape[0] / 8, L * shape[1] / 8, L * shape[2] / 8),
                              perturb=perturb)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, f0)
    tf = L / c0 + 8.0 / f0                                   # cpu_planar3d/main.cpp:64
    uo, vo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    so, to = orc.rk4(mesh, P, Go, m, m1, m2, c0, f0, p0, 0.0, tf, dt, uo, vo, max_steps=steps,
                     sumfact=True, nthreads=orc.max_threads())
    eqn = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    eqn.init()
    s, t = eqn.rk4(0.0, tf, dt, max_steps=steps)
    u, v = eqn.get_state()
    assert (s, t) == (so, to) and s == steps
    assert np.abs(uo).max() > 0
    assert rel_l2(u, uo) < TOL64 and rel_l2(v, vo) < TOL64


def test_rk4_final_short_step(wfx, orc, torch):
    # `while (t < tf)` with dt = min(dt, tf - t) (LinearGLL.hpp:241-242): last step shortened
    P, c0, f0, p0 = 2, 1500.0, 0.5e6, 6e4
    mesh = wfx.create_box_hex(4, P, (0.01,) * 3)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, f0)
    tf = 10.4 * dt
    uo, vo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    so, to = orc.rk4(mesh, P, Go, m, m1, m2, c0, f0, p0, 0.0, tf, dt, uo, vo)
    eqn = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    eqn.init()
    s, t = eqn.rk4(0.0, tf, dt)
    u, v = eqn.get_state()
    assert s == so == 11 and t == to
    assert rel_l2(u, uo) < TOL64 and rel_l2(v, vo) < TOL64


# ---- L1 primitives --------------------------------------------------------------------------------
def test_gather_and_scatter_add(wfx, torch):
    import ctypes as C
    capi = wfx.capi
    ctx = wfx.Context.get()
    mesh = _mesh(wfx, 3, 2)
    idx = np.ascontiguousarray(mesh.dofmap.reshape(-1), dtype=np.int32)
    # demo/gpu_scatter_local/main.cpp:70-90: gather of iota reproduces the dofmap
    x = torch.arange(mesh.ndofs, dtype=torch.float64, device="cuda")
    xe = torch.empty(idx.size, dtype=torch.float64, device="cuda")
    didx = torch.from_numpy(idx).cuda()
    capi.call("wfx_gather", ctx.handle, capi.F64, idx.size, C.c_void_p(didx.data_ptr()),
              C.c_void_p(x.data_ptr()), C.c_void_p(xe.data_ptr()), None)
    assert np.array_equal(xe.cpu().numpy(), idx.astype(np.float64))
    # scatter-add without atomics equals the serial loop, bitwise
    plan = C.c_void_p()
    capi.call("wfx_scatter_plan_create", ctx.handle, idx.size, capi.i32p(idx), mesh.ndofs, C.byref(plan))
    vals = np.random.default_rng(0).standard_normal(idx.size)
    want = np.zeros(mesh.ndofs)
    for i, j in enumerate(idx):
        want[j] += vals[i]
    out = torch.zeros(mesh.ndofs, dtype=torch.float64, device="cuda")
    capi.call("wfx_scatter_add", plan, capi.F64, C.c_void_p(dev(torch, vals).data_ptr()),
              C.c_void_p(out.data_ptr()), 1, None)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), want)
    capi.call("wfx_scatter_plan_destroy", plan)


# ---- e: multi-GPU (NCCL halo) -- runs when the box has at least two GPUs ---------------------------
def test_multi_gpu_halo_and_rk4(torch):
    import os
    import subprocess
    import sys
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.join(root, "tests", "mgpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "mgpu_check ok" in r.stdout


def test_planar3d_demo_full_run_matches_oracle(wfx, orc, torch):
    """BASELINE config 1 (cpu_planar3d in miniature): the whole run to t_f = L/c0 + 8/f0 -- 1 000+
    RK4 steps with source ramp, propagation and absorption -- against the oracle's time stepper."""
    P, c0, f0, p0, Lx = 4, 1500.0, 0.5e6, 6e4, 0.1
    nx = 24
    side = Lx / nx
    mesh = wfx.create_box_hex((nx, 1, 1), P, (Lx, side, side))
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, f0)
    tf = Lx / c0 + 8.0 / f0
    uo, vo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    so, to = orc.rk4(mesh, P, Go, m, m1, m2, c0, f0, p0, 0.0, tf, dt, uo, vo, sumfact=True,
                     nthreads=orc.max_threads())
    eqn = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    eqn.init()
    s, t = eqn.rk4(0.0, tf, dt)
    u, v = eqn.get_state()
    assert s == so and s > 300 and t == to
    assert np.abs(uo).max() > 1e3  # the wave (kPa scale) has crossed the domain
    assert rel_l2(u, uo) < TOL64 and rel_l2(v, vo) < TOL64


@pytest.mark.parametrize("streamed", [False, True])
def test_stiffness_interface_interior_split(wfx, orc, torch, monkeypatch, streamed):
    """The distributed-mesh schedule on one GPU: with an (artificial) set of rank-shared dofs the
    interface part followed by the interior part equals the plain apply, and the fused scaling
    skips exactly the shared dofs.  Same for the brick-ordered streamed-cell kernel."""
    import copy
    P = 4
    if streamed:
        monkeypatch.setenv("WFX_CELL2", "1")
    mesh = copy.copy(_mesh(wfx, 6, P))
    M = P * 6 + 1
    shared = (np.arange(M * M) + (M // 2) * M * M).astype(np.int32)  # the lattice plane x = L/2
    mesh.halo = {"send_indices": shared, "recv_indices": np.zeros(0, dtype=np.int32)}
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    assert op.nshared == len(shared) and op.info()["ncolours"] == 16
    assert (op.kernel_info()["variant"] == "brick-streamed") == streamed
    mass = wfx.MassOperator(mesh, P, geometry=geo)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(5).standard_normal(mesh.ndofs)
    kx = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, kx, dense=False)
    xd = dev(torch, x)
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply_part(xd, y, 0)
    got0 = y.cpu().numpy()
    # after the interface part every shared dof is complete, interior-only dofs are untouched
    assert rel_l2(got0[shared], kx[shared]) < TOL64
    op.apply_part(xd, y, 1)
    assert rel_l2(y.cpu().numpy(), kx) < TOL64
    y2 = torch.full_like(y, float("nan"))
    op.apply(xd, y2, beta=0)  # both parts in one call
    assert torch.equal(y, y2)
    y3 = torch.full_like(y, float("nan"))
    op.apply_scaled(xd, mass.inverse_diagonal_ptr(), y3)
    want = kx / mass.diagonal()
    want[shared] = kx[shared]  # shared dofs are left for the ghost reduction to scale
    assert rel_l2(y3.cpu().numpy(), want) < TOL64


# ---- kernel variants behind environment switches stay correct -----------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"WFX_REGULAR": "0"}, {"WFX_TUNED_STRIDES": "1"}, {"WFX_NO_UNIFORM": "1"},
                                 {"WFX_PERSISTENT": "1"}, {"WFX_PERSISTENT": "1", "WFX_NO_UNIFORM": "1"}])
def test_stiffness_kernel_variants(wfx, orc, torch, monkeypatch, env):
    """The generic (staged local dofmap) kernel, the conflict-free P4 layout with reordered G columns
    and the loaded batch headers are not the default on structured meshes: force each and compare
    with the default kernel (bitwise for the generic kernel: same arithmetic, same order) and the
    oracle."""
    P, N = 4, 6
    mesh = _mesh(wfx, N, P, 0.15, renumber=11)
    rng = np.random.default_rng(7)
    x = rng.standard_normal(mesh.ndofs)
    ref = wfx.StiffnessOperator(mesh, P, {"c0": 1500.0})
    y_ref = torch.empty(mesh.ndofs, dtype=torch.float64, device="cuda")
    ref.apply(dev(torch, x), y_ref, beta=0)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, {"c0": 1500.0}, geometry=geo)
    y = torch.full_like(y_ref, float("nan"))
    op.apply(dev(torch, x), y, beta=0)
    if "WFX_PERSISTENT" in env:
        assert op.info()["nlaunches"] == 1
        # the single-launch form in a time loop (not graph-replayed: its epoch is a kernel argument)
        eqn_a = wfx.LinearGLLOpt(mesh, None, P, 1500.0, 0.5e6, 6e4)
        eqn_a.init()
        dtw = wfx.cfl_timestep(mesh.h_min, 1500.0, P, 0.5e6)
        eqn_a.rk4(0.0, 1.0, dtw, max_steps=12)
        ua, va = eqn_a.get_state()
        for k in env:
            monkeypatch.delenv(k)
        eqn_b = wfx.LinearGLLOpt(mesh, None, P, 1500.0, 0.5e6, 6e4)
        eqn_b.init()
        eqn_b.rk4(0.0, 1.0, dtw, max_steps=12)
        ub, vb = eqn_b.get_state()
        assert np.abs(ub).max() > 0 and np.array_equal(ua, ub) and np.array_equal(va, vb)
    if "WFX_TUNED_STRIDES" in env:
        assert rel_l2(y.cpu().numpy(), y_ref.cpu().numpy()) < 1e-14
        # the geometry's columns were reordered in place: the exported G must not change
        Go, _ = orc.precompute_geometric_data(mesh, P)
        iu = np.triu_indices(3)
        assert np.array_equal(geo.get()[0][:, :, iu[0], iu[1]], Go[:, :, iu[0], iu[1]])
        # and a second operator on the same (reordered) geometry with the simple kernel agrees
        op2 = wfx.StiffnessOperator(mesh, P, {"c0": 1500.0}, mode=wfx.capi.STIFF_CELL_COLOUR, geometry=geo)
        y2 = torch.zeros_like(y_ref)
        op2.apply(dev(torch, x), y2, beta=0)
        assert rel_l2(y2.cpu().numpy(), y_ref.cpu().numpy()) < 1e-14
    else:
        assert torch.equal(y, y_ref)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    yo = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, yo, dense=True)
    assert rel_l2(y.cpu().numpy(), yo) < TOL64


@pytest.mark.gpu
def test_right_hand_sides_f0_f1(wfx, orc, torch):
    """LinearGLLOpt::f0 / f1 (LinearGLL.hpp:141-192) on their own: f1 = (K u + c0^2 g(t) m1 - c0 m2 v) / m
    composed from the oracle's pieces."""
    P, c0, f0, p0 = 4, 1500.0, 0.5e6, 6e4
    mesh = _mesh(wfx, 4, P, 0.15)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    rng = np.random.default_rng(3)
    u, v = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    eqn = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    ud, vd = dev(torch, u), dev(torch, v)
    res = torch.full_like(ud, float("nan"))
    for t in (0.3e-6, 2.0e-5):                       # inside and after the Hann ramp (4 periods = 8 us)
        w0, T, alpha = 2.0 * np.pi * f0, 1.0 / f0, 4.0
        window = 0.5 * (1.0 - np.cos(f0 * np.pi * t / alpha)) if t < T * alpha else 1.0
        g = window * p0 * w0 / c0 * np.cos(w0 * t)
        b = np.zeros(mesh.ndofs)
        orc.stiffness_apply(mesh, P, Go, u, b, dense=True)
        want = (b + c0 * c0 * g * m1 - c0 * m2 * v) / m
        eqn.f1(t, ud, vd, res)
        assert rel_l2(res.cpu().numpy(), want) < TOL64
    eqn.f0(0.0, ud, vd, res)
    assert torch.equal(res, vd)
    with pytest.raises(RuntimeError):
        eqn.f1(0.0, ud, vd, ud)


# ---- f3: probes and snapshots ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_probe_series_and_snapshots_match_oracle(wfx, orc, torch):
    """Probe time series and periodic snapshots of the GPU run against the oracle stepped one time
    step at a time; a snapshot fed back through set_state resumes the run bit for bit."""
    P, c0, f0, p0 = 4, 1500.0, 0.5e6, 6e4
    mesh = wfx.create_box_hex((6, 3, 3), P, (L * 6 / 8, L * 3 / 8, L * 3 / 8), perturb=0.1)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, f0)
    nsteps, every = 24, 8
    probes = np.array([0, 17, mesh.ndofs // 2, mesh.ndofs - 1], dtype=np.int32)
    uo, vo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    t, series, times, snaps_o = 0.0, [], [], {}
    for k in range(nsteps):
        s1, t = orc.rk4(mesh, P, Go, m, m1, m2, c0, f0, p0, t, 1.0, dt, uo, vo, max_steps=1, sumfact=True)
        assert s1 == 1
        series.append(uo[probes].copy())
        times.append(t)
        if (k + 1) % every == 0:
            snaps_o[k + 1] = (uo.copy(), vo.copy())
    eqn = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    eqn.init()
    eqn.set_probes(probes, max_records=nsteps + 5)
    snaps = {}
    eqn.set_snapshot(every, lambda step, tt, u, v: snaps.__setitem__(step, (tt, u.copy(), v.copy())))
    s, t_end = eqn.rk4(0.0, 1.0, dt, max_steps=10)
    s2, t_end = eqn.rk4(t_end, 1.0, dt, max_steps=nsteps - 10)      # the series continues across calls
    assert s + s2 == nsteps
    tt, vals = eqn.probe_series()
    assert vals.shape == (nsteps, len(probes)) and np.allclose(tt, times, rtol=1e-15, atol=0)
    scale = np.abs(np.array(series)).max()
    assert scale > 0 and np.abs(vals - np.array(series)).max() < 1e-11 * scale
    assert sorted(snaps) == sorted(snaps_o)
    for k in snaps:
        assert snaps[k][0] == times[k - 1]
        assert rel_l2(snaps[k][1], snaps_o[k][0]) < TOL64 and rel_l2(snaps[k][2], snaps_o[k][1]) < TOL64
    # restart from the snapshot at step 16: same final state as the uninterrupted run, bitwise
    u_end, v_end = eqn.get_state()
    eqn2 = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    eqn2.set_state(snaps[16][1], snaps[16][2])
    eqn2.rk4(snaps[16][0], 1.0, dt, max_steps=nsteps - 16)
    u2, v2 = eqn2.get_state()
    assert np.array_equal(u2, u_end) and np.array_equal(v2, v_end)


@pytest.mark.gpu
def test_stiffness_repeatable_under_concurrent_load(wfx, torch):
    """Race evidence without a sanitizer (compute-sanitizer is closed on the GPU pool): the apply is
    repeated while an unrelated kernel stream perturbs the CTA scheduling; every result must equal
    the first bit for bit (a shared-memory or write-back race would show as a changing bit pattern).
    Covers the regular-brick, generic and affine kernels."""
    P = 4
    side = torch.cuda.Stream()
    noise = torch.randn(2048, 2048, device="cuda")
    for perturb, env in ((0.15, {}), (0.0, {}), (0.15, {"WFX_REGULAR": "0"})):
        import os
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            mesh = _mesh(wfx, 12, P, perturb)
            geo = wfx.Geometry(mesh, P)
            op = wfx.StiffnessOperator(mesh, P, geometry=geo)
            mass = wfx.MassOperator(mesh, P, geometry=geo)
        finally:
            for k, v in old.items():
                os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
        x = torch.randn(mesh.ndofs, dtype=torch.float64, device="cuda")
        ref = torch.empty_like(x)
        op.apply_scaled(x, mass.inverse_diagonal_ptr(), ref)
        for it in range(25):
            if it % 2:
                with torch.cuda.stream(side):
                    for _ in range(3):
                        noise = noise @ noise * 1e-3
            y = torch.full_like(x, float("nan"))
            op.apply_scaled(x, mass.inverse_diagonal_ptr(), y)
            assert torch.equal(y, ref), f"apply {it} differs ({op.kernel_info()})"
        side.synchronize()


# ---- the reference's own CUDA primitives (oracle/_ref, compiled from the reference sources) -----------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_primitives_against_the_reference_cuda_kernels(wfx, orc, torch, dtype):
    """wfx_gather, wfx_scatter_add and the diagonal mass apply against the REFERENCE's kernels themselves:
    gather / scatter (common/cuda/scatter.cu) and SpectralMassOperator::apply = gather -> transform1 ->
    scatter (common/cuda/spectral_mass.hpp:84-89), compiled from the reference sources into oracle/_ref."""
    import ctypes as C
    ref = orc.ref_cuda()
    if ref is None:
        pytest.skip("oracle/_ref/libwfref_cuda.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    sfx = "f64" if dtype == np.float64 else "f32"
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    code = wfx.capi.dtype_code(dtype)
    capi, ctx = wfx.capi, wfx.Context.get()
    P = 4
    mesh = _mesh(wfx, 6, P, 0.15, renumber=4)
    tdm = np.ascontiguousarray(wfx.capi.reorder_dofmap(mesh.dofmap, P).reshape(-1), dtype=np.int32)  # permute.hpp:10-28
    n = tdm.size
    idx = torch.from_numpy(tdm).cuda()
    ptr = lambda t: C.c_void_p(t.data_ptr())
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(mesh.ndofs, dtype=tdt, device="cuda", generator=g)
    # gather: bit-identical
    xe_ref, xe = torch.empty(n, dtype=tdt, device="cuda"), torch.empty(n, dtype=tdt, device="cuda")
    getattr(ref, "ref_gather_" + sfx)(n, ptr(idx), ptr(x), ptr(xe_ref))
    capi.call("wfx_gather", ctx.handle, code, n, ptr(idx), ptr(x), ptr(xe), None)
    torch.cuda.synchronize()
    assert torch.equal(xe, xe_ref)
    # scatter-add: the reference adds with atomicAdd in arbitrary order -- exact for integer-valued data,
    # to rounding for random data
    plan = C.c_void_p()
    capi.call("wfx_scatter_plan_create", ctx.handle, n, capi.i32p(tdm), mesh.ndofs, C.byref(plan))
    for vals, exact in ((torch.randint(-8, 9, (n,), device="cuda", generator=g).to(tdt), True),
                        (torch.randn(n, dtype=tdt, device="cuda", generator=g), False)):
        y_ref = torch.zeros(mesh.ndofs, dtype=tdt, device="cuda")
        y = torch.zeros_like(y_ref)
        getattr(ref, "ref_scatter_" + sfx)(n, ptr(idx), ptr(vals), ptr(y_ref))
        capi.call("wfx_scatter_add", plan, code, ptr(vals), ptr(y), 1, None)
        torch.cuda.synchronize()
        if exact:
            assert torch.equal(y, y_ref)
        else:
            assert float((y - y_ref).norm() / y_ref.norm()) < (1e-15 if dtype == np.float64 else 1e-6)
    capi.call("wfx_scatter_plan_destroy", plan)
    # the reference's GPU mass operator: y += scatter(detJ .* gather(x)) in tensor-product dof order
    geo = wfx.Geometry(mesh, P, dtype=dtype)
    mass = wfx.MassOperator(mesh, P, dtype=dtype, geometry=geo)
    _, detJ = orc.precompute_geometric_data(mesh, P)            # [cell][tensor point], = detJ * w (precomputation.hpp:95)
    dj = torch.from_numpy(np.ascontiguousarray(detJ.reshape(-1))).to("cuda", tdt)
    y_ref = torch.zeros(mesh.ndofs, dtype=tdt, device="cuda")
    getattr(ref, "ref_gather_" + sfx)(n, ptr(idx), ptr(x), ptr(xe_ref))
    getattr(ref, "ref_transform1_" + sfx)(n, ptr(xe_ref), ptr(dj), ptr(xe_ref))
    getattr(ref, "ref_scatter_" + sfx)(n, ptr(idx), ptr(xe_ref), ptr(y_ref))
    y = torch.zeros_like(y_ref)
    mass(x, y)
    torch.cuda.synchronize()
    assert float((y - y_ref).norm() / y_ref.norm()) < (1e-14 if dtype == np.float64 else 2e-6)


# ---- the reference's own CPU code (oracle/_ref/libwfref_cpu.so, cut out of the reference's headers) -------
@pytest.mark.gpu
@pytest.mark.parametrize("P,shape,perturb", [(4, (4, 3, 2), 0.15), (2, (5, 4, 3), 0.15), (5, (2, 2, 2), 0.1)])
def test_cuda_operators_against_the_reference_cpu_code(wfx, orc, torch, P, shape, perturb):
    """The CUDA stiffness and mass operators against the REFERENCE's own StiffnessOperator::operator() /
    skernel and MassOperatorCPU::operator() / mkernel (common/operators.hpp), compiled from the reference
    sources (tests/test_reference_pins.py has the bit-for-bit pin of the oracle to the same code)."""
    if orc.ref_cpu() is None:
        pytest.skip("oracle/_ref/libwfref_cpu.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    mesh = wfx.create_box_hex(shape, P, (L, 0.7 * L, 1.3 * L), perturb=perturb)
    geo = wfx.Geometry(mesh, P)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    rng = np.random.default_rng(21)
    x, y0 = rng.standard_normal(mesh.ndofs), rng.standard_normal(mesh.ndofs)
    yr = y0.copy()
    orc.reference_stiffness_apply(mesh, P, Go, x, yr)
    for mode in (wfx.capi.STIFF_AUTO, wfx.capi.STIFF_CELL_STREAM, wfx.capi.STIFF_CELL_COLOUR):
        op = wfx.StiffnessOperator(mesh, P, geometry=geo, mode=mode)
        yd = dev(torch, y0)
        op(dev(torch, x), yd)                              # y += A x like the reference
        assert rel_l2(yd.cpu().numpy() - y0, yr - y0) < TOL64
    mr = np.zeros(mesh.ndofs)
    orc.reference_mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), mr)
    assert np.array_equal(wfx.MassOperator(mesh, P, geometry=geo).diagonal(), mr)   # lumped mass: bit-exact


@pytest.mark.gpu
@pytest.mark.parametrize("shape,perturb,nsteps,frac", [((4, 3, 2), 0.15, 40, 0.0), ((3, 3, 3), 0.0, 25, 0.4)])
def test_cuda_rk4_against_the_reference_time_stepper(wfx, orc, torch, capfd, shape, perturb, nsteps, frac):
    """The CUDA time stepper against the REFERENCE's own LinearGLLOpt::rk4 / f0 / f1 / kernels::axpy / copy
    (common/LinearGLL.hpp) over whole trajectories, including a shorter last step."""
    if orc.ref_cpu() is None:
        pytest.skip("oracle/_ref/libwfref_cpu.so was not built (needs the reference sources, WFX_REFERENCE, at build time)")
    P, c0, f0, p0 = 4, 1500.0, 0.5e6, 6e4
    mesh = wfx.create_box_hex(shape, P, (L * shape[0] / 8, L * shape[1] / 8, L * shape[2] / 8), perturb=perturb)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.reference_mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, c0, P, f0)
    tf = (nsteps + frac) * dt
    ur, vr = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    orc.reference_rk4(mesh, P, Go, m, m1, m2, c0, f0, p0, 0.0, tf, dt, ur, vr)
    capfd.readouterr()
    eqn = wfx.LinearGLLOpt(mesh, None, P, c0, f0, p0)
    eqn.init()
    s, t = eqn.rk4(0.0, tf, dt)
    u, v = eqn.get_state()
    # (the step count of `while (t < tf)` depends on the rounding of the accumulated t: take it from the
    # oracle's loop, which reproduces the reference's bit for bit)
    uo, vo = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    so, to = orc.rk4(mesh, P, Go, m, m1, m2, c0, f0, p0, 0.0, tf, dt, uo, vo, sumfact=True)
    assert (s, t) == (so, to) and s >= nsteps and np.abs(ur).max() > 0
    assert rel_l2(u, ur) < TOL64 and rel_l2(v, vr) < TOL64


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_rank_without_cells(wfx, torch, dtype):
    """A rank that owns no cell (only ghost dofs, or nothing): every operator is a no-op of the right kind --
    y = A x zeroes y, y += A x leaves it, the lumped mass is zero, gather / scatter of nothing succeed."""
    from wave_fenics_b200.mesh import HexMesh
    P, nd, ndofs = 4, 125, 7
    mesh = HexMesh(P=P, shape=(0, 0, 0), x=np.zeros((0, 3)), xdofs=np.zeros((0, 8), dtype=np.int32),
                   dofmap=np.zeros((0, nd), dtype=np.int32), ndofs=ndofs, size_local=0,
                   facet_cells=np.zeros(0, dtype=np.int32), facet_local=np.zeros(0, dtype=np.int32),
                   facet_tags=np.zeros(0, dtype=np.int32), h_min=1.0, lengths=(1.0, 1.0, 1.0), ndofs_global=ndofs)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    geo = wfx.Geometry(mesh, P, dtype)
    for mode in (wfx.capi.STIFF_AUTO, wfx.capi.STIFF_CELL_STREAM, wfx.capi.STIFF_CELL_COLOUR):
        op = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo, mode=mode)
        x = torch.ones(ndofs, dtype=tdt, device="cuda")
        y = torch.full_like(x, float("nan"))
        op.apply(x, y, beta=0)
        assert (y == 0).all()
        y.fill_(3.0)
        op(x, y)
        assert (y == 3.0).all()
    mass = wfx.MassOperator(mesh, P, dtype=dtype, geometry=geo)
    assert (mass.diagonal() == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 4, 7])
def test_single_cell_mesh(wfx, orc, torch, P):
    """The smallest mesh: one (perturbed) cell; every stiffness kernel, the lumped mass and one RK4 step."""
    mesh = wfx.create_box_hex((1, 1, 1), P, (L, 0.8 * L, 1.1 * L), perturb=0.0)
    mesh.x = mesh.x + 0.05 * L * np.random.default_rng(P).uniform(-1, 1, mesh.x.shape)   # a general hexahedron
    geo = wfx.Geometry(mesh, P)
    Go, detJ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(1).standard_normal(mesh.ndofs)
    kx = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Go, x, kx, dense=True)
    for mode in (wfx.capi.STIFF_AUTO, wfx.capi.STIFF_CELL_STREAM, wfx.capi.STIFF_CELL_COLOUR):
        op = wfx.StiffnessOperator(mesh, P, geometry=geo, mode=mode)
        y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
        op.apply(dev(torch, x), y, beta=0)
        assert rel_l2(y.cpu().numpy(), kx) < TOL64
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    assert np.array_equal(wfx.MassOperator(mesh, P, geometry=geo).diagonal(), m)
