"""Heterogeneous media: a per-cell coefficient folded into the geometric factors (wfx_geometry_scale_cells).

Scaling cell c's G by coeff[c] = (c[c] / c_ref)^2 makes every stiffness kernel apply -c_ref^2 K_c with
K_c = int c(x)^2 / c_ref^2 grad(phi_i) . grad(phi_j): the wave models then solve p_tt = div(c^2 grad p) (DESIGN.md
section 4.5a), and the thermal model uses the same route for a per-cell conductivity.  The coefficients are random
and log-uniform in [1/4, 4], so a mix-up between a plan's cell order and the cell ids, or a G copy that missed the
scaling, shows at O(1); the reference is always the oracle with G * coeff.

CPU: the premises of the bitwise checks on oracle data, and a known answer -- the lowest mode of a two-layer rigid
box, whose frequency pins down which interface condition the scaled form imposes (c^2 dp/dn continuous).
GPU: the stored scaled G bit for bit; every stiffness path against the dense reference kernel with the coefficient
set after the operator was created; after-creation against before-creation scaling bit for bit and a power-of-two
coefficient as an exact multiple; two operators sharing one geometry; the wave, ensemble and thermal models scaled
after construction against their CPU restatements; and the lossy model on the two-layer mode (delta_eff =
delta * coeff).
"""
import copy

import numpy as np
import pytest

L = 0.1
TOL64 = 1e-12
TOL32 = 2e-5          # as test_stiffness_fp32
TOL32_RUN = 1e-4      # fp32 model runs against the fp64 restatement (as test_ensemble_rk4_fp32)
C0, F0, P0 = 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 1e-2, 900.0, 1000.0
MODELS = {"linear": (0.0, 0.0, 1.0), "lossy": (DELTA, 0.0, 1.0), "westervelt": (DELTA, BETA, RHO0)}


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


def coefficients(ncells, seed):
    """log-uniform in [1/4, 4]"""
    return np.exp(np.random.default_rng(seed).uniform(np.log(0.25), np.log(4.0), ncells))


def scaled(G, coeff):
    return np.ascontiguousarray(G * np.asarray(coeff, dtype=np.float64)[:, None, None, None])


def _threads(orc):
    return orc.max_threads()


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


# ---- CPU --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dense", [True, False])
def test_power_of_two_coefficient_is_exact_on_the_oracle(wfx, orc, dense):
    """The premise of the GPU's exact-multiple check: a coefficient 4 scales every G entry exactly, and every
    product and sum of the apply by 4 as well, so K(4 G) x == 4 K(G) x bit for bit -- also in fp32 storage."""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (L, L, L), perturb=0.15)
    G, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(1).standard_normal(mesh.ndofs)
    y1, y4 = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, G, x, y1, dense=dense)
    orc.stiffness_apply(mesh, P, scaled(G, np.full(mesh.ncells, 4.0)), x, y4, dense=dense)
    assert np.abs(y1).max() > 0 and np.array_equal(y4, 4.0 * y1)
    g32 = G.astype(np.float32)
    assert np.array_equal((g32.astype(np.float64) * 4.0).astype(np.float32), g32 * np.float32(4.0))


def test_scaling_commutes_with_a_reordering_inside_each_cell(wfx, orc):
    """The premise of keeping private G copies by scaling them in place: an operator's copy holds each cell's
    values in another order (relabelled axes), and scaling per cell commutes with any such reordering bitwise, in
    fp64 and through fp32 storage."""
    P = 4
    mesh = wfx.create_box_hex((2, 2, 2), P, (L, L, L), perturb=0.15)
    G, _ = orc.precompute_geometric_data(mesh, P)
    coeff = coefficients(mesh.ncells, 3)
    n = P + 1
    # the point reordering of a relabelling of the tensor axes (x, y, z) -> (y, z, x), and the matching entries
    idx = np.arange(n ** 3).reshape(n, n, n).transpose(1, 2, 0).reshape(-1)
    ax = [1, 2, 0]
    relabel = lambda g: g[:, idx][:, :, ax][:, :, :, ax]  # noqa: E731
    assert np.array_equal(relabel(scaled(G, coeff)), scaled(relabel(G), coeff))
    s32 = lambda g: (g.astype(np.float32).astype(np.float64) * coeff[:, None, None, None]).astype(np.float32)  # noqa: E731
    assert np.array_equal(relabel(s32(G)), s32(relabel(G)))


# Two-layer rigid box, the interface at a cell face x = a: p = cos(k1 x) in layer 1, B cos(k2 (L - x)) in layer 2,
# with p and c^2 dp/dx continuous at x = a:  c1 tan(w a / c1) + c2 tan(w (L - a) / c2) = 0.
C1, C2 = 1500.0, 2100.0
NX, NA = 8, 3           # 8 cells along x, the interface after the third
WIDTH = 0.02            # cross-section modes lie far above the lowest x mode
# Measured on the CPU (P4, 8 x 1 x 1 cells, fp64), before the bounds were set:
#   lowest nonzero generalised eigenvalue of (-A, M):  |w_h^2 / w^2 - 1| = 3.1e-11
#   Rayleigh quotient of the exact mode's interpolant: |lam / (w / c_ref)^2 - 1| = 2.8e-11
#   lossy run from that mode (restatement, delta = 0.72, 1500 steps):  decay exponent 7.1e-9, phase 3.2e-8
# Another interface condition moves w far outside these bounds: dp/dx continuous gives 5.66e4 rad/s against 5.82e4.
KNOWN_BOUNDS = dict(eig=1e-9, rayleigh=1e-9, decay=1e-6, phase=1e-6)


def two_layer_omega(L_, a):
    """lowest positive root of c1 tan(w a / c1) + c2 tan(w (L - a) / c2) = 0, written without its poles"""
    from scipy.optimize import brentq
    g = lambda w: (C1 * np.sin(w * a / C1) * np.cos(w * (L_ - a) / C2)  # noqa: E731
                   + C2 * np.sin(w * (L_ - a) / C2) * np.cos(w * a / C1))
    ws = np.linspace(1.0, 4 * np.pi * C2 / L_, 20001)
    v = g(ws)
    i = np.nonzero(np.sign(v[:-1]) != np.sign(v[1:]))[0][0]
    return brentq(g, ws[i], ws[i + 1], xtol=1e-14, rtol=1e-15)


def two_layer_case(wfx):
    P = 4
    mesh = wfx.create_box_hex((NX, 1, 1), P, (L, WIDTH, WIDTH), tags=())
    a = NA * L / NX
    cx = np.arange(mesh.ncells)                  # cell c = (cx * 1 + cy) * 1 + cz
    coeff = np.where(cx < NA, (C1 / C0) ** 2, (C2 / C0) ** 2)
    w = two_layer_omega(L, a)
    k1, k2 = w / C1, w / C2
    x = wfx.dof_coordinates(mesh)[:, 0]
    B = np.cos(k1 * a) / np.cos(k2 * (L - a))
    u0 = np.where(x <= a, np.cos(k1 * x), B * np.cos(k2 * (L - x)))
    return mesh, P, coeff, w, u0


def test_two_layer_lowest_mode_known_answer(wfx, orc):
    """The lowest nonzero eigenvalue of the dense scaled stiffness against the lumped mass is w^2 of the exact
    two-layer mode, and the exact mode's Rayleigh quotient is too.  A homogeneous box would give c1 pi / L or
    c2 pi / L; continuity of dp/dn in place of c^2 dp/dn another root of another equation."""
    mesh, P, coeff, w, u0 = two_layer_case(wfx)
    G, detJ = orc.precompute_geometric_data(mesh, P)
    Gs = scaled(G, coeff)
    n = mesh.ndofs
    A = np.empty((n, n))
    e = np.zeros(n)
    for j in range(n):
        e[:] = 0.0
        e[j] = 1.0
        y = np.zeros(n)
        orc.stiffness_apply(mesh, P, Gs, e, y, dense=True)
        A[:, j] = y                                              # A = -c_ref^2 K_c
    m = np.zeros(n)
    orc.mass_apply(mesh, P, detJ, np.ones(n), m)
    s = 1.0 / np.sqrt(m)
    ev = np.linalg.eigvalsh(-(A * s[:, None]) * s[None, :])
    assert abs(ev[0]) < 1e-6 * ev[1]                             # the constant mode
    assert abs(ev[1] / w ** 2 - 1) < KNOWN_BOUNDS["eig"], ev[1] / w ** 2 - 1
    lam = -(u0 @ (A @ u0)) / C0 ** 2 / (u0 @ (m * u0))
    assert abs(lam / (w / C0) ** 2 - 1) < KNOWN_BOUNDS["rayleigh"]
    # the alternative interface condition (dp/dx continuous) has another lowest root
    from scipy.optimize import brentq
    a = NA * L / NX
    g = lambda v: np.sin(v * a / C1) * np.cos(v * (L - a) / C2) / C1 + np.sin(v * (L - a) / C2) * np.cos(v * a / C1) / C2  # noqa: E731
    ws = np.linspace(1.0, 2 * w, 20001)
    i = np.nonzero(np.sign(g(ws[:-1])) != np.sign(g(ws[1:])))[0][0]
    assert abs(brentq(g, ws[i], ws[i + 1]) / w - 1) > 0.02


# ---- GPU --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _tdt(torch, dtype):
    return torch.float64 if dtype == np.float64 else torch.float32


def _sheared(wfx, N, P):
    mesh = wfx.create_box_hex(N, P, (L, 0.8 * L, 1.3 * L))
    mesh.x = mesh.x @ np.array([[1.0, 0.2, 0.1], [0.0, 1.0, 0.3], [0.0, 0.0, 1.0]]).T
    return mesh


def _mixed(wfx, N, P):
    """cells duplicated in place with fresh dofs: the bricks holding one are no lattice bricks"""
    base = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    dup = np.array([3, 77, 200, 201, 450], dtype=np.int64)
    mesh = copy.copy(base)
    nd = (P + 1) ** 3
    extra = base.ndofs + np.arange(len(dup) * nd, dtype=np.int32).reshape(len(dup), nd)
    mesh.xdofs = np.concatenate([base.xdofs, base.xdofs[dup]])
    mesh.dofmap = np.concatenate([base.dofmap, extra])
    mesh.ndofs = base.ndofs + len(dup) * nd
    return mesh


A_, CC, CS = 0, 1, 4     # capi.STIFF_AUTO, STIFF_CELL_COLOUR, STIFF_CELL_STREAM
BRICK = ("brick-regular", "brick-generic")   # AUTO on small meshes: the brick kernel, whichever form the plan allows
# (id, P, N, dtype, renumber, mesh kind, mode, env, expected variant)
PATHS = [
    ("generic", 3, 4, np.float64, None, "box", A_, {"WFX_REGULAR": "0"}, "brick-generic"),
    ("regular", 3, 8, np.float64, 7, "box", A_, {}, "brick-regular"),
    ("regular-fp32", 4, 8, np.float32, None, "box", A_, {}, "brick-regular"),
    ("affine", 5, 4, np.float64, None, "sheared", A_, {}, "brick-regular"),
    ("affine-fp32", 4, 8, np.float32, None, "sheared", A_, {}, "brick-regular"),
    ("mixed", 4, 8, np.float64, None, "mixed", A_, {}, "brick-generic"),
    ("persistent", 4, 6, np.float64, 11, "box", A_, {"WFX_PERSISTENT": "1"}, "brick-regular"),
    ("p4d", 4, 6, np.float64, None, "box", A_, {"WFX_TUNED_STRIDES": "1"}, "brick-regular-p4d"),
    ("cell", 6, 2, np.float64, 5, "box", CC, {}, "cell"),
    ("brick-streamed", 5, 3, np.float64, None, "box", CS, {}, "brick-streamed"),
    ("brick-streamed-renumbered", 4, 4, np.float64, 11, "box", CS, {}, "brick-streamed"),
    ("cell-streamed-auto-p7-fp32", 7, 2, np.float32, None, "box", A_, {}, "cell-streamed"),
    ("cell-streamed-cell2", 6, 3, np.float64, None, "box", A_, {"WFX_CELL2": "1"}, "cell-streamed"),
    ("cell-streamed-cell2-renumbered", 2, 5, np.float64, 3, "box", A_, {"WFX_CELL2": "1"}, "cell-streamed"),
    ("cell-streamed-fp32", 4, 4, np.float32, None, "box", CS, {"WFX_STREAM_ORDER": "colour"}, "cell-streamed"),
]


def _path_mesh(wfx, kind, N, P, renumber):
    if kind == "sheared":
        return _sheared(wfx, N, P)
    if kind == "mixed":
        return _mixed(wfx, N, P)
    return wfx.create_box_hex(N, P, (L, L, L), perturb=0.15, renumber=renumber)


def _ref_apply(orc, mesh, P, Gs, x, dtype):
    y = np.zeros(mesh.ndofs)
    orc.stiffness_apply(mesh, P, Gs, np.ascontiguousarray(x, dtype=np.float64), y, dense=dtype == np.float64,
                        nthreads=_threads(orc))
    return y


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("P", [2, 4, 7])
def test_scaled_geometric_factors_bitwise(wfx, orc, torch, P, dtype):
    """The stored entries of the scaled G: G * coeff in fp64, float32(float64(float32(G)) * coeff) in fp32; detJ and
    the lumped mass untouched; refused coefficients leave G as it was."""
    mesh = wfx.create_box_hex(3 if P < 7 else 2, P, (L, L, L), perturb=0.15)
    Go, detJo = orc.precompute_geometric_data(mesh, P)
    coeff = coefficients(mesh.ncells, P)
    geo = wfx.Geometry(mesh, P, dtype)
    geo.scale_cells(coeff)
    G, detJ = geo.get()
    iu = np.triu_indices(3)
    if dtype == np.float64:
        want = scaled(Go, coeff)
    else:
        want = (Go.astype(np.float32).astype(np.float64) * coeff[:, None, None, None]).astype(np.float32)
    assert np.array_equal(G[:, :, iu[0], iu[1]], want[:, :, iu[0], iu[1]])
    assert np.array_equal(detJ, detJo)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJo, np.ones(mesh.ndofs), m)
    assert np.array_equal(wfx.MassOperator(mesh, P, dtype, geometry=geo).diagonal(), m.astype(dtype))
    for bad in (np.zeros(mesh.ncells), -coeff, np.where(np.arange(mesh.ncells) == 1, np.nan, coeff),
                np.where(np.arange(mesh.ncells) == mesh.ncells - 1, np.inf, coeff), coeff[:-1],
                np.concatenate([coeff, coeff[:1]])):
        with pytest.raises(wfx.WfxError):
            geo.scale_cells(bad)
        assert np.array_equal(geo.get()[0], G)


@pytest.mark.gpu
def test_scaled_geometric_factors_after_a_column_reorder(wfx, orc, torch, monkeypatch):
    """A P4 fp64 operator with the conflict-free layout reorders the geometry's G columns in place; a scale after
    that still gives G * coeff at every point, and a second scale composes."""
    monkeypatch.setenv("WFX_TUNED_STRIDES", "1")
    P = 4
    mesh = wfx.create_box_hex(6, P, (L, L, L), perturb=0.15)
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    assert op.kernel_info()["variant"] == "brick-regular-p4d"
    Go, _ = orc.precompute_geometric_data(mesh, P)
    c1, c2 = coefficients(mesh.ncells, 1), coefficients(mesh.ncells, 2)
    geo.scale_cells(c1)
    iu = np.triu_indices(3)
    assert np.array_equal(geo.get()[0][:, :, iu[0], iu[1]], scaled(Go, c1)[:, :, iu[0], iu[1]])
    geo.scale_cells(c2)
    assert np.array_equal(geo.get()[0][:, :, iu[0], iu[1]], scaled(scaled(Go, c1), c2)[:, :, iu[0], iu[1]])


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATHS, ids=[c[0] for c in PATHS])
def test_every_path_on_scaled_media(wfx, orc, torch, monkeypatch, case):
    """Each stiffness path (checked through kernel_info) with the coefficient set AFTER the operator was created:
    y = A x and (except on the simple kernel) y = (1/m) .* A x against the dense reference kernel with G * coeff;
    bitwise equal to an operator created after the scaling; and a coefficient 4 on a third geometry gives exactly
    4 times the unscaled result."""
    _, P, N, dtype, renumber, kind, mode, env, variant = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    mesh = _path_mesh(wfx, kind, N, P, renumber)
    coeff = coefficients(mesh.ncells, P + N)
    tdt = _tdt(torch, dtype)
    tol = TOL64 if dtype == np.float64 else TOL32

    geo_a = wfx.Geometry(mesh, P, dtype)
    op_a = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo_a, mode=mode)
    ki = op_a.kernel_info()
    assert ki["variant"] == variant, ki
    if kind == "sheared":
        assert ki["affine"]
    if kind == "mixed":
        assert ki["mixed"] and 0 < ki["regular_batches"] < ki["batches"]
    if "WFX_PERSISTENT" in env:
        assert op_a.info()["nlaunches"] == 1
    mass = wfx.MassOperator(mesh, P, dtype, geometry=geo_a)
    geo_a.scale_cells(coeff)

    geo_b = wfx.Geometry(mesh, P, dtype)
    geo_b.scale_cells(coeff)
    op_b = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo_b, mode=mode)
    assert op_b.kernel_info()["variant"] == variant

    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(11).standard_normal(mesh.ndofs).astype(dtype)
    want = _ref_apply(orc, mesh, P, scaled(Go, coeff), x, dtype)
    xd = dev(torch, x)
    ya, yb = (torch.full((mesh.ndofs,), float("nan"), dtype=tdt, device="cuda") for _ in range(2))
    op_a.apply(xd, ya, beta=0)
    op_b.apply(xd, yb, beta=0)
    assert rel_l2(ya.cpu().numpy(), want) < tol, rel_l2(ya.cpu().numpy(), want)
    assert torch.equal(ya, yb)
    if mode != CC:                                       # the simple kernel has no fused scaling
        inv = mass.inverse_diagonal_ptr()
        op_a.apply_scaled(xd, inv, ya)
        op_b.apply_scaled(xd, inv, yb)
        assert rel_l2(ya.cpu().numpy(), want / mass.diagonal().astype(np.float64)) < tol
        assert torch.equal(ya, yb)

    geo_c = wfx.Geometry(mesh, P, dtype)
    op_c = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo_c, mode=mode)
    y1, y4 = (torch.full((mesh.ndofs,), float("nan"), dtype=tdt, device="cuda") for _ in range(2))
    op_c.apply(xd, y1, beta=0)
    geo_c.scale_cells(np.full(mesh.ncells, 4.0))
    op_c.apply(xd, y4, beta=0)
    assert torch.equal(y4, 4 * y1)


@pytest.mark.gpu
@pytest.mark.parametrize("P,N,dtype,renumber,env,variant", [
    (3, 4, np.float64, None, {}, BRICK),                            # the ensemble's own plan
    (4, 3, np.float64, 9, {"WFX_REGULAR": "0"}, ("brick-generic",)),  # own plan, renumbered dofs
    (5, 3, np.float64, None, {"WFX_CELL2": "1"}, ("cell-streamed",)),  # the shared colour plan and its G copy
    (7, 2, np.float32, None, {}, ("cell-streamed",)),               # P7 fp32 AUTO: the shared plan
])
def test_apply_ensemble_on_scaled_media(wfx, orc, torch, monkeypatch, P, N, dtype, renumber, env, variant):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15, renumber=renumber)
    coeff = coefficients(mesh.ncells, 20 + P)
    tdt = _tdt(torch, dtype)
    tol = TOL64 if dtype == np.float64 else TOL32
    geo_a = wfx.Geometry(mesh, P, dtype)
    op_a = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo_a, ensemble=True)
    assert op_a.kernel_info()["variant"] in variant
    mass = wfx.MassOperator(mesh, P, dtype, geometry=geo_a)
    geo_a.scale_cells(coeff)
    geo_b = wfx.Geometry(mesh, P, dtype)
    geo_b.scale_cells(coeff)
    op_b = wfx.StiffnessOperator(mesh, P, dtype=dtype, geometry=geo_b, ensemble=True)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    Gs = scaled(Go, coeff)
    X = np.random.default_rng(P).standard_normal((mesh.ndofs, 8)).astype(dtype)
    KX = np.stack([_ref_apply(orc, mesh, P, Gs, X[:, m], dtype) for m in range(8)], axis=1)
    minv = 1.0 / mass.diagonal().astype(np.float64)
    for nv in (1, 3, 8):
        Xd = dev(torch, X[:, :nv])
        Ya, Yb = (torch.full((mesh.ndofs, nv), float("nan"), dtype=tdt, device="cuda") for _ in range(2))
        op_a.apply_ensemble(Xd, Ya, beta=0)
        op_b.apply_ensemble(Xd, Yb, beta=0)
        assert rel_l2(Ya.cpu().numpy(), KX[:, :nv]) < tol, nv
        assert torch.equal(Ya, Yb), nv
        op_a.apply_ensemble(Xd, Ya, beta=0, scale_ptr=mass.inverse_diagonal_ptr())
        op_b.apply_ensemble(Xd, Yb, beta=0, scale_ptr=mass.inverse_diagonal_ptr())
        assert rel_l2(Ya.cpu().numpy(), KX[:, :nv] * minv[:, None]) < tol, nv
        assert torch.equal(Ya, Yb), nv


@pytest.mark.gpu
@pytest.mark.parametrize("streamed", [False, True])
def test_interface_interior_parts_on_scaled_media(wfx, orc, torch, monkeypatch, streamed):
    """The distributed-mesh schedule on one GPU (an artificial rank-shared lattice plane), brick and streamed
    kernels, scaled after creation: the interface part completes the shared dofs, both parts the whole apply."""
    if streamed:
        monkeypatch.setenv("WFX_CELL2", "1")
    P, N = 4, 6
    mesh = copy.copy(wfx.create_box_hex(N, P, (L, L, L), perturb=0.15))
    M = P * N + 1
    shared = (np.arange(M * M) + (M // 2) * M * M).astype(np.int32)
    mesh.halo = {"send_indices": shared, "recv_indices": np.zeros(0, dtype=np.int32)}
    coeff = coefficients(mesh.ncells, 31)
    geo = wfx.Geometry(mesh, P)
    op = wfx.StiffnessOperator(mesh, P, geometry=geo)
    assert (op.kernel_info()["variant"] == "brick-streamed") == streamed
    geo.scale_cells(coeff)
    geo_b = wfx.Geometry(mesh, P)
    geo_b.scale_cells(coeff)
    op_b = wfx.StiffnessOperator(mesh, P, geometry=geo_b)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    x = np.random.default_rng(5).standard_normal(mesh.ndofs)
    kx = _ref_apply(orc, mesh, P, scaled(Go, coeff), x, np.float64)
    xd = dev(torch, x)
    y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
    op.apply_part(xd, y, 0)
    assert rel_l2(y.cpu().numpy()[shared], kx[shared]) < TOL64
    op.apply_part(xd, y, 1)
    assert rel_l2(y.cpu().numpy(), kx) < TOL64
    yb = torch.full_like(y, float("nan"))
    op_b.apply_part(xd, yb, 0)
    op_b.apply_part(xd, yb, 1)
    assert torch.equal(y, yb)


@pytest.mark.gpu
def test_two_operators_on_one_geometry(wfx, orc, torch, monkeypatch):
    """A colour-ordered streamed operator (private G copy in relabelled axes, with the ensemble path on its plan),
    then a conflict-free-layout operator that reorders the shared geometry's columns in place: the first operator's
    results do not change, and a coefficient set after both exist reaches both."""
    P, N = 4, 6
    mesh = wfx.create_box_hex(N, P, (L, L, L), perturb=0.15)
    geo = wfx.Geometry(mesh, P)
    monkeypatch.setenv("WFX_STREAM_ORDER", "colour")
    op1 = wfx.StiffnessOperator(mesh, P, geometry=geo, mode=wfx.capi.STIFF_CELL_STREAM, ensemble=True)
    assert op1.kernel_info()["variant"] == "cell-streamed"
    monkeypatch.delenv("WFX_STREAM_ORDER")
    rng = np.random.default_rng(4)
    x = rng.standard_normal(mesh.ndofs)
    X = rng.standard_normal((mesh.ndofs, 3))
    xd, Xd = dev(torch, x), dev(torch, X)

    def run(op):
        y = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64, device="cuda")
        op.apply(xd, y, beta=0)
        return y

    def run_ens(op):
        Y = torch.full(X.shape, float("nan"), dtype=torch.float64, device="cuda")
        op.apply_ensemble(Xd, Y, beta=0)
        return Y

    y1, Y1 = run(op1), run_ens(op1)
    monkeypatch.setenv("WFX_TUNED_STRIDES", "1")
    op2 = wfx.StiffnessOperator(mesh, P, geometry=geo)
    assert op2.kernel_info()["variant"] == "brick-regular-p4d"
    assert torch.equal(run(op1), y1) and torch.equal(run_ens(op1), Y1)
    Go, _ = orc.precompute_geometric_data(mesh, P)
    assert rel_l2(y1.cpu().numpy(), _ref_apply(orc, mesh, P, Go, x, np.float64)) < TOL64
    coeff = coefficients(mesh.ncells, 41)
    geo.scale_cells(coeff)
    Gs = scaled(Go, coeff)
    want = _ref_apply(orc, mesh, P, Gs, x, np.float64)
    for op in (op1, op2):
        assert rel_l2(run(op).cpu().numpy(), want) < TOL64, op.kernel_info()
    Ys = run_ens(op1).cpu().numpy()
    for m in range(3):
        assert rel_l2(Ys[:, m], _ref_apply(orc, mesh, P, Gs, X[:, m], np.float64)) < TOL64
    # an operator destroyed before the next scale leaves nothing behind that the scale would touch
    del op1
    geo.scale_cells(np.full(mesh.ncells, 0.5))
    assert rel_l2(run(op2).cpu().numpy(), 0.5 * want) < TOL64


# ---- models, scaled after construction (the Python route) --------------------------------------------------------
def _model_inputs(orc, mesh, P):
    G, detJ = orc.precompute_geometric_data(mesh, P)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    m1, m2 = orc.boundary_facet_mass(mesh, P)
    return G, m, m1, m2


def _make_model(wfx, name, mesh, P, dtype, mode):
    if name == "linear":
        return wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, stiffness_mode=mode)
    if name == "lossy":
        return wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, DELTA, dtype=dtype, stiffness_mode=mode)
    return wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype, stiffness_mode=mode)


MODEL_CASES = [  # (P, dtype, stiffness mode, graph replay, expected variants)
    (4, np.float64, A_, True, BRICK),
    (3, np.float64, CS, False, ("brick-streamed",)),
    (7, np.float32, A_, True, ("cell-streamed",)),
    (5, np.float32, CS, False, ("brick-streamed",)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", MODEL_CASES, ids=[f"P{c[0]}-{np.dtype(c[1]).name}-{c[4][0]}-graph{int(c[3])}"
                                                   for c in MODEL_CASES])
@pytest.mark.parametrize("model", list(MODELS))
def test_models_on_scaled_media(wfx, orc, mo, torch, monkeypatch, model, case):
    """Linear, lossy and Westervelt RK4 from a random state with a shortened last step, the geometry scaled after
    the model was built, against the restatement with G * coeff.  dt from the largest wave speed."""
    P, dtype, mode, graph, variant = case
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    coeff = coefficients(mesh.ncells, 50 + P)
    eqn = _make_model(wfx, model, mesh, P, dtype, mode)
    assert eqn.stiff_op.kernel_info()["variant"] in variant
    eqn.geometry.scale_cells(coeff)
    G, m, m1, m2 = _model_inputs(orc, mesh, P)
    dt = wfx.cfl_timestep(mesh.h_min, C0 * np.sqrt(coeff.max()), P, F0)
    rng = np.random.default_rng(P)
    u = (P0 * rng.standard_normal(mesh.ndofs)).astype(dtype).astype(np.float64)
    v = (P0 * 2 * np.pi * F0 * rng.standard_normal(mesh.ndofs)).astype(dtype).astype(np.float64)
    t0, steps = 5e-6, 12
    tf = t0 + (steps - 0.5) * dt
    uo, vo = u.copy(), v.copy()
    so, to = mo.rk4_westervelt(mesh, P, scaled(G, coeff), m, m1, m2, C0, F0, P0, *MODELS[model], t0, tf, dt, uo, vo,
                               sumfact=True, nthreads=_threads(orc))
    eqn.set_state(u, v)
    s, t = eqn.rk4(t0, tf, dt)
    ug, vg = eqn.get_state()
    assert (s, t) == (so, to) and s == steps
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    assert rel_l2(ug, uo) < tol and rel_l2(vg, vo) < tol, (rel_l2(ug, uo), rel_l2(vg, vo))


@pytest.mark.gpu
@pytest.mark.parametrize("P,dtype,mode,variant", [(4, np.float64, A_, BRICK),
                                                  (4, np.float64, CS, ("brick-streamed",)),
                                                  (7, np.float32, A_, ("cell-streamed",))])
def test_ensemble_model_on_scaled_media(wfx, orc, torch, P, dtype, mode, variant):
    """LinearGLLEnsemble on a geometry scaled after construction: every member equals a single-field model scaled
    the same way (P7 fp32: the ensemble shares the streamed operator's plan and G copy)."""
    f0s, p0s = (0.5e6, 0.3e6, 0.8e6), (6e4, 1e4, 3e4)
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    coeff = coefficients(mesh.ncells, 60 + P)
    n, nv = mesh.ndofs, len(f0s)
    dt = wfx.cfl_timestep(mesh.h_min, C0 * np.sqrt(coeff.max()), P, max(f0s))
    tf = 10.6 * dt
    rng = np.random.default_rng(7)
    U0, V0 = 1e-3 * rng.standard_normal((n, nv)), rng.standard_normal((n, nv))
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s, p0s, dtype=dtype, stiffness_mode=mode)
    assert ens.stiff_op.kernel_info()["variant"] in variant
    ens.geometry.scale_cells(coeff)
    ens.set_state(U0, V0)
    s, t = ens.rk4(0.0, tf, dt)
    U, V = ens.get_state()
    assert s == 11
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    G, m, m1, m2 = _model_inputs(orc, mesh, P)
    for k in range(nv):
        one = wfx.LinearGLLOpt(mesh, None, P, C0, f0s[k], p0s[k], dtype=dtype, stiffness_mode=mode)
        one.geometry.scale_cells(coeff)
        one.set_state(U0[:, k], V0[:, k])
        assert one.rk4(0.0, tf, dt) == (s, t)
        u1, v1 = one.get_state()
        assert rel_l2(U[:, k], u1.astype(np.float64)) < tol and rel_l2(V[:, k], v1.astype(np.float64)) < tol
        uo, vo = U0[:, k].astype(dtype).astype(np.float64), V0[:, k].astype(dtype).astype(np.float64)
        orc.rk4(mesh, P, scaled(G, coeff), m, m1, m2, C0, f0s[k], p0s[k], 0.0, tf, dt, uo, vo, sumfact=True)
        assert rel_l2(U[:, k], uo) < tol and rel_l2(V[:, k], vo) < tol


@pytest.mark.gpu
@pytest.mark.parametrize("P,dtype,mode,variant", [(7, np.float32, A_, "cell-streamed"),
                                                  (4, np.float64, CS, "brick-streamed")])
def test_thermal_per_cell_conductivity_on_streamed_paths(wfx, orc, mo, torch, P, dtype, mode, variant):
    """PennesGLL with a per-cell conductivity on the streamed kernels (P7 fp32 AUTO, STIFF_CELL_STREAM), both Robin
    tags and per-cell rhoC / perfusion, against the restatement with G * k / max k."""
    T_art, rhoc0, wb0 = 37.0, 3.6e6, 2.0e4
    h, T_ext = (300.0, 40.0), (20.0, 45.0)
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.015, 0.01, 0.01), perturb=0.15)
    rng = np.random.default_rng(P)
    k = 0.5 * coefficients(mesh.ncells, 70 + P)
    rhoc_c = rhoc0 * (1 + 0.4 * rng.random(mesh.ncells))
    perf_c = wb0 * rng.random(mesh.ncells)
    th = wfx.PennesGLL(mesh, P, k, rhoc_c, perf_c, T_art, h, T_ext, dtype=dtype, stiffness_mode=mode)
    assert th.stiff_op.kernel_info()["variant"] == variant
    G, m, m1, m2 = _model_inputs(orc, mesh, P)
    args = (mesh, P, scaled(G, k / th.k), m, m1, m2, th.k, th.rhoc, th.perf, T_art, h, T_ext)
    Q = 3e6 * rng.random(mesh.ndofs)
    th.set_heat_source(Q)
    theta0 = (4.0 + 5.0 * rng.random(mesh.ndofs)).astype(dtype).astype(np.float64)
    dt = 0.5 * th.max_eigenvalue(300)[1]
    tf = 15.4 * dt
    th.set_state(T_art + theta0)
    steps, t_end = th.rk4(0.0, tf, dt)
    u, cem, mx = theta0.copy(), np.zeros(mesh.ndofs), np.full(mesh.ndofs, -np.inf)
    so, to = mo.rk4_pennes(*args, Q, 1.0, 0.0, tf, dt, u, cem, mx, sumfact=True, nthreads=_threads(orc))
    assert (steps, t_end) == (so, to) == (16, to)
    rel = lambda a, b: np.abs(np.asarray(a, dtype=np.float64) - b).max() / np.abs(b).max()  # noqa: E731
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    d = th.dose()
    assert rel(th.rise(), u) <= tol and rel(d.cem43, cem) <= tol and rel(d.T_max - T_art, mx) <= tol


@pytest.mark.gpu
def test_two_layer_mode_decays_like_a_damped_oscillator(wfx, torch):
    """The lossy model from the exact two-layer mode with v = 0.  With delta_eff = delta * coeff the damping term
    is (delta / c_ref^2) div(c^2 grad p_t), so the mode's projection follows a'' + delta lam a' + c_ref^2 lam a = 0
    with lam = w^2 / c_ref^2 (from the GPU operators; the CPU test pins it to the exact w).  Bounds: see
    KNOWN_BOUNDS, measured on the restatement, which the GPU matches to 1e-12."""
    mesh, P, coeff, w, u0 = two_layer_case(wfx)
    dt, nsteps, delta = wfx.cfl_timestep(mesh.h_min, C2, P, F0), 1500, 0.72
    eqn = wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, delta)
    eqn.geometry.scale_cells(coeff)
    mdiag = eqn.mass_op.diagonal()
    y = torch.zeros(mesh.ndofs, dtype=torch.float64, device="cuda")
    eqn.stiff_op.apply(dev(torch, u0), y, beta=0)           # y = -c_ref^2 K_c u0
    nrm = u0 @ (mdiag * u0)
    lam = -(u0 @ y.cpu().numpy()) / C0 ** 2 / nrm
    assert abs(lam / (w / C0) ** 2 - 1) < KNOWN_BOUNDS["rayleigh"]
    g = delta * lam / 2
    wd = np.sqrt(C0 ** 2 * lam - g ** 2)
    eqn.set_state(u0, np.zeros(mesh.ndofs))
    assert eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)[0] == nsteps
    u, v = eqn.get_state()
    T = nsteps * dt
    a, ad = (u @ (mdiag * u0)) / nrm, (v @ (mdiag * u0)) / nrm
    env = lambda a_, ad_: a_ * a_ + ((ad_ + g * a_) / wd) ** 2  # noqa: E731
    g_meas = -np.log(env(a, ad) / env(1.0, 0.0)) / (2 * T)
    assert np.exp(-g * T) < 0.8                              # a visible loss of amplitude
    assert abs(g_meas / g - 1) < KNOWN_BOUNDS["decay"], (g_meas, g)
    a_exact = np.exp(-g * T) * (np.cos(wd * T) + g / wd * np.sin(wd * T))
    assert abs(a - a_exact) < KNOWN_BOUNDS["phase"] * np.exp(-g * T)
