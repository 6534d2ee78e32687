"""Volume sources (DESIGN.md section 4.5h): an additive pressure source on any dofs,

    b_j += c0^2 q_j g(t - tau_j),   g = 0 before the delay,

added at every stage after the boundary term and before the layer, Gamma2 and stage-quotient terms.  For a point source
q_j = phi_j(x0) (point_source).

CPU: the restatement (model_oracle wo_*_westervelt_source) against a textbook RK4 of the augmented system and, without a
source, against wo_rk4_westervelt_pml bit for bit; point_source weights; phase_conjugate_delays; discrete reciprocity.
GPU: every model against the restatement, the bitwise identities, reciprocity on the device, the free-space Green's
function, time-reversal focusing through a bone slab, refusals, the demo and the C++ wrapper.
"""
import importlib.util
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL64 = 1e-12
TOL32_RUN = 1e-4
C0, F0, P0 = 1500.0, 0.5e6, 6e4
DELTA, BETA, RHO0 = 1e-2, 900.0, 1000.0
KAPPA = 2.0 * BETA / (RHO0 * C0 * C0)


def _helpers():
    """the restatement's input builders of the layer's tests (tests/test_pml.py), loaded by path"""
    spec = importlib.util.spec_from_file_location("_pml_helpers", os.path.join(ROOT, "tests", "test_pml.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


H = _helpers()
rel_l2 = H.rel_l2


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


def _no_relax(mesh):
    return np.zeros(0), np.zeros((0, mesh.ndofs))


def _source_dofs(mesh, zeta, m1, rng, kinds=("interior", "tag1", "layer"), m2=None):
    """one dof of each kind: off every boundary and layer, on tag 1, on tag 2 (Gamma2, absorbing), in the layer"""
    x = __import__("wave_fenics_b200").dof_coordinates(mesh)
    lo, hi = x.min(0), x.max(0)
    inner = np.all((x > lo + 1e-12) & (x < hi - 1e-12), axis=1) & ~np.any(zeta > 0, axis=0)
    pick = dict(interior=np.nonzero(inner)[0], tag1=np.nonzero(m1 > 0)[0], layer=np.nonzero(np.any(zeta > 0, 0))[0],
                tag2=np.nonzero(m2 > 0)[0] if m2 is not None else None)
    return np.array([rng.choice(pick[k]) for k in kinds], dtype=np.int32)


# ---- CPU: the restatement ------------------------------------------------------------------------------------------
TEXTBOOK = [(2, "linear", 0), (3, "lossy", 1), (4, "westervelt", 2)]


@pytest.mark.parametrize("case", TEXTBOOK, ids=[f"P{c[0]}-{c[1]}-M{c[2]}" for c in TEXTBOOK])
def test_restatement_matches_textbook_rk4(wfx, orc, mo, case):
    """wo_rk4_westervelt_source against a textbook RK4 of the augmented system (dense stiffness, dense physical
    gradients, a random medium, relaxation, both tags, a layer on three faces), with sources on an interior, a tag-1 and
    a layer dof, random weights and delays that start the sources inside the run"""
    P, kind, M = case
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.15)
    med = H.random_medium(wfx, mesh.ncells, 11 + P, beta=kind == "westervelt")
    G, m, m1, m2, mu, detJ = H.weighted_inputs(orc, mo, mesh, P, med)
    kap = med.kappa(mesh, detJ, C0) if kind == "westervelt" else np.zeros(mesh.ndofs)
    delta = 0.0 if kind == "linear" else DELTA
    if M:
        rel = H.random_relaxation(wfx, mesh.ncells, M, 3)
        eps, tau = rel.eps_dofs(mesh, detJ, mu), rel.tau
    else:
        tau, eps = _no_relax(mesh)
    pml = wfx.PML.box(mesh, 0.011, [(0, 1), (1, 0), (2, 1)], C0)
    zeta = pml.zeta
    sw = med.stiffness_weight(mesh.ncells)
    inp = H.pml_inputs(orc, mo, mesh, P, zeta, sw)
    A = H.dense_stiffness(orc, mesh, P, G)
    Gr, dJw = H.first_principles_gradients(orc, mesh, P)
    perm = orc.perm(P)
    cell_on = np.array([np.any(zeta[:, mesh.dofmap[c]] > 0) for c in range(mesh.ncells)])
    dof_on = np.zeros(mesh.ndofs, dtype=bool)
    dof_on[mesh.dofmap[cell_on].reshape(-1)] = True
    Gr = Gr * cell_on[:, None, None, None]
    zq = zeta[:, mesh.dofmap[:, perm]].transpose(1, 2, 0)
    g1 = np.stack([zq[..., 1] + zq[..., 2] - zq[..., 0], zq[..., 0] + zq[..., 2] - zq[..., 1],
                   zq[..., 0] + zq[..., 1] - zq[..., 2]], -1)
    g2 = np.stack([zq[..., 1] * zq[..., 2], zq[..., 0] * zq[..., 2], zq[..., 0] * zq[..., 1]], -1)
    a = 1500.0 ** 2 * sw[:, None, None]
    z1, z2, z3 = zeta.sum(0), zeta[0] * zeta[1] + zeta[0] * zeta[2] + zeta[1] * zeta[2], zeta.prod(0)
    s = delta / 1500.0 ** 2
    rng = np.random.default_rng(P)
    sdofs = _source_dofs(mesh, zeta, m1, rng)
    dt = 0.5 * min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), pml.max_dt())
    t0, nsteps = 1.0e-6, 6
    sq = rng.uniform(0.2, 1.0, len(sdofs)) * rng.choice([-1, 1], len(sdofs))
    sdel = np.array([0.0, t0 + 1.3 * dt, t0 + 3.6 * dt])   # the last two start during the run

    def src(t):
        out = np.zeros(mesh.ndofs)
        for j, qj, tj in zip(sdofs, sq, sdel):
            if t - tj >= 0:
                out[j] = C0 ** 2 * qj * mo.source(t - tj, F0, P0, C0)[0]
        return out

    def rhs(t, p, pd, q, psi, phi):
        kq = (eps * p - q) / tau[:, None]
        R = ((eps * pd - kq) / tau[:, None]).sum(0)
        g, gd = mo.source(t, F0, P0, C0)
        grad = lambda f: np.einsum("cqld,d->cql", Gr, f)  # noqa: E731
        dtphi = -np.einsum("cqld,cql->d", Gr, dJw[..., None] * phi)
        layer = np.where(dof_on, dtphi - m * (z1 * pd + z2 * p + z3 * psi), 0.0)
        num = (A @ p + s * (A @ pd) + (C0 ** 2 * g + delta * gd) * m1 - C0 * m2 * pd + src(t) + layer
               + kap * m * pd ** 2 - m * R)
        kphi = a * (g1 * grad(p + s * pd) + g2 * grad(psi + s * p)) - zq * phi
        kphi = kphi * cell_on[:, None, None]
        return pd, num / (m * (1.0 - kap * p) + delta / C0 * m2), kq, np.where(dof_on, p, 0.0), kphi

    n = mesh.ndofs
    p, pd = 0.1 * P0 * rng.standard_normal(n), 0.1 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)
    q = eps * p * rng.uniform(0.5, 1.5, eps.shape)
    psi = np.where(dof_on, p * rng.uniform(0.5, 1.5, n) / (2 * np.pi * F0), 0.0)
    phi = a * np.einsum("cqld,d->cql", Gr, p) * rng.uniform(0.5, 1.5, (mesh.ncells, len(perm), 3)) / pml.zeta_max
    st = [x.copy() for x in (p, pd, q, psi, phi)]
    steps, _ = mo.rk4_westervelt_source(mesh, P, G, m, m1, m2, kap, C0, F0, P0, delta, tau, eps, inp, sdofs, sq, sdel,
                                        t0, 1.0, dt, *st, max_steps=nsteps)
    assert steps == nsteps
    y, t = [p, pd, q, psi, phi], t0
    for _ in range(nsteps):
        k1 = rhs(t, *y)
        k2 = rhs(t + dt / 2, *[x + dt / 2 * k for x, k in zip(y, k1)])
        k3 = rhs(t + dt / 2, *[x + dt / 2 * k for x, k in zip(y, k2)])
        k4 = rhs(t + dt, *[x + dt * k for x, k in zip(y, k3)])
        y = [x + dt / 6 * (a_ + 2 * b_ + 2 * c_ + d_) for x, a_, b_, c_, d_ in zip(y, k1, k2, k3, k4)]
        t += dt
    errs = [rel_l2(o, e) for o, e in zip(st, y) if np.any(e)]
    assert max(errs) < 1e-13, errs
    tf1 = t0 + 2.2 * dt
    fo = mo.f1_westervelt_source(mesh, P, G, m, m1, m2, kap, C0, F0, P0, delta, tau, eps, inp, sdofs, sq, sdel, tf1,
                                 *y)
    assert rel_l2(fo, rhs(tf1, *y)[1]) < 1e-13
    # the source matters at this bound: the same run without it is far off
    st0 = [x.copy() for x in (p, pd, q, psi, phi)]
    mo.rk4_westervelt_pml(mesh, P, G, m, m1, m2, kap, C0, F0, P0, delta, tau, eps, inp, t0, 1.0, dt, *st0,
                          max_steps=nsteps)
    assert rel_l2(st0[1], y[1]) > 1e3 * max(errs)


def test_restatement_without_a_source_is_the_layer_restatement_bitwise(wfx, orc, mo):
    P = 2
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = H.random_medium(wfx, mesh.ncells, 9)
    G, m, m1, m2, mu, detJ = H.weighted_inputs(orc, mo, mesh, P, med)
    kap = med.kappa(mesh, detJ, C0)
    pml = wfx.PML.box(mesh, 0.011, [(0, 1), (1, 0)], C0)
    inp = H.pml_inputs(orc, mo, mesh, P, pml.zeta, med.stiffness_weight(mesh.ncells))
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), pml.max_dt())
    rng = np.random.default_rng(2)
    u, v = 0.3 * P0 * rng.standard_normal(mesh.ndofs), 1e6 * rng.standard_normal(mesh.ndofs)
    for M in (0, 2):
        rel = H.random_relaxation(wfx, mesh.ncells, M, 1) if M else None
        tau = rel.tau if M else np.zeros(0)
        eps = rel.eps_dofs(mesh, detJ, mu) if M else np.zeros((0, mesh.ndofs))
        runs = []
        for fn, extra in ((mo.rk4_westervelt_pml, ()), (mo.rk4_westervelt_source, (None, None, None))):
            st = [u.copy(), v.copy(), np.zeros((M, mesh.ndofs)), *mo.pml_state(mesh, P)]
            r = fn(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, tau, eps, inp, *extra, 1e-6, 1e-6 + 9.5 * dt, dt, *st)
            runs.append((r, st))
        assert runs[0][0] == runs[1][0]
        assert all(np.array_equal(a, b) for a, b in zip(runs[0][1], runs[1][1])), M


# ---- CPU: point_source and phase_conjugate_delays ------------------------------------------------------------------
@pytest.mark.parametrize("P", [2, 4])
def test_point_source_weights(wfx, P):
    """sum q = 1 and sum q_j x_j = x0 (the trilinear map lies in Q_P), on a perturbed mesh"""
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.2)
    x = wfx.dof_coordinates(mesh)
    rng = np.random.default_rng(P)
    for _ in range(12):
        x0 = rng.uniform((0, 0, 0), (0.03, 0.03, 0.02))
        dofs, q = wfx.point_source(mesh, x0)
        assert dofs.dtype == np.int32 and np.all(np.diff(dofs) > 0)
        assert abs(q.sum() - 1.0) < 1e-14
        assert np.abs(q @ x[dofs] - x0).max() < 1e-14 * 0.03
    # a point at a dof: weight 1 there and nothing else
    for j in rng.choice(mesh.ndofs, 10, replace=False):
        dofs, q = wfx.point_source(mesh, x[j])
        assert list(dofs) == [j] and q[0] == 1.0


def test_point_source_on_shared_faces_edges_and_vertices(wfx):
    """either cell that holds the point gives the same weights"""
    from wave_fenics_b200 import operators as ops
    P = 3
    mesh = wfx.create_box_hex((2, 2, 2), P, (0.02, 0.02, 0.02), perturb=0.2)
    xv = mesh.x
    centre = [v for v in range(len(xv)) if np.all(np.abs(xv[v] - 0.01) < 0.004)][0]   # the interior vertex
    cells = [c for c in range(mesh.ncells) if centre in mesh.xdofs[c]]
    assert len(cells) == 8
    # a vertex (8 cells), an edge midpoint and a face point (from the trilinear map of one cell)
    c0 = cells[0]
    loc = list(mesh.xdofs[c0]).index(centre)
    b = np.array([(loc >> a) & 1 for a in range(3)], dtype=float)
    edge = b.copy()
    edge[0] = 0.37
    face = b.copy()
    face[:2] = (0.29, 0.61)
    for xi in (b, edge, face):
        x0, _ = ops._trilinear(xv[mesh.xdofs[c0]], xi)
        got = []
        for c in cells:
            r = ops._locate_in_cell(mesh, c, x0)
            if r is None:
                continue
            d, w = ops._cell_weights(mesh, c, r)
            got.append({int(k): v for k, v in zip(d, w) if v != 0.0})
        assert len(got) >= 2
        for g in got[1:]:
            assert set(g) == set(got[0])
            assert max(abs(g[k] - got[0][k]) for k in g) < 1e-13
        ref = wfx.point_source(mesh, x0)
        assert {int(k): v for k, v in zip(*ref)}.keys() == got[0].keys()


def test_point_source_refuses_points_outside_the_mesh(wfx):
    mesh = wfx.create_box_hex((2, 2, 2), 2, (0.02, 0.02, 0.02), perturb=0.1)
    for x0 in ((0.021, 0.01, 0.01), (-1e-6, 0.0, 0.0), (0.01, 0.01, 0.5)):
        with pytest.raises(wfx.WfxError, match="outside"):
            wfx.point_source(mesh, x0)
    wfx.point_source(mesh, (0.02, 0.02, 0.02))   # the far corner is inside


def test_phase_conjugate_delays(wfx):
    rng = np.random.default_rng(1)
    p = rng.standard_normal(50) + 1j * rng.standard_normal(50)
    tau = wfx.phase_conjugate_delays(p, F0)
    assert tau.shape == p.shape and np.all(tau >= 0) and np.all(tau < 1 / F0)
    # firing with them aligns every phase: arg(p e^{-i w tau}) = 0
    assert np.abs(np.angle(p * np.exp(-2j * np.pi * F0 * tau))).max() < 1e-12
    f = np.array([F0, 2 * F0, 0.7 * F0])
    pe = rng.standard_normal((20, 3)) + 1j * rng.standard_normal((20, 3))
    te = wfx.phase_conjugate_delays(pe, f)
    assert te.shape == pe.shape and np.all(te < 1 / f)
    assert np.abs(np.angle(pe * np.exp(-2j * np.pi * f * te))).max() < 1e-12


# ---- CPU: discrete reciprocity -------------------------------------------------------------------------------------
# Every linear model here has a symmetric transfer function (DESIGN.md section 4.5h), so the probe series at dof B under
# a unit source at A is the series at A under a unit source at B, step by step.  Measured on the restatement (fp64, P2,
# 60 steps, max |difference| / max |series|): 9.2e-14 without a layer, 2.8e-15 to 4.8e-13 with one, and 5.5e-14 between
# a tag-1 dof and a volume source.  That is roundoff: without a layer, the sum-factorised and the dense stiffness give
# series 6.3e-14 apart; with one, the run under a source scaled by 3 (series divided by 3) is 2.8e-13 from the unscaled
# run.  Bound 2e-12.
RECIP_STEPS = 60
RECIP_TOL = 2e-12
# fp32 on the device (max |difference| / max |series| over the same 60 steps): 1.1e-4 to 2.0e-4, fp32 roundoff
# (2^-24 = 6e-8) grown over the run; bound 5e-4
RECIP_TOL32 = 5e-4
RECIP = [("linear", 0, False), ("lossy", 0, True), ("lossy", 2, True), ("linear", 0, True)]


def _recip_setup(wfx, orc, mo, P, kind, M, with_pml, seed=5):
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.15)
    med = H.random_medium(wfx, mesh.ncells, 21 + seed, beta=False)
    G, m, m1, m2, mu, detJ = H.weighted_inputs(orc, mo, mesh, P, med)
    if M:
        rel = H.random_relaxation(wfx, mesh.ncells, M, 3)
        tau, eps = rel.tau, rel.eps_dofs(mesh, detJ, mu)
    else:
        rel, (tau, eps) = None, _no_relax(mesh)
    pml = wfx.PML.box(mesh, 0.011, [(0, 1), (1, 0)], C0) if with_pml else wfx.PML(mesh, np.zeros((3, mesh.ndofs)))
    inp = H.pml_inputs(orc, mo, mesh, P, pml.zeta, med.stiffness_weight(mesh.ncells))
    delta = DELTA if kind == "lossy" else 0.0
    dts = [wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)] + ([pml.max_dt()] if with_pml else [])
    if M:
        dts.append(rel.max_dt())
    return mesh, med, pml, (G, m, m1, m2, np.zeros(mesh.ndofs), C0, F0, P0, delta, tau, eps, inp), min(dts)


def _recip_series(mo, mesh, P, args, sdofs, sq, probe, dt, nsteps, m1=None):
    """u[probe] after every step of a run from rest under the volume source (sdofs, sq); m1 replaces the tag-1 mass"""
    a = list(args)
    if m1 is not None:
        a[2] = m1
    M = a[10].shape[0]
    st = [np.zeros(mesh.ndofs), np.zeros(mesh.ndofs), np.zeros((M, mesh.ndofs)), *mo.pml_state(mesh, P)]
    out, t = [], 0.0
    for _ in range(nsteps):
        _, t = mo.rk4_westervelt_source(mesh, P, *a, sdofs, sq, None, t, 1.0, dt, *st, max_steps=1, sumfact=True)
        out.append(st[0][probe])
    return np.array(out)


@pytest.mark.parametrize("case", RECIP, ids=[f"{c[0]}-M{c[1]}-pml{int(c[2])}" for c in RECIP])
def test_reciprocity_on_the_restatement(wfx, orc, mo, case):
    kind, M, with_pml = case
    P = 2
    mesh, med, pml, args, dt = _recip_setup(wfx, orc, mo, P, kind, M, with_pml)
    rng = np.random.default_rng(7)
    A, B = _source_dofs(mesh, pml.zeta if with_pml else np.zeros((3, mesh.ndofs)), args[2], rng,
                        ("interior", "layer" if with_pml else "interior"))
    args = list(args)
    args[2] = np.zeros(mesh.ndofs)                 # no tag-1 source: the volume sources alone
    ab = _recip_series(mo, mesh, P, args, [A], [1.0], B, dt, RECIP_STEPS)
    ba = _recip_series(mo, mesh, P, args, [B], [1.0], A, dt, RECIP_STEPS)
    scale = np.abs(ab).max()
    assert scale > 0
    assert np.abs(ab - ba).max() < RECIP_TOL * scale, np.abs(ab - ba).max() / scale


def test_reciprocity_between_tag1_and_a_volume_source_on_the_restatement(wfx, orc, mo):
    """the tag-1 term of dof i alone (profile amplitude 1 there, 0 elsewhere) against a volume source q = m1_i at B"""
    P = 2
    mesh, med, pml, args, dt = _recip_setup(wfx, orc, mo, P, "linear", 0, True)
    m1 = args[2]
    rng = np.random.default_rng(3)
    i, B = _source_dofs(mesh, pml.zeta, m1, rng, ("tag1", "interior"))
    only_i = np.where(np.arange(mesh.ndofs) == i, m1, 0.0)
    s1 = _recip_series(mo, mesh, P, args, [], [], B, dt, RECIP_STEPS, m1=only_i)
    s2 = _recip_series(mo, mesh, P, args, [B], [m1[i]], i, dt, RECIP_STEPS, m1=np.zeros(mesh.ndofs))
    scale = np.abs(s1).max()
    assert scale > 0 and np.abs(s1 - s2).max() < RECIP_TOL * scale, np.abs(s1 - s2).max() / scale


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


GPU_MESH = H.GPU_MESH
GPU_FACES = H.GPU_FACES


def _sources(wfx, mesh, eqn, pml, seed, nv=None, scale=1e-5):
    """a point source at a random interior point plus sources on a tag-1, a tag-2 (Gamma2: the term must be divided by
    m + q there) and a layer dof, random weights (a column per
    member for nv) and delays over two periods.  The weights are scaled by `scale`: a unit point source of this g gives
    GPa next to the point, far outside the Westervelt model's range (kappa p < 1)"""
    rng = np.random.default_rng(seed)
    x = wfx.dof_coordinates(mesh)
    lo, hi = x.min(0), x.max(0)
    dofs, q = wfx.point_source(mesh, lo + rng.uniform(0.3, 0.7, 3) * (hi - lo))
    m1, m2 = eqn.bnd_op.facet_masses()
    extra = _source_dofs(mesh, pml.zeta, m1, rng, ("tag1", "tag2", "layer"), m2)
    extra = extra[~np.isin(extra, dofs)]
    dofs = np.concatenate([dofs, extra]).astype(np.int32)
    q = np.concatenate([q, rng.uniform(-1, 1, len(extra))])
    shape = (len(dofs),) if nv is None else (len(dofs), nv)
    q = scale * q
    if nv is not None:
        q = q[:, None] * rng.uniform(0.5, 1.5, shape)
    delay = rng.uniform(0, 2 / F0, shape)
    delay[0] = 0.0
    return dofs, q, delay


PARITY = [
    (2, np.float64, True, 0, "linear"), (3, np.float64, False, 0, "linear"), (3, np.float64, True, 2, "lossy"),
    (4, np.float64, True, 0, "westervelt"), (4, np.float64, False, 1, "westervelt-kd"), (5, np.float64, True, 0, "lossy"),
    (5, np.float64, False, 0, "westervelt-kd"), (4, np.float32, True, 2, "lossy"), (4, np.float32, False, 0, "linear"),
    (7, np.float32, True, 1, "westervelt-kd"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY, ids=[f"P{c[0]}-{np.dtype(c[1]).name}-graph{int(c[2])}-M{c[3]}-{c[4]}"
                                              for c in PARITY])
def test_models_with_a_volume_source_match_the_restatement(wfx, orc, mo, torch, monkeypatch, case):
    """RK4 through the sources' delays and the ramp, on a perturbed mesh in a random medium with a layer, both tags;
    u, v against the restatement; f1 against wo_f1_westervelt_source"""
    P, dtype, graph, M, name = case
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh, eqn, pml, args, dt = H._parity_case(wfx, orc, mo, P, dtype, M, name)
    dofs, q, delay = _sources(wfx, mesh, eqn, pml, P)
    eqn.set_volume_source(dofs, q, delay)
    u, v = H._random_state(mesh.ndofs, P, dtype, 0.1 if name.startswith("westervelt") else 1.0)
    t0, steps = 1.5e-6, 14
    tf = t0 + (steps - 0.5) * dt
    uo, vo, qo = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
    psio, phio = mo.pml_state(mesh, P)
    so, to = mo.rk4_westervelt_source(mesh, P, *args, dofs, q, delay, t0, tf, dt, uo, vo, qo, psio, phio, sumfact=True,
                                      nthreads=orc.max_threads())
    eqn.set_state(u, v)
    s, t = eqn.rk4(t0, tf, dt)
    ug, vg = eqn.get_state()
    assert (s, t) == (so, to) and s == steps
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    assert max(rel_l2(ug, uo), rel_l2(vg, vo)) < tol, (rel_l2(ug, uo), rel_l2(vg, vo))
    # without the source the run is far from this one
    uw, vw, qw = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
    mo.rk4_westervelt_pml(mesh, P, *args, t0, tf, dt, uw, vw, qw, *mo.pml_state(mesh, P), sumfact=True,
                          nthreads=orc.max_threads())
    assert rel_l2(vw, vo) > 100 * tol
    # f1 at a time inside the delays, at the model's state
    qs = np.ascontiguousarray(eqn.relaxation_state(), dtype=np.float64) if M else None
    psi_full, phi_full = mo.pml_state(mesh, P)
    cell_on, dof_on = H._layer_masks(mesh, pml.zeta)
    psig, phig = eqn.pml_state()
    psi_full[dof_on] = psig
    phi_full[cell_on] = phig
    tf1 = 1.3 / F0
    fo = mo.f1_westervelt_source(mesh, P, *args, dofs, q, delay, tf1, u, v, qs, psi_full, phi_full)
    res = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64 if dtype == np.float64 else torch.float32,
                     device="cuda")
    tdev = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(dtype))).cuda()  # noqa: E731
    eqn.f1(tf1, tdev(u), tdev(v), res)
    torch.cuda.synchronize()
    assert rel_l2(res.cpu().numpy(), fo) < (TOL64 if dtype == np.float64 else 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("graph", [True, False])
def test_ensembles_with_per_member_columns(wfx, orc, mo, torch, monkeypatch, dtype, graph):
    """LinearGLLEnsemble with nv = 3 members of their own f0 / p0 and a column of weights and delays each, against the
    restatement of every member; f1 of the ensemble against it"""
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    P, nv = 3, 3
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.15)
    f0s, p0s = np.array([F0, 0.8 * F0, 1.3 * F0]), np.array([P0, 2 * P0, 0.5 * P0])
    med = H.random_medium(wfx, mesh.ncells, 61, beta=False)
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, f0s, p0s, dtype=dtype, medium=med)
    no_layer = wfx.PML(mesh, np.zeros((3, mesh.ndofs)))
    dofs, q, delay = _sources(wfx, mesh, ens, wfx.PML.box(mesh, 0.011, GPU_FACES, C0), 8, nv)
    ens.set_volume_source(dofs, q, delay)
    G, m, m1, m2, mu, detJ = H.weighted_inputs(orc, mo, mesh, P, med)
    inp = H.pml_inputs(orc, mo, mesh, P, no_layer.zeta, med.stiffness_weight(mesh.ncells))
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0 * 1.3)
    rng = np.random.default_rng(4)
    U = (0.3 * P0 * rng.standard_normal((mesh.ndofs, nv))).astype(dtype).astype(np.float64)
    V = (3e5 * rng.standard_normal((mesh.ndofs, nv))).astype(dtype).astype(np.float64)
    t0, steps = 1.0e-6, 12
    ens.set_state(U, V)
    ens.rk4(t0, t0 + (steps - 0.5) * dt, dt)
    ug, _ = ens.get_state()
    tf1 = 1.7 / F0
    res = torch.empty((mesh.ndofs * nv,), dtype=torch.float64 if dtype == np.float64 else torch.float32, device="cuda")
    tdev = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(dtype)).reshape(-1)).cuda()  # noqa: E731
    ens.f1(tf1, tdev(U), tdev(V), res)
    torch.cuda.synchronize()
    f1g = res.cpu().numpy().reshape(mesh.ndofs, nv)
    tau, eps = _no_relax(mesh)
    for mm in range(nv):
        a = (G, m, m1, m2, np.zeros(mesh.ndofs), C0, f0s[mm], p0s[mm], 0.0, tau, eps, inp)
        uo, vo = U[:, mm].copy(), V[:, mm].copy()
        mo.rk4_westervelt_source(mesh, P, *a, dofs, q[:, mm], delay[:, mm], t0, t0 + (steps - 0.5) * dt, dt, uo, vo,
                                 None, *mo.pml_state(mesh, P), sumfact=True)
        tol = TOL64 if dtype == np.float64 else TOL32_RUN
        assert rel_l2(ug[:, mm], uo) < tol, mm
        fo = mo.f1_westervelt_source(mesh, P, *a, dofs, q[:, mm], delay[:, mm], tf1, np.ascontiguousarray(U[:, mm]),
                                     np.ascontiguousarray(V[:, mm]))
        assert rel_l2(f1g[:, mm], fo) < (TOL64 if dtype == np.float64 else 2e-5), mm


def _run(eqn, u, v, t0, tf, dt, max_steps=0):
    eqn.set_state(u, v)
    st = eqn.rk4(t0, tf, dt, max_steps=max_steps)
    return st, eqn.get_state()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", ["linear", "lossy", "westervelt"])
def test_no_source_a_cleared_source_and_zero_weights_are_the_model_without_one(wfx, torch, dtype, name):
    P = 3
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.1)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    u, v = H._random_state(mesh.ndofs, 3, dtype, 0.1)
    args = (u, v, 7.5e-6, 7.5e-6 + 10.5 * dt, dt)
    ref = _run(H._model(wfx, name, mesh, P, dtype, None), *args)
    dofs, q = wfx.point_source(mesh, (0.011, 0.013, 0.007))
    empty = H._model(wfx, name, mesh, P, dtype, None)
    empty.set_volume_source(np.zeros(0, dtype=np.int32), np.zeros(0))
    cleared = H._model(wfx, name, mesh, P, dtype, None)
    cleared.set_volume_source(dofs, q)
    cleared.rk4(0.0, 1.0, dt, max_steps=3)
    cleared.set_volume_source()
    zero = H._model(wfx, name, mesh, P, dtype, None)
    zero.set_volume_source(dofs, np.zeros_like(q))
    for eqn in (empty, cleared, zero):
        got = _run(eqn, *args)
        assert got[0] == ref[0]
        assert np.array_equal(got[1][0], ref[1][0]) and np.array_equal(got[1][1], ref[1][1])
    on = H._model(wfx, name, mesh, P, dtype, None)
    on.set_volume_source(dofs, q)
    assert not np.array_equal(_run(on, *args)[1][0], ref[1][0])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_a_uniform_delay_shifts_the_run(wfx, torch, dtype):
    """from rest with a silent array, delays tau = k dt on every source: after N + k steps the state of the tau = 0 run
    after N steps (the stage times differ in their last bits only)"""
    P, k, N = 3, 7, 25
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.1)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    dofs, q = wfx.point_source(mesh, (0.013, 0.009, 0.011))
    z = np.zeros(mesh.ndofs)
    out = []
    for tau, n in ((0.0, N), (k * dt, N + k)):
        eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, pml=wfx.PML.box(mesh, 0.011, GPU_FACES, C0))
        eqn.set_source_profile(np.zeros(mesh.ndofs))
        eqn.set_volume_source(dofs, q, np.full(len(dofs), tau))
        out.append(_run(eqn, z, z, 0.0, 1.0, dt, max_steps=n)[1][0].astype(np.float64))
    assert np.abs(out[0]).max() > 0
    assert rel_l2(out[1], out[0]) < (1e-10 if dtype == np.float64 else 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_repeated_runs_and_checkpoint_restarts_are_bitwise(wfx, torch, dtype):
    P = 4
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.1)
    rel = H.random_relaxation(wfx, mesh.ncells, 2, 9)
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    eqn = H._model(wfx, "westervelt", mesh, P, dtype, None, rel, pml)
    dofs, q, delay = _sources(wfx, mesh, eqn, pml, 12)
    eqn.set_volume_source(dofs, q, delay)
    dt = min(wfx.cfl_timestep(mesh.h_min, C0, P, F0), rel.max_dt(), pml.max_dt())
    u, v = H._random_state(mesh.ndofs, 4, dtype, 0.1)
    full = []
    for _ in range(2):
        eqn.set_state(u, v)
        eqn.rk4(0.0, 1.0, dt, max_steps=30)
        full.append((eqn.get_state(), eqn.relaxation_state(), eqn.pml_state()))
    for a, b in zip(full[0], full[1]):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    eqn.set_state(u, v)
    _, t = eqn.rk4(0.0, 1.0, dt, max_steps=15)
    ck = (eqn.get_state(), eqn.relaxation_state(), eqn.pml_state())
    eqn.init()
    eqn.set_state(*ck[0])
    eqn.set_relaxation_state(ck[1])
    eqn.set_pml_state(*ck[2])
    eqn.rk4(t, 1.0, dt, max_steps=15)
    got = (eqn.get_state(), eqn.relaxation_state(), eqn.pml_state())
    for a, b in zip(full[0], got):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def _device_series(wfx, eqn, mesh, sdofs, sq, probe, dt, nsteps):
    eqn.set_volume_source(sdofs, sq)
    eqn.set_probes([probe], nsteps)
    eqn.init()
    eqn.rk4(0.0, 1.0, dt, max_steps=nsteps)
    return eqn.probe_series()[1][:, 0].astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("case", RECIP, ids=[f"{c[0]}-M{c[1]}-pml{int(c[2])}" for c in RECIP])
def test_reciprocity_on_the_device(wfx, orc, mo, torch, case, dtype):
    kind, M, with_pml = case
    P = 2
    mesh, med, pml, args, dt = _recip_setup(wfx, orc, mo, P, kind, M, with_pml)
    rel = H.random_relaxation(wfx, mesh.ncells, M, 3) if M else None
    m1 = args[2]
    rng = np.random.default_rng(7)
    A, B = _source_dofs(mesh, pml.zeta if with_pml else np.zeros((3, mesh.ndofs)), m1, rng,
                        ("interior", "layer" if with_pml else "interior"))
    mk = lambda: H._model(wfx, kind, mesh, P, dtype, med, rel, pml if with_pml else None)  # noqa: E731
    eqn = mk()
    eqn.set_source_profile(np.zeros(mesh.ndofs))          # no tag-1 source: the volume sources alone
    ab = _device_series(wfx, eqn, mesh, [A], [1.0], B, dt, RECIP_STEPS)
    ba = _device_series(wfx, eqn, mesh, [B], [1.0], A, dt, RECIP_STEPS)
    scale = np.abs(ab).max()
    tol = RECIP_TOL if dtype == np.float64 else RECIP_TOL32
    mismatch = np.abs(ab - ba).max() / scale
    assert scale > 0 and mismatch < tol, mismatch
    if dtype == np.float32:
        # the fp32 mismatch is fp32 roundoff: the fp32 series differ from the fp64 series of the same runs as much
        ref = H._model(wfx, kind, mesh, P, np.float64, med, rel, pml if with_pml else None)
        ref.set_source_profile(np.zeros(mesh.ndofs))
        ab64 = _device_series(wfx, ref, mesh, [A], [1.0], B, dt, RECIP_STEPS)
        ba64 = _device_series(wfx, ref, mesh, [B], [1.0], A, dt, RECIP_STEPS)
        rounding = max(np.abs(ab - ab64).max(), np.abs(ba - ba64).max()) / scale
        print(f"reciprocity fp32 {kind}-M{M}-pml{int(with_pml)}: A<->B mismatch {mismatch:.3e}, fp32 vs fp64 "
              f"{rounding:.3e}")
        assert mismatch <= 2.0 * rounding, (mismatch, rounding)
    if kind == "linear" and with_pml:
        # a tag-1 dof i (profile amplitude 1 there only) against a volume source q = m1_i at B
        i, = _source_dofs(mesh, pml.zeta, m1, np.random.default_rng(3), ("tag1",))
        eqn.set_source_profile(np.where(np.arange(mesh.ndofs) == i, 1.0, 0.0))
        s1 = _device_series(wfx, eqn, mesh, None, None, B, dt, RECIP_STEPS)
        eqn.set_source_profile(np.zeros(mesh.ndofs))
        s2 = _device_series(wfx, eqn, mesh, [B], [m1[i]], i, dt, RECIP_STEPS)
        sc = np.abs(s1).max()
        assert sc > 0 and np.abs(s1 - s2).max() < tol * sc, np.abs(s1 - s2).max() / sc


@pytest.mark.gpu
def test_refusals_on_the_device(wfx, torch):
    P = 2
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1])
    eqn = H._model(wfx, "lossy", mesh, P, np.float64, None)
    for dofs, q, delay, match in (([mesh.ndofs], [1.0], None, "outside"), ([-1], [1.0], None, "outside"),
                                  ([3, 7, 3], [1.0, 1.0, 1.0], None, "duplicate"), ([3], [np.nan], None, "non-finite"),
                                  ([3], [1.0], [np.inf], "non-finite"), ([3], [1.0], [-1e-9], "negative")):
        with pytest.raises(wfx.WfxError, match=match):
            eqn.set_volume_source(dofs, q, delay)
    with pytest.raises(wfx.WfxError, match="shape"):
        eqn.set_volume_source([3, 4], [1.0])
    # an index that int32 would wrap into range, weights without dofs, non-integer dofs
    with pytest.raises(wfx.WfxError, match="outside"):
        eqn.set_volume_source(np.array([2 ** 32 + 3], dtype=np.int64), [1.0])
    with pytest.raises(wfx.WfxError, match="without dofs"):
        eqn.set_volume_source([], [1.0])
    with pytest.raises(wfx.WfxError, match="integers"):
        eqn.set_volume_source([3.0], [1.0])
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, (F0, 2 * F0), (P0, P0))
    with pytest.raises(wfx.WfxError, match="shape"):
        ens.set_volume_source([3, 4], [1.0, 1.0])
    ens.set_volume_source([3, 4], np.ones((2, 2)), np.zeros((2, 2)))
    # snapshots stay allowed; the model still steps after the refusals
    eqn.set_volume_source(*wfx.point_source(mesh, (0.01, 0.01, 0.01)))
    eqn.set_snapshot(1, lambda *a: None)
    eqn.init()
    assert eqn.rk4(0.0, 1.0, wfx.cfl_timestep(mesh.h_min, C0, P, F0), max_steps=3)[0] == 3


# ---- GPU: the free-space Green's function --------------------------------------------------------------------------
# An undistorted octant [0, L]^3 with the source at the corner dof (q = 1), rigid symmetry faces through it, no tag-1
# facets and a one-wavelength PML.box on the three far faces: mirroring makes it a full-space source of strength 8, so
# p = 8 g(t - r / c0) / (4 pi r) and p_1 = (2 p0 k / (pi r)) exp(-i k r) (g = p0 k cos(w t) after the ramp).  Compared
# for r in [lambda, 2.5 lambda] along the three axes and the diagonal, sampled over two periods after 24.
# Measured on a B200 (fp64, P4): max |p_1 - exact| / max |exact| = 2.1e-2 at h = lambda / 2 (46 dofs) and 1.2e-4 at
# h = lambda / 4 (88 dofs), a 177-fold fall.  Sampled after 14 periods instead, h = lambda / 4 gives 6.8e-3: the
# transient left at that time, not the layer: a two-wavelength layer gives the same 6.8e-3 after 14 periods.  After 24
# the remaining 1.2e-4 is mostly the layer's reflection: a two-wavelength layer with R0 = 1e-6 gives 2.0e-5 (and 9.9e-7
# at h = lambda / 8).  h = lambda / 2 stays at 2.0e-2 to 2.1e-2 for every window and layer, its discretisation error.
# Bounds: 1e-3 at lambda / 4 and at least a 4-fold fall.
GREEN_N0, GREEN_PERIODS = 24, 2
GREEN_BOUNDS = dict(fine=1e-3, fall=4.0)


def _green_error(wfx, cells_per_lambda, P=4):
    lam = C0 / F0
    L = 3.5 * lam
    n = int(round(3.5 * cells_per_lambda))
    mesh = wfx.create_box_hex(n, P, (L, L, L), tags=())
    pml = wfx.PML.box(mesh, lam, [(0, 1), (1, 1), (2, 1)], C0)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, pml=pml)
    dofs, q = wfx.point_source(mesh, (0.0, 0.0, 0.0))
    assert len(dofs) == 1 and q[0] == 1.0
    eqn.set_volume_source(dofs, q)
    k_steps = int(np.ceil((1 / F0) / min(wfx.cfl_timestep(mesh.h_min, C0, P, F0), pml.max_dt())))
    dt = (1 / F0) / k_steps
    eqn.init()
    eqn.set_field_stats(GREEN_N0 * k_steps * dt + 0.5 * dt, harmonics=1)
    eqn.rk4(0.0, 1.0, dt, max_steps=(GREEN_N0 + GREEN_PERIODS) * k_steps)
    p1 = eqn.field_stats().harmonics[0]
    x = wfx.dof_coordinates(mesh)
    r = np.linalg.norm(x, axis=1)
    tol = 1e-9 * L
    on_axis = (np.sum(np.abs(x) < tol, axis=1) == 2)
    diag = (np.abs(x[:, 0] - x[:, 1]) < tol) & (np.abs(x[:, 1] - x[:, 2]) < tol)
    sel = (on_axis | diag) & (r >= lam * (1 - 1e-9)) & (r <= 2.5 * lam * (1 + 1e-9))
    k = 2 * np.pi / lam
    exact = 2 * P0 * k / (np.pi * r[sel]) * np.exp(-1j * k * r[sel])
    return np.abs(p1[sel] - exact).max() / np.abs(exact).max(), int(sel.sum())


@pytest.mark.gpu
def test_greens_function_known_answer(wfx, torch):
    e2, n2 = _green_error(wfx, 2)
    e4, n4 = _green_error(wfx, 4)
    print(f"green: h = lambda/2 error {e2:.3e} ({n2} dofs), h = lambda/4 error {e4:.3e} ({n4} dofs)")
    assert n2 > 10 and n4 > n2
    assert e4 < GREEN_BOUNDS["fine"] and e4 * GREEN_BOUNDS["fall"] <= e2


# ---- GPU: time reversal through a bone slab -------------------------------------------------------------------------
# A P4 box (4 lambda along x, 4 lambda across), the array on tag 1 at x = 0, a PML of 0.75 lambda on the five other
# faces, a bone slab (rho = 1900, c = 2800) over x in [1, 1.5] lambda and the target at x = 2.75 lambda on the axis.  The
# emission runs with the array silent (profile amplitude 0) and a point source at the target; p_1 on tag 1 is conjugated
# (phase_conjugate_delays).  By reciprocity the focal sum_j q_j p_1,j of a treatment with profile (a, tau) is
# sum_i m1_i a_i exp(-i w tau_i) p_1,i of the emission, m1 the model's weighted tag-1 facet mass.
TR_N0, TR_PERIODS = 16, 2
# Measured on a B200 (fp64): |focal - prediction| / |focal under the conjugate delays| is at most 1.4e-2 over the six
# runs (the transient left after 16 periods); bound 3e-2.  Focal |p_1| through the slab: 2.02e5 Pa with the conjugate
# delays, 1.55e5 with focus_delays (a gain of 1.31), 9.0e3 with random delays; in water 2.415e5 against 2.404e5 (1.004).
TR_BOUNDS = dict(prediction=3e-2)


def _tr_case(wfx, slab):
    lam = C0 / F0
    P, L = 4, 4 * lam
    mesh = wfx.create_box_hex(8, P, (L, L, L), tags=((0, 0, 1),))
    xc = mesh.x[mesh.xdofs].mean(axis=1)
    bone = (xc[:, 0] > lam) & (xc[:, 0] < 1.5 * lam) if slab else np.zeros(mesh.ncells, dtype=bool)
    med = wfx.Medium(np.where(bone, 1900.0, 1000.0), np.where(bone, 2800.0, C0), rho_ref=1000.0)
    pml = wfx.PML.box(mesh, 0.75 * lam, [(0, 1), (1, 0), (1, 1), (2, 0), (2, 1)], med.c_max)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, medium=med, pml=pml)
    k_steps = int(np.ceil((1 / F0) / min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), pml.max_dt())))
    focus = np.array([2.75 * lam, L / 2, L / 2])
    return mesh, eqn, (1 / F0) / k_steps, k_steps, focus


def _tr_run(eqn, dt, k_steps):
    eqn.init()
    eqn.set_field_stats(TR_N0 * k_steps * dt + 0.5 * dt, harmonics=1)
    eqn.rk4(0.0, 1.0, dt, max_steps=(TR_N0 + TR_PERIODS) * k_steps)
    return eqn.field_stats().harmonics[0]


def _time_reversal(wfx, slab):
    mesh, eqn, dt, k_steps, focus = _tr_case(wfx, slab)
    fd, fq = wfx.point_source(mesh, focus)
    m1 = eqn.bnd_op.facet_masses()[0]
    arr = m1 > 0
    # emission: the array silent, the point source at the target
    eqn.set_source_profile(np.zeros(mesh.ndofs))
    eqn.set_volume_source(fd, fq)
    pe = _tr_run(eqn, dt, k_steps)
    eqn.set_volume_source()
    x = wfx.dof_coordinates(mesh)
    rng = np.random.default_rng(5)
    delays = dict(conjugate=wfx.phase_conjugate_delays(pe, F0) * arr,
                  geometric=wfx.focus_delays(x, focus, C0) * arr,
                  random=rng.uniform(0, 1 / F0, mesh.ndofs) * arr)
    amp = arr.astype(np.float64)
    out = {}
    for name, tau in delays.items():
        tau = tau - tau[arr].min() * arr if name == "geometric" else tau
        eqn.set_source_profile(amp, tau)
        focal = fq @ _tr_run(eqn, dt, k_steps)[fd]
        pred = np.sum(m1 * amp * np.exp(-2j * np.pi * F0 * tau) * pe)
        out[name] = (focal, pred)
    return out


@pytest.mark.gpu
def test_time_reversal_through_a_bone_slab(wfx, torch):
    res, errs = {}, {}
    for slab in (True, False):
        out = _time_reversal(wfx, slab)
        for name, (focal, pred) in out.items():
            errs[slab, name] = abs(focal - pred) / abs(out["conjugate"][0])
            print(f"time reversal: slab={slab} {name}: |p1| focal {abs(focal):.4e}, prediction {abs(pred):.4e}, "
                  f"error {errs[slab, name]:.2e}")
        res[slab] = {k: abs(v[0]) for k, v in out.items()}
    assert max(errs.values()) < TR_BOUNDS["prediction"], errs
    for slab in (True, False):
        assert res[slab]["conjugate"] >= res[slab]["geometric"] and res[slab]["conjugate"] >= res[slab]["random"]
    print(f"time reversal gain over geometric delays: slab {res[True]['conjugate'] / res[True]['geometric']:.3f}, "
          f"water {res[False]['conjugate'] / res[False]['geometric']:.3f}")


# ---- GPU: the C++ wrapper ------------------------------------------------------------------------------------------
def _build_cpp(wfx, outdir):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_volume_source_hpp.cpp")
    exe = os.path.join(str(outdir), "test_wavefx_volume_source_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_volume_source_cpp_wrapper_compiles_and_links(wfx, tmp_path):
    assert os.path.exists(_build_cpp(wfx, tmp_path))


@pytest.mark.gpu
def test_volume_source_cpp_wrapper_reproduces_python(wfx, torch, tmp_path):
    """LossyGLLOpt with a medium, a layer and set_volume_source from C++, 15 steps, a restart, 15 more: the same u as
    the Python model bit for bit"""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = H.random_medium(wfx, mesh.ncells, 91, beta=False)
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), pml.max_dt())
    u, v = H._random_state(mesh.ndofs, 5, np.float64)
    lossy = H._model(wfx, "lossy", mesh, P, np.float64, med, pml=pml)
    sdofs, sq, sdelay = _sources(wfx, mesh, lossy, pml, 77)
    lossy.set_volume_source(sdofs, sq, sdelay)
    files = {"params.f64": np.array([P, C0, F0, P0, DELTA, dt]),
             "x.f64": mesh.x, "xdofs.i32": mesh.xdofs, "dofmap.i32": mesh.dofmap,
             "fcell.i32": mesh.facet_cells, "flocal.i32": mesh.facet_local, "ftag.i32": mesh.facet_tags,
             "u.f64": u, "v.f64": v, "stiffness.f64": med.stiffness_weight(mesh.ncells),
             "mass.f64": med.mass_weight(mesh.ncells, C0), "facet.f64": med.facet_weight(mesh, C0),
             "zeta.f64": pml.zeta, "sdofs.i32": sdofs, "sq.f64": sq, "sdelay.f64": sdelay}
    for name, a in files.items():
        np.ascontiguousarray(a, dtype=np.int32 if name.endswith("i32") else np.float64).tofile(str(tmp_path / name))
    r = subprocess.run([_build_cpp(wfx, tmp_path), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "volume source hpp ok" in r.stdout, r.stdout + r.stderr
    lossy.set_state(u, v)
    _, t1 = lossy.rk4(0.0, 1.0, dt, max_steps=15)
    cu, cv = lossy.get_state()
    cpsi, cphi = lossy.pml_state()
    lossy.set_state(cu, cv)
    lossy.set_pml_state(cpsi, cphi)
    lossy.rk4(t1, 1.0, dt, max_steps=15)
    assert np.array_equal(np.fromfile(str(tmp_path / "u.out.f64"), dtype=np.float64), lossy.get_state()[0])


# ---- GPU: the demo -------------------------------------------------------------------------------------------------
def _demo_tr(extra):
    r = subprocess.run(["python", os.path.join(ROOT, "demo", "planar3d.py"), "--nx", "16", "--nyz", "12",
                        "--length", "0.012", "--focus", "0.008", "--pml", "0.0015", "--stats-periods", "2",
                        "--time-reversal", *extra], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    vals = {}
    for ln in r.stdout.splitlines():
        if ln.startswith("time reversal: ") and " delays: focal |p1| = " in ln:
            name = ln.split("time reversal: ")[1].split(" delays")[0]
            focal = float(ln.split("focal |p1| = ")[1].split(",")[0])
            diff = float(ln.split("(difference ")[1].rstrip(")"))
            vals[name] = (focal, diff)
    assert set(vals) == {"geometric", "time-reversal"}, r.stdout
    return vals, r.stdout


# Measured on a B200 (the demo box: 4 lambda long, 3 lambda wide, h = lambda / 4, P4, a 0.5 lambda PML on five faces,
# focus at 2.67 lambda, the demo's run of L / c0 + 8 periods): through the slab (x in [1, 1.5] lambda) the focal |p1| is
# 1.314e5 Pa with the time-reversal delays and 1.188e5 with the geometric ones (gain 1.107), each |focal - prediction|
# at most 2.5e-2 of the time-reversal amplitude (the transient the shorter run leaves); in water 1.524e5 against
# 1.521e5 (gain 1.002), differences 7e-6.  Bound 5e-2 of the time-reversal focal amplitude.
DEMO_TR = dict(prediction=5e-2)


@pytest.mark.gpu
def test_demo_time_reversal_option(wfx, torch):
    """demo/planar3d.py --focus --pml --time-reversal, through a bone slab and in water: the time-reversal focal |p1|
    is at least the geometric one, and both match their reciprocity predictions"""
    for extra in (("--layer", "0.003", "0.0045"), ()):
        vals, out = _demo_tr(extra)
        tr, geo = vals["time-reversal"], vals["geometric"]
        print(out)
        assert tr[0] >= geo[0], out
        for focal, diff in vals.values():
            assert diff < DEMO_TR["prediction"] * tr[0], out
