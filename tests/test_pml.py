"""Perfectly matched layers (DESIGN.md section 4.5g): the second-order PML of Grote and Sim (2010) in the weighted form
of section 4.5e, with psi on the layer's dofs and phi at the GLL points of its cells,

    m~ (p_tt + sum zeta p_t + sum zeta zeta p + zeta1 zeta2 zeta3 psi) = b + div phi,   psi_t = p
    phi_t = -Z phi + a Gamma1 grad w + a Gamma2 grad(psi + s p).

CPU: the restatement (model_oracle wo_*_westervelt_pml) against a textbook RK4 of the augmented system built from
first principles and, without layer cells, against wo_rk4_westervelt_relax bit for bit; known answers on the
restatement -- oblique incidence in a duct against the outgoing field, the decay inside the layer, the long-time
stability of a closed box; PML.box.
GPU: every model against the restatement, the model without a layer bit for bit, repeatability, checkpoints,
scale_cells before and after the layer, field statistics, the oblique-incidence answer and the refusals.
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
KAPPA = 2.0 * BETA / (RHO0 * C0 * C0)


def rel_l2(a, b):
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


@pytest.fixture(scope="module")
def mo():
    from model_oracle import model_oracle
    return model_oracle


def random_medium(wfx, ncells, seed, beta=True):
    rng = np.random.default_rng(seed)
    lu = lambda lo, hi: np.exp(rng.uniform(np.log(lo), np.log(hi), ncells))  # noqa: E731
    b = None
    if beta:
        b = lu(0.1, 8.0)
        b[rng.random(ncells) < 0.2] = 0.0
    return wfx.Medium(lu(900.0, 2000.0), lu(1400.0, 3000.0), b, rho_ref=RHO_REF)


def random_relaxation(wfx, ncells, M, seed):
    rng = np.random.default_rng(seed)
    tau = 1.0 / (2 * np.pi * np.geomspace(0.3e6, 3e6, M))
    eps = rng.uniform(0.0, 0.05, (M, ncells))
    return wfx.Relaxation(tau, eps, 1500.0)


def weighted_inputs(orc, mo, mesh, P, medium):
    """(G * sigma, m~, m1~, m2~, mu, detJ w) of the restatement; an identity medium without one"""
    G, detJ = orc.precompute_geometric_data(mesh, P)
    if medium is None:
        medium = __import__("wave_fenics_b200").Medium(RHO_REF, C0, rho_ref=RHO_REF)
    Gs = np.ascontiguousarray(G * medium.stiffness_weight(mesh.ncells)[:, None, None, None])
    mu = medium.mass_weight(mesh.ncells, C0)
    m = np.zeros(mesh.ndofs)
    orc.mass_apply(mesh, P, np.ascontiguousarray(detJ * mu[:, None]), np.ones(mesh.ndofs), m)
    m1, m2 = mo.boundary_facet_mass_weighted(mesh, P, medium.facet_weight(mesh, C0))
    return Gs, m, m1, m2, mu, detJ


def pml_inputs(orc, mo, mesh, P, zeta, coeff=None):
    """the restatement's layer inputs: J^-1 from the oracle at the GLL points in tensor order, |detJ| w"""
    pts, wts = orc.gll(P)
    n = P + 1
    a, b, c = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
    X = np.stack([pts[a.reshape(-1)], pts[b.reshape(-1)], pts[c.reshape(-1)]], -1)
    W = (wts[a] * wts[b] * wts[c]).reshape(-1)
    K = orc.jacobian_data(mesh, X, W)["K"]
    _, detJ = orc.precompute_geometric_data(mesh, P)
    return mo.PMLInputs(mesh, P, zeta, K, detJ, coeff)


def dense_stiffness(orc, mesh, P, G):
    n = mesh.ndofs
    A = np.zeros((n, n))
    for j in range(n):
        e, col = np.zeros(n), np.zeros(n)
        e[j] = 1.0
        orc.stiffness_apply(mesh, P, G, e, col, dense=True)
        A[:, j] = col
    return A


def first_principles_gradients(orc, mesh, P):
    """Gr [ncells, nq, 3, ndofs]: the physical gradient at every GLL point (tensor order) of the field with the given
    dof values, and dJw [ncells, nq] = |det J| w.  Independent of the library's tables: GLL nodes from the roots of
    P_n', weights 2 / (n (n+1) P_n(x)^2), Lagrange derivatives by barycentric formulas, the trilinear Jacobian
    differentiated by hand (tests/test_oracle_kat.py)."""
    from numpy.polynomial import legendre as Lg
    n = P + 1
    cP = np.zeros(P + 1)
    cP[P] = 1.0
    xi = np.concatenate([[-1.0], np.sort(Lg.legroots(Lg.legder(cP))), [1.0]])
    w = 2.0 / (P * (P + 1) * Lg.legval(xi, cP) ** 2)
    x01, w01 = (xi + 1) / 2, w / 2
    bw = np.array([1.0 / np.prod([x01[i] - x01[j] for j in range(n) if j != i]) for i in range(n)])
    Dasc = np.zeros((n, n))
    for q in range(n):
        for i in range(n):
            if i != q:
                Dasc[q, i] = bw[i] / bw[q] / (x01[q] - x01[i])
        Dasc[q, q] = -Dasc[q].sum()
    pos = np.array([0, P] + list(range(1, P)))
    pts, wts, D = x01[pos], w01[pos], Dasc[np.ix_(pos, pos)]
    perm = orc.perm(P)
    A, B, Cc = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
    X = np.stack([pts[A], pts[B], pts[Cc]], -1)
    nq = n ** 3
    I = np.eye(n)
    # reference gradient operator on a cell's tensor-ordered values: R[a] [nq, nq]
    R = [np.einsum("qm,bc,de->qbdmce", D, I, I).reshape(nq, nq), np.einsum("ab,qm,de->aqdbme", I, D, I).reshape(nq, nq),
         np.einsum("ab,cd,qm->acqbdm", I, I, D).reshape(nq, nq)]
    Gr = np.zeros((mesh.ncells, nq, 3, mesh.ndofs))
    dJw = np.zeros((mesh.ncells, nq))
    for c in range(mesh.ncells):
        xv = mesh.x[mesh.xdofs[c]]
        J = np.zeros((n, n, n, 3, 3))
        for vtx in range(8):
            bits = [(vtx >> a) & 1 for a in range(3)]
            f = [X[..., a] if bits[a] else 1.0 - X[..., a] for a in range(3)]
            for a in range(3):
                g = (1.0 if bits[a] else -1.0) * f[(a + 1) % 3] * f[(a + 2) % 3]
                J[..., :, a] += xv[vtx][None, None, None, :] * g[..., None]
        J = J.reshape(nq, 3, 3)
        Kq = np.linalg.inv(J)                                   # K[a][l] = dX_a / dx_l
        dJw[c] = np.abs(np.linalg.det(J)) * (wts[A] * wts[B] * wts[Cc]).reshape(-1)
        dofs = mesh.dofmap[c][perm]
        for l in range(3):
            loc = sum(Kq[:, a, l][:, None] * R[a] for a in range(3))   # [nq, nq] on the cell's values
            np.add.at(Gr[c, :, l, :], (slice(None), dofs), loc)
    return Gr, dJw


# ---- CPU: the restatement ------------------------------------------------------------------------------------------
TEXTBOOK = [(2, "linear", 0), (3, "lossy", 1), (4, "westervelt", 2)]


@pytest.mark.parametrize("case", TEXTBOOK, ids=[f"P{c[0]}-{c[1]}-M{c[2]}" for c in TEXTBOOK])
def test_restatement_matches_textbook_rk4(wfx, orc, mo, case):
    """wo_rk4_westervelt_pml against a textbook RK4 of the augmented system (dense stiffness, dense physical
    gradients, a random medium, relaxation, both tags), on a perturbed mesh with a layer on three faces: zeta on
    faces, edges and a corner"""
    P, kind, M = case
    mesh = wfx.create_box_hex((3, 3, 2), P, (0.03, 0.03, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 11 + P, beta=kind == "westervelt")
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    kap = med.kappa(mesh, detJ, C0) if kind == "westervelt" else np.zeros(mesh.ndofs)
    delta = 0.0 if kind == "linear" else DELTA
    if M:
        rel = random_relaxation(wfx, mesh.ncells, M, 3)
        eps, tau = rel.eps_dofs(mesh, detJ, mu), rel.tau
    else:
        eps, tau = np.zeros((0, mesh.ndofs)), np.zeros(0)
    pml = wfx.PML.box(mesh, 0.011, [(0, 1), (1, 0), (2, 1)], C0)
    zeta = pml.zeta
    assert np.any(np.count_nonzero(zeta, axis=0) == 3) and np.any(np.count_nonzero(zeta, axis=0) == 2)
    sw = med.stiffness_weight(mesh.ncells)
    inp = pml_inputs(orc, mo, mesh, P, zeta, sw)
    A = dense_stiffness(orc, mesh, P, G)
    Gr, dJw = first_principles_gradients(orc, mesh, P)
    perm = orc.perm(P)
    cell_on = np.array([np.any(zeta[:, mesh.dofmap[c]] > 0) for c in range(mesh.ncells)])
    dof_on = np.zeros(mesh.ndofs, dtype=bool)
    dof_on[mesh.dofmap[cell_on].reshape(-1)] = True
    Gr = Gr * cell_on[:, None, None, None]
    zq = zeta[:, mesh.dofmap[:, perm]].transpose(1, 2, 0)            # zeta at every point [ncells, nq, 3]
    g1 = np.stack([zq[..., 1] + zq[..., 2] - zq[..., 0], zq[..., 0] + zq[..., 2] - zq[..., 1],
                   zq[..., 0] + zq[..., 1] - zq[..., 2]], -1)
    g2 = np.stack([zq[..., 1] * zq[..., 2], zq[..., 0] * zq[..., 2], zq[..., 0] * zq[..., 1]], -1)
    a = 1500.0 ** 2 * sw[:, None, None]
    z1, z2, z3 = zeta.sum(0), zeta[0] * zeta[1] + zeta[0] * zeta[2] + zeta[1] * zeta[2], zeta.prod(0)
    s = delta / 1500.0 ** 2

    def rhs(t, p, pd, q, psi, phi):
        kq = (eps * p - q) / tau[:, None]
        R = ((eps * pd - kq) / tau[:, None]).sum(0)
        g, gd = mo.source(t, F0, P0, C0)
        grad = lambda f: np.einsum("cqld,d->cql", Gr, f)  # noqa: E731
        dtphi = -np.einsum("cqld,cql->d", Gr, dJw[..., None] * phi)
        layer = np.where(dof_on, dtphi - m * (z1 * pd + z2 * p + z3 * psi), 0.0)
        num = (A @ p + s * (A @ pd) + (C0 ** 2 * g + delta * gd) * m1 - C0 * m2 * pd + layer + kap * m * pd ** 2
               - m * R)
        kphi = a * (g1 * grad(p + s * pd) + g2 * grad(psi + s * p)) - zq * phi
        kphi = kphi * cell_on[:, None, None]
        return pd, num / (m * (1.0 - kap * p) + delta / C0 * m2), kq, np.where(dof_on, p, 0.0), kphi

    dt = 0.5 * min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), pml.max_dt())
    rng = np.random.default_rng(5)
    n = mesh.ndofs
    p, pd = 0.1 * P0 * rng.standard_normal(n), 0.1 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)
    q = eps * p * rng.uniform(0.5, 1.5, eps.shape)
    psi = np.where(dof_on, p * rng.uniform(0.5, 1.5, n) / (2 * np.pi * F0), 0.0)
    phi = a * np.einsum("cqld,d->cql", Gr, p) * rng.uniform(0.5, 1.5, (mesh.ncells, len(perm), 3)) / pml.zeta_max
    st = [x.copy() for x in (p, pd, q, psi, phi)]
    t0, nsteps = 1.0e-6, 5
    steps, _ = mo.rk4_westervelt_pml(mesh, P, G, m, m1, m2, kap, C0, F0, P0, delta, tau, eps, inp, t0, 1.0, dt, *st,
                                     max_steps=nsteps)
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
    assert np.abs(y[3]).max() > 0 and np.abs(y[4]).max() > 0
    fo = mo.f1_westervelt_pml(mesh, P, G, m, m1, m2, kap, C0, F0, P0, delta, tau, eps, inp, 3e-6, y[0], y[1], y[2],
                              y[3], y[4])
    assert rel_l2(fo, rhs(3e-6, *y)[1]) < 1e-13


def test_restatement_without_layer_cells_is_the_relaxation_restatement_bitwise(wfx, orc, mo):
    P = 2
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 9)
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    kap = med.kappa(mesh, detJ, C0)
    dt = wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0)
    rng = np.random.default_rng(2)
    u, v = 0.3 * P0 * rng.standard_normal(mesh.ndofs), 1e6 * rng.standard_normal(mesh.ndofs)
    inp = pml_inputs(orc, mo, mesh, P, np.zeros((3, mesh.ndofs)))
    for M in (0, 2):
        rel = random_relaxation(wfx, mesh.ncells, M, 1) if M else None
        tau = rel.tau if M else np.zeros(0)
        eps = rel.eps_dofs(mesh, detJ, mu) if M else np.zeros((0, mesh.ndofs))
        u1, v1, q1 = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
        r1 = mo.rk4_westervelt_relax(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, tau, eps, 1e-6, 1e-6 + 9.5 * dt, dt,
                                     u1, v1, q1)
        u2, v2, q2 = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
        psi, phi = mo.pml_state(mesh, P)
        r2 = mo.rk4_westervelt_pml(mesh, P, G, m, m1, m2, kap, C0, F0, P0, DELTA, tau, eps, inp, 1e-6, 1e-6 + 9.5 * dt,
                                   dt, u2, v2, q2, psi, phi)
        assert r1 == r2 and np.array_equal(u1, u2) and np.array_equal(v1, v2) and np.array_equal(q1, q2), M
        assert not np.any(psi) and not np.any(phi)


# ---- CPU: known answers --------------------------------------------------------------------------------------------
# Oblique incidence: the duct of tests/test_source_profile.py (Lx = 2 lambda, Ly = lambda, two cells thick, P4, four
# cells per wavelength, rigid lateral faces, source a(y) = cos(pi y / Ly) on tag 1 at x = 0) carries only the first
# duct mode, a pair of plane waves at theta = asin(pi / (k Ly)) = 30 degrees, with k_x = sqrt(k^2 - (pi / Ly)^2).  The
# purely outgoing field is |p_1| = p0 (k / k_x) |cos(pi y / Ly)|.  Its first-order absorbing end (tag 2 at x = 2 lambda)
# reflects R = (k_x - k) / (k_x + k) = -0.072; here it is replaced by one wavelength of layer (PML.box, R0 = 1e-4,
# order 2) and a rigid end at x = 3 lambda.  Sampled over two periods from 24 periods on, as the duct test.
# Measured on the CPU restatement (fp64), before the bounds were set: max | |p_1| - outgoing | / max outgoing over
# x <= 2 lambda is 0.152 with the absorbing end and 4.9e-4 with the layer (a ratio of 3.2e-3); in the first half of the
# layer, on y = 0, |p_1(x)| / |p_1(2 lambda)| follows exp(-(k_x / w) int zeta_x dx) to 4.1e-4 (it falls to 0.61 there).
DUCT_N0, DUCT_PERIODS = 24, 2
DUCT_BOUNDS = dict(pml=1e-3, ratio=0.1, decay=1e-3)


def _duct(wfx, with_layer):
    P, lam = 4, C0 / F0
    L, Ly = 2 * lam, lam
    if with_layer:
        mesh = wfx.create_box_hex((12, 4, 2), P, (L + lam, Ly, Ly / 2), tags=((0, 0, 1),))
        pml = wfx.PML.box(mesh, lam, [(0, 1)], C0, R0=1e-4)
    else:
        mesh = wfx.create_box_hex((8, 4, 2), P, (L, Ly, Ly / 2))
        pml = wfx.PML(mesh, np.zeros((3, mesh.ndofs)))
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    k = int(round(1.0 / F0 / dt))
    X = wfx.dof_coordinates(mesh)
    kk = 2 * np.pi / lam
    kx = np.sqrt(kk ** 2 - (np.pi / Ly) ** 2)
    outgoing = P0 * kk / kx * np.abs(np.cos(np.pi * X[:, 1] / Ly))
    return mesh, P, pml, dt, k, X, np.cos(np.pi * X[:, 1] / Ly), outgoing, kx, L


def _duct_error(p1, X, outgoing, L):
    sel = X[:, 0] <= L + 1e-12
    return np.abs(np.abs(p1[sel]) - outgoing[sel]).max() / outgoing.max()


def _duct_restatement(wfx, orc, mo, with_layer):
    mesh, P, pml, dt, k, X, amp, outgoing, kx, L = _duct(wfx, with_layer)
    G, m, m1, m2, _, _ = weighted_inputs(orc, mo, mesh, P, None)
    inp = pml_inputs(orc, mo, mesh, P, pml.zeta)
    z = np.zeros(mesh.ndofs)
    # the apodised source: a(y) g(t) on tag 1 is the boundary term with a m1 (no delay)
    args = (mesh, P, G, m, amp * m1, m2, z, C0, F0, P0, 0.0, np.zeros(0), np.zeros((0, mesh.ndofs)), inp)
    kw = dict(sumfact=True, nthreads=orc.max_threads())
    u, v = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    psi, phi = mo.pml_state(mesh, P)
    _, t = mo.rk4_westervelt_pml(*args, 0.0, 1.0, dt, u, v, None, psi, phi, max_steps=DUCT_N0 * k, **kw)
    acc = np.zeros(mesh.ndofs, dtype=np.complex128)
    n = DUCT_PERIODS * k
    for _ in range(n):
        _, t = mo.rk4_westervelt_pml(*args, t, 1.0, dt, u, v, None, psi, phi, max_steps=1, **kw)
        acc += u * np.exp(-2j * np.pi * F0 * t)
    return acc * 2 / n, mesh, pml, X, outgoing, kx, L


def test_oblique_incidence_known_answer(wfx, orc, mo):
    p1, _, _, X, outgoing, _, L = _duct_restatement(wfx, orc, mo, False)
    e_abc = _duct_error(p1, X, outgoing, L)
    p1, mesh, pml, X, outgoing, kx, L = _duct_restatement(wfx, orc, mo, True)
    e_pml = _duct_error(p1, X, outgoing, L)
    assert e_pml < DUCT_BOUNDS["pml"] and e_pml < DUCT_BOUNDS["ratio"] * e_abc, (e_pml, e_abc)
    # decay over the first half of the layer on y = z = 0: zeta_x = zeta_max (d / lam)^2, int_0^d = zeta_max d^3 / (3 lam^2)
    lam = C0 / F0
    on = (np.abs(X[:, 1]) < 1e-12) & (np.abs(X[:, 2]) < 1e-12) & (X[:, 0] >= L - 1e-12) & (X[:, 0] <= L + lam / 2 + 1e-12)
    line = np.nonzero(on)[0]
    line = line[np.argsort(X[line, 0])]
    d = X[line, 0] - L
    pred = np.exp(-(kx / (2 * np.pi * F0)) * pml.zeta_max * d ** 3 / (3 * lam ** 2))
    got = np.abs(p1[line]) / np.abs(p1[line[0]])
    assert np.abs(got - pred).max() < DUCT_BOUNDS["decay"] and pred.min() < 0.7


# Stability: a Gaussian pulse (sigma 0.7 mm) at the centre of a closed, rigid 8 mm box, 8^3 cells at P2, with a two-cell
# layer (PML.box, R0 = 1e-4) on all six faces, run for 20 crossing times (747 CFL steps, dt max zeta = 1.48).  Measured
# on the CPU restatement before the bounds were set: the energy of the field outside the layer falls to 8.1e-13 of its
# start, and max |p| falls monotonically over the last half (1.8e-5 to 1.5e-7 of the initial peak).
STAB_BOUNDS = dict(energy=1e-6)


def test_closed_box_with_a_layer_on_every_face_is_stable(wfx, orc, mo):
    P, N, H, NL = 2, 8, 1e-3, 2
    mesh = wfx.create_box_hex(N, P, (N * H,) * 3, tags=())
    pml = wfx.PML.box(mesh, NL * H, [(a, s) for a in range(3) for s in (0, 1)], C0)
    G, m, m1, m2, _, _ = weighted_inputs(orc, mo, mesh, P, None)
    inp = pml_inputs(orc, mo, mesh, P, pml.zeta)
    X = wfx.dof_coordinates(mesh)
    inner = np.all((X > NL * H - 1e-12) & (X < (N - NL) * H + 1e-12), axis=1)
    u, v = np.exp(-np.sum((X - N * H / 2) ** 2, axis=1) / (2 * 0.7e-3 ** 2)), np.zeros(mesh.ndofs)

    def energy(u, v):
        ui = np.where(inner, u, 0.0)
        au = np.zeros(mesh.ndofs)
        orc.stiffness_apply(mesh, P, G, ui, au, dense=False)
        return 0.5 * np.sum(m[inner] * v[inner] ** 2) - 0.5 * ui @ au

    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    nsteps = int(np.ceil(20 * N * H / C0 / dt))
    assert dt < pml.max_dt()
    e0 = energy(u, v)
    psi, phi = mo.pml_state(mesh, P)
    z = np.zeros(mesh.ndofs)
    args = (mesh, P, G, m, m1, m2, z, C0, F0, 0.0, 0.0, np.zeros(0), np.zeros((0, mesh.ndofs)), inp)
    t, peaks = 0.0, []
    for _ in range(20):
        _, t = mo.rk4_westervelt_pml(*args, t, 1.0, dt, u, v, None, psi, phi, max_steps=nsteps // 20, sumfact=True,
                                     nthreads=orc.max_threads())
        peaks.append(np.abs(u).max())
    assert energy(u, v) < STAB_BOUNDS["energy"] * e0
    assert np.all(np.diff(peaks[9:]) <= 0), peaks


# ---- CPU: PML.box ---------------------------------------------------------------------------------------------------
def test_box_profile_values_and_corners(wfx):
    P = 2
    mesh = wfx.create_box_hex((4, 4, 4), P, (0.04, 0.04, 0.04))
    L = 0.01
    pml = wfx.PML.box(mesh, L, [(0, 0), (0, 1), (1, 1)], C0, R0=1e-3, order=3)
    x = wfx.dof_coordinates(mesh)
    zmax = 4 * C0 * np.log(1e3) / (2 * L)
    dx = np.maximum(np.maximum(L - x[:, 0], x[:, 0] - (0.04 - L)), 0.0)
    dy = np.maximum(x[:, 1] - (0.04 - L), 0.0)
    np.testing.assert_allclose(pml.zeta[0], zmax * (dx / L) ** 3, rtol=1e-12, atol=1e-9 * zmax)
    np.testing.assert_allclose(pml.zeta[1], zmax * (dy / L) ** 3, rtol=1e-12, atol=1e-9 * zmax)
    assert not np.any(pml.zeta[2])
    corner = np.argmin(np.linalg.norm(x - [0.04, 0.04, 0.0], axis=1))
    assert np.allclose(pml.zeta[:2, corner], zmax) and pml.zeta[2, corner] == 0
    assert abs(pml.zeta_max - zmax) <= 1e-12 * zmax
    assert pml.max_dt() == 2.5 / pml.zeta_max
    assert wfx.PML(mesh, np.zeros((3, mesh.ndofs))).max_dt() == np.inf


def test_refusals_on_the_host(wfx):
    mesh = wfx.create_box_hex((4, 2, 2), 2, (0.04, 0.02, 0.02))
    for args in ((0.0, [(0, 1)], C0), (np.nan, [(0, 1)], C0), (0.01, [(3, 1)], C0), (0.01, [(0, 2)], C0),
                 (0.01, [], C0), (0.01, [(0, 1), (0, 1)], C0), (0.01, [(0, 1)], 0.0), (0.011, [(1, 0), (1, 1)], C0),
                 (0.03, [(1, 1)], C0)):
        with pytest.raises(wfx.WfxError):
            wfx.PML.box(mesh, *args)
    for kw in (dict(R0=0.0), dict(R0=1.0), dict(order=-1.0)):
        with pytest.raises(wfx.WfxError):
            wfx.PML.box(mesh, 0.01, [(0, 1)], C0, **kw)
    z = np.zeros((3, mesh.ndofs))
    for bad in (np.zeros((2, mesh.ndofs)), np.zeros((3, mesh.ndofs + 1))):
        with pytest.raises(wfx.WfxError):
            wfx.PML(mesh, bad)
    for val in (-1.0, np.nan, np.inf):
        zb = z.copy()
        zb[1, 3] = val
        with pytest.raises(wfx.WfxError):
            wfx.PML(mesh, zb)
    pml = wfx.PML.box(mesh, 0.01, [(0, 1)], C0)
    with pytest.raises(wfx.WfxError, match="ensemble"):
        wfx.LinearGLLEnsemble(mesh, None, 2, C0, (F0,), (P0,), pml=pml)
    # a distributed model refuses the layer before touching the halo
    with pytest.raises(wfx.WfxError, match="distributed"):
        wfx.LinearGLLOpt(mesh, None, 2, C0, F0, P0, halo=object(), pml=pml)


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


GPU_MESH = ((3, 2, 2), (0.03, 0.02, 0.02))
GPU_FACES = [(0, 1), (1, 0), (2, 1)]


def _layer_masks(mesh, zeta):
    cell_on = np.array([np.any(zeta[:, mesh.dofmap[c]] > 0) for c in range(mesh.ncells)])
    dof_on = np.zeros(mesh.ndofs, dtype=bool)
    dof_on[mesh.dofmap[cell_on].reshape(-1)] = True
    return cell_on, dof_on


def _model(wfx, name, mesh, P, dtype, medium, relaxation=None, pml=None):
    if name.startswith("linear"):
        return wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, dtype=dtype, medium=medium, pml=pml)
    if name.startswith("lossy"):
        delta = 0.0 if name == "lossy0" else DELTA
        return wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, delta, dtype=dtype, medium=medium, relaxation=relaxation,
                               pml=pml)
    return wfx.WesterveltGLLOpt(mesh, None, P, C0, F0, P0, DELTA, BETA, RHO0, dtype=dtype, medium=medium,
                                relaxation=relaxation, pml=pml)


def _random_state(n, seed, dtype, scale=1.0):
    rng = np.random.default_rng(seed)
    u = (scale * 0.3 * P0 * rng.standard_normal(n)).astype(dtype).astype(np.float64)
    v = (scale * 0.3 * P0 * 2 * np.pi * F0 * rng.standard_normal(n)).astype(dtype).astype(np.float64)
    return u, v


# (P, dtype, graph, M, model): linear / lossy0 (delta = 0) / lossy / westervelt (scalar kappa, no medium) /
# westervelt-kd (per-dof kappa of a random medium); every model but `westervelt` in a random medium
PARITY = [
    (2, np.float64, True, 0, "linear"), (3, np.float64, False, 0, "linear"), (2, np.float64, False, 1, "lossy0"),
    (3, np.float64, True, 2, "lossy"), (4, np.float64, True, 0, "westervelt"), (4, np.float64, False, 3, "westervelt-kd"),
    (5, np.float64, True, 1, "lossy"), (5, np.float64, False, 0, "westervelt-kd"), (4, np.float64, True, 0, "lossy0"),
    (4, np.float32, True, 2, "lossy"), (4, np.float32, False, 0, "linear"), (7, np.float32, True, 1, "westervelt-kd"),
]


def _parity_case(wfx, orc, mo, P, dtype, M, name, seed=0):
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.15)
    rel = random_relaxation(wfx, mesh.ncells, M, 50 + P) if M else None
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    med = None if name == "westervelt" else random_medium(wfx, mesh.ncells, 40 + P + seed, beta=name == "westervelt-kd")
    eqn = _model(wfx, name, mesh, P, dtype, med, rel, pml)
    G, m, m1, m2, mu, detJ = weighted_inputs(orc, mo, mesh, P, med)
    sw = np.ones(mesh.ncells) if med is None else med.stiffness_weight(mesh.ncells)
    inp = pml_inputs(orc, mo, mesh, P, pml.zeta, sw)
    eps = eqn.relaxation_eps if M else np.zeros((0, mesh.ndofs))
    tau = rel.tau if M else np.zeros(0)
    delta = 0.0 if name in ("linear", "lossy0") else DELTA
    if name.startswith("westervelt"):
        kappa = eqn.kappa if eqn.kappa is not None else np.full(mesh.ndofs, KAPPA)
    else:
        kappa = np.zeros(mesh.ndofs)
    dts = [wfx.cfl_timestep(mesh.h_min, C0 if med is None else med.c_max, P, F0), pml.max_dt()]
    if M:
        dts.append(rel.max_dt())
    return mesh, eqn, pml, (G, m, m1, m2, kappa, C0, F0, P0, delta, tau, eps, inp), min(dts)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY, ids=[f"P{c[0]}-{np.dtype(c[1]).name}-graph{int(c[2])}-M{c[3]}-{c[4]}"
                                              for c in PARITY])
def test_models_with_a_layer_match_the_restatement(wfx, orc, mo, torch, monkeypatch, case):
    """RK4 with a shortened last step through the ramp's end, on a perturbed mesh in a random medium with a layer on
    three faces (faces, edges, a corner), both tags; u, v, the memory variables, psi and phi against the restatement;
    f1 at the model's psi and phi against wo_f1_westervelt_pml"""
    P, dtype, graph, M, name = case
    if not graph:
        monkeypatch.setenv("WFX_WAVE_GRAPH", "0")
    mesh, eqn, pml, args, dt = _parity_case(wfx, orc, mo, P, dtype, M, name)
    cell_on, dof_on = _layer_masks(mesh, pml.zeta)
    info = eqn.pml_info()
    assert info == dict(cells=int(cell_on.sum()), dofs=int(dof_on.sum()), zeta_max=info["zeta_max"])
    assert abs(info["zeta_max"] - pml.zeta_max) <= 1e-15 * pml.zeta_max
    u, v = _random_state(mesh.ndofs, P, dtype, 0.1 if name.startswith("westervelt") else 1.0)
    t0, steps = 7.5e-6, 12
    tf = t0 + (steps - 0.5) * dt
    uo, vo, qo = u.copy(), v.copy(), np.zeros((M, mesh.ndofs))
    psio, phio = mo.pml_state(mesh, P)
    so, to = mo.rk4_westervelt_pml(mesh, P, *args, t0, tf, dt, uo, vo, qo, psio, phio, sumfact=True,
                                   nthreads=orc.max_threads())
    eqn.set_state(u, v)
    s, t = eqn.rk4(t0, tf, dt)
    ug, vg = eqn.get_state()
    psig, phig = eqn.pml_state()
    assert (s, t) == (so, to) and s == steps
    tol = TOL64 if dtype == np.float64 else TOL32_RUN
    errs = [rel_l2(ug, uo), rel_l2(vg, vo), rel_l2(psig, psio[dof_on]), rel_l2(phig, phio[cell_on])]
    if M:
        errs.append(rel_l2(eqn.relaxation_state(), qo))
    assert max(errs) < tol, errs
    # f1 at the model's memory variables, psi and phi
    q = np.ascontiguousarray(eqn.relaxation_state(), dtype=np.float64) if M else None
    psi_full, phi_full = mo.pml_state(mesh, P)
    psi_full[dof_on] = psig
    phi_full[cell_on] = phig
    fo = mo.f1_westervelt_pml(mesh, P, *args, 3e-6, u, v, q, psi_full, phi_full)
    res = torch.full((mesh.ndofs,), float("nan"), dtype=torch.float64 if dtype == np.float64 else torch.float32,
                     device="cuda")
    tdev = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(dtype))).cuda()  # noqa: E731
    eqn.f1(3e-6, tdev(u), tdev(v), res)
    torch.cuda.synchronize()
    assert rel_l2(res.cpu().numpy(), fo) < (TOL64 if dtype == np.float64 else 2e-5)


def _run(eqn, u, v, t0, tf, dt):
    eqn.set_state(u, v)
    st = eqn.rk4(t0, tf, dt)
    return st, eqn.get_state()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", ["linear", "lossy", "westervelt"])
def test_no_cells_and_a_cleared_layer_are_the_model_without_one(wfx, torch, dtype, name):
    P = 3
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.1)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    u, v = _random_state(mesh.ndofs, 3, dtype, 0.1)
    ref = _run(_model(wfx, name, mesh, P, dtype, None), u, v, 7.5e-6, 7.5e-6 + 10.5 * dt, dt)
    empty = _model(wfx, name, mesh, P, dtype, None, pml=wfx.PML(mesh, np.zeros((3, mesh.ndofs))))
    assert empty.pml_info() == dict(cells=0, dofs=0, zeta_max=0.0)
    cleared = _model(wfx, name, mesh, P, dtype, None, pml=wfx.PML.box(mesh, 0.011, GPU_FACES, C0))
    cleared.set_pml(None)
    for eqn in (empty, cleared):
        got = _run(eqn, u, v, 7.5e-6, 7.5e-6 + 10.5 * dt, dt)
        assert got[0] == ref[0]
        assert np.array_equal(got[1][0], ref[1][0]) and np.array_equal(got[1][1], ref[1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_repeated_runs_and_checkpoint_restarts_are_bitwise(wfx, torch, dtype):
    P = 4
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.1)
    rel = random_relaxation(wfx, mesh.ncells, 2, 9)
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    eqn = _model(wfx, "westervelt", mesh, P, dtype, None, rel, pml)
    dt = min(wfx.cfl_timestep(mesh.h_min, C0, P, F0), rel.max_dt(), pml.max_dt())
    u, v = _random_state(mesh.ndofs, 4, dtype, 0.1)
    full = []
    for _ in range(2):
        eqn.set_state(u, v)
        eqn.rk4(0.0, 1.0, dt, max_steps=20)
        full.append((eqn.get_state(), eqn.relaxation_state(), eqn.pml_state()))
    for a, b in zip(full[0], full[1]):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    eqn.set_state(u, v)
    _, t = eqn.rk4(0.0, 1.0, dt, max_steps=10)
    ck = (eqn.get_state(), eqn.relaxation_state(), eqn.pml_state())
    eqn.init()
    assert not np.any(eqn.pml_state()[0]) and not np.any(eqn.pml_state()[1])
    eqn.set_state(*ck[0])
    assert not np.any(eqn.pml_state()[1])
    eqn.set_relaxation_state(ck[1])
    eqn.set_pml_state(*ck[2])
    eqn.rk4(t, 1.0, dt, max_steps=10)
    got = (eqn.get_state(), eqn.relaxation_state(), eqn.pml_state())
    for a, b in zip(full[0], got):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.gpu
def test_scale_cells_before_and_after_the_layer(wfx, orc, mo, torch):
    """the layer's a_c = cK^2 coeff_c follows wfx_geometry_scale_cells whether it is called before or after the layer
    is built: bitwise the same run, and the restatement with the scaled a"""
    P = 3
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.15)
    w = np.exp(np.random.default_rng(3).uniform(np.log(0.25), np.log(4.0), mesh.ncells))
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    before = _model(wfx, "linear", mesh, P, np.float64, None)
    before.geometry.scale_cells(w)
    before.set_pml(pml)
    after = _model(wfx, "linear", mesh, P, np.float64, None, pml=pml)
    after.geometry.scale_cells(w)
    dt = min(wfx.cfl_timestep(mesh.h_min, 2 * C0, P, F0), pml.max_dt())
    u, v = _random_state(mesh.ndofs, 8, np.float64)
    out = []
    for eqn in (before, after):
        eqn.set_state(u, v)
        eqn.rk4(1e-6, 1.0, dt, max_steps=10)
        out.append((eqn.get_state(), eqn.pml_state()))
    assert all(np.array_equal(x, y) for x, y in zip(out[0][0] + out[0][1], out[1][0] + out[1][1]))
    G, m, m1, m2, _, _ = weighted_inputs(orc, mo, mesh, P, None)
    G = np.ascontiguousarray(G * w[:, None, None, None])
    inp = pml_inputs(orc, mo, mesh, P, pml.zeta, w)
    uo, vo = u.copy(), v.copy()
    psio, phio = mo.pml_state(mesh, P)
    mo.rk4_westervelt_pml(mesh, P, G, m, m1, m2, np.zeros(mesh.ndofs), C0, F0, P0, 0.0, np.zeros(0),
                          np.zeros((0, mesh.ndofs)), inp, 1e-6, 1.0, dt, uo, vo, None, psio, phio, max_steps=10,
                          sumfact=True)
    cell_on, _ = _layer_masks(mesh, pml.zeta)
    assert rel_l2(out[0][0][0], uo) < TOL64 and rel_l2(out[0][1][1], phio[cell_on]) < TOL64


@pytest.mark.gpu
def test_field_stats_with_a_layer(wfx, torch):
    """the statistics of a model with a layer sample the stepped field: peaks equal the running max / min of the
    states of single-step calls"""
    P = 3
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1], perturb=0.1)
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    eqn = _model(wfx, "lossy", mesh, P, np.float64, None, pml=pml)
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    eqn.init()
    eqn.set_field_stats(0.0, harmonics=1)
    pmax, pmin, t = np.full(mesh.ndofs, -np.inf), np.full(mesh.ndofs, np.inf), 0.0
    for _ in range(15):
        _, t = eqn.rk4(t, 1.0, dt, max_steps=1)
        u = eqn.get_state()[0]
        pmax, pmin = np.maximum(pmax, u), np.minimum(pmin, u)
    fs = eqn.field_stats()
    assert fs.samples == 15 and np.array_equal(fs.pmax, pmax) and np.array_equal(fs.pmin, pmin)
    assert np.abs(fs.pmax).max() > 0


@pytest.mark.gpu
def test_refusals_on_the_device(wfx, torch):
    import ctypes as C
    P = 2
    mesh = wfx.create_box_hex(GPU_MESH[0], P, GPU_MESH[1])
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    eqn = _model(wfx, "lossy", mesh, P, np.float64, None, pml=pml)
    def layer_of(model):
        x = np.ascontiguousarray(mesh.x, dtype=np.float64)
        h = C.c_void_p()
        wfx.capi.call("wfx_pml_create", model.ctx.handle, model.geometry.handle, mesh.ndofs,
                      wfx.capi.i32p(np.ascontiguousarray(mesh.dofmap, dtype=np.int32).reshape(-1)), x.shape[0],
                      wfx.capi.f64p(x.reshape(-1)),
                      wfx.capi.i32p(np.ascontiguousarray(mesh.xdofs, dtype=np.int32).reshape(-1)),
                      wfx.capi.f64p(pml.zeta.reshape(-1)), C.byref(h))
        return h

    # a layer built on another model's geometry, in another dtype or in another context; an ensemble model
    ens = wfx.LinearGLLEnsemble(mesh, None, P, C0, (F0, 2 * F0), (P0, P0))
    other_ctx = wfx.LossyGLLOpt(mesh, None, P, C0, F0, P0, DELTA, ctx=wfx.Context(0))
    cases = [(_model(wfx, "lossy", mesh, P, np.float64, None), eqn, "geometry"),
             (_model(wfx, "lossy", mesh, P, np.float32, None), eqn, "geometry"),
             (other_ctx, eqn, "context"), (ens, ens, "ensemble")]
    for owner, target, match in cases:
        h = layer_of(owner)
        with pytest.raises(wfx.WfxError, match=match):
            wfx.capi.call("wfx_wave_set_pml", target.handle, h)
        wfx.capi.lib.wfx_pml_destroy(h)
    # negative or non-finite zeta reach the C ABI too
    bad = pml.zeta.copy()
    bad[0, 0] = -1.0
    h = C.c_void_p()
    with pytest.raises(wfx.WfxError, match="zeta"):
        wfx.capi.call("wfx_pml_create", eqn.ctx.handle, eqn.geometry.handle, mesh.ndofs,
                      wfx.capi.i32p(np.ascontiguousarray(mesh.dofmap, dtype=np.int32).reshape(-1)), mesh.x.shape[0],
                      wfx.capi.f64p(np.ascontiguousarray(mesh.x, dtype=np.float64).reshape(-1)),
                      wfx.capi.i32p(np.ascontiguousarray(mesh.xdofs, dtype=np.int32).reshape(-1)),
                      wfx.capi.f64p(bad.reshape(-1)), C.byref(h))
    # a profile of another mesh
    small = wfx.create_box_hex((2, 2, 2), P, (0.02, 0.02, 0.02))
    with pytest.raises(wfx.WfxError, match="dofs"):
        eqn.set_pml(wfx.PML.box(small, 0.01, [(0, 1)], C0))
    # snapshots either way round
    with pytest.raises(wfx.WfxError, match="snapshot"):
        eqn.set_snapshot(1, lambda *a: None)
    plain = _model(wfx, "linear", mesh, P, np.float64, None)
    plain.set_snapshot(1, lambda *a: None)
    with pytest.raises(wfx.WfxError, match="snapshot"):
        plain.set_pml(pml)
    # the step bound, the state without a layer, state shapes
    with pytest.raises(wfx.WfxError, match="zeta"):
        eqn.rk4(0.0, 1.0, pml.max_dt())
    with pytest.raises(wfx.WfxError, match="no perfectly matched layer"):
        _model(wfx, "linear", mesh, P, np.float64, None).pml_state()
    psi, phi = eqn.pml_state()
    with pytest.raises(wfx.WfxError, match="shape"):
        eqn.set_pml_state(psi[1:], phi)
    with pytest.raises(wfx.WfxError, match="must be a PML"):
        eqn.set_pml(pml.zeta)
    # the model still steps after the refusals
    dt = wfx.cfl_timestep(mesh.h_min, C0, P, F0)
    eqn.init()
    assert eqn.rk4(0.0, 1.0, dt, max_steps=3)[0] == 3


@pytest.mark.gpu
def test_oblique_incidence_known_answer_on_the_gpu(wfx, torch):
    """the duct with its one-wavelength layer on the device (source profile, field statistics) at the restatement's
    bound"""
    mesh, P, pml, dt, k, X, amp, outgoing, _, L = _duct(wfx, True)
    eqn = wfx.LinearGLLOpt(mesh, None, P, C0, F0, P0, pml=pml)
    eqn.set_source_profile(amp, None)
    eqn.init()
    t = 0.0
    for _ in range(DUCT_N0 * k):
        t += dt
    eqn.set_field_stats(t + dt, harmonics=1)
    assert eqn.rk4(0.0, 1.0, dt, max_steps=(DUCT_N0 + DUCT_PERIODS) * k)[0] == (DUCT_N0 + DUCT_PERIODS) * k
    fs = eqn.field_stats()
    assert fs.samples == DUCT_PERIODS * k
    assert _duct_error(fs.harmonics[0], X, outgoing, L) < DUCT_BOUNDS["pml"]


@pytest.mark.gpu
def test_demo_pml_option(wfx, torch):
    """demo/planar3d.py --focus with --pml: the lateral faces and the far end become a layer with rigid outer faces; it
    runs, reports the layer and the on-axis maximum"""
    r = subprocess.run(["python", os.path.join(ROOT, "demo", "planar3d.py"), "--nx", "8", "--nyz", "8",
                        "--length", "0.012", "--focus", "0.006", "--pml", "0.0015", "--stats-periods", "2"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    out = r.stdout
    line = [ln for ln in out.splitlines() if ln.startswith("pml: ")][0]
    cells = int(line.split()[1])
    assert 0 < cells < 8 * 8 * 8 and "5 faces" in line and "zeta_max" in line, out
    assert "on-axis maximum" in out, out


# ---- C++ wrapper ---------------------------------------------------------------------------------------------------
def _build_cpp(wfx, outdir):
    src = os.path.join(ROOT, "tests", "cpp", "test_wavefx_pml_hpp.cpp")
    exe = os.path.join(str(outdir), "test_wavefx_pml_hpp")
    libdir = os.path.dirname(wfx.capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "wave-fenics_b200", "hpp"), src, "-o", exe,
           "-L", libdir, "-l:libwavefx.so", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_pml_cpp_wrapper_compiles_and_links(wfx, tmp_path):
    assert os.path.exists(_build_cpp(wfx, tmp_path))


@pytest.mark.gpu
def test_pml_cpp_wrapper_reproduces_python(wfx, torch, tmp_path):
    """LossyGLLOpt with a medium and set_pml from C++, 15 steps, get / set of psi and phi through a restart, 15 more:
    the same u, psi and phi as the Python model bit for bit"""
    P = 3
    mesh = wfx.create_box_hex((3, 2, 2), P, (0.03, 0.02, 0.02), perturb=0.15)
    med = random_medium(wfx, mesh.ncells, 91, beta=False)
    pml = wfx.PML.box(mesh, 0.011, GPU_FACES, C0)
    dt = min(wfx.cfl_timestep(mesh.h_min, med.c_max, P, F0), pml.max_dt())
    u, v = _random_state(mesh.ndofs, 5, np.float64)
    lossy = _model(wfx, "lossy", mesh, P, np.float64, med, pml=pml)
    files = {"params.f64": np.array([P, C0, F0, P0, DELTA, dt]),
             "x.f64": mesh.x, "xdofs.i32": mesh.xdofs, "dofmap.i32": mesh.dofmap,
             "fcell.i32": mesh.facet_cells, "flocal.i32": mesh.facet_local, "ftag.i32": mesh.facet_tags,
             "u.f64": u, "v.f64": v, "stiffness.f64": med.stiffness_weight(mesh.ncells),
             "mass.f64": med.mass_weight(mesh.ncells, C0), "facet.f64": med.facet_weight(mesh, C0),
             "zeta.f64": pml.zeta}
    for name, a in files.items():
        np.ascontiguousarray(a, dtype=np.int32 if name.endswith("i32") else np.float64).tofile(str(tmp_path / name))
    r = subprocess.run([_build_cpp(wfx, tmp_path), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "pml hpp ok" in r.stdout, r.stdout + r.stderr
    lossy.set_state(u, v)
    _, t1 = lossy.rk4(0.0, 1.0, dt, max_steps=15)
    cu, cv = lossy.get_state()
    cpsi, cphi = lossy.pml_state()
    lossy.set_state(cu, cv)
    lossy.set_pml_state(cpsi, cphi)
    lossy.rk4(t1, 1.0, dt, max_steps=15)
    got = lambda name: np.fromfile(str(tmp_path / name), dtype=np.float64)  # noqa: E731
    psi, phi = lossy.pml_state()
    assert np.array_equal(got("u.out.f64"), lossy.get_state()[0])
    assert np.array_equal(got("psi.out.f64"), psi) and np.array_equal(got("phi.out.f64"), phi.reshape(-1))
