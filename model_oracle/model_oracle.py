"""ctypes loader for the CPU restatement of the lossy and Westervelt models and of the Pennes thermal model
(model_oracle.c).

TEST INFRASTRUCTURE ONLY -- imported by tests/, the demo's --check and tools/, never by the product package.
Built with the strict flags of oracle/oracle.py, so that its linear part computes what the oracle computes.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

from oracle import oracle as _orc

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "model_oracle.c")
DEPS = (SRC, _orc.SRC)
OUT = os.path.join(HERE, "_build")

_i32p = C.POINTER(C.c_int32)
_f64p = C.POINTER(C.c_double)


def _out_dir():
    """model_oracle/_build, or the oracle's temporary directory when the checkout is read-only."""
    try:
        os.makedirs(OUT, exist_ok=True)
        if os.access(OUT, os.W_OK):
            return OUT
    except OSError:
        pass
    return _orc._out_dir()


def build(force=False):
    h = hashlib.sha256()
    for f in DEPS:
        with open(f, "rb") as fh:
            h.update(fh.read())
    name = f"libmodel_oracle_{h.hexdigest()[:12]}.so"
    path = os.path.join(OUT, name)
    if force or not os.path.exists(path):
        path = os.path.join(_out_dir(), name)
    if force or not os.path.exists(path):
        cmd = [_orc.GCC, "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC",
               "-o", path + ".tmp", SRC, "-lm"]
        subprocess.run(cmd, check=True)
        os.replace(path + ".tmp", path)
    return path


_lib = []


def lib():
    if not _lib:
        L = C.CDLL(build())
        i, l, d = C.c_int, C.c_int64, C.c_double
        L.wo_source.restype, L.wo_source.argtypes = None, [d, d, d, d, _f64p, _f64p]
        L.wo_f1_westervelt.restype = None
        L.wo_f1_westervelt.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d, d, _f64p, _f64p,
                                       _f64p, i, i]
        L.wo_rk4_westervelt.restype = l
        L.wo_rk4_westervelt.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d, d, d, d, l,
                                        _f64p, _f64p, i, i, _f64p]
        L.wo_f1_westervelt_profile.restype = None
        L.wo_f1_westervelt_profile.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d, _f64p,
                                               _f64p, d, _f64p, _f64p, _f64p, i, i]
        L.wo_rk4_westervelt_profile.restype = l
        L.wo_rk4_westervelt_profile.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d, _f64p,
                                                _f64p, d, d, d, l, _f64p, _f64p, i, i, _f64p]
        L.wo_rhs_pennes.restype = None
        L.wo_rhs_pennes.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, _f64p, _f64p, d, d, d, d, d, _f64p,
                                    d, _f64p, _f64p, i, i]
        L.wo_rk4_pennes.restype = l
        L.wo_rk4_pennes.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, _f64p, _f64p, d, d, d, d, d, _f64p,
                                    d, d, d, d, l, _f64p, _f64p, _f64p, i, i, _f64p]
        L.wo_boundary_facet_mass_weighted.restype = i
        L.wo_boundary_facet_mass_weighted.argtypes = [i, l, _i32p, _i32p, _i32p, _f64p, _i32p, _i32p, _f64p, _f64p,
                                                      _f64p]
        L.wo_f1_westervelt_medium.restype = None
        L.wo_f1_westervelt_medium.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, _f64p,
                                              _f64p, _f64p, i, i]
        L.wo_rk4_westervelt_medium.restype = l
        L.wo_rk4_westervelt_medium.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d, d,
                                               l, _f64p, _f64p, i, i, _f64p]
        L.wo_f1_westervelt_relax.restype = None
        L.wo_f1_westervelt_relax.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, i, _f64p,
                                             _f64p, d, _f64p, _f64p, _f64p, _f64p, i, i]
        L.wo_rk4_westervelt_relax.restype = l
        L.wo_rk4_westervelt_relax.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, i, _f64p,
                                              _f64p, d, d, d, l, _f64p, _f64p, _f64p, i, i, _f64p]
        L.wo_f1_westervelt_pml.restype = None
        L.wo_f1_westervelt_pml.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, i, _f64p,
                                           _f64p, _f64p, _f64p, _f64p, _f64p, d, _f64p, _f64p, _f64p, _f64p, _f64p,
                                           _f64p, i, i]
        L.wo_rk4_westervelt_pml.restype = l
        L.wo_rk4_westervelt_pml.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, i, _f64p,
                                            _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, l, _f64p, _f64p, _f64p, _f64p,
                                            _f64p, i, i, _f64p]
        L.wo_f1_westervelt_source.restype = None
        L.wo_f1_westervelt_source.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, i, _f64p,
                                              _f64p, _f64p, _f64p, _f64p, _f64p, l, _i32p, _f64p, _f64p, d, _f64p,
                                              _f64p, _f64p, _f64p, _f64p, _f64p, i, i]
        L.wo_rk4_westervelt_source.restype = l
        L.wo_rk4_westervelt_source.argtypes = [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, i, _f64p,
                                               _f64p, _f64p, _f64p, _f64p, _f64p, l, _i32p, _f64p, _f64p, d, d, d, l,
                                               _f64p, _f64p, _f64p, _f64p, _f64p, i, i, _f64p]
        _lib.append(L)
    return _lib[0]


def _f(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_f64p)


def source(t, f0, p0, c0):
    """(g(t), g'(t)) of the source: g as wfx_wave.cu's source_amplitude, g' analytic."""
    g, gd = C.c_double(), C.c_double()
    lib().wo_source(float(t), float(f0), float(p0), float(c0), C.byref(g), C.byref(gd))
    return g.value, gd.value


def f1_westervelt(mesh, P, G, m, m1, m2, c0, f0, p0, delta, beta, rho0, t, u, v, sumfact=False, nthreads=1):
    """p_tt of the lumped lossy / Westervelt system at (t, u, v)."""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    out = np.empty(mesh.ndofs)
    lib().wo_f1_westervelt(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m), _f(m1),
                           _f(m2), c0, f0, p0, delta, beta, rho0, t, _f(u), _f(v), _f(out), int(sumfact), nthreads)
    return out


def rk4_westervelt(mesh, P, G, m, m1, m2, c0, f0, p0, delta, beta, rho0, t0, tf, dt, u, v, max_steps=0,
                   sumfact=False, nthreads=1):
    """RK4 of the lossy / Westervelt model; u, v updated in place.  -> (steps, t_end)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    t_end = C.c_double()
    steps = lib().wo_rk4_westervelt(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m),
                                    _f(m1), _f(m2), c0, f0, p0, delta, beta, rho0, t0, tf, dt, max_steps, _f(u),
                                    _f(v), int(sumfact), nthreads, C.byref(t_end))
    return steps, t_end.value



def _profile(mesh, amp, delay):
    amp = np.ones(mesh.ndofs) if amp is None else np.ascontiguousarray(amp, dtype=np.float64)
    delay = np.zeros(mesh.ndofs) if delay is None else np.ascontiguousarray(delay, dtype=np.float64)
    assert amp.shape == delay.shape == (mesh.ndofs,)
    return amp, delay


def f1_westervelt_profile(mesh, P, G, m, m1, m2, c0, f0, p0, delta, beta, rho0, amp, delay, t, u, v, sumfact=False,
                          nthreads=1):
    """f1_westervelt with the source amp[i] g(t - delay[i]) at dof i (zero before the delay); None: 1 / 0."""
    amp, delay = _profile(mesh, amp, delay)
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    out = np.empty(mesh.ndofs)
    lib().wo_f1_westervelt_profile(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m),
                                   _f(m1), _f(m2), c0, f0, p0, delta, beta, rho0, _f(amp), _f(delay), t, _f(u), _f(v),
                                   _f(out), int(sumfact), nthreads)
    return out


def rk4_westervelt_profile(mesh, P, G, m, m1, m2, c0, f0, p0, delta, beta, rho0, amp, delay, t0, tf, dt, u, v,
                           max_steps=0, sumfact=False, nthreads=1):
    """rk4_westervelt with a source profile (see f1_westervelt_profile); u, v updated in place.  -> (steps, t_end)"""
    amp, delay = _profile(mesh, amp, delay)
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    t_end = C.c_double()
    steps = lib().wo_rk4_westervelt_profile(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)),
                                            _f(m), _f(m1), _f(m2), c0, f0, p0, delta, beta, rho0, _f(amp), _f(delay),
                                            t0, tf, dt, max_steps, _f(u), _f(v), int(sumfact), nthreads,
                                            C.byref(t_end))
    return steps, t_end.value


def _opt(a):
    return None if a is None else _f(np.ascontiguousarray(a, dtype=np.float64))


def rhs_pennes(mesh, P, G, m, m1, m2, k, rhoc, perf, T_art, h, T_ext, Q, s, theta, sumfact=False, nthreads=1):
    """theta' of the lumped Pennes system (DESIGN.md section 4.5d) at theta = T - T_art.  rhoc [ndofs]; perf, Q
    [ndofs] or None (0); h, T_ext: the two Robin tags' (h1, h2) and (T_ext1, T_ext2)."""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    rhoc = np.ascontiguousarray(rhoc, dtype=np.float64)
    perf = None if perf is None else np.ascontiguousarray(perf, dtype=np.float64)
    Q = None if Q is None else np.ascontiguousarray(Q, dtype=np.float64)
    out = np.empty(mesh.ndofs)
    lib().wo_rhs_pennes(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m), _f(m1), _f(m2),
                        k, _f(rhoc), _opt(perf), T_art, h[0], h[1], T_ext[0], T_ext[1], _opt(Q), s,
                        _f(np.ascontiguousarray(theta, dtype=np.float64)), _f(out), int(sumfact), nthreads)
    return out


def rk4_pennes(mesh, P, G, m, m1, m2, k, rhoc, perf, T_art, h, T_ext, Q, s, t0, tf, dt, theta, cem43, theta_max,
               max_steps=0, sumfact=False, nthreads=1):
    """RK4 of the Pennes model with the CEM43 dose and the peak rise; theta, cem43, theta_max updated in place.
    -> (steps, t_end)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    rhoc = np.ascontiguousarray(rhoc, dtype=np.float64)
    perf = None if perf is None else np.ascontiguousarray(perf, dtype=np.float64)
    Q = None if Q is None else np.ascontiguousarray(Q, dtype=np.float64)
    t_end = C.c_double()
    steps = lib().wo_rk4_pennes(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m), _f(m1),
                                _f(m2), k, _f(rhoc), _opt(perf), T_art, h[0], h[1], T_ext[0], T_ext[1], _opt(Q), s,
                                t0, tf, dt, max_steps, _f(theta), _f(cem43), _f(theta_max), int(sumfact), nthreads,
                                C.byref(t_end))
    return steps, t_end.value


# ---- layered media (DESIGN.md section 4.5e) -------------------------------------------------------------------------
def boundary_facet_mass_weighted(mesh, P, facet_weight):
    """(m1, m2) of oracle.boundary_facet_mass with facet f's GLL facet mass multiplied by facet_weight[f]"""
    x = np.ascontiguousarray(mesh.x, dtype=np.float64)
    xd = np.ascontiguousarray(mesh.xdofs, dtype=np.int32)
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    fc = np.ascontiguousarray(mesh.facet_cells, dtype=np.int32)
    fl = np.ascontiguousarray(mesh.facet_local, dtype=np.int32)
    ft = np.ascontiguousarray(mesh.facet_tags, dtype=np.int32)
    fw = np.ascontiguousarray(facet_weight, dtype=np.float64)
    assert fw.shape == (len(fc),)
    m1, m2 = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    ip = lambda a: a.ctypes.data_as(_i32p)  # noqa: E731
    assert lib().wo_boundary_facet_mass_weighted(P, len(fc), ip(fc), ip(fl), ip(ft), _f(x.reshape(-1)),
                                                 ip(xd.reshape(-1)), ip(dm.reshape(-1)), _f(fw), _f(m1), _f(m2)) == 0
    return m1, m2


def f1_westervelt_medium(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, t, u, v, sumfact=False, nthreads=1):
    """f1_westervelt in a layered medium: G, m, m1, m2 weighted as given, kappa [ndofs] per dof"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    out = np.empty(mesh.ndofs)
    lib().wo_f1_westervelt_medium(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m),
                                  _f(m1), _f(m2), _f(np.ascontiguousarray(kappa, dtype=np.float64)), c0, f0, p0, delta,
                                  t, _f(u), _f(v), _f(out), int(sumfact), nthreads)
    return out


def rk4_westervelt_medium(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, t0, tf, dt, u, v, max_steps=0,
                          sumfact=False, nthreads=1):
    """rk4_westervelt in a layered medium (see f1_westervelt_medium); u, v updated in place.  -> (steps, t_end)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    kappa = np.ascontiguousarray(kappa, dtype=np.float64)
    assert kappa.shape == (mesh.ndofs,)
    t_end = C.c_double()
    steps = lib().wo_rk4_westervelt_medium(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)),
                                           _f(m), _f(m1), _f(m2), _f(kappa), c0, f0, p0, delta, t0, tf, dt, max_steps,
                                           _f(u), _f(v), int(sumfact), nthreads, C.byref(t_end))
    return steps, t_end.value


# ---- relaxation absorption (DESIGN.md section 4.5f) -----------------------------------------------------------------
def _relax(mesh, tau, eps, q):
    tau = np.ascontiguousarray(tau, dtype=np.float64).reshape(-1)
    M = len(tau)
    eps = np.ascontiguousarray(eps, dtype=np.float64).reshape(M, mesh.ndofs)
    q = np.zeros((M, mesh.ndofs)) if q is None else q
    assert q.dtype == np.float64 and q.shape == (M, mesh.ndofs) and q.flags["C_CONTIGUOUS"]
    p = lambda a: _f(a.reshape(-1)) if a.size else _f(np.zeros(1))  # noqa: E731
    return M, p(tau), p(eps), q, p(q)


def f1_westervelt_relax(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, tau, eps, t, u, v, q=None, sumfact=False,
                        nthreads=1):
    """f1_westervelt_medium with M relaxation processes: tau [M], eps [M, ndofs], memory variables q [M, ndofs]
    (None: 0)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    M, tp, ep, _, qp = _relax(mesh, tau, eps, q)
    out = np.empty(mesh.ndofs)
    lib().wo_f1_westervelt_relax(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m),
                                 _f(m1), _f(m2), _f(np.ascontiguousarray(kappa, dtype=np.float64)), c0, f0, p0, delta,
                                 M, tp, ep, t, _f(u), _f(v), qp, _f(out), int(sumfact), nthreads)
    return out


def rk4_westervelt_relax(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, tau, eps, t0, tf, dt, u, v, q, max_steps=0,
                         sumfact=False, nthreads=1):
    """rk4_westervelt_medium with relaxation (see f1_westervelt_relax); u, v and q [M, ndofs] updated in place.
    -> (steps, t_end)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    kappa = np.ascontiguousarray(kappa, dtype=np.float64)
    assert kappa.shape == (mesh.ndofs,)
    M, tp, ep, q, qp = _relax(mesh, tau, eps, q)
    t_end = C.c_double()
    steps = lib().wo_rk4_westervelt_relax(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)),
                                          _f(m), _f(m1), _f(m2), _f(kappa), c0, f0, p0, delta, M, tp, ep, t0, tf, dt,
                                          max_steps, _f(u), _f(v), qp, int(sumfact), nthreads, C.byref(t_end))
    return steps, t_end.value


# ---- perfectly matched layer (DESIGN.md section 4.5g) --------------------------------------------------------------
class PMLInputs:
    """The layer's inputs of the restatement: zeta [3, ndofs], K = J^-1 [ncells, nq, 3, 3] and dJw = |detJ| w
    [ncells, nq] at the GLL points in tensor order (the reference layout of oracle.precompute_geometric_data), and the
    cells' composed stiffness coefficient coeff [ncells] (a_c = 1500^2 coeff_c)."""

    def __init__(self, mesh, P, zeta, K, dJw, coeff=None):
        nq = (P + 1) ** 3
        self.zeta = np.ascontiguousarray(zeta, dtype=np.float64).reshape(3, mesh.ndofs)
        self.K = np.ascontiguousarray(K, dtype=np.float64).reshape(mesh.ncells, nq, 3, 3)
        self.dJw = np.ascontiguousarray(dJw, dtype=np.float64).reshape(mesh.ncells, nq)
        self.coeff = (np.ones(mesh.ncells) if coeff is None
                      else np.ascontiguousarray(coeff, dtype=np.float64).reshape(mesh.ncells))

    def args(self):
        return (_f(self.zeta.reshape(-1)), _f(self.K.reshape(-1)), _f(self.dJw.reshape(-1)), _f(self.coeff))


def pml_state(mesh, P):
    """zero (psi [ndofs], phi [ncells, nq, 3])"""
    return np.zeros(mesh.ndofs), np.zeros((mesh.ncells, (P + 1) ** 3, 3))


def f1_westervelt_pml(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, tau, eps, pml, t, u, v, q=None, psi=None,
                      phi=None, sumfact=False, nthreads=1):
    """f1_westervelt_relax with a perfectly matched layer (pml: PMLInputs) at psi [ndofs], phi [ncells, nq, 3]
    (None: 0)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    M, tp, ep, _, qp = _relax(mesh, tau, eps, q)
    z_psi, z_phi = pml_state(mesh, P)
    psi = z_psi if psi is None else np.ascontiguousarray(psi, dtype=np.float64)
    phi = z_phi if phi is None else np.ascontiguousarray(phi, dtype=np.float64)
    out = np.empty(mesh.ndofs)
    lib().wo_f1_westervelt_pml(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m), _f(m1),
                               _f(m2), _f(np.ascontiguousarray(kappa, dtype=np.float64)), c0, f0, p0, delta, M, tp, ep,
                               *pml.args(), t, _f(u), _f(v), qp, _f(psi), _f(phi.reshape(-1)), _f(out), int(sumfact),
                               nthreads)
    return out


def rk4_westervelt_pml(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, tau, eps, pml, t0, tf, dt, u, v, q, psi, phi,
                       max_steps=0, sumfact=False, nthreads=1):
    """rk4_westervelt_relax with a perfectly matched layer (see f1_westervelt_pml); u, v, q, psi [ndofs] and phi
    [ncells, nq, 3] updated in place.  -> (steps, t_end)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    kappa = np.ascontiguousarray(kappa, dtype=np.float64)
    assert kappa.shape == (mesh.ndofs,)
    M, tp, ep, q, qp = _relax(mesh, tau, eps, q)
    for a in (psi, phi):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    assert psi.shape == (mesh.ndofs,) and phi.shape == (mesh.ncells, (P + 1) ** 3, 3)
    t_end = C.c_double()
    steps = lib().wo_rk4_westervelt_pml(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)),
                                        _f(m), _f(m1), _f(m2), _f(kappa), c0, f0, p0, delta, M, tp, ep, *pml.args(),
                                        t0, tf, dt, max_steps, _f(u), _f(v), qp, _f(psi), _f(phi.reshape(-1)),
                                        int(sumfact), nthreads, C.byref(t_end))
    return steps, t_end.value


# ---- volume sources (DESIGN.md section 4.5h) -----------------------------------------------------------------------
def _vsrc(dofs, q, delay):
    dofs = np.ascontiguousarray(np.zeros(0) if dofs is None else dofs, dtype=np.int32).reshape(-1)
    q = np.ascontiguousarray(np.zeros(0) if q is None else q, dtype=np.float64).reshape(-1)
    delay = np.zeros(len(dofs)) if delay is None else np.ascontiguousarray(delay, dtype=np.float64).reshape(-1)
    assert len(dofs) == len(q) == len(delay)
    return len(dofs), dofs.ctypes.data_as(_i32p), _f(q), _f(delay), (dofs, q, delay)


def f1_westervelt_source(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, tau, eps, pml, dofs, q_src, delay, t, u, v,
                         q=None, psi=None, phi=None, sumfact=False, nthreads=1):
    """f1_westervelt_pml with a volume source: c0^2 q_src[p] g(t - delay[p]) added at dof dofs[p] (delay None: 0)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    M, tp, ep, _, qp = _relax(mesh, tau, eps, q)
    z_psi, z_phi = pml_state(mesh, P)
    psi = z_psi if psi is None else np.ascontiguousarray(psi, dtype=np.float64)
    phi = z_phi if phi is None else np.ascontiguousarray(phi, dtype=np.float64)
    ns, sd, sq, sl, _keep = _vsrc(dofs, q_src, delay)
    out = np.empty(mesh.ndofs)
    lib().wo_f1_westervelt_source(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)), _f(m),
                                  _f(m1), _f(m2), _f(np.ascontiguousarray(kappa, dtype=np.float64)), c0, f0, p0, delta,
                                  M, tp, ep, *pml.args(), ns, sd, sq, sl, t, _f(u), _f(v), qp, _f(psi),
                                  _f(phi.reshape(-1)), _f(out), int(sumfact), nthreads)
    return out


def rk4_westervelt_source(mesh, P, G, m, m1, m2, kappa, c0, f0, p0, delta, tau, eps, pml, dofs, q_src, delay, t0, tf,
                          dt, u, v, q, psi, phi, max_steps=0, sumfact=False, nthreads=1):
    """rk4_westervelt_pml with a volume source (see f1_westervelt_source); u, v, q, psi and phi updated in place.
    -> (steps, t_end)"""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    kappa = np.ascontiguousarray(kappa, dtype=np.float64)
    assert kappa.shape == (mesh.ndofs,)
    M, tp, ep, q, qp = _relax(mesh, tau, eps, q)
    for a in (psi, phi):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    assert psi.shape == (mesh.ndofs,) and phi.shape == (mesh.ncells, (P + 1) ** 3, 3)
    ns, sd, sq, sl, _keep = _vsrc(dofs, q_src, delay)
    t_end = C.c_double()
    steps = lib().wo_rk4_westervelt_source(P, mesh.ncells, mesh.ndofs, dm.ctypes.data_as(_i32p), _f(G.reshape(-1)),
                                           _f(m), _f(m1), _f(m2), _f(kappa), c0, f0, p0, delta, M, tp, ep, *pml.args(),
                                           ns, sd, sq, sl, t0, tf, dt, max_steps, _f(u), _f(v), qp, _f(psi),
                                           _f(phi.reshape(-1)), int(sumfact), nthreads, C.byref(t_end))
    return steps, t_end.value
