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
