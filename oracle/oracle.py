"""ctypes loader for the CPU oracle (oracle/wave_oracle.c).

TEST INFRASTRUCTURE ONLY -- imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  Never imported by the product package.
PARITY UNPINNED for the C restatement (see the header of wave_oracle.c); the reference's own CUDA
primitives, the one part of the path that compiles here, are available through ref_cuda().
"""
import atexit
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "wave_oracle.c")
OUT = os.path.join(HERE, "_build")
GCC = os.environ.get("ORACLE_GCC", "/usr/bin/gcc")
_tmp_out = []

_i32p = C.POINTER(C.c_int32)
_f64p = C.POINTER(C.c_double)


def _cpu_tag():
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags"):
                    return hashlib.sha256(line.encode()).hexdigest()[:12]
    except OSError:
        pass
    return "unknown"


def _out_dir():
    """oracle/_build, or a private temporary directory (removed at exit) when the checkout is read-only."""
    try:
        os.makedirs(OUT, exist_ok=True)
        if os.access(OUT, os.W_OK):
            return OUT
    except OSError:
        pass
    if not _tmp_out:
        _tmp_out.append(tempfile.mkdtemp(prefix="wfx_oracle_"))
        atexit.register(shutil.rmtree, _tmp_out[0], True)
    return _tmp_out[0]


def build(fast=False, force=False):
    """strict: IEEE build for parity.  fast: the reference's -Ofast -march=native flags
    (demo/cpu_planar3d/CMakeLists.txt:27) for CPU-baseline timing; rebuilt per host CPU."""
    with open(SRC, "rb") as fh:
        dig = hashlib.sha256(fh.read()).hexdigest()[:12]
    if fast:
        name, flags = f"liboracle_fast_{_cpu_tag()}_{dig}.so", ["-Ofast", "-march=native", "-mprefer-vector-width=512"]
    else:
        name, flags = f"liboracle_{dig}.so", ["-O2", "-march=x86-64-v3", "-ffp-contract=off"]
    path = os.path.join(OUT, name)
    if force or not os.path.exists(path):
        path = os.path.join(_out_dir(), name)
    if force or not os.path.exists(path):
        cmd = [GCC, *flags, "-fopenmp", "-shared", "-fPIC", "-o", path + ".tmp", SRC, "-lm"]
        subprocess.run(cmd, check=True)
        os.replace(path + ".tmp", path)
    return path


_libs = {}


def lib(fast=False):
    if fast not in _libs:
        L = C.CDLL(build(fast))
        i, l, d = C.c_int, C.c_int64, C.c_double
        sig = {
            "wo_gll": (i, [i, _f64p, _f64p]),
            "wo_deriv_1d": (i, [i, _f64p, i]),
            "wo_perm": (i, [i, _i32p]),
            "wo_tabulate_dphi": (i, [i, _f64p]),
            "wo_reorder_dofmap": (None, [i, l, _i32p, _i32p]),
            "wo_precompute_geometric_data": (i, [i, l, _f64p, _i32p, _f64p, _f64p]),
            "wo_compute_jacobian": (None, [l, i, _f64p, _f64p, _i32p, _f64p]),
            "wo_compute_jacobian_determinant": (None, [l, _f64p, _f64p]),
            "wo_compute_jacobian_inverse": (None, [l, _f64p, _f64p]),
            "wo_compute_geometrical_factor": (None, [l, i, _f64p, _f64p, _f64p, _f64p]),
            "wo_gauss_legendre": (i, [i, _f64p, _f64p]),
            "wo_tabulate_1d": (i, [i, i, _f64p, i, _f64p]),
            "wo_mass_apply": (None, [i, l, _i32p, _f64p, _f64p, _f64p]),
            "wo_stiffness_apply_dense": (None, [i, l, l, _i32p, _f64p, _f64p, _f64p, i]),
            "wo_stiffness_apply_sumfact": (None, [i, l, l, _i32p, _f64p, _f64p, _f64p, i]),
            "wo_boundary_facet_mass": (i, [i, l, _i32p, _i32p, _i32p, _f64p, _i32p, _i32p, _f64p, _f64p]),
            "wo_rk4": (l, [i, l, l, _i32p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d, l, _f64p, _f64p,
                           i, i, _f64p]),
            "wo_max_threads": (i, []),
            "wo_clamp_value": (d, [d]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _libs[fast] = L
    return _libs[fast]


def ref_cuda():
    """ctypes handle of oracle/_ref/libwfref_cuda.so -- the REFERENCE's own CUDA primitives (gather,
    atomic scatter, transform1; common/cuda/scatter.cu, transform.cu) compiled from /root/reference by
    oracle/build_ref.py -- or None when it has not been built.  Device pointers, default stream,
    synchronous (the reference calls cudaDeviceSynchronize after every launch)."""
    from . import build_ref
    path = build_ref.build()
    if not path or not os.path.exists(path):
        return None
    L = C.CDLL(path)
    vp, i32 = C.c_void_p, C.c_int32
    for name in ("ref_gather_f64", "ref_gather_f32", "ref_scatter_f64", "ref_scatter_f32"):
        getattr(L, name).argtypes = [i32, vp, vp, vp]
        getattr(L, name).restype = None
    for name in ("ref_transform1_f64", "ref_transform1_f32"):
        getattr(L, name).argtypes = [i32, vp, vp, vp]
        getattr(L, name).restype = None
    return L


def ref_cpu(fast=False):
    """ctypes handle of oracle/_ref/libwfref_cpu.so (fast: libwfref_cpu_fast.so, the same code at -Ofast for timing) -- the REFERENCE's own cell kernels skernel and mkernel
    (common/operators.hpp:113-133, 36-40), cut out of the header where it lies under /root/reference and
    compiled by oracle/build_ref.py -- or None when it has not been built.
      wfref_skernel(A[nd] (+=), w[nd], G[nq][3][3], dphi[3][nq][nd], nq, nd)
      wfref_mkernel(A[nq] (=), w[nq], detJ[nq], nq, nd)"""
    from . import build_ref
    path = build_ref.build_cpu()
    if fast and path:
        path = build_ref.LIB_CPU_FAST
    if not path or not os.path.exists(path):
        return None
    L = C.CDLL(path)
    L.wfref_skernel.argtypes = [_f64p, _f64p, _f64p, _f64p, C.c_int, C.c_int]
    L.wfref_skernel.restype = None
    L.wfref_mkernel.argtypes = [_f64p, _f64p, _f64p, C.c_int, C.c_int]
    L.wfref_mkernel.restype = None
    L.wfref_stiffness_apply.argtypes = [C.c_int, C.c_int, C.c_int, _i32p, _f64p, _f64p, _f64p, _f64p]
    L.wfref_stiffness_apply.restype = None
    L.wfref_mass_apply.argtypes = [C.c_int, C.c_int, C.c_int, _i32p, _f64p, _i32p, _f64p, _f64p]
    L.wfref_mass_apply.restype = None
    d = C.c_double
    L.wfref_rk4.argtypes = [C.c_int, C.c_int, C.c_int, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d, d, d,
                            _f64p, _f64p]
    L.wfref_rk4.restype = None
    L.wfref_f1.argtypes = [C.c_int, C.c_int, C.c_int, _i32p, _f64p, _f64p, _f64p, _f64p, _f64p, d, d, d, d,
                           _f64p, _f64p, _f64p]
    L.wfref_f1.restype = None
    return L


def ref_mesh():
    """ctypes handle of oracle/_ref/libwfref_mesh.so -- the REFERENCE's own decompose3d and
    compute_cartesian_indices (demo/gpu_cg/mesh.hpp:37-62) -- or None when it has not been built."""
    from . import build_ref
    path = build_ref.build_mesh()
    if not path or not os.path.exists(path):
        return None
    L = C.CDLL(path)
    L.wfref_decompose3d.argtypes = [C.c_int, C.POINTER(C.c_int)]
    L.wfref_decompose3d.restype = None
    L.wfref_cartesian_indices.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_longlong)]
    L.wfref_cartesian_indices.restype = None
    L.wfref_reorder_dofmap.argtypes = [C.c_int, C.c_int, C.c_int, _i32p, _i32p, _i32p]
    L.wfref_reorder_dofmap.restype = None
    L.wfref_demo_time_parameters.argtypes = [C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, _f64p, _f64p,
                                             C.POINTER(C.c_int)]
    L.wfref_demo_time_parameters.restype = None
    L.wfref_dot.argtypes = [_f64p, C.c_int, C.c_int, _f64p, C.c_int, C.c_int, _f64p, C.c_int]
    L.wfref_dot.restype = None
    return L


def reference_stiffness_apply(mesh, P, G, x, y):
    """y += A x through the REFERENCE's own StiffnessOperator::operator() and skernel
    (common/operators.hpp:182-200, 113-133), compiled into oracle/_ref/libwfref_cpu.so."""
    nd = (P + 1) ** 3
    dphi = np.ascontiguousarray(tabulate_dphi(P))
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    G = np.ascontiguousarray(G, dtype=np.float64)
    ref_cpu().wfref_stiffness_apply(mesh.ncells, mesh.ndofs, nd, _i(dm.reshape(-1)), _f(G.reshape(-1)),
                                    _f(dphi.reshape(-1)), _f(x), _f(y))


def reference_mass_apply(mesh, P, detJ, x, y):
    """y += M x through the REFERENCE's own MassOperatorCPU::operator() and mkernel
    (common/operators.hpp:85-108, 36-40)."""
    nd = (P + 1) ** 3
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    detJ = np.ascontiguousarray(detJ, dtype=np.float64)
    pm = np.ascontiguousarray(perm(P), dtype=np.int32)
    ref_cpu().wfref_mass_apply(mesh.ncells, mesh.ndofs, nd, _i(dm.reshape(-1)), _f(detJ.reshape(-1)), _i(pm),
                               _f(x), _f(y))


def reference_rk4(mesh, P, G, m, m1, m2, c0, f0, p0, t0, tf, dt, u, v):
    """The REFERENCE's own LinearGLLOpt::rk4 / f0 / f1 / kernels::copy / axpy (common/LinearGLL.hpp:15-35,
    130-287) around its own stiffness operator; u, v updated in place.  The boundary form (FFCx kernel in
    the reference) is the diagonal GLL facet form with the facet masses m1, m2."""
    nd = (P + 1) ** 3
    dphi = np.ascontiguousarray(tabulate_dphi(P))
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    G = np.ascontiguousarray(G, dtype=np.float64)
    ref_cpu().wfref_rk4(mesh.ncells, mesh.ndofs, nd, _i(dm.reshape(-1)), _f(G.reshape(-1)), _f(dphi.reshape(-1)),
                        _f(m), _f(m1), _f(m2), c0, f0, p0, t0, tf, dt, _f(u), _f(v))


def reference_f1(mesh, P, G, m, m1, m2, c0, f0, p0, t, u, v):
    """dv/dt = f1(t, u, v) through the REFERENCE's own LinearGLLOpt::f1 (common/LinearGLL.hpp:151-192)."""
    nd = (P + 1) ** 3
    dphi = np.ascontiguousarray(tabulate_dphi(P))
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    G = np.ascontiguousarray(G, dtype=np.float64)
    out = np.empty(mesh.ndofs)
    ref_cpu().wfref_f1(mesh.ncells, mesh.ndofs, nd, _i(dm.reshape(-1)), _f(G.reshape(-1)), _f(dphi.reshape(-1)),
                       _f(m), _f(m1), _f(m2), c0, f0, p0, t, _f(u), _f(v), _f(out))
    return out


def _f(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_f64p)


def _i(a):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_i32p)


def max_threads():
    return lib().wo_max_threads()


def gll(P):
    p, w = np.empty(P + 1), np.empty(P + 1)
    assert lib().wo_gll(P, _f(p), _f(w)) == 0
    return p, w


def deriv_1d(P, clamp=True):
    D = np.empty((P + 1, P + 1))
    assert lib().wo_deriv_1d(P, _f(D), int(clamp)) == 0
    return D


def perm(P):
    out = np.empty((P + 1) ** 3, dtype=np.int32)
    assert lib().wo_perm(P, _i(out)) == 0
    return out


def tabulate_dphi(P):
    nd = (P + 1) ** 3
    out = np.empty((3, nd, nd))
    assert lib().wo_tabulate_dphi(P, _f(out)) == 0
    return out


def reorder_dofmap(dofmap, P):
    dofmap = np.ascontiguousarray(dofmap, dtype=np.int32)
    out = np.empty_like(dofmap)
    lib().wo_reorder_dofmap(P, dofmap.size // (P + 1) ** 3, _i(dofmap.reshape(-1)), _i(out.reshape(-1)))
    return out


def precompute_geometric_data(mesh, P):
    """-> (G [nc,nq,3,3], detJ [nc,nq])   common/precomputation.hpp:18-110"""
    nq = (P + 1) ** 3
    x = np.ascontiguousarray(mesh.x, dtype=np.float64)
    xd = np.ascontiguousarray(mesh.xdofs, dtype=np.int32)
    G, detJ = np.empty((mesh.ncells, nq, 3, 3)), np.empty((mesh.ncells, nq))
    assert lib().wo_precompute_geometric_data(P, mesh.ncells, _f(x.reshape(-1)), _i(xd.reshape(-1)),
                                              _f(G.reshape(-1)), _f(detJ.reshape(-1))) == 0
    return G, detJ


def jacobian_data(mesh, points, weights):
    """common/precompute.hpp:49-176 at arbitrary points -> dict J, detJ, K, G"""
    points = np.ascontiguousarray(points, dtype=np.float64)
    nq, nc = points.shape[0], mesh.ncells
    x = np.ascontiguousarray(mesh.x, dtype=np.float64)
    xd = np.ascontiguousarray(mesh.xdofs, dtype=np.int32)
    J, detJ = np.empty((nc, nq, 3, 3)), np.empty((nc, nq))
    K, G = np.empty((nc, nq, 3, 3)), np.empty((nc, nq, 3, 3))
    L = lib()
    L.wo_compute_jacobian(nc, nq, _f(points.reshape(-1)), _f(x.reshape(-1)), _i(xd.reshape(-1)), _f(J.reshape(-1)))
    L.wo_compute_jacobian_determinant(nc * nq, _f(J.reshape(-1)), _f(detJ.reshape(-1)))
    L.wo_compute_jacobian_inverse(nc * nq, _f(J.reshape(-1)), _f(K.reshape(-1)))
    w = np.ascontiguousarray(weights, dtype=np.float64)
    L.wo_compute_geometrical_factor(nc, nq, _f(J.reshape(-1)), _f(detJ.reshape(-1)), _f(w), _f(G.reshape(-1)))
    return dict(J=J, detJ=detJ, K=K, G=G)


def gauss_legendre(m):
    p, w = np.empty(m), np.empty(m)
    assert lib().wo_gauss_legendre(m, _f(p), _f(w)) == 0
    return p, w


def tabulate_1d(P, q, derivative):
    m = (q + 2) // 2
    pts, _ = gauss_legendre(m)
    out = np.empty((m, P + 1))
    assert lib().wo_tabulate_1d(P, m, _f(pts), derivative, _f(out)) == 0
    return out


def mass_apply(mesh, P, detJ, x, y):
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    lib().wo_mass_apply(P, mesh.ncells, _i(dm.reshape(-1)), _f(detJ.reshape(-1)), _f(x), _f(y))


def stiffness_apply(mesh, P, G, x, y, dense=True, nthreads=1, fast=False):
    """y += -c0^2 K x (c0 = 1500).  dense=True: the reference's skernel."""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    fn = lib(fast).wo_stiffness_apply_dense if dense else lib(fast).wo_stiffness_apply_sumfact
    fn(P, mesh.ncells, mesh.ndofs, _i(dm.reshape(-1)), _f(G.reshape(-1)), _f(x), _f(y), nthreads)


def boundary_facet_mass(mesh, P):
    m1, m2 = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    x = np.ascontiguousarray(mesh.x, dtype=np.float64)
    xd = np.ascontiguousarray(mesh.xdofs, dtype=np.int32)
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    fc = np.ascontiguousarray(mesh.facet_cells, dtype=np.int32)
    fl = np.ascontiguousarray(mesh.facet_local, dtype=np.int32)
    ft = np.ascontiguousarray(mesh.facet_tags, dtype=np.int32)
    assert lib().wo_boundary_facet_mass(P, len(fc), _i(fc), _i(fl), _i(ft), _f(x.reshape(-1)),
                                        _i(xd.reshape(-1)), _i(dm.reshape(-1)), _f(m1), _f(m2)) == 0
    return m1, m2


def rk4(mesh, P, G, m, m1, m2, c0, f0, p0, t0, tf, dt, u, v, max_steps=0, sumfact=False, nthreads=1,
        fast=False):
    """LinearGLLOpt::rk4 (common/LinearGLL.hpp:198-287); u, v updated in place."""
    dm = np.ascontiguousarray(mesh.dofmap, dtype=np.int32)
    t_end = C.c_double()
    steps = lib(fast).wo_rk4(P, mesh.ncells, mesh.ndofs, _i(dm.reshape(-1)), _f(G.reshape(-1)), _f(m),
                             _f(m1), _f(m2), c0, f0, p0, t0, tf, dt, max_steps, _f(u), _f(v),
                             int(sumfact), nthreads, C.byref(t_end))
    return steps, t_end.value
