"""Host-side mirror of the reference operator interface over the C ABI.

Same names, argument meaning and call shape as the reference classes:

  MassOperator(V, degree)(x, y)                 common/operators.hpp:43-109 (MassOperatorCPU)
  StiffnessOperator(V, degree, params)(x, y)    common/operators.hpp:136-201
  LinearGLLOpt(mesh, meshtags, degree, c0, f0, p0).init() / .rk4(t0, tf, dt)
                                                common/LinearGLL.hpp:37-287
  LinearGLLEnsemble(mesh, meshtags, degree, c0, f0s, p0s)
                                                nv LinearGLLOpt models on one mesh, stepped together
  WesterveltGLLOpt(mesh, meshtags, degree, c0, f0, p0, delta, beta, rho0), LossyGLLOpt (beta = 0)
                                                lossy and nonlinear (Westervelt) models, DESIGN.md 4.5a
  Medium(rho, c, beta)                          layered media (per-cell density, sound speed and nonlinearity),
                                                the `medium=` keyword of every wave model, DESIGN.md 4.5e
  Relaxation(tau, eps, c), Medium.relaxation   power-law absorption by relaxation processes, the `relaxation=`
                                                keyword of LossyGLLOpt / WesterveltGLLOpt, DESIGN.md 4.5f
  PML(mesh, zeta), PML.box                      perfectly matched layers, the `pml=` keyword of the single-field
                                                wave models, DESIGN.md 4.5g

`V` is a HexMesh (mesh.py): it carries what the reference pulls out of the DOLFINx
FunctionSpace (geometry, geometry dofmap, cell dofmap, index-map sizes).  Vectors are
DOLFINx-layout arrays: torch CUDA tensors (device path, asynchronous on the current torch
stream) or numpy arrays (host path: copied to the GPU and back inside the call, like the
reference functor applied to host la::Vectors).  All compute happens in libwavefx.so.
"""
import ctypes as C
from collections import namedtuple

import numpy as np

from . import capi

# field statistics of a wave model (LinearGLLOpt.field_stats, DESIGN.md section 4.5b)
FieldStats = namedtuple("FieldStats", "samples t_first t_last pmax pmin harmonics")


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Context:
    """One per GPU (role of utils::set_device, common/cuda/utils.hpp:22-38)."""
    _cache = {}

    def __init__(self, device=0):
        self.device = int(device)
        self.handle = C.c_void_p()
        capi.call("wfx_ctx_create", self.device, C.byref(self.handle))

    @classmethod
    def get(cls, device=0):
        device = int(device)
        if device not in cls._cache:
            cls._cache[device] = cls(device)
        return cls._cache[device]

    def synchronize(self):
        capi.call("wfx_ctx_sync", self.handle)


class Geometry:
    """precompute_geometric_data (common/precomputation.hpp:18-110) on the GPU."""

    def __init__(self, V, degree, dtype=np.float64, ctx=None):
        self.ctx = ctx or Context.get()
        self.P = int(degree)
        self.dtype = np.dtype(dtype)
        self.ncells = V.ncells
        self.handle = C.c_void_p()
        x = np.ascontiguousarray(V.x, dtype=np.float64)
        xd = np.ascontiguousarray(V.xdofs, dtype=np.int32)
        capi.call("wfx_geometry_create", self.ctx.handle, self.P, capi.dtype_code(self.dtype),
                  V.ncells, x.shape[0], capi.f64p(x.reshape(-1)), capi.i32p(xd.reshape(-1)),
                  C.byref(self.handle))

    def info(self):
        nc, na = C.c_int64(), C.c_int64()
        capi.call("wfx_geometry_info", self.handle, C.byref(nc), C.byref(na))
        return dict(ncells=nc.value, n_affine=na.value)

    def scale_cells(self, coeff):
        """G[c] *= coeff[c]: a piecewise-constant coefficient, e.g. (c0[c] / c0_ref)^2.  Reaches the operators and
        models already built on this geometry (their next applies), on every kernel path."""
        coeff = np.ascontiguousarray(coeff, dtype=np.float64)
        if coeff.size != self.ncells:
            raise capi.WfxError("one coefficient per cell expected")
        capi.call("wfx_geometry_scale_cells", self.handle, capi.f64p(coeff))
        self.scaled = True

    def detJw(self):
        """detJ * w [ncells, nq] (fp64, reference layout): the lumped mass's per-point weights."""
        detJ = np.empty((self.ncells, (self.P + 1) ** 3))
        capi.call("wfx_geometry_get", self.handle, None, capi.f64p(detJ.reshape(-1)))
        return detJ

    def get(self):
        """(G [ncells,nq,3,3], detJ [ncells,nq]) in the reference layout."""
        nq = (self.P + 1) ** 3
        G = np.empty((self.ncells, nq, 3, 3))
        detJ = np.empty((self.ncells, nq))
        capi.call("wfx_geometry_get", self.handle, capi.f64p(G.reshape(-1)), capi.f64p(detJ.reshape(-1)))
        return G, detJ

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_geometry_destroy(self.handle)
            self.handle = None


def compute_jacobian_data(V, points, weights=None, ctx=None, want=("J", "detJ", "K", "G")):
    """compute_jacobian / _determinant / _inverse / compute_geometrical_factor
    (common/precompute.hpp:49-176) at arbitrary reference points, on the GPU."""
    ctx = ctx or Context.get()
    points = np.ascontiguousarray(points, dtype=np.float64)
    nq = points.shape[0]
    nc = V.ncells
    out = {}
    J = np.empty((nc, nq, 3, 3)) if "J" in want else None
    detJ = np.empty((nc, nq)) if "detJ" in want else None
    K = np.empty((nc, nq, 3, 3)) if "K" in want else None
    G = np.empty((nc, nq, 3, 3)) if "G" in want and weights is not None else None
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
    x = np.ascontiguousarray(V.x, dtype=np.float64)
    xd = np.ascontiguousarray(V.xdofs, dtype=np.int32)
    flat = lambda a: None if a is None else capi.f64p(a.reshape(-1))
    capi.call("wfx_compute_jacobian_data", ctx.handle, nc, x.shape[0], capi.f64p(x.reshape(-1)),
              capi.i32p(xd.reshape(-1)), nq, capi.f64p(points.reshape(-1)), flat(w), flat(J),
              flat(detJ), flat(K), flat(G))
    for k, v in (("J", J), ("detJ", detJ), ("K", K), ("G", G)):
        if v is not None:
            out[k] = v
    return out


class _Operator:
    dtype = np.dtype(np.float64)
    ndofs = 0

    def _check(self, x, y):
        if _is_torch(x) != _is_torch(y):
            raise capi.WfxError("x and y must both be torch CUDA tensors or both numpy arrays")
        if _is_torch(x):
            import torch
            want = torch.float64 if self.dtype == np.float64 else torch.float32
            for v in (x, y):
                if not v.is_cuda or v.dtype != want or not v.is_contiguous() or v.numel() != self.ndofs:
                    raise capi.WfxError("vector must be a contiguous CUDA tensor of the operator's dtype and size")
            return True
        for v in (x, y):
            if v.dtype != self.dtype or not v.flags["C_CONTIGUOUS"] or v.size != self.ndofs:
                raise capi.WfxError("vector must be a contiguous numpy array of the operator's dtype and size")
        return False


class StiffnessOperator(_Operator):
    """y += -c0^2 K x  (common/operators.hpp:183-200).  `params` is accepted and ignored for
    the speed of sound exactly as the reference does (c0 = 1500 hard-coded, :113-115) unless
    honour_params=True."""

    def __init__(self, V, degree, params=None, dtype=np.float64, ctx=None, geometry=None,
                 mode=capi.STIFF_AUTO, honour_params=False, split=True, ensemble=False):
        self.ctx = ctx or Context.get()
        self.P = int(degree)
        self.dtype = np.dtype(dtype)
        self.geometry = geometry or Geometry(V, degree, dtype, self.ctx)
        self.ndofs = int(V.ndofs)
        c0 = 1500.0
        if honour_params and params and "c0" in params:
            c0 = float(params["c0"])
        self.c0 = c0
        self.handle = C.c_void_p()
        dm = np.ascontiguousarray(V.dofmap, dtype=np.int32)
        # distributed mesh: the dofs that also live on another rank (halo send + receive lists)
        halo = getattr(V, "halo", None) or {}
        shared = None
        if len(halo.get("send_indices", ())) or len(halo.get("recv_indices", ())):
            shared = np.unique(np.concatenate([halo["send_indices"], halo["recv_indices"]])).astype(np.int32)
        self.nshared = 0 if shared is None else len(shared)
        capi.call("wfx_stiffness_create_partitioned", self.ctx.handle, self.geometry.handle, self.ndofs,
                  capi.i32p(dm.reshape(-1)), c0,
                  mode | (0 if split else capi.STIFF_NO_SPLIT) | (capi.STIFF_ENSEMBLE if ensemble else 0), self.nshared,
                  capi.i32p(shared), C.byref(self.handle))
        self.split = bool(split) and self.nshared > 0

    def __call__(self, x, y):
        self.apply(x, y, beta=1)

    def apply(self, x, y, beta=1):
        if self._check(x, y):
            capi.call("wfx_stiffness_apply", self.handle, C.c_void_p(x.data_ptr()),
                      C.c_void_p(y.data_ptr()), int(beta), _stream_ptr())
        else:
            capi.call("wfx_stiffness_apply_host", self.handle, C.c_void_p(x.ctypes.data),
                      C.c_void_p(y.ctypes.data), int(beta))

    def apply_part(self, x, y, part, beta=0, scale_ptr=None, stream=None):
        """Distributed meshes: part 0 = cells touching rank-shared dofs, 1 = the rest, -1 = both.
        scale_ptr (1/m) is applied on the last touch of NON-shared dofs only."""
        self._check(x, y)
        capi.call("wfx_stiffness_apply_part", self.handle, C.c_void_p(x.data_ptr()),
                  C.c_void_p(scale_ptr) if scale_ptr else None, C.c_void_p(y.data_ptr()), int(beta),
                  int(part), stream if stream is not None else _stream_ptr())

    def apply_scaled(self, x, scale_ptr, y):
        """y = scale .* (-c0^2 K x): the fused stiffness + lumped-mass-inverse apply."""
        self._check(x, y)
        capi.call("wfx_stiffness_apply_scaled", self.handle, C.c_void_p(x.data_ptr()),
                  C.c_void_p(scale_ptr), C.c_void_p(y.data_ptr()), _stream_ptr())

    def apply_ensemble(self, X, Y, beta=0, scale_ptr=None):
        """Y[:, m] (+)= scale .* (-c0^2 K X[:, m]) for every member m, in one pass over the geometric
        factors: X, Y contiguous CUDA tensors of shape (ndofs, nv), 1 <= nv <= 8 (member-interleaved, the
        DOLFINx blocked layout with bs = nv).  scale_ptr: device pointer to ndofs values (e.g. 1/m) or None;
        a scale needs beta == 0.  Needs ensemble=True at construction."""
        import torch
        want = torch.float64 if self.dtype == np.float64 else torch.float32
        for v in (X, Y):
            if (not _is_torch(v) or not v.is_cuda or v.dtype != want or not v.is_contiguous() or v.dim() != 2
                    or v.shape[0] != self.ndofs):
                raise capi.WfxError("ensemble vectors must be contiguous (ndofs, nv) CUDA tensors of the operator's dtype")
        if X.shape != Y.shape:
            raise capi.WfxError("ensemble vectors X and Y differ in shape")
        capi.call("wfx_stiffness_apply_ensemble", self.handle, int(X.shape[1]), C.c_void_p(X.data_ptr()),
                  C.c_void_p(scale_ptr) if scale_ptr else None, C.c_void_p(Y.data_ptr()), int(beta), _stream_ptr())

    def info(self):
        nc, nd, ndofs = C.c_int64(), C.c_int(), C.c_int64()
        fl, by, ncol, nl = C.c_double(), C.c_double(), C.c_int(), C.c_int()
        capi.call("wfx_stiffness_info", self.handle, C.byref(nc), C.byref(nd), C.byref(ndofs),
                  C.byref(fl), C.byref(by), C.byref(ncol), C.byref(nl))
        return dict(num_cells=nc.value, num_dofs=nd.value, ndofs=ndofs.value, flops=fl.value,
                    bytes=by.value, ncolours=ncol.value, nlaunches=nl.value)

    def kernel_info(self):
        v, a, m, nr, nb, sm = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int64()
        capi.call("wfx_stiffness_kernel_info", self.handle, C.byref(v), C.byref(a), C.byref(m), C.byref(nr),
                  C.byref(nb), C.byref(sm))
        names = {-1: "cell", 0: "brick-generic", 1: "brick-regular", 2: "brick-regular-p4d", 3: "cell-streamed", 4: "brick-streamed"}
        return dict(variant=names.get(v.value, str(v.value)), affine=bool(a.value), mixed=bool(m.value),
                    regular_batches=nr.value, batches=nb.value, smem_bytes=sm.value)

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_stiffness_destroy(self.handle)
            self.handle = None


class MassOperator(_Operator):
    """y += M x with the collocated (diagonal) GLL mass (common/operators.hpp:86-108).  cell_weight: one positive
    weight per cell, m_i = sum_c w_c (detJ w)_{c,i} (the weighted mass of a layered medium, Medium.mass_weight)."""

    def __init__(self, V, degree, dtype=np.float64, ctx=None, geometry=None, cell_weight=None):
        self.ctx = ctx or Context.get()
        self.P = int(degree)
        self.dtype = np.dtype(dtype)
        self.geometry = geometry or Geometry(V, degree, dtype, self.ctx)
        self.ndofs = int(V.ndofs)
        self.handle = C.c_void_p()
        dm = np.ascontiguousarray(V.dofmap, dtype=np.int32)
        if cell_weight is not None:
            cell_weight = np.ascontiguousarray(cell_weight, dtype=np.float64).reshape(-1)
            if cell_weight.size != V.ncells:
                raise capi.WfxError("one mass weight per cell expected")
        capi.call("wfx_mass_create_weighted", self.ctx.handle, self.geometry.handle, self.ndofs,
                  capi.i32p(dm.reshape(-1)), capi.f64p(cell_weight), C.byref(self.handle))

    def __call__(self, x, y):
        self.apply(x, y, beta=1)

    def apply(self, x, y, beta=1):
        if self._check(x, y):
            capi.call("wfx_mass_apply", self.handle, C.c_void_p(x.data_ptr()),
                      C.c_void_p(y.data_ptr()), int(beta), _stream_ptr())
        else:
            capi.call("wfx_mass_apply_host", self.handle, C.c_void_p(x.ctypes.data),
                      C.c_void_p(y.ctypes.data), int(beta))

    def apply_inverse(self, x, y):
        """y = x ./ m (x and y may be the same tensor)."""
        self._check(x, y)
        capi.call("wfx_mass_apply_inverse", self.handle, C.c_void_p(x.data_ptr()),
                  C.c_void_p(y.data_ptr()), _stream_ptr())

    def assemble(self, halo):
        """Distributed meshes: sum the diagonal over the ranks sharing a dof (fp64 halo)."""
        capi.call("wfx_mass_assemble", self.handle, halo.handle)

    def _ptr(self, name):
        p = C.c_void_p()
        capi.call(name, self.handle, C.byref(p))
        return p.value

    def diagonal_ptr(self):
        return self._ptr("wfx_mass_diagonal")

    def inverse_diagonal_ptr(self):
        return self._ptr("wfx_mass_inverse_diagonal")

    def _download(self, ptr):
        out = np.empty(self.ndofs, dtype=self.dtype)
        capi.call("wfx_memcpy_d2h", self.ctx.handle, C.c_void_p(out.ctypes.data), C.c_void_p(ptr), out.nbytes)
        return out

    def diagonal(self):
        return self._download(self.diagonal_ptr())

    def inverse_diagonal(self):
        return self._download(self.inverse_diagonal_ptr())

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_mass_destroy(self.handle)
            self.handle = None


# the reference names both spellings (LinearGLL.hpp:63 vs operators.hpp:44)
MassOperatorCPU = MassOperator


class BoundaryOperator(_Operator):
    """b += c0^2 g m1 - c0 m2 .* v_n  (forms.ufl:21-24 via assemble_vector, LinearGLL.hpp:175).  facet_weight: one
    positive weight per facet triplet multiplying its facet mass (a layered medium, Medium.facet_weight)."""

    def __init__(self, V, degree, dtype=np.float64, ctx=None, facet_weight=None):
        self.ctx = ctx or Context.get()
        self.P = int(degree)
        self.dtype = np.dtype(dtype)
        self.ndofs = int(V.ndofs)
        self.handle = C.c_void_p()
        x = np.ascontiguousarray(V.x, dtype=np.float64)
        xd = np.ascontiguousarray(V.xdofs, dtype=np.int32)
        dm = np.ascontiguousarray(V.dofmap, dtype=np.int32)
        fc = np.ascontiguousarray(V.facet_cells, dtype=np.int32)
        fl = np.ascontiguousarray(V.facet_local, dtype=np.int32)
        ft = np.ascontiguousarray(V.facet_tags, dtype=np.int32)
        if facet_weight is not None:
            facet_weight = np.ascontiguousarray(facet_weight, dtype=np.float64).reshape(-1)
            if facet_weight.size != len(fc):
                raise capi.WfxError("one facet weight per facet triplet expected")
        capi.call("wfx_boundary_create_weighted", self.ctx.handle, self.P, capi.dtype_code(self.dtype), len(fc),
                  capi.i32p(fc), capi.i32p(fl), capi.i32p(ft), x.shape[0], capi.f64p(x.reshape(-1)),
                  capi.i32p(xd.reshape(-1)), self.ndofs, capi.i32p(dm.reshape(-1)), capi.f64p(facet_weight),
                  C.byref(self.handle))

    def apply(self, c0, g, vn, b):
        self._check(vn, b)
        capi.call("wfx_boundary_apply", self.handle, float(c0), float(g), C.c_void_p(vn.data_ptr()),
                  C.c_void_p(b.data_ptr()), _stream_ptr())

    def assemble(self, halo):
        """Distributed meshes: sum the facet masses over the ranks sharing a boundary dof (fp64 halo)."""
        capi.call("wfx_boundary_assemble", self.handle, halo.handle)

    def facet_masses(self):
        m1, m2 = np.empty(self.ndofs), np.empty(self.ndofs)
        capi.call("wfx_boundary_get", self.handle, capi.f64p(m1), capi.f64p(m2))
        return m1, m2

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_boundary_destroy(self.handle)
            self.handle = None


def focus_delays(points, focus, c0):
    """Delays that focus a phased-array source at `focus`: tau_i = (max_j d_j - d_i) / c0 with d_i = |x_i - focus|,
    for points [n, 3] (e.g. dof_coordinates(mesh)).  Every tau_i >= 0; the farthest point fires first (tau = 0), so
    all contributions reach the focus at the same time."""
    x = np.asarray(points, dtype=np.float64)
    d = np.linalg.norm(x - np.asarray(focus, dtype=np.float64).reshape(1, -1), axis=1)
    return (d.max() - d) / float(c0) if len(d) else d


def _trilinear(xv, xi):
    """x(xi) and dx/dxi [3, 3] of the cell with vertices xv [8, 3] (vertex v = ix + 2 iy + 4 iz) at xi in [0, 1]^3"""
    f = [(1.0 - xi[a], xi[a]) for a in range(3)]
    x, J = np.zeros(3), np.zeros((3, 3))
    for v in range(8):
        b = (v & 1, (v >> 1) & 1, (v >> 2) & 1)
        w = [f[a][b[a]] for a in range(3)]
        x += w[0] * w[1] * w[2] * xv[v]
        for a in range(3):
            d = (1.0 if b[a] else -1.0) * w[(a + 1) % 3] * w[(a + 2) % 3]
            J[:, a] += d * xv[v]
    return x, J


def _locate_in_cell(mesh, c, point, tol=1e-10):
    """xi in [0, 1]^3 with x_c(xi) = point by Newton iteration on cell c's trilinear map, or None when the point lies
    outside the cell.  Reference coordinates within 1e-14 of a GLL node are put on it, so that a point at a dof or on a
    face, edge or vertex gives exact zeros at the dofs whose basis functions vanish there."""
    xv = mesh.x[mesh.xdofs[c]]
    x0 = np.asarray(point, dtype=np.float64)
    xi = np.full(3, 0.5)
    for _ in range(60):
        x, J = _trilinear(xv, xi)
        try:
            step = np.linalg.solve(J, x - x0)
        except np.linalg.LinAlgError:
            return None
        xi = xi - step
        if np.any(np.abs(xi - 0.5) > 10.0):
            return None
        if np.abs(step).max() < 1e-15:
            break
    if np.any(xi < -tol) or np.any(xi > 1.0 + tol):
        return None
    nodes, _ = capi.gll(mesh.P)
    for a in range(3):
        k = np.argmin(np.abs(nodes - xi[a]))
        if abs(nodes[k] - xi[a]) < 1e-14:
            xi[a] = nodes[k]
    return np.clip(xi, 0.0, 1.0)


def _cell_weights(mesh, c, xi):
    """(dofs, phi_dofs(x(xi))) of cell c: the GLL Lagrange basis at reference point xi, in the cell's dof order"""
    P = mesh.P
    nodes, _ = capi.gll(P)
    perm = capi.compute_permutations(P)
    L = np.ones((3, P + 1))
    for a in range(3):
        for i in range(P + 1):
            for j in range(P + 1):
                if j != i:
                    L[a, i] *= (xi[a] - nodes[j]) / (nodes[i] - nodes[j])
    phi = np.einsum("a,b,c->abc", L[0], L[1], L[2]).reshape(-1)   # tensor order t = (i0 n + i1) n + i2
    return np.asarray(mesh.dofmap[c])[perm], phi


def point_source(mesh, point):
    """(dofs, q) of a point source at a physical point: q_j = phi_j(point), the GLL basis functions of the cell that
    holds the point (located by Newton iteration on its trilinear map), at the dofs where they do not vanish, dofs
    ascending.  On a shared face, edge or vertex either cell gives the same weights.  The same weights make the
    interpolating sensor p(point) = sum_j q_j p_j.  Feed them to set_volume_source (DESIGN.md section 4.5h).  A point
    outside the mesh raises WfxError."""
    x0 = np.asarray(point, dtype=np.float64).reshape(3)
    xc = mesh.x[mesh.xdofs]
    lo, hi = xc.min(axis=1), xc.max(axis=1)
    pad = 1e-10 * (hi - lo).max(axis=1, keepdims=True)
    for c in np.nonzero(np.all((x0 >= lo - pad) & (x0 <= hi + pad), axis=1))[0]:
        xi = _locate_in_cell(mesh, int(c), x0)
        if xi is None:
            continue
        dofs, phi = _cell_weights(mesh, int(c), xi)
        keep = phi != 0.0
        order = np.argsort(dofs[keep])
        return dofs[keep][order].astype(np.int32), phi[keep][order]
    raise capi.WfxError(f"point_source: the point {tuple(x0)} lies outside the mesh")


def phase_conjugate_delays(p_hat, f0):
    """Time-reversal delays for a source profile: tau = mod(arg p_hat, 2 pi) / (2 pi f0), in [0, 1 / f0), shaped like
    p_hat.  p_hat: the first-harmonic map (field_stats().harmonics[0]) of an emission from a point source at the
    target; f0: the model's source frequency, or the members' frequencies [nv] for an ensemble's (ndofs, nv) map.
    Firing every element with these delays aligns the phases of all contributions at the target (DESIGN.md section
    4.5h)."""
    p = np.asarray(p_hat)
    f = np.broadcast_to(np.asarray(f0, dtype=np.float64), p.shape[-1:] if p.ndim > 1 else ())
    tau = np.mod(np.angle(p), 2.0 * np.pi) / (2.0 * np.pi * f)
    return np.where(tau * f < 1.0, tau, 0.0)


def _refuse_pml(pml):
    if pml is not None:
        raise capi.WfxError("pml: ensemble models are not supported (LinearGLLOpt, LossyGLLOpt, WesterveltGLLOpt)")


def _refuse_relaxation(relaxation):
    if relaxation is not None:
        raise capi.WfxError("relaxation: needs LossyGLLOpt or WesterveltGLLOpt (for linear tissue, LossyGLLOpt with "
                            "delta = 0)")


class LinearGLLOpt:
    """The wave model + RK4 driver (common/LinearGLL.hpp:37-287) on the GPU.

    mesh carries the facet tags (`meshtags` may be None or a (cells, local, tags) triple that
    overrides them).  medium: a Medium (layered media, DESIGN.md section 4.5e) or None; one rank only."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency,
                 pressureAmplitude, dtype=np.float64, ctx=None, halo=None, stiffness_mode=capi.STIFF_AUTO,
                 setup_halo=None, medium=None, relaxation=None, pml=None):
        _refuse_relaxation(relaxation)
        if pml is not None and halo is not None:
            raise capi.WfxError("pml: distributed models are not supported (one rank only)")
        self.ctx = ctx or Context.get()
        self.V = mesh
        if meshtags is not None:
            import copy
            mesh = copy.copy(mesh)
            mesh.facet_cells, mesh.facet_local, mesh.facet_tags = meshtags
        if medium is not None and halo is not None:
            raise capi.WfxError("medium: distributed models are not supported (one rank only)")
        self.k_ = int(degreeOfBasis)
        self.c0_, self.freq0_, self.p0_ = float(speedOfSound), float(sourceFrequency), float(pressureAmplitude)
        self.dtype = np.dtype(dtype)
        self._medium_geometry(mesh, medium)
        self.mass_op = MassOperator(mesh, self.k_, dtype, self.ctx, self.geometry,
                                    cell_weight=self._mass_weight)                      # :105
        params = {"c0": self.c0_}
        self.stiff_op = StiffnessOperator(mesh, self.k_, params, dtype, self.ctx, self.geometry,
                                          mode=stiffness_mode)                           # :120
        self.bnd_op = BoundaryOperator(mesh, self.k_, dtype, self.ctx,
                                       facet_weight=self._facet_weight)                  # :113-115
        self.halo = halo
        if halo is not None:
            # the masses are summed over the ranks in fp64: an fp32 model needs a second, fp64 halo
            # for this one-off set-up step (`setup_halo`, built here on the same mesh if not given)
            if setup_halo is None:
                if self.dtype == np.float64:
                    setup_halo = halo
                else:
                    from .partition import Halo
                    setup_halo = Halo(mesh, self.ctx, np.float64, comm=halo.comm)
            self.setup_halo = setup_halo
            self.mass_op.assemble(setup_halo)                                            # :110
            self.bnd_op.assemble(setup_halo)
        self.handle = C.c_void_p()
        capi.call("wfx_wave_create", self.ctx.handle, self.stiff_op.handle, self.mass_op.handle,
                  self.bnd_op.handle, halo.handle if halo is not None else None, int(mesh.size_local),
                  self.c0_, self.freq0_, self.p0_, C.byref(self.handle))
        self.ndofs = int(mesh.ndofs)
        self.pml = None
        if pml is not None:
            self.set_pml(pml)

    def _medium_geometry(self, mesh, medium):
        """The model's geometry, scaled by the medium's stiffness weight, and the medium's mass and facet weights
        (None without a medium)."""
        if medium is not None and not isinstance(medium, Medium):
            raise capi.WfxError("medium must be a Medium")
        self.medium = medium
        self.geometry = Geometry(mesh, self.k_, self.dtype, self.ctx)
        self._mass_weight = self._facet_weight = None
        if medium is None:
            return
        self.geometry.scale_cells(medium.stiffness_weight(mesh.ncells))
        self._mass_weight = medium.mass_weight(mesh.ncells, self.c0_)
        self._facet_weight = medium.facet_weight(mesh, self.c0_)

    def init(self):
        capi.call("wfx_wave_init", self.handle)

    def set_state(self, u, v):
        u = np.ascontiguousarray(u, dtype=self.dtype)
        v = np.ascontiguousarray(v, dtype=self.dtype)
        capi.call("wfx_wave_set_state", self.handle, C.c_void_p(u.ctypes.data), C.c_void_p(v.ctypes.data))

    def get_state(self):
        u, v = np.empty(self.ndofs, dtype=self.dtype), np.empty(self.ndofs, dtype=self.dtype)
        capi.call("wfx_wave_get_state", self.handle, C.c_void_p(u.ctypes.data), C.c_void_p(v.ctypes.data))
        return u, v

    def set_probes(self, dofs, max_records):
        """Record u[dofs] after every completed time step (kept on the device, up to max_records)."""
        dofs = np.ascontiguousarray(dofs, dtype=np.int32)
        self._nprobes = len(dofs)
        capi.call("wfx_wave_set_probes", self.handle, len(dofs), capi.i32p(dofs), int(max_records))

    def probe_series(self):
        """(t [nrec], u [nrec, nprobes]) recorded so far."""
        n = C.c_int64()
        capi.call("wfx_wave_get_probe_series", self.handle, C.byref(n), None, None)
        t = np.empty(n.value)
        vals = np.empty((n.value, getattr(self, "_nprobes", 0)), dtype=self.dtype)
        capi.call("wfx_wave_get_probe_series", self.handle, C.byref(n), capi.f64p(t), C.c_void_p(vals.ctypes.data))
        return t, vals

    def set_field_stats(self, t_start, harmonics=0):
        """Accumulate field statistics (DESIGN.md section 4.5b) on the device after every completed step whose
        reached time is >= t_start - dt/2: peak positive and negative pressure and the complex amplitudes of
        harmonics 1..`harmonics` (<= 8) of the model's source frequency at every dof.  Resets the accumulators,
        as do init and set_state.  set_field_stats(None) switches them off and frees them."""
        if t_start is None:
            capi.call("wfx_wave_set_field_stats", self.handle, 0, 0.0, 0)
            return
        capi.call("wfx_wave_set_field_stats", self.handle, 1, float(t_start), int(harmonics))

    def _entry_shape(self):
        return (self.ndofs,)

    def field_stats(self):
        """FieldStats(samples, t_first, t_last, pmax, pmin, harmonics) accumulated so far: pmax, pmin in the model
        dtype, shaped like the state; harmonics complex128 [H, *state shape], harmonics[h - 1] the amplitude
        p_h = (2 / N) sum_n u(t_n) exp(-i h w t_n) of harmonic h."""
        shape = self._entry_shape()
        on, nharm = C.c_int(), C.c_int()
        capi.call("wfx_wave_field_stats_info", self.handle, C.byref(on), None, C.byref(nharm))
        if not on.value:
            raise capi.WfxError("field statistics are off (set_field_stats)")
        nharm = nharm.value
        pmax, pmin = np.empty(shape, dtype=self.dtype), np.empty(shape, dtype=self.dtype)
        harm = np.empty((nharm, *shape), dtype=np.complex128)
        n, t0, t1 = C.c_int64(), C.c_double(), C.c_double()
        capi.call("wfx_wave_get_field_stats", self.handle, C.byref(n), C.byref(t0), C.byref(t1),
                  C.c_void_p(pmax.ctypes.data), C.c_void_p(pmin.ctypes.data),
                  C.cast(C.c_void_p(harm.ctypes.data), capi._c_f64p))
        return FieldStats(n.value, t0.value, t1.value, pmax, pmin, harm)

    def set_source_profile(self, amplitude=None, delay=None):
        """Phased-array source on tag 1 (DESIGN.md section 4.5c): the boundary term uses amplitude[i] g(t - delay[i])
        at every entry i in place of g(t), with g(s) = g'(s) = 0 for s < 0.  Arrays shaped like the state
        ((ndofs,), or (ndofs, nv) for an ensemble); entries off tag 1 are ignored.  None stands for 1 (amplitude)
        or 0 (delay); set_source_profile() clears the profile.  The profile survives init, set_state and
        restarts.  Delays are >= 0, see focus_delays."""
        shape = self._entry_shape()

        def arr(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.float64)
            if a.shape != shape:
                raise capi.WfxError(f"source profile arrays must have shape {shape}")
            return a

        amplitude, delay = arr(amplitude), arr(delay)
        capi.call("wfx_wave_set_source_profile", self.handle, capi.f64p(amplitude), capi.f64p(delay))

    def set_volume_source(self, dofs=None, q=None, delay=None):
        """Volume source (DESIGN.md section 4.5h): at every stage b_j += c0^2 q_j g(t - delay_j) on the n distinct dofs
        `dofs`, g the model's source (g = 0 before the delay), added before the layer, Gamma2 and quotient terms.
        q and delay have shape (n,), or (n, nv) for an ensemble (a column per member); delay None stands for 0.  A
        point source at x0 is point_source(mesh, x0).  set_volume_source() clears the source.  Model configuration:
        it survives init, set_state and restarts."""
        d = np.asarray([] if dofs is None else dofs)
        if d.ndim != 1 or (d.size and not np.issubdtype(d.dtype, np.integer)):
            raise capi.WfxError("volume source: dofs must be a 1-D array of integers")
        if d.size == 0:
            if any(a is not None and np.size(a) for a in (q, delay)):
                raise capi.WfxError("volume source: weights or delays without dofs (set_volume_source() clears)")
            capi.call("wfx_wave_set_volume_source", self.handle, 0, None, None, None)
            return
        # checked before the int32 conversion, which would wrap indices of 2^31 and above
        bad = np.nonzero((d < 0) | (d >= self.ndofs))[0]
        if len(bad):
            raise capi.WfxError(f"volume source: dof {int(d[bad[0]])} at entry {int(bad[0])} outside [0, {self.ndofs})")
        dofs = np.ascontiguousarray(d, dtype=np.int32)
        shape = (len(dofs),) + self._entry_shape()[1:]

        def arr(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.float64)
            if a.shape != shape:
                raise capi.WfxError(f"volume source weights and delays must have shape {shape}")
            return a

        q, delay = arr(q), arr(delay)
        if q is None:
            raise capi.WfxError("volume source: weights q are required")
        capi.call("wfx_wave_set_volume_source", self.handle, len(dofs), capi.i32p(dofs), capi.f64p(q),
                  capi.f64p(delay))

    def set_snapshot(self, every, fn):
        """fn(step, t, u, v) with numpy views of the pinned host copies (copy them to keep them), every
        `every` completed steps; the device -> host copy overlaps the time stepping."""
        if fn is None or not every:
            self._snap_cb = None
            capi.call("wfx_wave_set_snapshot", self.handle, 0, None, None)
            return
        n, dt = self.ndofs, self.dtype

        def tramp(_user, step, t, up, vp):
            ctype = C.c_double if dt == np.float64 else C.c_float
            u = np.ctypeslib.as_array(C.cast(up, C.POINTER(ctype)), shape=(n,))
            v = np.ctypeslib.as_array(C.cast(vp, C.POINTER(ctype)), shape=(n,))
            fn(int(step), float(t), u, v)

        self._snap_cb = capi.SNAPSHOT_FN(tramp)  # keep the trampoline alive
        capi.call("wfx_wave_set_snapshot", self.handle, int(every), C.cast(self._snap_cb, C.c_void_p), None)

    def f0(self, t, u, v, result):
        """result = v (LinearGLL.hpp:141-144); device tensors."""
        capi.call("wfx_wave_f0", self.handle, float(t), C.c_void_p(u.data_ptr()), C.c_void_p(v.data_ptr()),
                  C.c_void_p(result.data_ptr()), _stream_ptr())

    def f1(self, t, u, v, result):
        """result = M^-1 (-c0^2 K u + boundary(g(t), v)) (LinearGLL.hpp:151-192); device tensors."""
        capi.call("wfx_wave_f1", self.handle, float(t), C.c_void_p(u.data_ptr()), C.c_void_p(v.data_ptr()),
                  C.c_void_p(result.data_ptr()), _stream_ptr())

    def rk4(self, startTime, finalTime, timeStep, max_steps=0, stream=None):
        steps, t_end = C.c_int64(), C.c_double()
        capi.call("wfx_wave_rk4", self.handle, float(startTime), float(finalTime), float(timeStep),
                  int(max_steps), C.byref(steps), C.byref(t_end), stream if stream is not None else _stream_ptr())
        return steps.value, t_end.value

    def set_pml(self, pml=None):
        """A perfectly matched layer (DESIGN.md section 4.5g): a PML built on this model's mesh, whose layer is then
        built on the device on the model's own geometry (so a medium's stiffness weight reaches it); None removes it.
        Model configuration: it survives init, set_state and restarts.  psi and phi start at 0 here, at init and at
        set_state; a checkpoint restores them with set_pml_state after set_state.  rk4 then refuses steps of
        PML.max_dt and above; snapshots are refused (they carry u and v only)."""
        if pml is not None:
            if not isinstance(pml, PML):
                raise capi.WfxError("pml must be a PML")
            if pml.zeta.shape != (3, self.ndofs):
                raise capi.WfxError(f"pml: the profile has {pml.zeta.shape[1]} dofs, the model {self.ndofs}")
        capi.call("wfx_wave_set_pml", self.handle, None)
        self._destroy_pml()
        self.pml = None
        if pml is None:
            return
        V = self.V
        x = np.ascontiguousarray(V.x, dtype=np.float64)
        h = C.c_void_p()
        capi.call("wfx_pml_create", self.ctx.handle, self.geometry.handle, self.ndofs,
                  capi.i32p(np.ascontiguousarray(V.dofmap, dtype=np.int32).reshape(-1)), x.shape[0],
                  capi.f64p(x.reshape(-1)), capi.i32p(np.ascontiguousarray(V.xdofs, dtype=np.int32).reshape(-1)),
                  capi.f64p(pml.zeta.reshape(-1)), C.byref(h))
        try:
            capi.call("wfx_wave_set_pml", self.handle, h)
        except capi.WfxError:
            capi.lib.wfx_pml_destroy(h)
            raise
        self._pml_handle = h
        self.pml = pml

    def pml_info(self):
        """dict(cells, dofs, zeta_max) of the model's layer (the cells where zeta > 0 at a point, their dofs)"""
        if self.pml is None:
            raise capi.WfxError("pml: the model has no perfectly matched layer (set_pml)")
        nc, nd, zm = C.c_int64(), C.c_int64(), C.c_double()
        capi.call("wfx_pml_info", self._pml_handle, C.byref(nc), C.byref(nd), C.byref(zm))
        return dict(cells=nc.value, dofs=nd.value, zeta_max=zm.value)

    def _pml_shapes(self):
        info = self.pml_info()
        return (info["dofs"],), (info["cells"], (self.k_ + 1) ** 3, 3)

    def pml_state(self):
        """(psi [layer dofs], phi [layer cells, (P+1)^3, 3]) in the model dtype; the layer's dofs ascending, its cells
        in mesh order, points in the tensor order of the reference's dof permutation"""
        sp, sf = self._pml_shapes()
        psi, phi = np.empty(sp, dtype=self.dtype), np.empty(sf, dtype=self.dtype)
        capi.call("wfx_wave_get_pml_state", self.handle, C.c_void_p(psi.ctypes.data), C.c_void_p(phi.ctypes.data))
        return psi, phi

    def set_pml_state(self, psi, phi):
        """psi, phi of a checkpoint (after set_state, which zeroes them), shaped as pml_state returns them"""
        sp, sf = self._pml_shapes()
        psi = np.ascontiguousarray(psi, dtype=self.dtype)
        phi = np.ascontiguousarray(phi, dtype=self.dtype)
        if psi.shape != sp or phi.shape != sf:
            raise capi.WfxError(f"pml state must have shapes {sp} and {sf}")
        capi.call("wfx_wave_set_pml_state", self.handle, C.c_void_p(psi.ctypes.data), C.c_void_p(phi.ctypes.data))

    def _destroy_pml(self):
        h = getattr(self, "_pml_handle", None)
        if h and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_pml_destroy(h)
        self._pml_handle = None

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_wave_destroy(self.handle)
            self.handle = None
        self._destroy_pml()


class LinearGLLEnsemble(LinearGLLOpt):
    """nv wave models (1 <= nv <= 8) on one mesh with one speed of sound, stepped together: member m is
    LinearGLLOpt(mesh, meshtags, degree, c0, f0s[m], p0s[m]).  One rank.  The stiffness apply of a stage
    reads the geometric factors once for all members.  States are (ndofs, nv) arrays (member-interleaved,
    entry (dof i, member m) at i*nv + m); probe values come as (nrecords, nprobes, nv).  Snapshots are not
    available for ensembles."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequencies, pressureAmplitudes,
                 dtype=np.float64, ctx=None, stiffness_mode=capi.STIFF_AUTO, medium=None, relaxation=None, pml=None):
        _refuse_relaxation(relaxation)
        _refuse_pml(pml)
        self.ctx = ctx or Context.get()
        self.V = mesh
        if meshtags is not None:
            import copy
            mesh = copy.copy(mesh)
            mesh.facet_cells, mesh.facet_local, mesh.facet_tags = meshtags
        f0s = np.ascontiguousarray(sourceFrequencies, dtype=np.float64).reshape(-1)
        p0s = np.ascontiguousarray(pressureAmplitudes, dtype=np.float64).reshape(-1)
        if f0s.shape != p0s.shape:
            raise capi.WfxError("one source frequency and one pressure amplitude per member expected")
        self.nv = len(f0s)
        self.k_ = int(degreeOfBasis)
        self.c0_ = float(speedOfSound)
        self.freq0s_, self.p0s_ = f0s, p0s
        self.dtype = np.dtype(dtype)
        self._medium_geometry(mesh, medium)
        self.mass_op = MassOperator(mesh, self.k_, dtype, self.ctx, self.geometry, cell_weight=self._mass_weight)
        self.stiff_op = StiffnessOperator(mesh, self.k_, {"c0": self.c0_}, dtype, self.ctx, self.geometry,
                                          mode=stiffness_mode, ensemble=True)
        self.bnd_op = BoundaryOperator(mesh, self.k_, dtype, self.ctx, facet_weight=self._facet_weight)
        self.halo = None
        self.handle = C.c_void_p()
        capi.call("wfx_wave_create_ensemble", self.ctx.handle, self.stiff_op.handle, self.mass_op.handle,
                  self.bnd_op.handle, self.nv, int(mesh.size_local), self.c0_, capi.f64p(f0s), capi.f64p(p0s),
                  C.byref(self.handle))
        self.ndofs = int(mesh.ndofs)

    def _state(self, a):
        a = np.ascontiguousarray(a, dtype=self.dtype)
        if a.shape != (self.ndofs, self.nv):
            raise capi.WfxError(f"ensemble state must have shape ({self.ndofs}, {self.nv})")
        return a

    def set_state(self, u, v):
        u, v = self._state(u), self._state(v)
        capi.call("wfx_wave_set_state", self.handle, C.c_void_p(u.ctypes.data), C.c_void_p(v.ctypes.data))

    def get_state(self):
        u = np.empty((self.ndofs, self.nv), dtype=self.dtype)
        v = np.empty((self.ndofs, self.nv), dtype=self.dtype)
        capi.call("wfx_wave_get_state", self.handle, C.c_void_p(u.ctypes.data), C.c_void_p(v.ctypes.data))
        return u, v

    def _entry_shape(self):
        return (self.ndofs, self.nv)

    def probe_series(self):
        """(t [nrec], u [nrec, nprobes, nv]) recorded so far."""
        n = C.c_int64()
        capi.call("wfx_wave_get_probe_series", self.handle, C.byref(n), None, None)
        t = np.empty(n.value)
        vals = np.empty((n.value, getattr(self, "_nprobes", 0), self.nv), dtype=self.dtype)
        capi.call("wfx_wave_get_probe_series", self.handle, C.byref(n), capi.f64p(t), C.c_void_p(vals.ctypes.data))
        return t, vals

    def set_snapshot(self, every, fn):
        capi.call("wfx_wave_set_snapshot", self.handle, int(every), None, None)

    def set_pml(self, pml=None):
        _refuse_pml(pml)


class WesterveltGLLOpt(LinearGLLOpt):
    """The Westervelt model on one rank, with the surface of LinearGLLOpt (DESIGN.md section 4.5a):

        (1 - kappa p) p_tt - c0^2 lap p - delta lap p_t = kappa p_t^2,   kappa = 2 beta / (rho0 c0^2)

    dp/dn = g(t) on tag 1 (the source of LinearGLLOpt), dp/dn = -p_t / c0 on tag 2.  diffusivityOfSound
    delta [m^2/s] >= 0, coefficientOfNonlinearity beta >= 0, density rho0 [kg/m^3] > 0 when beta > 0.
    delta = beta = 0 is LinearGLLOpt bit for bit.  A per-cell coefficient set with Geometry.scale_cells
    multiplies the delta term too (delta_eff = delta * coeff).  With a Medium the nonlinearity is per dof
    (set_nonlinearity), from the medium's beta, which defaults to coefficientOfNonlinearity; delta_eff = delta
    (c / c0)^2 (DESIGN.md section 4.5e).  relaxation: a Relaxation (power-law absorption, DESIGN.md section 4.5f),
    see set_relaxation.  pml: a PML (perfectly matched layer, DESIGN.md section 4.5g), see set_pml."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                 diffusivityOfSound, coefficientOfNonlinearity, density, dtype=np.float64, ctx=None,
                 stiffness_mode=capi.STIFF_AUTO, medium=None, relaxation=None, pml=None):
        self.ctx = ctx or Context.get()
        self.V = mesh
        if meshtags is not None:
            import copy
            mesh = copy.copy(mesh)
            mesh.facet_cells, mesh.facet_local, mesh.facet_tags = meshtags
        self.k_ = int(degreeOfBasis)
        self.c0_, self.freq0_, self.p0_ = float(speedOfSound), float(sourceFrequency), float(pressureAmplitude)
        self.delta_, self.beta_, self.rho0_ = (float(diffusivityOfSound), float(coefficientOfNonlinearity),
                                               float(density))
        self.dtype = np.dtype(dtype)
        self._medium_geometry(mesh, medium)
        self.mass_op = MassOperator(mesh, self.k_, dtype, self.ctx, self.geometry, cell_weight=self._mass_weight)
        self.stiff_op = StiffnessOperator(mesh, self.k_, {"c0": self.c0_}, dtype, self.ctx, self.geometry,
                                          mode=stiffness_mode)
        self.bnd_op = BoundaryOperator(mesh, self.k_, dtype, self.ctx, facet_weight=self._facet_weight)
        self.halo = None
        self.handle = C.c_void_p()
        capi.call("wfx_wave_create_westervelt", self.ctx.handle, self.stiff_op.handle, self.mass_op.handle,
                  self.bnd_op.handle, int(mesh.size_local), self.c0_, self.freq0_, self.p0_, self.delta_,
                  self.beta_, self.rho0_, C.byref(self.handle))
        self.ndofs = int(mesh.ndofs)
        self.kappa = None
        if medium is not None:
            kappa = medium.kappa(mesh, self.geometry.detJw(), self.c0_, self.beta_)
            # the medium's kappa replaces the scalar one whenever either is nonzero; only a model created with
            # beta = 0 in a medium without nonlinearity keeps the lossy update
            if self.beta_ > 0 or np.any(kappa > 0):
                self.set_nonlinearity(kappa)
        self.relaxation = None
        if relaxation is not None:
            self.set_relaxation(relaxation)
        self.pml = None
        if pml is not None:
            self.set_pml(pml)

    def set_nonlinearity(self, kappa=None):
        """kappa [ndofs] >= 0: a per-dof kappa in place of 2 beta / (rho0 c0^2) (the model then steps the nonlinear
        update even with beta = 0); None restores the scalar.  Survives init, set_state and restarts."""
        k = None if kappa is None else np.ascontiguousarray(kappa, dtype=np.float64)
        if k is not None and k.shape != (self.ndofs,):
            raise capi.WfxError(f"kappa must have shape ({self.ndofs},)")
        capi.call("wfx_wave_set_nonlinearity", self.handle, capi.f64p(k))
        self.kappa = k

    def set_relaxation(self, relaxation=None):
        """Relaxation absorption (DESIGN.md section 4.5f): a Relaxation whose per-cell strengths become per-dof ones
        with this model's mass weights (Relaxation.eps_dofs); None switches it off.  Model configuration: it survives
        init, set_state and restarts.  The memory variables start at 0 here, at init and at set_state; a checkpoint
        restores them with set_relaxation_state after set_state.  rk4 then refuses steps of Relaxation.max_dt and
        above; snapshots are refused (they carry u and v only)."""
        if relaxation is None:
            capi.call("wfx_wave_set_relaxation", self.handle, 0, None, None)
            self.relaxation, self.relaxation_eps = None, None
            return
        if not isinstance(relaxation, Relaxation):
            raise capi.WfxError("relaxation must be a Relaxation")
        eps = relaxation.eps_dofs(self.V, self.geometry.detJw(), self._mass_weight)
        capi.call("wfx_wave_set_relaxation", self.handle, relaxation.M, capi.f64p(relaxation.tau),
                  capi.f64p(np.ascontiguousarray(eps)))
        self.relaxation, self.relaxation_eps = relaxation, eps

    def _relax_shape(self):
        if self.relaxation is None:
            raise capi.WfxError("relaxation state: the model has no relaxation (set_relaxation)")
        return (self.relaxation.M, self.ndofs)

    def relaxation_state(self):
        """the memory variables q [M, ndofs] in the model dtype"""
        q = np.empty(self._relax_shape(), dtype=self.dtype)
        capi.call("wfx_wave_get_relaxation_state", self.handle, C.c_void_p(q.ctypes.data))
        return q

    def set_relaxation_state(self, q):
        """q [M, ndofs]: the memory variables of a checkpoint (after set_state, which zeroes them)"""
        shape = self._relax_shape()
        q = np.ascontiguousarray(q, dtype=self.dtype)
        if q.shape != shape:
            raise capi.WfxError(f"relaxation state must have shape {shape}")
        capi.call("wfx_wave_set_relaxation_state", self.handle, C.c_void_p(q.ctypes.data))


class LossyGLLOpt(WesterveltGLLOpt):
    """The lossy wave model (WesterveltGLLOpt with beta = 0):  p_tt - c0^2 lap p - delta lap p_t = 0.  In a Medium
    that gives beta per cell the model steps the Westervelt update with the medium's per-dof kappa (the medium's
    beta replaces the model's beta = 0, as for WesterveltGLLOpt); a Medium without beta keeps it lossy."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                 diffusivityOfSound, dtype=np.float64, ctx=None, stiffness_mode=capi.STIFF_AUTO, medium=None,
                 relaxation=None, pml=None):
        super().__init__(mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                         diffusivityOfSound, 0.0, 1.0, dtype=dtype, ctx=ctx, stiffness_mode=stiffness_mode,
                         medium=medium, relaxation=relaxation, pml=pml)


# dose of a thermal model (PennesGLL.dose): steps since init / set_state, CEM43 [min] and peak temperature per dof
ThermalDose = namedtuple("ThermalDose", "steps cem43 T_max")


def cell_to_dof_average(mesh, detJw, coeff, weight=None):
    """Per-dof mass-weighted average of a per-cell coefficient, sum_c coeff_c (detJ w)_{c,i} / m_i with
    m_i = sum_c (detJ w)_{c,i}, the lumped mass: then coeff_i m_i is the GLL quadrature of the piecewise-constant
    coefficient.  detJw [ncells, nq] in the reference layout (Geometry.detJw, oracle.precompute_geometric_data).
    weight: per-cell weights w_c of a weighted mass, sum_c coeff_c w_c (detJ w)_{c,i} / sum_c w_c (detJ w)_{c,i}."""
    coeff = np.asarray(coeff, dtype=np.float64).reshape(-1)
    if coeff.size != mesh.ncells:
        raise capi.WfxError("one coefficient per cell expected")
    perm = capi.compute_permutations(mesh.P)
    dofs = np.asarray(mesh.dofmap)[:, perm].reshape(-1)
    w = np.asarray(detJw, dtype=np.float64).reshape(mesh.ncells, -1)
    if weight is not None:
        weight = np.asarray(weight, dtype=np.float64).reshape(-1)
        if weight.size != mesh.ncells:
            raise capi.WfxError("one weight per cell expected")
        w = weight[:, None] * w
    m = np.bincount(dofs, weights=w.reshape(-1), minlength=mesh.ndofs)
    return np.bincount(dofs, weights=(coeff[:, None] * w).reshape(-1), minlength=mesh.ndofs) / m


class Medium:
    """A layered acoustic medium (DESIGN.md section 4.5e): per-cell density rho [kg/m^3] > 0, speed of sound c [m/s]
    > 0 and, optionally, coefficient of nonlinearity beta >= 0, each a scalar or one value per cell, solving

        (1 / (rho c^2)) p_tt - div((1 / rho) grad p) [- loss] = (beta / (rho^2 c^4)) (p^2)_tt

    with p and (1 / rho) dp/dn continuous at interfaces.  Multiplied by rho_ref c0^2 it maps onto per-cell and
    per-facet weights of the existing operators: stiffness rho_ref / rho_c (Geometry.scale_cells), mass
    rho_ref c0^2 / (rho_c c_c^2) (MassOperator cell_weight), facet masses rho_ref / rho_f on tag 1 and
    rho_ref c0 / (rho_f c_f) on tag 2 (BoundaryOperator facet_weight, f the facet's cell), and a per-dof kappa for
    the Westervelt model.  With rho = rho_ref and c = c0 every weight is exactly 1.  The loss term becomes
    delta (c / c0)^2.  Pass it as `medium=` to a wave model; cfl_timestep(h, medium.c_max, ...) gives its step.
    alpha0 [Np/m at 1 MHz] >= 0 and y > 0 (scalars or per cell, given together): the tissue's power-law absorption
    alpha0 (f / 1 MHz)^y, which Medium.relaxation fits with relaxation processes (DESIGN.md section 4.5f) and
    PennesGLL.heat_from_wave(..., medium=) heats with."""

    def __init__(self, rho, c, beta=None, rho_ref=1000.0, alpha0=None, y=None):
        def arr(name, a, positive):
            a = np.asarray(a, dtype=np.float64)
            if a.ndim > 1:
                raise capi.WfxError(f"medium: {name} must be a scalar or one value per cell")
            if not np.all(np.isfinite(a)) or not np.all(a > 0 if positive else a >= 0):
                need = "positive" if positive else "not negative"
                raise capi.WfxError(f"medium: {name} must be finite and {need}")
            return a
        self.rho, self.c = arr("rho", rho, True), arr("c", c, True)
        self.beta = None if beta is None else arr("beta", beta, False)
        if np.ndim(rho_ref):
            raise capi.WfxError("medium: rho_ref must be a scalar")
        self.rho_ref = float(arr("rho_ref", rho_ref, True))
        if (alpha0 is None) != (y is None):
            raise capi.WfxError("medium: alpha0 and y go together")
        self.alpha0 = None if alpha0 is None else arr("alpha0", alpha0, False)
        self.y = None if y is None else arr("y", y, True)
        sizes = {a.size for a in (self.rho, self.c, self.beta, self.alpha0, self.y) if a is not None and a.ndim == 1}
        if len(sizes) > 1:
            raise capi.WfxError("medium: per-cell arrays differ in length")
        self.ncells = sizes.pop() if sizes else None

    @property
    def c_max(self):
        """the largest speed of sound, for the CFL step"""
        return float(np.max(self.c))

    def _cells(self, a, ncells):
        if self.ncells is not None and self.ncells != ncells:
            raise capi.WfxError(f"medium: {self.ncells} cells given, the mesh has {ncells}")
        return np.broadcast_to(a, (ncells,)).astype(np.float64)

    def cell_impedance(self, ncells):
        """Z_c = rho_c c_c, one value per cell"""
        return self._cells(self.rho, ncells) * self._cells(self.c, ncells)

    def stiffness_weight(self, ncells):
        """sigma_c = rho_ref / rho_c"""
        return self.rho_ref / self._cells(self.rho, ncells)

    def mass_weight(self, ncells, c0):
        """mu_c = rho_ref c0^2 / (rho_c c_c^2)"""
        rho, c = self._cells(self.rho, ncells), self._cells(self.c, ncells)
        return (self.rho_ref * c0 * c0) / (rho * c * c)

    def facet_weight(self, mesh, c0):
        """one weight per facet triplet: rho_ref / rho_f on tag 1, rho_ref c0 / (rho_f c_f) = Z_ref / Z_f on tag 2,
        1 elsewhere (f the facet's cell)"""
        rho, c = self._cells(self.rho, mesh.ncells), self._cells(self.c, mesh.ncells)
        fc = np.asarray(mesh.facet_cells, dtype=np.int64)
        tag = np.asarray(mesh.facet_tags)
        w = np.ones(len(fc))
        w[tag == 1] = self.rho_ref / rho[fc[tag == 1]]
        w[tag == 2] = (self.rho_ref * c0) / (rho[fc[tag == 2]] * c[fc[tag == 2]])
        return w

    def cell_kappa(self, ncells, beta=0.0):
        """kappa_c = 2 beta_c / (rho_c c_c^2); beta: the value where the medium has none"""
        b = self._cells(beta if self.beta is None else self.beta, ncells)
        rho, c = self._cells(self.rho, ncells), self._cells(self.c, ncells)
        return 2.0 * b / (rho * c * c)

    def kappa(self, mesh, detJw, c0, beta=0.0):
        """kappa_i = sum_c kappa_c mu_c (detJ w)_{c,i} / m~_i with m~ the weighted mass (host set-up).  A dof whose
        cells all carry the same kappa_c gets that value exactly, so that a homogeneous region (the reference medium
        in particular) steps with the scalar kappa bit for bit."""
        return _shared_exact_average(mesh, detJw, self.cell_kappa(mesh.ncells, beta), self.mass_weight(mesh.ncells, c0))

    def relaxation(self, f_lo, f_hi, mechanisms=3):
        """Relaxation processes that reproduce alpha0 (f / 1 MHz)^y over the band [f_lo, f_hi] [Hz] in every cell
        (DESIGN.md section 4.5f).  The `mechanisms` (1..3) relaxation frequencies are log-spaced over
        [f_lo / s, s f_hi] and shared by all cells, with the spread s in 1.5..3 that fits best.  Per cell, eps >= 0 is
        the minimax fit of the first-order attenuation (a linear program), refined on the exact alpha from
        k(w) = (w / c) sqrt(1 + sum eps / (1 + i w tau)).  Returns a Relaxation whose fit_error is the largest
        relative error of the exact alpha over the band, over all cells."""
        if self.alpha0 is None:
            raise capi.WfxError("relaxation: the medium has no absorption (alpha0, y)")
        if not (0 < f_lo < f_hi and np.isfinite(f_hi)):
            raise capi.WfxError("relaxation: the band needs 0 < f_lo < f_hi")
        if mechanisms not in (1, 2, 3):
            raise capi.WfxError("relaxation: 1 to 3 mechanisms")
        n = self.ncells or 1
        a0, y, c = (np.broadcast_to(a, (n,)) for a in (self.alpha0, self.y, self.c))
        groups, inv = np.unique(np.stack([a0, y, c], 1), axis=0, return_inverse=True)
        best = None
        for spread in (1.5, 2.0, 2.5, 3.0):
            fr = np.geomspace(f_lo / spread, spread * f_hi, mechanisms) if mechanisms > 1 else np.array(
                [np.sqrt(f_lo * f_hi)])
            tau = 1.0 / (2.0 * np.pi * fr)
            fits = [_fit_relaxation(tau, g[0], g[1], g[2], f_lo, f_hi) for g in groups]
            err = max(e for _, e in fits)
            if best is None or err < best[0]:
                best = (err, tau, np.stack([e for e, _ in fits], 1))
        err, tau, eps_groups = best
        return Relaxation(tau, eps_groups[:, inv.reshape(-1)], c, fit_error=err)


def _shared_exact_average(mesh, detJw, coeff, weight):
    """cell_to_dof_average with `weight`, except that a dof whose cells all carry the same value gets it exactly"""
    avg = cell_to_dof_average(mesh, detJw, coeff, weight)
    perm = capi.compute_permutations(mesh.P)
    dofs = np.asarray(mesh.dofmap)[:, perm].reshape(-1)
    cpt = np.repeat(coeff, len(perm))
    lo, hi = np.full(mesh.ndofs, np.inf), np.full(mesh.ndofs, -np.inf)
    np.minimum.at(lo, dofs, cpt)
    np.maximum.at(hi, dofs, cpt)
    return np.where(lo == hi, lo, avg)


def _relax_k(f, tau, eps, c):
    """k(w) = (w / c) sqrt(1 + sum_nu eps_nu / (1 + i w tau_nu)), shape f.shape + (ncells,); eps [M, ncells]"""
    w = 2.0 * np.pi * np.asarray(f, dtype=np.float64)[..., None]
    x = sum(eps[j] / (1.0 + 1j * w * tau[j]) for j in range(len(tau)))
    return w / c * np.sqrt(1.0 + x)


def _fit_relaxation(tau, a0, y, c, f_lo, f_hi, iters=8):
    """(eps [M], max relative error of the exact alpha) for alpha0 (f / 1 MHz)^y over [f_lo, f_hi] at speed c"""
    from scipy.optimize import linprog
    M = len(tau)
    if a0 == 0:
        return np.zeros(M), 0.0
    f = np.geomspace(f_lo, f_hi, 96)
    w = 2.0 * np.pi * f
    target = a0 * (f / 1e6) ** y
    A = (w / (2.0 * c))[:, None] * (w[:, None] * tau[None, :]) / (1.0 + (w[:, None] * tau[None, :]) ** 2)
    exact = lambda e: -_relax_k(f, tau, e[:, None], c)[:, 0].imag  # noqa: E731
    goal = target.copy()
    eps = np.zeros(M)
    for _ in range(iters):
        # minimise t subject to |A eps / goal - 1| <= t, eps >= 0
        Ar = A / goal[:, None]
        one = np.ones((len(f), 1))
        res = linprog(np.r_[np.zeros(M), 1.0], A_ub=np.block([[Ar, -one], [-Ar, -one]]),
                      b_ub=np.r_[np.ones(len(f)), -np.ones(len(f))], bounds=[(0, None)] * (M + 1), method="highs")
        if res.status != 0:
            raise capi.WfxError(f"relaxation: the fit failed ({res.message})")
        eps = res.x[:M]
        # the exact alpha differs from the first-order one by a smooth factor: aim the first-order fit past it
        goal = target * (A @ eps) / exact(eps)
    fd = np.geomspace(f_lo, f_hi, 1024)
    return eps, float(np.abs(-_relax_k(fd, tau, eps[:, None], c)[:, 0].imag / (a0 * (fd / 1e6) ** y) - 1.0).max())


class Relaxation:
    """M = 1..3 relaxation processes (DESIGN.md section 4.5f) with shared relaxation times tau [M] > 0 [s] and
    strengths eps [M, ncells] >= 0 (or [M]: the same in every cell), in cells with the high-frequency sound speed c
    (scalar or per cell):  tau_nu q_nu' + q_nu = eps_nu p,  (1 / (rho c^2)) (p + sum_nu q_nu)_tt - ... .  For
    p ~ e^{i w t}:  k(w) = (w / c) sqrt(1 + sum_nu eps_nu / (1 + i w tau_nu)),  alpha = -Im k,  phase speed w / Re k
    (below c, rising to c at high frequency).  fit_error: Medium.relaxation's largest relative error of alpha."""

    def __init__(self, tau, eps, c, fit_error=None):
        tau = np.asarray(tau, dtype=np.float64).reshape(-1)
        if not 1 <= tau.size <= capi.RELAX_MAX:
            raise capi.WfxError(f"relaxation: 1 to {capi.RELAX_MAX} processes")
        if not np.all(np.isfinite(tau)) or not np.all(tau > 0):
            raise capi.WfxError("relaxation: tau must be finite and positive")
        eps = np.asarray(eps, dtype=np.float64)
        if eps.ndim == 1:
            eps = eps[:, None]
        if eps.ndim != 2 or eps.shape[0] != tau.size:
            raise capi.WfxError("relaxation: eps must have shape [M] or [M, ncells]")
        if not np.all(np.isfinite(eps)) or not np.all(eps >= 0):
            raise capi.WfxError("relaxation: eps must be finite and not negative")
        c = np.asarray(c, dtype=np.float64)
        if c.ndim > 1 or not np.all(np.isfinite(c)) or not np.all(c > 0):
            raise capi.WfxError("relaxation: c must be finite and positive, a scalar or one value per cell")
        if c.ndim and eps.shape[1] not in (1, c.size):
            raise capi.WfxError("relaxation: eps and c differ in the number of cells")
        self.tau, self.eps, self.c = np.ascontiguousarray(tau), np.ascontiguousarray(eps), c
        self.fit_error = fit_error

    @property
    def M(self):
        return self.tau.size

    def eps_cells(self, ncells):
        """eps [M, ncells]"""
        if self.eps.shape[1] not in (1, ncells):
            raise capi.WfxError(f"relaxation: {self.eps.shape[1]} cells given, the mesh has {ncells}")
        return np.ascontiguousarray(np.broadcast_to(self.eps, (self.M, ncells)))

    def alpha(self, f):
        """attenuation [Np/m] per cell at frequency f [Hz] (shape f.shape + (ncells,)), from the exact k(w)"""
        return -_relax_k(f, self.tau, self.eps, self.c).imag

    def phase_speed(self, f):
        """phase speed w / Re k [m/s] per cell at frequency f [Hz]"""
        return 2.0 * np.pi * np.asarray(f, dtype=np.float64)[..., None] / _relax_k(f, self.tau, self.eps, self.c).real

    def max_dt(self):
        """just below the step at which rk4 refuses: dt (1 + sum_nu max eps_nu) / tau_min = 2.5 (a lone dof's
        eigenvalue -(1 + eps) / tau; RK4 is unstable beyond 2.785).  The per-dof eps are averages of the per-cell
        ones, so this bound holds for every mesh."""
        return 2.5 * (1.0 - 1e-9) * self.tau.min() / (1.0 + self.eps.max(axis=1).sum())

    def eps_dofs(self, mesh, detJw, mass_weight=None):
        """eps_nu,i = sum_c eps_nu,c mu_c (detJ w)_{c,i} / m~_i [M, ndofs] with the weighted mass m~ (mass_weight: mu_c,
        None for 1), exact for the lumped system; a dof whose cells share one eps gets it exactly"""
        e = self.eps_cells(mesh.ncells)
        return np.ascontiguousarray(np.stack([_shared_exact_average(mesh, detJw, e[j], mass_weight)
                                              for j in range(self.M)]))


class PML:
    """A perfectly matched layer (DESIGN.md section 4.5g): damping profiles zeta [3, ndofs] >= 0 [1/s], zeta[j] along
    physical axis j, on the dofs of `mesh`.  The layer is the cells where some zeta_j > 0 at one of their points; a
    wave model given it (`pml=`, set_pml) stretches its stiffness term there with the second-order PML of Grote and
    Sim (2010).  The Westervelt and relaxation terms are not stretched: the layer reflects O(kappa p) and O(eps)."""

    def __init__(self, mesh, zeta):
        z = np.array(zeta, dtype=np.float64)
        if z.shape != (3, mesh.ndofs):
            raise capi.WfxError(f"pml: zeta must have shape (3, {mesh.ndofs})")
        if not np.all(np.isfinite(z)) or np.any(z < 0):
            raise capi.WfxError("pml: zeta must be finite and not negative")
        self.zeta = np.ascontiguousarray(z)

    @classmethod
    def box(cls, mesh, thickness, faces, c, R0=1e-4, order=2):
        """A layer `thickness` deep inside the mesh from each named face (axis 0..2, side 0 (low) or 1 (high)) of the
        bounding box of the dof coordinates: zeta_j = zeta_max (d_j / L)^order at depth d_j into a layer on axis j,
        zeta_max = (order + 1) c ln(1 / R0) / (2 L), the normal-incidence reflection R0 of the continuous layer with a
        rigid end for waves of speed c.  Edges and corners get two or three nonzero zeta_j."""
        from .mesh import dof_coordinates
        L = float(thickness)
        if not (np.isfinite(L) and L > 0):
            raise capi.WfxError("pml: thickness must be finite and positive")
        if not (np.isfinite(c) and c > 0):
            raise capi.WfxError("pml: c must be finite and positive")
        if not (0 < R0 < 1):
            raise capi.WfxError("pml: R0 must lie in (0, 1)")
        if not (np.isfinite(order) and order >= 0):
            raise capi.WfxError("pml: order must be finite and not negative")
        faces = [tuple(int(v) for v in f) for f in faces]
        if not faces or any(len(f) != 2 or f[0] not in (0, 1, 2) or f[1] not in (0, 1) for f in faces) \
                or len(set(faces)) != len(faces):
            raise capi.WfxError("pml: faces must be distinct (axis 0..2, side 0 or 1) pairs")
        x = dof_coordinates(mesh)
        lo, hi = x.min(axis=0), x.max(axis=0)
        zmax = (order + 1) * float(c) * np.log(1.0 / R0) / (2.0 * L)
        zeta = np.zeros((3, mesh.ndofs))
        for axis, side in faces:
            sides = sum(1 for a, _ in faces if a == axis)
            if sides * L > hi[axis] - lo[axis]:
                raise capi.WfxError("pml: the layers are thicker than the mesh")
            d = (lo[axis] + L - x[:, axis]) if side == 0 else (x[:, axis] - (hi[axis] - L))
            d = np.clip(d, 0.0, L)
            zeta[axis] = np.maximum(zeta[axis], zmax * (d / L) ** order * (d > 0))
        return cls(mesh, zeta)

    @property
    def zeta_max(self):
        return float(self.zeta.max()) if self.zeta.size else 0.0

    def max_dt(self):
        """The largest time step rk4 accepts with this layer: dt max zeta < 2.5 (a lone dof has the eigenvalues
        -zeta_j; RK4 is stable on the real axis to 2.785)"""
        zm = self.zeta_max
        return 2.5 / zm if zm > 0 else np.inf


class PennesGLL:
    """The Pennes bioheat model with a CEM43 thermal dose (DESIGN.md section 4.5d), one rank:

        rhoC T_t = div(k grad T) - wbCb (T - T_art) + s Q        -k dT/dn = h_j (T - T_ext_j) on tag j = 1, 2

    other faces insulated.  conductivity k [W/(m K)], heat_capacity rhoC [J/(m^3 K)] and perfusion wbCb
    [W/(m^3 K)] are scalars or one value per cell: a per-cell k scales this model's own geometry (k_c / max k), a
    per-cell rhoC or wbCb becomes its mass-weighted per-dof average (cell_to_dof_average).  h = (h1, h2)
    [W/(m^2 K)], T_ext = (T_ext1, T_ext2); boundary=None builds the facet operator only when h != 0.  The state is
    held as the rise over T_art; temperatures in and out are T = T_art + rise.  The heat source Q starts at 0 and
    the heat scale s at 1."""

    def __init__(self, mesh, degree, conductivity, heat_capacity, perfusion=0.0, T_art=37.0, h=(0.0, 0.0),
                 T_ext=None, dtype=np.float64, ctx=None, stiffness_mode=capi.STIFF_AUTO, boundary=None, _ops=None):
        self.ctx = ctx or Context.get()
        self.V = mesh
        self.P = int(degree)
        self.dtype = np.dtype(dtype)
        self.ndofs = int(mesh.ndofs)
        self.T_art = float(T_art)
        k = np.asarray(conductivity, dtype=np.float64)
        h = np.asarray(h, dtype=np.float64).reshape(2)
        T_ext = np.full(2, self.T_art) if T_ext is None else np.asarray(T_ext, dtype=np.float64).reshape(2)
        if boundary is None:
            boundary = bool(np.any(h != 0))
        if _ops is None:
            self.geometry = Geometry(mesh, self.P, dtype, self.ctx)
            if k.ndim:
                self.k = float(k.max())
                self.geometry.scale_cells(k / self.k)
            else:
                self.k = float(k)
            self.mass_op = MassOperator(mesh, self.P, dtype, self.ctx, self.geometry)
            self.stiff_op = StiffnessOperator(mesh, self.P, None, dtype, self.ctx, self.geometry, mode=stiffness_mode)
            self.bnd_op = BoundaryOperator(mesh, self.P, dtype, self.ctx) if boundary else None
        else:
            self.geometry, self.mass_op, self.stiff_op, self.bnd_op = _ops
            if k.ndim:
                raise capi.WfxError("shared operators: a per-cell conductivity needs the model's own geometry")
            self.k = float(k)
            if not boundary:
                self.bnd_op = None
        detJw = None

        def per_dof(c):
            nonlocal detJw
            c = np.asarray(c, dtype=np.float64)
            if not c.ndim:
                return np.full(self.ndofs, float(c))
            if detJw is None:
                detJw = self.geometry.detJw()
            return cell_to_dof_average(mesh, detJw, c)

        self.rhoc = per_dof(heat_capacity)
        self.perf = per_dof(perfusion)
        self.handle = C.c_void_p()
        capi.call("wfx_thermal_create", self.ctx.handle, self.stiff_op.handle, self.mass_op.handle,
                  self.bnd_op.handle if self.bnd_op is not None else None, self.k, capi.f64p(self.rhoc),
                  capi.f64p(self.perf), self.T_art, capi.f64p(np.ascontiguousarray(h)),
                  capi.f64p(np.ascontiguousarray(T_ext)), C.byref(self.handle))

    @classmethod
    def from_wave(cls, model, conductivity, heat_capacity, perfusion=0.0, T_art=37.0, h=(0.0, 0.0), T_ext=None,
                  boundary=None):
        """A thermal model on a wave model's mesh that shares its geometry, stiffness, mass and boundary operators
        (none keeps per-apply state).  Refused when the wave model's geometry was scaled (wfx_geometry_scale_cells):
        the diffusion term would carry the acoustic coefficient."""
        if getattr(model.geometry, "scaled", False):
            raise capi.WfxError("from_wave: the wave model's geometry is scaled; build the thermal model's own operators")
        ops = (model.geometry, model.mass_op, model.stiff_op, model.bnd_op)
        return cls(model.V, model.k_, conductivity, heat_capacity, perfusion, T_art, h, T_ext, dtype=model.dtype,
                   ctx=model.ctx, boundary=boundary, _ops=ops)

    def init(self):
        """T = T_art everywhere; resets the dose"""
        capi.call("wfx_thermal_init", self.handle)

    def set_state(self, T):
        """T [ndofs] (temperatures); resets the dose"""
        rise = np.ascontiguousarray(np.asarray(T, dtype=np.float64) - self.T_art, dtype=self.dtype)
        if rise.shape != (self.ndofs,):
            raise capi.WfxError(f"thermal state must have shape ({self.ndofs},)")
        capi.call("wfx_thermal_set_state", self.handle, C.c_void_p(rise.ctypes.data))

    def rise(self):
        """theta = T - T_art in the model dtype, as held on the device"""
        out = np.empty(self.ndofs, dtype=self.dtype)
        capi.call("wfx_thermal_get_state", self.handle, C.c_void_p(out.ctypes.data))
        return out

    def get_state(self):
        """T = T_art + theta, fp64"""
        return self.T_art + self.rise().astype(np.float64)

    def state_ptr(self):
        p = C.c_void_p()
        capi.call("wfx_thermal_state_ptr", self.handle, C.byref(p))
        return p.value

    def set_heat_source(self, Q=None):
        """Q [W/m^3] per dof (None: 0)"""
        q = None if Q is None else np.ascontiguousarray(Q, dtype=np.float64)
        if q is not None and q.shape != (self.ndofs,):
            raise capi.WfxError(f"heat source must have shape ({self.ndofs},)")
        capi.call("wfx_thermal_set_heat_source", self.handle, capi.f64p(q))

    def heat_from_wave(self, model, alpha0, y=None, rho0=None, c0=None, member=0, medium=None):
        """Q = sum_h alpha0 (h f0 / 1 MHz)^y |p_h|^2 / (rho0 c0) from the harmonic maps of `model`'s field statistics,
        computed on the device.  alpha0 [Np/m at 1 MHz]: a scalar or one value per dof; member: the ensemble member.
        medium: a Medium on this mesh; 1 / (rho0 c0) is then the per-dof mass-weighted average of 1 / (rho_c c_c),
        folded into alpha0 (rho0 and c0 are not used).  alpha0 = None takes alpha0 from the medium, as its per-dof
        mass-weighted average, and y from the medium too when y is None; the medium must then have one y everywhere
        (a per-cell y is refused)."""
        if alpha0 is None:
            if medium is None or medium.alpha0 is None:
                raise capi.WfxError("heat_from_wave: alpha0 = None needs a medium with alpha0 and y")
            ys = np.unique(medium.y)
            if ys.size != 1:
                raise capi.WfxError("heat_from_wave: the medium's y varies per cell; pass alpha0 and y")
            if y is None:
                y = float(ys[0])
            elif float(y) != float(ys[0]):
                raise capi.WfxError("heat_from_wave: y differs from the medium's")
            nc = self.V.ncells
            alpha0 = cell_to_dof_average(self.V, self.geometry.detJw(), np.broadcast_to(medium.alpha0, (nc,)))
        if y is None or (medium is None and (rho0 is None or c0 is None)):
            raise capi.WfxError("heat_from_wave: needs y, and rho0 and c0 without a medium")
        a = np.asarray(alpha0, dtype=np.float64)
        a_host = None
        if a.ndim:
            a_host = np.ascontiguousarray(a.reshape(-1))
            if a_host.size != self.ndofs:
                raise capi.WfxError(f"alpha0 must be a scalar or have shape ({self.ndofs},)")
        if medium is not None:
            nc = self.V.ncells
            inv_z = 1.0 / medium.cell_impedance(nc)
            a_host = np.ascontiguousarray(np.broadcast_to(a, (self.ndofs,)) *
                                          cell_to_dof_average(self.V, self.geometry.detJw(), inv_z))
            a, rho0, c0 = np.asarray(0.0), 1.0, 1.0
        capi.call("wfx_thermal_heat_from_wave", self.handle, model.handle, int(member), float(a) if not a.ndim else 0.0,
                  capi.f64p(a_host), float(y), float(rho0), float(c0))

    def heat_source(self):
        q = np.empty(self.ndofs)
        capi.call("wfx_thermal_get_heat_source", self.handle, capi.f64p(q))
        return q

    def set_heat_scale(self, s):
        """s >= 0 multiplies Q (duty cycles: heating with s = 1, cooling with s = 0)"""
        capi.call("wfx_thermal_set_heat_scale", self.handle, float(s))

    def rhs(self, theta, out):
        """out = theta' at theta (rises), CUDA tensors of the model dtype"""
        capi.call("wfx_thermal_rhs", self.handle, C.c_void_p(theta.data_ptr()), C.c_void_p(out.data_ptr()),
                  _stream_ptr())

    def rk4(self, startTime, finalTime, timeStep, max_steps=0, stream=None):
        steps, t_end = C.c_int64(), C.c_double()
        capi.call("wfx_thermal_rk4", self.handle, float(startTime), float(finalTime), float(timeStep), int(max_steps),
                  C.byref(steps), C.byref(t_end), stream if stream is not None else _stream_ptr())
        return steps.value, t_end.value

    def dose(self):
        """ThermalDose(steps, cem43 [min], T_max = T_art + max rise) accumulated since init / set_state"""
        n = C.c_int64()
        cem = np.empty(self.ndofs)
        thmax = np.empty(self.ndofs, dtype=self.dtype)
        capi.call("wfx_thermal_get_dose", self.handle, C.byref(n), capi.f64p(cem), C.c_void_p(thmax.ctypes.data))
        return ThermalDose(n.value, cem, self.T_art + thmax.astype(np.float64))

    def max_eigenvalue(self, iters=200):
        """(lambda, dt_max) of the power iteration (wfx_thermal_stable_dt): lambda approaches the largest eigenvalue
        from below, so dt_max = 2.785293563405282 / lambda may lie above the true RK4 limit."""
        lam, dtm = C.c_double(), C.c_double()
        capi.call("wfx_thermal_stable_dt", self.handle, int(iters), C.byref(lam), C.byref(dtm))
        return lam.value, dtm.value

    def stable_dt(self, safety=0.8, iters=200):
        """safety * dt_max: a time step inside the RK4 stability limit (the safety factor covers the estimate's
        shortfall)"""
        return safety * self.max_eigenvalue(iters)[1]

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_thermal_destroy(self.handle)
            self.handle = None
