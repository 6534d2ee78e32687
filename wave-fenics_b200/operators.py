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
    """y += M x with the collocated (diagonal) GLL mass (common/operators.hpp:86-108)."""

    def __init__(self, V, degree, dtype=np.float64, ctx=None, geometry=None):
        self.ctx = ctx or Context.get()
        self.P = int(degree)
        self.dtype = np.dtype(dtype)
        self.geometry = geometry or Geometry(V, degree, dtype, self.ctx)
        self.ndofs = int(V.ndofs)
        self.handle = C.c_void_p()
        dm = np.ascontiguousarray(V.dofmap, dtype=np.int32)
        capi.call("wfx_mass_create", self.ctx.handle, self.geometry.handle, self.ndofs,
                  capi.i32p(dm.reshape(-1)), C.byref(self.handle))

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
    """b += c0^2 g m1 - c0 m2 .* v_n  (forms.ufl:21-24 via assemble_vector, LinearGLL.hpp:175)."""

    def __init__(self, V, degree, dtype=np.float64, ctx=None):
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
        capi.call("wfx_boundary_create", self.ctx.handle, self.P, capi.dtype_code(self.dtype), len(fc),
                  capi.i32p(fc), capi.i32p(fl), capi.i32p(ft), x.shape[0], capi.f64p(x.reshape(-1)),
                  capi.i32p(xd.reshape(-1)), self.ndofs, capi.i32p(dm.reshape(-1)), C.byref(self.handle))

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


class LinearGLLOpt:
    """The wave model + RK4 driver (common/LinearGLL.hpp:37-287) on the GPU.

    mesh carries the facet tags (`meshtags` may be None or a (cells, local, tags) triple that
    overrides them)."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency,
                 pressureAmplitude, dtype=np.float64, ctx=None, halo=None, stiffness_mode=capi.STIFF_AUTO,
                 setup_halo=None):
        self.ctx = ctx or Context.get()
        self.V = mesh
        if meshtags is not None:
            import copy
            mesh = copy.copy(mesh)
            mesh.facet_cells, mesh.facet_local, mesh.facet_tags = meshtags
        self.k_ = int(degreeOfBasis)
        self.c0_, self.freq0_, self.p0_ = float(speedOfSound), float(sourceFrequency), float(pressureAmplitude)
        self.dtype = np.dtype(dtype)
        self.geometry = Geometry(mesh, self.k_, dtype, self.ctx)
        self.mass_op = MassOperator(mesh, self.k_, dtype, self.ctx, self.geometry)      # :105
        params = {"c0": self.c0_}
        self.stiff_op = StiffnessOperator(mesh, self.k_, params, dtype, self.ctx, self.geometry,
                                          mode=stiffness_mode)                           # :120
        self.bnd_op = BoundaryOperator(mesh, self.k_, dtype, self.ctx)                   # :113-115
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

    def __del__(self):
        if getattr(self, "handle", None) and getattr(capi, "lib", None) is not None:
            capi.lib.wfx_wave_destroy(self.handle)
            self.handle = None


class LinearGLLEnsemble(LinearGLLOpt):
    """nv wave models (1 <= nv <= 8) on one mesh with one speed of sound, stepped together: member m is
    LinearGLLOpt(mesh, meshtags, degree, c0, f0s[m], p0s[m]).  One rank.  The stiffness apply of a stage
    reads the geometric factors once for all members.  States are (ndofs, nv) arrays (member-interleaved,
    entry (dof i, member m) at i*nv + m); probe values come as (nrecords, nprobes, nv).  Snapshots are not
    available for ensembles."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequencies, pressureAmplitudes,
                 dtype=np.float64, ctx=None, stiffness_mode=capi.STIFF_AUTO):
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
        self.geometry = Geometry(mesh, self.k_, dtype, self.ctx)
        self.mass_op = MassOperator(mesh, self.k_, dtype, self.ctx, self.geometry)
        self.stiff_op = StiffnessOperator(mesh, self.k_, {"c0": self.c0_}, dtype, self.ctx, self.geometry,
                                          mode=stiffness_mode, ensemble=True)
        self.bnd_op = BoundaryOperator(mesh, self.k_, dtype, self.ctx)
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


class WesterveltGLLOpt(LinearGLLOpt):
    """The Westervelt model on one rank, with the surface of LinearGLLOpt (DESIGN.md section 4.5a):

        (1 - kappa p) p_tt - c0^2 lap p - delta lap p_t = kappa p_t^2,   kappa = 2 beta / (rho0 c0^2)

    dp/dn = g(t) on tag 1 (the source of LinearGLLOpt), dp/dn = -p_t / c0 on tag 2.  diffusivityOfSound
    delta [m^2/s] >= 0, coefficientOfNonlinearity beta >= 0, density rho0 [kg/m^3] > 0 when beta > 0.
    delta = beta = 0 is LinearGLLOpt bit for bit.  A per-cell coefficient set with Geometry.scale_cells
    multiplies the delta term too (delta_eff = delta * coeff)."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                 diffusivityOfSound, coefficientOfNonlinearity, density, dtype=np.float64, ctx=None,
                 stiffness_mode=capi.STIFF_AUTO):
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
        self.geometry = Geometry(mesh, self.k_, dtype, self.ctx)
        self.mass_op = MassOperator(mesh, self.k_, dtype, self.ctx, self.geometry)
        self.stiff_op = StiffnessOperator(mesh, self.k_, {"c0": self.c0_}, dtype, self.ctx, self.geometry,
                                          mode=stiffness_mode)
        self.bnd_op = BoundaryOperator(mesh, self.k_, dtype, self.ctx)
        self.halo = None
        self.handle = C.c_void_p()
        capi.call("wfx_wave_create_westervelt", self.ctx.handle, self.stiff_op.handle, self.mass_op.handle,
                  self.bnd_op.handle, int(mesh.size_local), self.c0_, self.freq0_, self.p0_, self.delta_,
                  self.beta_, self.rho0_, C.byref(self.handle))
        self.ndofs = int(mesh.ndofs)


class LossyGLLOpt(WesterveltGLLOpt):
    """The lossy wave model (WesterveltGLLOpt with beta = 0):  p_tt - c0^2 lap p - delta lap p_t = 0."""

    def __init__(self, mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                 diffusivityOfSound, dtype=np.float64, ctx=None, stiffness_mode=capi.STIFF_AUTO):
        super().__init__(mesh, meshtags, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                         diffusivityOfSound, 0.0, 1.0, dtype=dtype, ctx=ctx, stiffness_mode=stiffness_mode)


# dose of a thermal model (PennesGLL.dose): steps since init / set_state, CEM43 [min] and peak temperature per dof
ThermalDose = namedtuple("ThermalDose", "steps cem43 T_max")


def cell_to_dof_average(mesh, detJw, coeff):
    """Per-dof mass-weighted average of a per-cell coefficient, sum_c coeff_c (detJ w)_{c,i} / m_i with
    m_i = sum_c (detJ w)_{c,i}, the lumped mass: then coeff_i m_i is the GLL quadrature of the piecewise-constant
    coefficient.  detJw [ncells, nq] in the reference layout (Geometry.detJw, oracle.precompute_geometric_data)."""
    coeff = np.asarray(coeff, dtype=np.float64).reshape(-1)
    if coeff.size != mesh.ncells:
        raise capi.WfxError("one coefficient per cell expected")
    perm = capi.compute_permutations(mesh.P)
    dofs = np.asarray(mesh.dofmap)[:, perm].reshape(-1)
    w = np.asarray(detJw, dtype=np.float64).reshape(mesh.ncells, -1)
    m = np.bincount(dofs, weights=w.reshape(-1), minlength=mesh.ndofs)
    return np.bincount(dofs, weights=(coeff[:, None] * w).reshape(-1), minlength=mesh.ndofs) / m


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

    def heat_from_wave(self, model, alpha0, y, rho0, c0, member=0):
        """Q = sum_h alpha0 (h f0 / 1 MHz)^y |p_h|^2 / (rho0 c0) from the harmonic maps of `model`'s field statistics,
        computed on the device.  alpha0 [Np/m at 1 MHz]: a scalar or one value per dof; member: the ensemble member."""
        a = np.asarray(alpha0, dtype=np.float64)
        a_host = None
        if a.ndim:
            a_host = np.ascontiguousarray(a.reshape(-1))
            if a_host.size != self.ndofs:
                raise capi.WfxError(f"alpha0 must be a scalar or have shape ({self.ndofs},)")
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
