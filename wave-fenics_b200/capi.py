"""ctypes binding of include/wavefx.h (libwavefx.so).

There is no CPU fallback: if the shared library is missing this module raises, and every
device entry point fails when no B200 is present.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WFX_LIB") or os.path.join(HERE, "libwavefx.so")

F64, F32 = 0, 1
STIFF_AUTO, STIFF_CELL_COLOUR, STIFF_NO_SPLIT, STIFF_CELL_STREAM, STIFF_ENSEMBLE = 0, 1, 2, 4, 8
ENSEMBLE_MAX = 8
HARMONICS_MAX = 8
RELAX_MAX = 3

_c_i32p = C.POINTER(C.c_int32)
_c_i64p = C.POINTER(C.c_int64)
_c_f64p = C.POINTER(C.c_double)
_vp = C.c_void_p
_vpp = C.POINTER(C.c_void_p)


class WfxError(RuntimeError):
    pass


SNAPSHOT_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p)


def _load():
    if not os.path.exists(LIB_PATH):
        raise WfxError(
            f"{LIB_PATH} not found: build it with `python wave-fenics_b200/build.py` "
            "(the B200 path has no CPU fallback)")
    return C.CDLL(LIB_PATH)


lib = _load()

# name -> argtypes; every function returns int status except wfx_last_error / wfx_version
_SIG = {
    "wfx_gll": [C.c_int, _c_f64p, _c_f64p],
    "wfx_deriv_1d": [C.c_int, _c_f64p],
    "wfx_compute_permutations": [C.c_int, _c_i32p],
    "wfx_tabulate_basis_and_permutation": [C.c_int, _c_f64p, _c_i32p],
    "wfx_reorder_dofmap": [C.c_int, C.c_int64, _c_i32p, _c_i32p],
    "wfx_tabulate_1d": [C.c_int, C.c_int, C.c_int, _c_f64p, C.POINTER(C.c_int)],
    "wfx_ctx_create": [C.c_int, _vpp],
    "wfx_ctx_destroy": [_vp],
    "wfx_ctx_sync": [_vp],
    "wfx_malloc": [_vp, C.c_int64, _vpp],
    "wfx_free": [_vp, _vp],
    "wfx_memcpy_h2d": [_vp, _vp, _vp, C.c_int64],
    "wfx_memcpy_d2h": [_vp, _vp, _vp, C.c_int64],
    "wfx_geometry_create": [_vp, C.c_int, C.c_int, C.c_int64, C.c_int64, _c_f64p, _c_i32p, _vpp],
    "wfx_geometry_get": [_vp, _c_f64p, _c_f64p],
    "wfx_geometry_info": [_vp, _c_i64p, _c_i64p],
    "wfx_geometry_scale_cells": [_vp, _c_f64p],
    "wfx_geometry_destroy": [_vp],
    "wfx_compute_jacobian_data": [_vp, C.c_int64, C.c_int64, _c_f64p, _c_i32p, C.c_int, _c_f64p,
                                  _c_f64p, _c_f64p, _c_f64p, _c_f64p, _c_f64p],
    "wfx_stiffness_create": [_vp, _vp, C.c_int64, _c_i32p, C.c_double, C.c_int, _vpp],
    "wfx_stiffness_apply": [_vp, _vp, _vp, C.c_int, _vp],
    "wfx_stiffness_create_partitioned": [_vp, _vp, C.c_int64, _c_i32p, C.c_double, C.c_int, C.c_int64,
                                         _c_i32p, _vpp],
    "wfx_stiffness_apply_part": [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp],
    "wfx_halo_update_rev_fwd_scaled": [_vp, _vp, _vp, _vp],
    "wfx_boundary_assemble": [_vp, _vp],
    "wfx_stiffness_apply_scaled": [_vp, _vp, _vp, _vp, _vp],
    "wfx_stiffness_apply_ensemble": [_vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp],
    "wfx_stiffness_apply_host": [_vp, _vp, _vp, C.c_int],
    "wfx_stiffness_mass_apply_host": [_vp, _vp, _vp, _vp],
    "wfx_stiffness_mass_apply_host_batch": [_vp, _vp, C.c_int, _vpp, _vpp],
    "wfx_stiffness_info": [_vp, _c_i64p, C.POINTER(C.c_int), _c_i64p, _c_f64p, _c_f64p,
                           C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "wfx_stiffness_kernel_info": [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_int), C.POINTER(C.c_int), _c_i64p],
    "wfx_stiffness_destroy": [_vp],
    "wfx_mass_create": [_vp, _vp, C.c_int64, _c_i32p, _vpp],
    "wfx_mass_create_weighted": [_vp, _vp, C.c_int64, _c_i32p, _c_f64p, _vpp],
    "wfx_mass_apply": [_vp, _vp, _vp, C.c_int, _vp],
    "wfx_mass_apply_host": [_vp, _vp, _vp, C.c_int],
    "wfx_mass_apply_inverse": [_vp, _vp, _vp, _vp],
    "wfx_mass_assemble": [_vp, _vp],
    "wfx_mass_diagonal": [_vp, _vpp],
    "wfx_mass_inverse_diagonal": [_vp, _vpp],
    "wfx_mass_destroy": [_vp],
    "wfx_gather": [_vp, C.c_int, C.c_int64, _vp, _vp, _vp, _vp],
    "wfx_scatter_plan_create": [_vp, C.c_int64, _c_i32p, C.c_int64, _vpp],
    "wfx_scatter_add": [_vp, C.c_int, _vp, _vp, C.c_int, _vp],
    "wfx_scatter_plan_destroy": [_vp],
    "wfx_boundary_create": [_vp, C.c_int, C.c_int, C.c_int64, _c_i32p, _c_i32p, _c_i32p, C.c_int64,
                            _c_f64p, _c_i32p, C.c_int64, _c_i32p, _vpp],
    "wfx_boundary_create_weighted": [_vp, C.c_int, C.c_int, C.c_int64, _c_i32p, _c_i32p, _c_i32p, C.c_int64,
                                     _c_f64p, _c_i32p, C.c_int64, _c_i32p, _c_f64p, _vpp],
    "wfx_boundary_apply": [_vp, C.c_double, C.c_double, _vp, _vp, _vp],
    "wfx_boundary_get": [_vp, _c_f64p, _c_f64p],
    "wfx_boundary_destroy": [_vp],
    "wfx_comm_unique_id": [C.c_char_p],
    "wfx_comm_create": [_vp, C.c_char_p, C.c_int, C.c_int, _vpp],
    "wfx_comm_destroy": [_vp],
    "wfx_halo_create": [_vp, _vp, C.c_int, C.c_int64, C.c_int64, C.c_int, _c_i32p, _c_i32p, _c_i32p, C.c_int,
                        _c_i32p, _c_i32p, _c_i32p, _vpp],
    "wfx_halo_transport": [_vp, C.POINTER(C.c_int)],
    "wfx_halo_update_fwd": [_vp, _vp, _vp],
    "wfx_halo_update_rev": [_vp, _vp, _vp],
    "wfx_halo_update_rev_fwd": [_vp, _vp, _vp],
    "wfx_halo_destroy": [_vp],
    "wfx_wave_create": [_vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_double, C.c_double, C.c_double, _vpp],
    "wfx_wave_create_ensemble": [_vp, _vp, _vp, _vp, C.c_int, C.c_int64, C.c_double, _c_f64p, _c_f64p, _vpp],
    "wfx_wave_create_westervelt": [_vp, _vp, _vp, _vp, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_double, C.c_double, _vpp],
    "wfx_wave_set_nonlinearity": [_vp, _c_f64p],
    "wfx_wave_set_relaxation": [_vp, C.c_int, _c_f64p, _c_f64p],
    "wfx_wave_get_relaxation_state": [_vp, _vp],
    "wfx_wave_set_relaxation_state": [_vp, _vp],
    "wfx_pml_create": [_vp, _vp, C.c_int64, _c_i32p, C.c_int64, _c_f64p, _c_i32p, _c_f64p, _vpp],
    "wfx_pml_info": [_vp, _c_i64p, _c_i64p, _c_f64p],
    "wfx_pml_destroy": [_vp],
    "wfx_wave_set_pml": [_vp, _vp],
    "wfx_wave_get_pml_state": [_vp, _vp, _vp],
    "wfx_wave_set_pml_state": [_vp, _vp, _vp],
    "wfx_wave_init": [_vp],
    "wfx_wave_set_state": [_vp, _vp, _vp],
    "wfx_wave_get_state": [_vp, _vp, _vp],
    "wfx_wave_state_ptrs": [_vp, _vpp, _vpp],
    "wfx_wave_f0": [_vp, C.c_double, _vp, _vp, _vp, _vp],
    "wfx_wave_f1": [_vp, C.c_double, _vp, _vp, _vp, _vp],
    "wfx_wave_rk4": [_vp, C.c_double, C.c_double, C.c_double, C.c_int64, _c_i64p, _c_f64p, _vp],
    "wfx_wave_set_probes": [_vp, C.c_int64, _c_i32p, C.c_int64],
    "wfx_wave_get_probe_series": [_vp, _c_i64p, _c_f64p, _vp],
    "wfx_wave_set_field_stats": [_vp, C.c_int, C.c_double, C.c_int],
    "wfx_wave_get_field_stats": [_vp, _c_i64p, _c_f64p, _c_f64p, _vp, _vp, _c_f64p],
    "wfx_wave_field_stats_info": [_vp, C.POINTER(C.c_int), _c_f64p, C.POINTER(C.c_int)],
    "wfx_wave_set_source_profile": [_vp, _c_f64p, _c_f64p],
    "wfx_wave_set_volume_source": [_vp, C.c_int64, _c_i32p, _c_f64p, _c_f64p],
    "wfx_wave_set_snapshot": [_vp, C.c_int64, _vp, _vp],
    "wfx_wave_destroy": [_vp],
    "wfx_thermal_create": [_vp, _vp, _vp, _vp, C.c_double, _c_f64p, _c_f64p, C.c_double, _c_f64p, _c_f64p, _vpp],
    "wfx_thermal_init": [_vp],
    "wfx_thermal_set_state": [_vp, _vp],
    "wfx_thermal_get_state": [_vp, _vp],
    "wfx_thermal_state_ptr": [_vp, _vpp],
    "wfx_thermal_set_heat_source": [_vp, _c_f64p],
    "wfx_thermal_heat_from_wave": [_vp, _vp, C.c_int, C.c_double, _c_f64p, C.c_double, C.c_double, C.c_double],
    "wfx_thermal_get_heat_source": [_vp, _c_f64p],
    "wfx_thermal_set_heat_scale": [_vp, C.c_double],
    "wfx_thermal_rhs": [_vp, _vp, _vp, _vp],
    "wfx_thermal_rk4": [_vp, C.c_double, C.c_double, C.c_double, C.c_int64, _c_i64p, _c_f64p, _vp],
    "wfx_thermal_get_dose": [_vp, _c_i64p, _c_f64p, _vp],
    "wfx_thermal_stable_dt": [_vp, C.c_int, _c_f64p, _c_f64p],
    "wfx_thermal_destroy": [_vp],
    "wfx_debug_structured_coords": [C.c_int64, C.c_int64, _c_i32p, _c_i32p, C.POINTER(C.c_int)],
    # debug helper (not in wavefx.h): host-only plan construction + verification
    "wfx_debug_stream_plan_check": [C.c_int, C.c_int64, C.c_int64, _c_i32p, C.POINTER(C.c_float), C.c_int, C.c_int,
                                    C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.POINTER(C.c_int), _c_i64p],
    "wfx_debug_plan_stats": [C.c_int, C.c_int64, C.c_int64, _c_i32p, C.POINTER(C.c_float), C.c_int,
                             C.c_int, C.c_int, _c_i64p],
}

lib.wfx_last_error.restype = C.c_char_p
lib.wfx_last_error.argtypes = []
lib.wfx_version.restype = C.c_int
lib.wfx_version.argtypes = []
_missing = set()
for _name, _args in _SIG.items():
    try:
        _f = getattr(lib, _name)
    except AttributeError:
        # an older experiment build named by WFX_LIB: its missing entry points fail when called
        _missing.add(_name)
        continue
    _f.argtypes = _args
    _f.restype = C.c_int


def check(status):
    if status != 0:
        raise WfxError(lib.wfx_last_error().decode(errors="replace"))


def call(name, *args):
    if name in _missing:
        raise WfxError(f"{LIB_PATH} does not export {name}")
    check(getattr(lib, name)(*args))


def i32p(a):
    if a is None:
        return None
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_c_i32p)


def f64p(a):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_c_f64p)


def dtype_code(dtype):
    dt = np.dtype(dtype)
    if dt == np.float64:
        return F64
    if dt == np.float32:
        return F32
    raise WfxError(f"unsupported scalar type {dt}")


# ---- host tables ---------------------------------------------------------------------------
def gll(P):
    pts, wts = np.empty(P + 1), np.empty(P + 1)
    call("wfx_gll", P, f64p(pts), f64p(wts))
    return pts, wts


def deriv_1d(P):
    D = np.empty((P + 1, P + 1))
    call("wfx_deriv_1d", P, f64p(D))
    return D


def compute_permutations(P):
    perm = np.empty((P + 1) ** 3, dtype=np.int32)
    call("wfx_compute_permutations", P, i32p(perm))
    return perm


def tabulate_basis_and_permutation(P):
    """(table [4, nq, nd], perm [nd]) as common/operators.hpp:13-32 returns them."""
    nd = (P + 1) ** 3
    table = np.empty((4, nd, nd))
    perm = np.empty(nd, dtype=np.int32)
    call("wfx_tabulate_basis_and_permutation", P, f64p(table.reshape(-1)), i32p(perm))
    return table, perm


def reorder_dofmap(dofmap, P):
    dofmap = np.ascontiguousarray(dofmap, dtype=np.int32)
    out = np.empty_like(dofmap)
    nd = (P + 1) ** 3
    call("wfx_reorder_dofmap", P, dofmap.size // nd, i32p(dofmap.reshape(-1)), i32p(out.reshape(-1)))
    return out


def tabulate_1d(P, q, derivative):
    m = C.c_int(0)
    call("wfx_tabulate_1d", P, q, derivative, None, C.byref(m))
    table = np.empty((m.value, P + 1))
    call("wfx_tabulate_1d", P, q, derivative, f64p(table), C.byref(m))
    return table


def debug_structured_coords(xdofs, npts):
    """(ok, ijk [ncells, 3]) -- integer grid coordinates from the connectivity (host only)."""
    xdofs = np.ascontiguousarray(xdofs, dtype=np.int32)
    ijk = np.zeros((xdofs.shape[0], 3), dtype=np.int32)
    ok = C.c_int()
    call("wfx_debug_structured_coords", xdofs.shape[0], int(npts), i32p(xdofs.reshape(-1)), i32p(ijk.reshape(-1)),
         C.byref(ok))
    return bool(ok.value), ijk


def debug_stream_plan_check(P, dofmap, ndofs, centroid=None, brick_order=True, brick=(4, 4, 4), W=8, shared=None,
                            relabel_axes=True):
    """Builds the streamed-cell kernel's plan on the host and verifies every invariant the kernel relies on
    (verify_stream_plan); raises WfxError on a violation."""
    dofmap = np.ascontiguousarray(dofmap, dtype=np.int32)
    nd = (P + 1) ** 3
    ncells = dofmap.size // nd
    stats = np.zeros(8, dtype=np.int64)
    axes = np.zeros(3, dtype=np.int32)
    cptr = None
    if centroid is not None:
        centroid = np.ascontiguousarray(centroid, dtype=np.float32)
        cptr = centroid.ctypes.data_as(C.POINTER(C.c_float))
    sptr = None
    if shared is not None:
        flags = np.zeros(ndofs, dtype=np.uint8)
        flags[np.asarray(shared, dtype=np.int64)] = 1
        sptr = flags.ctypes.data_as(C.POINTER(C.c_uint8))
    call("wfx_debug_stream_plan_check", P, ncells, ndofs, i32p(dofmap.reshape(-1)), cptr, int(bool(brick_order)),
         int(brick[0]), int(brick[1]), int(brick[2]), W, sptr, int(bool(relabel_axes)),
         axes.ctypes.data_as(C.POINTER(C.c_int)), stats.ctypes.data_as(_c_i64p))
    keys = ["colours", "batches", "part_split", "uni_nr", "untouched"]
    return dict(zip(keys, stats.tolist()), axis_perm=axes.tolist())


def debug_plan_stats(P, dofmap, ndofs, centroid=None, brick_edge=4, W=8, nloc_cap=65535):
    dofmap = np.ascontiguousarray(dofmap, dtype=np.int32)
    nd = (P + 1) ** 3
    ncells = dofmap.size // nd
    stats = np.zeros(16, dtype=np.int64)
    cptr = None
    if centroid is not None:
        centroid = np.ascontiguousarray(centroid, dtype=np.float32)
        cptr = centroid.ctypes.data_as(C.POINTER(C.c_float))
    call("wfx_debug_plan_stats", P, ncells, ndofs, i32p(dofmap.reshape(-1)), cptr, brick_edge, W,
         nloc_cap, stats.ctypes.data_as(_c_i64p))
    keys = ["cell_colours", "batches", "batch_colours", "nloc_max", "rounds", "padded_slots",
            "private_dofs", "batch_dofs", "untouched", "regular_batches", "Sx", "Sy", "ms_cell_plan", "ms_brick_plan"]
    return dict(zip(keys, stats.tolist()))
