"""wave-fenics_b200: B200-native matrix-free hot path of waveFEniCS behind its operator API.

The directory name carries a hyphen, so it is imported through the `wave_fenics_b200`
shim module at the repository root.  All compute lives in libwavefx.so (csrc/); this
package is the Python host-side mirror of the reference's operator interface.
"""
from . import capi  # noqa: F401  (raises when libwavefx.so is missing: no CPU fallback)
from .capi import WfxError  # noqa: F401
from .mesh import HexMesh, create_box_hex, cfl_timestep, dof_coordinates  # noqa: F401
from .operators import (BoundaryOperator, Context, FieldStats, Geometry, LinearGLLEnsemble, LinearGLLOpt,  # noqa: F401
                        LossyGLLOpt, MassOperator, MassOperatorCPU, PennesGLL, StiffnessOperator, ThermalDose,
                        WesterveltGLLOpt, cell_to_dof_average, compute_jacobian_data, focus_delays)
