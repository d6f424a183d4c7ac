"""lsm_b200 — B200-native engine for LevelSetMethods.jl's dense-grid time-integration path.

The directory is called ``levelsetmethods.jl_b200`` (not an importable name); import it through the
``lsm_b200`` shim at the repository root.  Contents: ``csrc/`` (CUDA kernels + the C ABI of
``include/lsm_b200.h``), ``_lib.py`` (ctypes binding), ``api.py`` (host mirror of the reference's
Julia API for this path), ``julia/`` (the ccall glue for the real package).
"""
from . import _lib
from ._lib import LSMError, CFLError, TimeError, BCError, build
from .api import (Context, MultiContext, integrate_multi, compute_cfl_multi, default_context, set_default_context, CartesianGrid, BoundaryCondition, PeriodicBC,
                  ExtrapolationBC, NeumannBC, LinearExtrapolationBC, SymmetryBC, MeshField, Upwind, WENO5,
                  TimeScaled, DeviceExpr, SeparableVelocity, LevelSetTerm, AdvectionTerm, CurvatureTerm, NormalMotionTerm,
                  EikonalReinitializationTerm, update_term, compute_cfl, step_plan, TimeIntegrator, ForwardEuler, RK2, RK3,
                  LevelSetEquation, current_state, current_time, integrate, integrate_bang, volume, perimeter, eikonal_reinitialize, extend_along_normals,
                  InterfaceMesh, extract_interface, merge_interfaces, extract_interface_multi, redistance, extend_closest_point,
                  CubicInterpolation, interpolate, LevelSetIntegrals, level_set_integrals, level_set_integrals_multi,
    union, union_, intersect, intersect_, setdiff, setdiff_, complement, complement_,
                  _normalize_bc, _add_boundary_conditions)

__all__ = [n for n in dir() if not n.startswith("__")]
