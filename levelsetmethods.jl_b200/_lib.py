"""ctypes binding of ``liblsm_b200.so`` (the C ABI in ``include/lsm_b200.h``).

There is no CPU fallback: if the shared library is missing, importing this module raises, and if
no sm_100 device is present every compute call raises :class:`LSMError` with ``LSM_ERR_CUDA``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("LSM_B200_SO") or os.path.join(_HERE, "liblsm_b200.so")   # override: tuning builds only
CSRC = os.path.join(_HERE, "csrc")

# ---- enums (mirror include/lsm_b200.h) -----------------------------------------------------------
OK, ERR_ARG, ERR_CFL, ERR_TIME, ERR_BC, ERR_CUDA, ERR_NCCL, ERR_OOM, ERR_UNSUPPORTED = range(9)
F32, F64 = 0, 1
BC_NONE, BC_PERIODIC, BC_EXTRAP, BC_SYMMETRY = -1, 0, 1, 2
TERM_ADVECTION, TERM_NORMAL, TERM_CURVATURE, TERM_EIKONAL = 0, 1, 2, 3
UPWIND, WENO5 = 0, 1
COEF_CONST, COEF_FIELD, COEF_SEPARABLE, COEF_NONE, COEF_EXPR = 0, 1, 2, 3, 4
TS_NONE, TS_COS, TS_HOST = 0, 1, 2
SHAPE_SPHERE, SHAPE_BOX, SHAPE_PLANE, SHAPE_CONST = 0, 1, 2, 3
FORWARD_EULER, RK2, RK3 = 0, 1, 2
OPT_KERNEL, OPT_TIME_STAGES, OPT_CFL_CACHE, OPT_OVERLAP, OPT_GRAPH, OPT_CFL_CANDIDATES, OPT_RESIDENT = 0, 1, 2, 3, 5, 6, 7
MAX_TERMS = 4


class lsm_bc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("P", C.c_int32)]


class lsm_term(C.Structure):
    _fields_ = [("kind", C.c_int32), ("scheme", C.c_int32), ("coef_kind", C.c_int32), ("tscale_kind", C.c_int32),
                ("cval", C.c_double * 3), ("tparam", C.c_double), ("field", C.c_void_p)]


class lsm_counters(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("stage_launches", C.c_int64), ("cfl_passes", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("halo_bytes_sent", C.c_int64),
                ("last_stage_ms", C.c_double), ("sum_stage_ms", C.c_double), ("timed_stages", C.c_int64),
                ("pair_launches", C.c_int64), ("resident_steps", C.c_int64)]


class LSMError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[lsm_b200 status {code}] {msg}")
        self.code = code


class CFLError(LSMError, ArithmeticError):
    """ArgumentError of levelsetterms.jl:26."""


class TimeError(LSMError, ValueError):
    """ArgumentError of levelsetequation.jl:196."""


class BCError(LSMError, ValueError):
    """ArgumentError of boundaryconditions.jl:184-186 / levelsetequation.jl:69-70 / meshfield.jl:222-232."""


# every symbol include/lsm_b200.h declares: name -> (restype, argtypes)
_i32, _i64, _dbl, _vp = C.c_int32, C.c_int64, C.c_double, C.c_void_p
_pi32, _pdbl = C.POINTER(C.c_int32), C.POINTER(C.c_double)
SYMBOLS = {
    "lsm_abi_version": (_i32, []),
    "lsm_last_error": (C.c_char_p, []),
    "lsm_device_count": (_i32, [_pi32]),
    "lsm_ctx_create": (_i32, [_i32, C.POINTER(_vp)]),
    "lsm_nccl_unique_id": (_i32, [_vp]),
    "lsm_ctx_create_rank": (_i32, [_i32, _i32, _i32, _vp, C.POINTER(_vp)]),
    "lsm_ctx_create_multi": (_i32, [_i32, _pi32, C.POINTER(_vp)]),
    "lsm_multi_compute_cfl": (_i32, [_i32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.POINTER(lsm_term)), _i32, C.c_double, _pdbl, _pdbl]),
    "lsm_multi_integrate": (_i32, [_i32, C.POINTER(_vp), _i32, C.c_double, C.POINTER(_vp), C.POINTER(C.POINTER(lsm_term)), _i32, C.c_double, C.c_double,
                                   C.c_double, _i64, _pdbl, C.POINTER(_i64)]),
    "lsm_ctx_destroy": (_i32, [_vp]),
    "lsm_sync": (_i32, [_vp]),
    "lsm_set_option": (_i32, [_vp, _i32, _i32]),
    "lsm_get_counters": (_i32, [_vp, C.POINTER(lsm_counters)]),
    "lsm_reset_counters": (_i32, [_vp]),
    "lsm_event_record": (_i32, [_vp, _i32]),
    "lsm_event_elapsed_ms": (_i32, [_vp, _i32, _i32, _pdbl]),
    "lsm_host_register": (_i32, [_vp, _i64]),
    "lsm_host_unregister": (_i32, [_vp]),
    "lsm_slab_plan": (_i32, [_i32, _i32, _i32, _pi32, _pi32]),
    "lsm_step_plan": (_i32, [_dbl, _dbl, _dbl, _dbl, _dbl, _i64, _i32, _pdbl, C.POINTER(C.c_int64), _pi32, C.POINTER(C.c_int64), _pdbl]),
    "lsm_field_create": (_i32, [_vp, _i32, _pi32, _i32, _i32, _pdbl, _pdbl, C.POINTER(_vp)]),
    "lsm_field_create_separable": (_i32, [_vp, _i32, _pi32, _pdbl, _pdbl, _pdbl, _pdbl, C.POINTER(_vp)]),
    "lsm_field_destroy": (_i32, [_vp]),
    "lsm_field_fill_shape": (_i32, [_vp, _i32, _pdbl, _i32]),
    "lsm_field_fill_separable": (_i32, [_vp, _vp]),
    "lsm_expr_check": (_i32, [_i32, _i32, C.POINTER(C.c_char_p)]),
    "lsm_field_set_expr": (_i32, [_vp, C.POINTER(C.c_char_p)]),
    "lsm_field_fill_expr": (_i32, [_vp, _dbl]),
    "lsm_field_set_bc": (_i32, [_vp, C.POINTER(lsm_bc)]),
    "lsm_field_local_extent": (_i32, [_vp, _pi32, _pi32]),
    "lsm_field_upload": (_i32, [_vp, _vp]),
    "lsm_field_download": (_i32, [_vp, _vp]),
    "lsm_field_copy": (_i32, [_vp, _vp]),
    "lsm_field_meshsize": (_i32, [_vp, _pdbl]),
    "lsm_field_getindex": (_i32, [_vp, _pi32, _i32, _pdbl]),
    "lsm_field_stage_buffer": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "lsm_compute_cfl": (_i32, [_vp, _vp, C.POINTER(lsm_term), _i32, _dbl, _pdbl, _pdbl]),
    "lsm_nstages": (_i32, [_i32]),
    "lsm_stage": (_i32, [_vp, _i32, _i32, _vp, C.POINTER(lsm_term), _i32, _dbl, _dbl, _pdbl]),
    "lsm_advance": (_i32, [_vp, _i32, _vp, C.POINTER(lsm_term), _i32, _dbl, _dbl]),
    "lsm_integrate": (_i32, [_vp, _i32, _dbl, _vp, C.POINTER(lsm_term), _i32, _dbl, _dbl, _dbl, _i64, _pdbl,
                             C.POINTER(_i64)]),
    "lsm_eikonal_s0": (_i32, [_vp, _vp]),
    "lsm_volume": (_i32, [_vp, _vp, _pdbl]),
    "lsm_perimeter": (_i32, [_vp, _vp, _pdbl]),
    "lsm_extend_along_normals": (_i32, [_vp, _vp, _vp, _i32, _dbl, _vp, _dbl, _dbl]),
    "lsm_field_csg": (_i32, [_vp, _vp, _vp, _i32]),
    "lsm_interface_extract": (_i32, [_vp, _vp, _dbl, C.POINTER(_i64), C.POINTER(_i64)]),
    "lsm_interface_fetch": (_i32, [_vp, _pdbl, C.POINTER(_i64), _pi32]),
    "lsm_multi_interface_extract": (_i32, [_i32, C.POINTER(_vp), C.POINTER(_vp), _dbl, C.POINTER(_i64), C.POINTER(_i64)]),
    "lsm_redistance": (_i32, [_vp, _vp, _i32, C.POINTER(_i64)]),
    "lsm_extend_closest_point": (_i32, [_vp, _vp, _vp, _i32, _i32, C.POINTER(_i64)]),
    "lsm_interpolate_cubic": (_i32, [_vp, _vp, _i64, _pdbl, _pdbl, _pdbl, _pdbl]),
    "lsm_redistance_cubic": (_i32, [_vp, _vp, _i32, C.POINTER(_i64), C.POINTER(_i64)]),
    "lsm_level_set_integrals": (_i32, [_vp, _vp, _vp, _dbl, _pdbl]),
    "lsm_multi_level_set_integrals": (_i32, [_i32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _dbl, _pdbl]),
    "lsm_max_abs_diff": (_i32, [_vp, _vp, _vp, _pdbl]),
}


def build(force: bool = False) -> str:
    """Compile liblsm_b200.so for sm_100a with the committed Makefile (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", "Makefile"))]
    srcs.append(os.path.join(os.path.dirname(_HERE), "include", "lsm_b200.h"))
    stale = (not os.path.exists(SO_PATH)) or os.path.getmtime(SO_PATH) < max(os.path.getmtime(s) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", CSRC, "-s", f"-j{min(8, os.cpu_count() or 4)}"] + (["-B"] if force else []), check=True)
    return SO_PATH


_lib = None


def lib():
    """The loaded shared library with typed entry points.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `make -C {CSRC}` (or __graft_entry__.build()). "
                "lsm_b200 has no CPU fallback.")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)      # AttributeError if the ABI and the header ever drift apart
            fn.restype, fn.argtypes = res, args
        if L.lsm_abi_version() != 1:
            raise ImportError("liblsm_b200.so ABI version mismatch")
        _lib = L
    return _lib


def last_error() -> str:
    return (lib().lsm_last_error() or b"").decode()


def check(rc: int):
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_CFL:
        raise CFLError(rc, msg)
    if rc == ERR_TIME:
        raise TimeError(rc, msg)
    if rc == ERR_BC:
        raise BCError(rc, msg)
    raise LSMError(rc, msg)
