"""ctypes binding of the C ABI declared in ``include/tssplat_b200.h``.

There is no CPU fallback: if ``libtssplat_b200.so`` is missing or does not load, importing the
product modules raises.  Build it with ``python -m tssplat_b200.build`` (needs nvcc, no GPU).
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

# TSSPLAT_B200_LIB: developer override (e.g. the -DTSB_TRACE profiling build of tools/trace_phases.py)
LIB_PATH = os.environ.get("TSSPLAT_B200_LIB") or _build.LIB_PATH

TSB_OK, TSB_E_INVALID, TSB_E_MESH, TSB_E_CUDA, TSB_E_NOMEM = 0, -1, -2, -3, -4

# every symbol include/tssplat_b200.h declares (tests check the library exports each one)
EXPORTED_SYMBOLS = (
    "tsb_create", "tsb_destroy", "tsb_last_error", "tsb_get_info", "tsb_energy_grad", "tsb_energy_grad_ex", "tsb_energy_grad_host", "tsb_scale",
    "tsb_grad_limit", "tsb_adam_uniform_step", "tsb_train_step",
    "tsb_surface_create", "tsb_surface_destroy", "tsb_surface_last_error", "tsb_surface_forward", "tsb_surface_backward",
    "tsb_surface_extract", "tsb_free_host", "tsb_setup_last_error",
)


class tsb_options_t(C.Structure):
    _fields_ = [("warps_per_cta", C.c_int32), ("laplacian_scale", C.c_int32), ("ring_slots", C.c_int32),
                ("force_global", C.c_int32), ("tet_cost_x100", C.c_int32), ("enable_amips", C.c_int32), ("reserved", C.c_int32 * 2)]


class tsb_terms_t(C.Structure):
    _fields_ = [("c1", C.c_float), ("c2", C.c_float), ("order", C.c_int32), ("c3", C.c_float), ("reserved", C.c_int32 * 4)]


class tsb_info_t(C.Structure):
    _fields_ = [
        ("n", C.c_int32), ("nele", C.c_int32), ("n_components", C.c_int32), ("grid", C.c_int32),
        ("warps_per_cta", C.c_int32), ("ctas_per_sm", C.c_int32), ("mode_global", C.c_int32),
        ("smem_bytes", C.c_int32), ("ring_slots", C.c_int32), ("n_segments", C.c_int32),
        ("n_boundary_faces", C.c_int32), ("max_component_vertices", C.c_int32),
        ("nnz", C.c_int64), ("nnz_padded", C.c_int64), ("device_bytes", C.c_int64), ("stream_bytes", C.c_int64),
    ]


class tsb_train_state_t(C.Structure):
    _fields_ = [("g1", C.c_void_p), ("g2", C.c_void_p), ("grad", C.c_void_p), ("energy", C.c_void_p),
                ("schedule", C.c_void_p), ("history", C.c_void_p), ("step", C.c_void_p), ("work", C.c_void_p),
                ("n_steps", C.c_int32), ("beta1", C.c_double), ("beta2", C.c_double)]


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the B200 CUDA library has not been built "
            "(run `python -m tssplat_b200.build`); tssplat_b200 has no CPU fallback")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise ImportError(f"cannot load {LIB_PATH}: {e}; tssplat_b200 has no CPU fallback") from e
    vp, f32, i32, i64 = C.c_void_p, C.c_float, C.c_int32, C.c_int64
    lib.tsb_create.restype = C.c_int
    lib.tsb_create.argtypes = [vp, vp, i32, i32, C.POINTER(tsb_options_t), C.c_int, C.POINTER(vp)]
    lib.tsb_destroy.restype = None
    lib.tsb_destroy.argtypes = [vp]
    lib.tsb_last_error.restype = C.c_char_p
    lib.tsb_last_error.argtypes = [vp]
    lib.tsb_get_info.restype = C.c_int
    lib.tsb_get_info.argtypes = [vp, C.POINTER(tsb_info_t)]
    lib.tsb_energy_grad.restype = C.c_int
    lib.tsb_energy_grad.argtypes = [vp, vp, f32, f32, i32, f32, vp, vp, vp, vp]
    lib.tsb_energy_grad_ex.restype = C.c_int
    lib.tsb_energy_grad_ex.argtypes = [vp, vp, C.POINTER(tsb_terms_t), f32, vp, vp, vp, vp]
    lib.tsb_energy_grad_host.restype = C.c_int
    lib.tsb_energy_grad_host.argtypes = [vp, vp, f32, f32, i32, f32, vp, vp, vp]
    lib.tsb_scale.restype = C.c_int
    lib.tsb_scale.argtypes = [vp, i64, f32, vp, vp, vp]
    lib.tsb_grad_limit.restype = C.c_int
    lib.tsb_grad_limit.argtypes = [vp, i64, f32, f32, vp, vp]
    lib.tsb_adam_uniform_step.restype = C.c_int
    lib.tsb_adam_uniform_step.argtypes = [vp, vp, vp, vp, i64, C.c_double, C.c_double, C.c_double, i32, C.c_double, vp, vp]
    lib.tsb_train_step.restype = C.c_int
    lib.tsb_train_step.argtypes = [vp, vp, vp, f32, f32, i32, C.POINTER(tsb_train_state_t), vp]
    lib.tsb_surface_create.restype = C.c_int
    lib.tsb_surface_create.argtypes = [vp, i32, vp, i32, i32, C.c_int, C.POINTER(vp)]
    lib.tsb_surface_destroy.restype = None
    lib.tsb_surface_destroy.argtypes = [vp]
    lib.tsb_surface_last_error.restype = C.c_char_p
    lib.tsb_surface_last_error.argtypes = [vp]
    lib.tsb_surface_forward.restype = C.c_int
    lib.tsb_surface_forward.argtypes = [vp, vp, vp, vp, vp]
    lib.tsb_surface_backward.restype = C.c_int
    lib.tsb_surface_backward.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.tsb_surface_extract.restype = C.c_int
    lib.tsb_surface_extract.argtypes = [vp, C.c_int32, C.c_int32, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                        C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32))]
    lib.tsb_free_host.restype = None
    lib.tsb_free_host.argtypes = [vp]
    lib.tsb_setup_last_error.restype = C.c_char_p
    lib.tsb_setup_last_error.argtypes = []
    return lib


lib = _load()


def last_error(handle=None) -> str:
    msg = lib.tsb_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, handle=None, what: str = "tssplat_b200") -> None:
    """Non-zero return codes become exceptions, like the reference's throw std::runtime_error
    (``tssplat_ext/tet_spheres/tet_spheres.cpp:152-202``)."""
    if rc == TSB_OK:
        return
    raise RuntimeError(f"{what}: {last_error(handle)} (code {rc})")
