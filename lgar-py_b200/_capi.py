"""ctypes binding of liblgar_b200.so (C ABI in include/lgar_b200.h).

This is the stub a maintainer of the reference adds to call the B200 path (INTEGRATION.md).
The library is built in-tree by build.py / __graft_entry__.build(); importing it never
touches a GPU, every compute entry point fails loudly without an sm_100 device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LGAR_B200_LIB: developer override used to A/B two builds of the same library on one GPU box
LIB_PATH = os.environ.get("LGAR_B200_LIB") or os.path.join(_HERE, "liblgar_b200.so")

ABI_VERSION = 3
MAX_LAYERS, MAX_FRONTS, MAX_GIUH, NUM_OUTPUTS = 4, 16, 8, 10
MAX_DEPTHS = 8  # sensor depths of the soil-moisture output (lgar_problem.moisture_depths)
OUT_NAMES = ("runoff", "percolation", "AET", "infiltration", "ending_volume", "ponded_water",
             "giuh_runoff", "precip", "PET", "discharge")
STATUS_NAMES = ("OK", "NEG_POW", "NAN", "THETA_ORDER", "BOTTOM_REACHED", "NULL_NEIGHBOUR",
                "FRONT_OVERFLOW", "ITER_CAP", "INDEX_ERROR")
FRONT_OVERFLOW = STATUS_NAMES.index("FRONT_OVERFLOW")
# statuses that are capacity limits of this library rather than states in which the reference raises (its front lists
# are unbounded and its root finders have no iteration cap)
CAPACITY_STATUSES = (FRONT_OVERFLOW, STATUS_NAMES.index("ITER_CAP"))


def status_message(column, status: int, step=None) -> str:
    """Report of a column that ended with a non-zero status (and, if known, the forcing step it crashed at)."""
    at = "" if step is None else f" at forcing step {step}"
    msg = f"LGAR column {column}: status {STATUS_NAMES[status]}{at}"
    if status in CAPACITY_STATUSES:
        return (msg + ": a capacity limit of the CUDA library (16 wetting fronts per column in the differentiable path "
                "/ 1e6 root-finder iterations), not a reference exception; mask the column (the agent's "
                "on_column_error='mask') or rerun it forward-only with max_fronts=32")
    return msg + " (the reference raises here)"
EXPORTS = ("lgar_abi_version", "lgar_device_check", "lgar_last_error_string", "lgar_workspace_bytes",
           "lgar_forward", "lgar_backward", "lgar_backward_ex", "lgar_forward_host", "lgar_measure_fp64_flops")

_dp = C.c_void_p  # device or host pointer, passed as an integer address


class Problem(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_columns", C.c_int32), ("num_layers", C.c_int32),
        ("num_steps", C.c_int32), ("num_subcycles", C.c_int32), ("num_sites", C.c_int32),
        ("nint", C.c_int32), ("num_giuh", C.c_int32), ("max_fronts", C.c_int32),
        ("chunk_steps", C.c_int32), ("resume", C.c_int32), ("use_closed_form_G", C.c_int32),
        ("step_begin", C.c_int32), ("step_end", C.c_int32), ("pipeline_seq", C.c_int32), ("num_depths", C.c_int32),
        ("iter_cap", C.c_int64),
        ("subcycle_length_h", C.c_double), ("wilting_point_psi", C.c_double),
        ("frozen_factor", C.c_double), ("giuh_ordinates", C.c_double * MAX_GIUH),
        ("alpha", _dp), ("n", _dp), ("ksat", _dp), ("theta_r", _dp), ("theta_e", _dp),
        ("thickness", _dp), ("initial_psi", _dp), ("ponded_depth_max", _dp),
        ("forcing", _dp), ("site_index", _dp), ("column_order", _dp),
        ("moisture_depths", C.c_double * MAX_DEPTHS),
    ]


class Outputs(C.Structure):
    _fields_ = [
        ("per_step", _dp), ("per_step_mask", C.c_uint32), ("tile_diag_rows", C.c_int32),
        ("sums", _dp), ("start_volume", _dp), ("status", _dp), ("crash_step", _dp),
        ("num_fronts", _dp), ("fronts", _dp), ("front_layer", _dp), ("front_to_bottom", _dp),
        ("counters", _dp), ("tile_cycles", _dp), ("moisture", _dp), ("layer_water", _dp),
    ]


class Gradients(C.Structure):
    _fields_ = [
        ("grad_per_step", _dp), ("grad_mask", C.c_uint32), ("reduce", C.c_int32), ("grad_sums", _dp),
        ("grad_alpha", _dp), ("grad_n", _dp), ("grad_ksat", _dp), ("partials", _dp), ("tape_overflow", _dp),
        ("counters", _dp), ("grad_ponded_depth_max", _dp), ("grad_moisture", _dp), ("grad_layer_water", _dp),
    ]


class LGARLibraryError(RuntimeError):
    pass


_lib = None


def lib():
    """Load liblgar_b200.so (raises if it has not been built: there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LGARLibraryError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.lgar_abi_version.restype = C.c_int
        L.lgar_device_check.restype = C.c_int
        L.lgar_last_error_string.restype = C.c_char_p
        L.lgar_workspace_bytes.restype = C.c_size_t
        L.lgar_workspace_bytes.argtypes = [C.POINTER(Problem), C.c_int]
        L.lgar_forward.restype = C.c_int
        L.lgar_forward.argtypes = [C.POINTER(Problem), C.POINTER(Outputs), C.c_void_p, C.c_size_t,
                                   C.c_int, C.c_void_p]
        L.lgar_backward.restype = C.c_int
        L.lgar_backward.argtypes = [C.POINTER(Problem), C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.lgar_backward_ex.restype = C.c_int
        L.lgar_backward_ex.argtypes = [C.POINTER(Problem), C.POINTER(Gradients), C.c_void_p, C.c_size_t, C.c_void_p]
        L.lgar_forward_host.restype = C.c_int
        L.lgar_forward_host.argtypes = [C.POINTER(Problem), C.POINTER(Outputs)]
        L.lgar_measure_fp64_flops.restype = C.c_double
        L.lgar_measure_fp64_flops.argtypes = [C.c_int]
        if L.lgar_abi_version() != ABI_VERSION:
            raise LGARLibraryError("liblgar_b200.so ABI version mismatch; rebuild")
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().lgar_last_error_string().decode(errors="replace")
        raise LGARLibraryError(f"{what} failed (code {rc}): {msg}")
