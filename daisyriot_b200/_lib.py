"""ctypes loader for libdaisy_b200.so (the C-ABI of include/daisy_b200.h).

There is no CPU fallback: if the CUDA library is missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("DAISY_B200_LIB") or os.path.join(_HERE, "libdaisy_b200.so")  # override: A/B builds of the library
CSRC = os.path.join(_HERE, "csrc")

HIT_DTYPE = np.dtype([("t", np.float32), ("triangleId", np.int32), ("u", np.float32), ("v", np.float32)])
TRIPL_DTYPE = np.dtype([("m_row", np.int32), ("m_col", np.int32), ("m_value", np.float64)])

FF_DEVICE, FF_HOST = 0, 1


class DaisyError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a into daisyriot_b200/libdaisy_b200.so (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", CSRC, "-j4"], stdout=None if verbose else subprocess.DEVNULL)
    return SO_PATH


# every symbol include/daisy_b200.h declares: (restype, argtypes)
_vp, _i, _i64p, _fp, _ip, _dp = C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)
SYMBOLS = {
    "daisy_last_error": (C.c_char_p, []),
    "daisy_version": (_i, []),
    "daisy_device_count": (_i, []),
    "daisy_ctx_create": (_i, [_fp, _i, _fp, _i, _ip, _i, _i, C.POINTER(_vp)]),
    "daisy_ctx_destroy": (None, [_vp]),
    "daisy_ctx_set_samples": (_i, [_vp, _fp, _i]),
    "daisy_ctx_set_partition": (_i, [_vp, _i, _i]),
    "daisy_ctx_row_range": (_i, [_vp, _ip, _ip, _ip]),
    "daisy_ctx_set_stream": (_i, [_vp, _vp]),
    "daisy_plane_ids": (_i, [_fp, _i, _ip, _i, _ip]),
    "daisy_ctx_face_count": (_i, [_vp]),
    "daisy_face_grid_dump": (_i, [_fp, _i, _ip, _i, _i, _fp, C.POINTER(C.c_int8), _ip, C.c_int64]),
    "daisy_face_grid_stats": (_i, [_fp, _i, _ip, _i, _i, _i64p, _ip, _ip]),
    "daisy_query_closest": (_i, [_vp, _i, _fp, _vp]),
    "daisy_query_closest_device": (_i, [_vp, _i, _vp, _vp]),
    "daisy_trace_screen": (_i, [_vp, _i, _i, _i, _fp, _fp, _fp, _i, _fp, _vp]),
    "daisy_unoccluded_rows": (_i, [_vp, _i, _i, _i, _vp]),
    "daisy_formfactors_build": (_i, [_vp, _i]),
    "daisy_formfactors_ld": (_i, [_vp, _i64p]),
    "daisy_formfactors_read_rows": (_i, [_vp, _i, _i, _fp]),
    "daisy_formfactors_to_csc": (_i, [_vp, _i64p, _fp, _ip, _ip]),
    "daisy_formfactors_write_rows": (_i, [_vp, _i, _i, _fp]),
    "daisy_formfactors_write_csc": (_i, [_vp, C.c_int64, _fp, _ip, _ip]),
    "daisy_formfactors_csc_uploads": (_i, [_vp]),
    "daisy_visibility_masks": (_i, [_vp, _i, _i, _i, C.POINTER(C.c_uint64)]),
    "daisy_formfactors_row_digest": (_i, [_vp, _i, _i, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "daisy_formfactors_stats": (_i, [_vp, _i64p, _i64p, _i64p, _dp, _dp]),
    "daisy_formfactors_alloc": (_i, [_vp]),
    "daisy_formfactors_ipc_handle": (_i, [_vp, _vp]),
    "daisy_formfactors_set_peers": (_i, [_vp, _vp, _i]),
    "daisy_formfactors_pairs_fallback": (C.c_int64, [_vp]),
    "daisy_ctx_update_geometry": (_i, [_vp, _fp, _i, _fp, _i]),
    "daisy_formfactors_update": (_i, [_vp, _i]),
    "daisy_ctx_replace_mesh": (_i, [_vp, _fp, _i, _fp, _i, _ip, _i, _ip]),
    "daisy_formfactors_update_stats": (_i, [_vp, _i64p, _i64p, _i64p, _dp]),
    "daisy_solver_create": (_i, [_vp, _i, _fp, _fp, _i, _ip, C.POINTER(_vp)]),
    "daisy_solver_destroy": (None, [_vp]),
    "daisy_solver_reset": (_i, [_vp]),
    "daisy_solver_step": (_i, [_vp, _dp]),
    "daisy_solver_converge": (_i, [_vp, C.c_double, _i, _i, _ip]),
    "daisy_solver_converge_device": (_i, [_vp, C.c_double, _i, _i, _ip]),
    "daisy_solver_numpasses": (_i, [_vp]),
    "daisy_solver_band_sums": (_i, [_vp, _dp]),
    "daisy_solver_read": (_i, [_vp, _fp, _fp]),
    "daisy_solver_write": (_i, [_vp, _fp, _fp]),
    "daisy_solver_step_local": (_i, [_vp]),
    "daisy_solver_write_partitioned": (_i, [_vp, _fp, _fp]),
    "daisy_solver_write_slices": (_i, [_vp, _fp, _fp]),
    "daisy_solver_launches_per_pass": (_i, [_vp]),
    "daisy_solver_tile_map": (_i, [_vp, _ip, C.POINTER(C.c_uint8), C.c_int64, _i64p, _dp]),
    "daisy_gather_plan_dump": (_i, [C.POINTER(C.c_uint8), _i, _i, _i, _ip, _ip, _ip, _ip, C.c_int64]),
    "daisy_group_create": (_i, [_fp, _i, _fp, _i, _ip, _i, _ip, _i, C.POINTER(_vp)]),
    "daisy_group_destroy": (None, [_vp]),
    "daisy_group_size": (_i, [_vp]),
    "daisy_group_ctx": (_vp, [_vp, _i]),
    "daisy_group_set_samples": (_i, [_vp, _fp, _i]),
    "daisy_group_formfactors_build": (_i, [_vp, _i]),
    "daisy_group_formfactors_read_rows": (_i, [_vp, _i, _i, _fp]),
    "daisy_group_formfactors_write_rows": (_i, [_vp, _i, _i, _fp]),
    "daisy_group_formfactors_to_csc": (_i, [_vp, _i64p, _fp, _ip, _ip]),
    "daisy_group_formfactors_write_csc": (_i, [_vp, C.c_int64, _fp, _ip, _ip]),
    "daisy_group_formfactors_stats": (_i, [_vp, _i64p, _i64p, _dp, _dp]),
    "daisy_group_update_geometry": (_i, [_vp, _fp, _i, _fp, _i]),
    "daisy_group_formfactors_update": (_i, [_vp, _i]),
    "daisy_group_replace_mesh": (_i, [_vp, _fp, _i, _fp, _i, _ip, _i, _ip]),
    "daisy_group_solver_create": (_i, [_vp, _i, _fp, _fp, _i, _ip, C.POINTER(_vp)]),
    "daisy_group_solver_destroy": (None, [_vp]),
    "daisy_group_solver_reset": (_i, [_vp]),
    "daisy_group_solver_step": (_i, [_vp, _dp]),
    "daisy_group_solver_converge": (_i, [_vp, C.c_double, _i, _i, _ip]),
    "daisy_group_solver_converge_device": (_i, [_vp, C.c_double, _i, _i, _ip]),
    "daisy_group_solver_numpasses": (_i, [_vp]),
    "daisy_group_solver_band_sums": (_i, [_vp, _dp]),
    "daisy_group_solver_read": (_i, [_vp, _fp, _fp]),
    "daisy_group_solver_write": (_i, [_vp, _fp, _fp]),
    "daisy_solver_ipc_handles": (_i, [_vp, C.c_char_p]),
    "daisy_solver_set_peers": (_i, [_vp, C.c_char_p, _i]),
    "daisy_solver_step_fused": (_i, [_vp, _dp]),
    "daisy_solver_exchange_info": (_i, [_vp, C.POINTER(_vp), _i64p, _i64p]),
    "daisy_solver_step_finish": (_i, [_vp, _dp]),
    "daisy_solver_last_step_ms": (_i, [_vp, _dp]),
    "daisy_solver_set_chained": (_i, [_vp, _i]),
    "daisy_solver_restart": (_i, [_vp, _fp]),
    "daisy_solver_set_emission": (_i, [_vp, _fp]),
    "daisy_solver_set_materials": (_i, [_vp, _fp, _i, _ip]),
    "daisy_group_solver_restart": (_i, [_vp, _fp]),
    "daisy_group_solver_set_emission": (_i, [_vp, _fp]),
    "daisy_group_solver_set_materials": (_i, [_vp, _fp, _i, _ip]),
}

_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise DaisyError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(there is no CPU fallback for this path)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().daisy_last_error()
        raise DaisyError(f"{what or 'daisy call'} failed ({rc}): {msg.decode() if msg else ''}")


def fptr(a: np.ndarray):
    return a.ctypes.data_as(_fp)


def iptr(a: np.ndarray):
    return a.ctypes.data_as(_ip)
