"""ctypes binding of libsphmw.so — the same symbols the Julia shim binds with `ccall`
(sph_mountain_waves_b200/julia/SmoothedParticlesB200.jl, INTEGRATION.md).

There is no CPU fallback: if the library is missing or no CUDA device is present
the calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libsphmw.so"

OK = 0
E_INVALID, E_CUDA, E_UNSUPPORTED_OP, E_UNKNOWN_FIELD, E_CAPACITY, E_STATE, E_IO = -1, -2, -3, -4, -5, -6, -7


class SphmwError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libsphmw error {code}: {msg}")
        self.code = code


class UnsupportedOperator(SphmwError):
    """The closure is not in the device operator menu (there is no CPU fallback)."""


class Config(C.Structure):
    _fields_ = [
        ("box_min", C.c_double * 3),
        ("box_max", C.c_double * 3),
        ("h", C.c_double),
        ("capacity", C.c_int64),
        ("device", C.c_int32),
        ("flags", C.c_int32),
        ("slab_lo", C.c_int64),
        ("slab_hi", C.c_int64),
    ]


class LatticeSetup(C.Structure):
    _fields_ = [
        ("grid", C.c_int32), ("mountain", C.c_int32), ("dr", C.c_double),
        ("dom_min", C.c_double * 3), ("dom_max", C.c_double * 3), ("bc_width", C.c_double),
        ("h_m", C.c_double), ("a", C.c_double), ("U", C.c_double),
        ("type_fluid", C.c_double), ("type_wall", C.c_double), ("type_mountain", C.c_double),
        ("h0", C.c_double),
    ]


_lib = None

_P = C.c_void_p
_SIGS = {
    "sphmw_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "sphmw_destroy": (C.c_int, [_P]),
    "sphmw_last_error": (C.c_char_p, []),
    "sphmw_version": (C.c_char_p, []),
    "sphmw_set_stream": (C.c_int, [_P, C.c_void_p]),
    "sphmw_sync": (C.c_int, [_P]),
    "sphmw_set_flags": (C.c_int, [_P, C.c_int32]),
    "sphmw_set_param": (C.c_int, [_P, C.c_char_p, C.c_double]),
    "sphmw_get_param": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_double)]),
    "sphmw_key_tables": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "sphmw_resize": (C.c_int, [_P, C.c_int64]),
    "sphmw_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_upload": (C.c_int, [_P, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]),
    "sphmw_download": (C.c_int, [_P, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]),
    "sphmw_create_cell_list": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_apply": (C.c_int, [_P, C.c_char_p, C.c_int32]),
    "sphmw_op_list": (C.c_int64, [C.c_char_p, C.c_int64]),
    "sphmw_step": (C.c_int, [_P, C.c_char_p, C.c_int32]),
    "sphmw_generate_mountain_wave": (C.c_int, [_P, C.POINTER(LatticeSetup), C.POINTER(C.c_int64),
                                               C.POINTER(C.c_int64)]),
    "sphmw_flow_add_new_particles": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_aflow_add_new_particles": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_cell_keys": (C.c_int, [_P, C.c_void_p, C.c_int64]),
    "sphmw_cell_entries": (C.c_int, [_P, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "sphmw_pairs_dump": (C.c_int, [_P, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "sphmw_count_pairs": (C.c_int, [_P, C.c_int32]),
    "sphmw_pair_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_pretest_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_int32, C.c_void_p]),
    "sphmw_swap_removal_moves": (C.c_int, [C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "sphmw_pretest_pairs_q6": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_int32, C.c_void_p]),
    "sphmw_slab_column_sets": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "sphmw_pair_list_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_tile_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_timing_filter": (C.c_int, [_P, C.c_char_p]),
    "sphmw_frame_capture": (C.c_int, [_P, C.POINTER(C.c_char_p), C.c_int32, C.POINTER(C.c_int32)]),
    "sphmw_frame_wait": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_void_p), C.c_int32, C.POINTER(C.c_int64)]),
    "sphmw_upload_async": (C.c_int, [_P, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]),
    "sphmw_upload_commit": (C.c_int, [_P]),
    "sphmw_upload_index_async": (C.c_int, [_P, C.c_void_p, C.c_int64]),
    "sphmw_comm_unique_id": (C.c_int, [C.c_void_p]),
    "sphmw_comm_init": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_char_p, C.c_int64]),
    "sphmw_comm_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_comm_open_box": (C.c_int, [_P, C.c_int32]),
    "sphmw_reduce": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_double)]),
    "sphmw_kernel_eval": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]),
    "sphmw_pvd_open": (C.c_int, [_P, C.c_char_p]),
    "sphmw_pvd_save_frame": (C.c_int, [_P, C.POINTER(C.c_char_p), C.c_int32]),
    "sphmw_pvd_close": (C.c_int, [_P]),
    "sphmw_vtp_open": (C.c_int, [C.c_char_p, C.POINTER(_P)]),
    "sphmw_vtp_close": (C.c_int, [_P]),
    "sphmw_vtp_info": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "sphmw_vtp_array": (C.c_int, [_P, C.c_int32, C.c_char_p, C.c_int64, C.POINTER(C.c_int32)]),
    "sphmw_vtp_read": (C.c_int, [_P, C.c_char_p, C.c_void_p, C.c_int64]),
    "sphmw_vtp_write": (C.c_int, [C.c_char_p, C.c_int64, C.c_void_p, C.c_int32, C.POINTER(C.c_char_p),
                                  C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]),
    "sphmw_timing_enable": (C.c_int, [_P, C.c_int32]),
    "sphmw_timing_reset": (C.c_int, [_P]),
    "sphmw_timing_report": (C.c_int64, [_P, C.c_char_p, C.c_int64, C.POINTER(C.c_double),
                                        C.POINTER(C.c_int64), C.c_int32]),
    "sphmw_launch_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sphmw_step_phase": (C.c_int, [_P, C.c_char_p, C.c_int32]),
    "sphmw_halo_record_doubles": (C.c_int, []),
    "sphmw_halo_record_width": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "sphmw_halo_pack": (C.c_int, [_P, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "sphmw_halo_pack_begin": (C.c_int, [_P, C.c_void_p, C.c_void_p, C.c_int64]),
    "sphmw_halo_pack_finish": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int64)]),
    "sphmw_halo_pack_wait": (C.c_int, [_P, C.c_void_p]),
    "sphmw_halo_unpack": (C.c_int, [_P, C.c_void_p, C.c_int64, C.c_int64]),
    "sphmw_slab_counts": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "sphmw_set_index": (C.c_int, [_P, C.c_void_p, C.c_int64]),
    "sphmw_download_index": (C.c_int, [_P, C.c_void_p, C.c_void_p, C.c_int64]),
    "sphmw_download_raw": (C.c_int, [_P, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]),
}


def lib() -> C.CDLL:
    """Load libsphmw.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m sph_mountain_waves_b200.build` "
                "(needs nvcc).  There is no CPU fallback.")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def exported_symbols():
    return sorted(_SIGS)


def check(rc: int) -> int:
    if rc < 0:
        msg = lib().sphmw_last_error().decode("utf-8", "replace")
        if rc == E_UNSUPPORTED_OP:
            raise UnsupportedOperator(rc, msg)
        raise SphmwError(rc, msg)
    return rc


def as_f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
