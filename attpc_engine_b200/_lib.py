"""ctypes binding of ``libattpc_b200.so`` (C ABI: ``include/attpc_b200.h``).

There is no CPU fallback: if the shared library is missing or no CUDA device is usable, the
functions here raise.  Build the library with ``python -c "import __graft_entry__ as g; g.build()"``
(or ``python -m attpc_engine_b200.build``).
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_NAME = "libattpc_b200.so"
LIB_PATH = Path(__file__).resolve().parent / LIB_NAME
ABI_VERSION = 8

# flags (include/attpc_b200.h)
KEEP_ALL_TB = 1 << 0
SPYRAL_ROWS = 1 << 1
NO_WIGGLE = 1 << 2
SKIP_HOST_COPY = 1 << 3
ROWS_KEEP_ALL = 1 << 4
SKIP_CLOUD_COPY = 1 << 5
COLUMNS = 1 << 6
EXACT_MESH = 1 << 7
COLUMNS32 = 1 << 8
SPYRAL_COLUMNS = 1 << 9
COLUMNS_PACKED = 1 << 10


class AttpcConfig(C.Structure):
    _fields_ = [
        ("length", C.c_double),
        ("efield", C.c_double),
        ("bfield", C.c_double),
        ("mpgd_gain", C.c_int64),
        ("diffusion", C.c_double),
        ("fano_factor", C.c_double),
        ("w_value", C.c_double),
        ("gas_density", C.c_double),
        ("micromegas_edge", C.c_int32),
        ("windows_edge", C.c_int32),
        ("adc_threshold", C.c_double),
        ("drift_velocity", C.c_double),
        ("grid_low_mm", C.c_double),
        ("grid_high_mm", C.c_double),
        ("lut_origin_mm", C.c_int32),
        ("lut_n", C.c_int32),
        ("ode_rtol", C.c_double),
        ("ode_atol", C.c_double),
        ("freeze_ke_mev", C.c_double),
        ("max_events_per_launch", C.c_int32),
        ("hash_capacity", C.c_int32),
        ("copy_events_per_launch", C.c_int32),
        ("unit_points", C.c_int32),
        ("table_spill_keys", C.c_int32),
        ("longitudinal_diffusion", C.c_double),
    ]


class AttpcSpecies(C.Structure):
    _fields_ = [
        ("z", C.c_int32),
        ("a", C.c_int32),
        ("mass", C.c_double),
        ("lm", C.c_int32),
        ("e_min", C.c_int32),
        ("n_oct", C.c_int32),
        ("reserved0", C.c_int32),
        ("dedx", C.POINTER(C.c_double)),
    ]


class AttpcReplay(C.Structure):
    _fields_ = [
        ("u_offsets", C.POINTER(C.c_int64)),
        ("u_keys", C.POINTER(C.c_int64)),
        ("u_vals", C.POINTER(C.c_double)),
    ]


class AttpcResult(C.Structure):
    _fields_ = [
        ("n_events", C.c_int64),
        ("n_points", C.c_int64),
        ("offsets", C.POINTER(C.c_int64)),
        ("cloud", C.POINTER(C.c_double)),
        ("labels", C.POINTER(C.c_int64)),
        ("n_rows", C.c_int64),
        ("row_offsets", C.POINTER(C.c_int64)),
        ("rows", C.POINTER(C.c_double)),
        ("row_labels", C.POINTER(C.c_int64)),
        ("offsets_dev", C.c_void_p),
        ("cloud_dev", C.c_void_p),
        ("labels_dev", C.c_void_p),
        ("n_tracks", C.c_int64),
        ("n_trajectory_points", C.c_int64),
        ("n_active_points", C.c_int64),
        ("n_primary_electrons", C.c_int64),
        ("n_deposits", C.c_int64),
        ("n_keys", C.c_int64),
        ("ms_h2d", C.c_float),
        ("ms_tracks", C.c_float),
        ("ms_deposit", C.c_float),
        ("ms_finalize", C.c_float),
        ("ms_d2h", C.c_float),
        ("ms_total", C.c_float),
        ("n_kernel_launches", C.c_int32),
        ("n_retries", C.c_int32),
        ("n_track_launches", C.c_int32),
        ("n_group_launches", C.c_int32),
        ("n_hash_probes", C.c_int64),
        ("hash_capacity", C.c_int32),
        ("reserved1", C.c_int32),
        ("n_table_flushes", C.c_int64),
        ("col_pad", C.POINTER(C.c_int16)),
        ("col_tb_q16", C.POINTER(C.c_uint32)),
        ("col_electrons", C.POINTER(C.c_int64)),
        ("col_label", C.POINTER(C.c_int8)),
        ("n_rk_steps", C.c_int64),
        ("n_rk_rejects", C.c_int64),
        ("max_track_passes", C.c_int64),
        ("col_electrons32", C.POINTER(C.c_uint32)),
        ("n_big", C.c_int64),
        ("big_rows", C.POINTER(C.c_int64)),
        ("big_electrons", C.POINTER(C.c_int64)),
        ("ms_order", C.c_float),
        ("reserved2", C.c_float),
        ("row_col_pad", C.POINTER(C.c_int16)),
        ("row_col_tb_q16", C.POINTER(C.c_uint32)),
        ("row_col_e_lo", C.POINTER(C.c_uint32)),
        ("row_col_e_hi", C.POINTER(C.c_uint16)),
        ("row_col_label", C.POINTER(C.c_int8)),
        ("col_wiggle", C.POINTER(C.c_uint16)),
        ("tb_counts", C.POINTER(C.c_uint16)),
        ("pad_rank_shift", C.c_int32),
        ("reserved3", C.c_int32),
    ]


_P_D = C.POINTER(C.c_double)
_P_I64 = C.POINTER(C.c_int64)
_P_I32 = C.POINTER(C.c_int32)
_P_I16 = C.POINTER(C.c_int16)

# name -> (restype, argtypes); every symbol include/attpc_b200.h declares
SIGNATURES = {
    "attpc_abi_version": (C.c_int, []),
    "attpc_device_count": (C.c_int, []),
    "attpc_create": (
        C.c_int,
        [C.POINTER(AttpcConfig), _P_I16, _P_D, _P_D, C.c_int32, _P_D, C.c_int32, C.POINTER(AttpcSpecies),
         C.c_int32, C.c_int32, C.POINTER(C.c_void_p)],
    ),  # fmt: skip
    "attpc_destroy": (None, [C.c_void_p]),
    "attpc_last_error": (C.c_char_p, [C.c_void_p]),
    "attpc_simulate": (
        C.c_int,
        [C.c_void_p, _P_D, _P_D, C.c_int64, C.c_int32, _P_I32, _P_I32, C.c_int32, C.c_uint64, C.c_int64,
         C.c_uint32, C.POINTER(AttpcResult)],
    ),  # fmt: skip
    "attpc_simulate_dev": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, _P_I32, _P_I32, C.c_int32, C.c_uint64,
         C.c_int64, C.c_uint32, C.POINTER(AttpcResult)],
    ),  # fmt: skip
    "attpc_simulate_replay": (
        C.c_int,
        [C.c_void_p, _P_I64, _P_D, _P_D, _P_I32, _P_I32, _P_I32, _P_I32, C.c_int64, C.c_int64,
         C.POINTER(AttpcReplay), C.c_uint32, _P_I64, C.POINTER(AttpcResult)],
    ),  # fmt: skip
    "attpc_trajectories": (
        C.c_int,
        [C.c_void_p, _P_D, _P_D, _P_I32, C.c_int64, C.c_int32, C.c_int32, _P_D, _P_I32],
    ),
    "attpc_convert_to_spyral": (
        C.c_int,
        [C.c_void_p, _P_I64, _P_D, _P_I64, C.c_int64, C.c_uint32, C.POINTER(AttpcResult)],
    ),
    "attpc_lookup_pads": (C.c_int, [C.c_void_p, _P_D, C.c_int64, _P_I32]),
    "attpc_read_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
}

_lib = None


class AttpcLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once) and declare every prototype.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise AttpcLibraryError(
            f"{LIB_PATH} not found: the CUDA library is not built (run __graft_entry__.build()). "
            "attpc_engine_b200 has no CPU fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.attpc_abi_version() != ABI_VERSION:
        raise AttpcLibraryError(f"{LIB_NAME} has ABI {lib.attpc_abi_version()}, binding expects {ABI_VERSION}")
    _lib = lib
    return lib


def last_error(handle) -> str:
    msg = load().attpc_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(code: int, handle=None) -> None:
    """Map C status codes onto the exceptions the reference raises (ValueError) or RuntimeError."""
    if code == 0:
        return
    msg = last_error(handle)
    if code == -1:
        raise ValueError(msg or "attpc_b200: bad argument")
    if code == -4:
        raise MemoryError(msg or "attpc_b200: out of memory")
    raise RuntimeError(f"attpc_b200 error {code}: {msg}")
