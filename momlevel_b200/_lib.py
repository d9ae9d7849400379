"""ctypes binding of libmomlevel_b200.so (the C ABI declared in include/momlevel_b200.h).

There is no CPU implementation behind this module: if the CUDA library cannot be loaded
the import of any compute entry point raises, it never falls back.
"""

import ctypes
import os
import pathlib

from . import _build

__all__ = ["lib", "check", "MLError", "F32", "F64", "EOS_IDS", "FUNC_IDS", "P_SCALAR", "P_PER_LEVEL", "P_FULL",
           "PATH_DIRECT", "PATH_TMA", "MAX_LAYERS", "MAX_REGIONS",
           "EXPORTS"]

F32, F64 = 0, 1
EOS_IDS = {"wright": 0, "linear": 1}
FUNC_IDS = {"density": 0, "drho_dtemp": 1, "drho_dsal": 2, "alpha": 3, "beta": 4}
P_SCALAR, P_PER_LEVEL, P_FULL = 0, 1, 2
DOMAIN_LOCAL, DOMAIN_GLOBAL = 0, 1
PATH_DIRECT, PATH_TMA = 1, 2
MAX_LAYERS = 8  # ML_MAX_LAYERS
MAX_REGIONS = 15  # ML_MAX_REGIONS

_vp, _i, _i64, _d, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol include/momlevel_b200.h declares
EXPORTS = {
    "ml_version": (_i, []),
    "ml_last_error": (ctypes.c_char_p, []),
    "ml_last_path": (_i, []),
    "ml_launch_count": (_i64, []),
    "ml_set_force_direct": (_i, [_i]),
    "ml_set_variants_chunk": (_i, [_i]),
    "ml_set_column_pressure": (_i, [_vp, _i64]),
    "ml_eos_eval": (_i, [_i, _i, _i, _vp, _vp, _i, _i, _vp, _i, _i64, _i64, _i64, _vp, _vp]),
    "ml_flament_spice": (_i, [_i, _vp, _vp, _i64, _vp, _vp]),
    "ml_calc_dz": (_i, [_vp, _vp, _d, _d, _i, _i, _i64, _i64, _vp, _vp]),
    "ml_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ml_reference_state": (_i, [_i, _i, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ml_steric_local": (_i, [_i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _d, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ml_steric_local_layers": (_i, [_i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _d, _vp, _i, _i64, _i64, _i64, _vp,
                                    _vp]),
    "ml_steric_local_layers_variants": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _d, _vp, _i, _i64,
                                             _i64, _i64, _vp, _vp, _vp, _vp]),
    "ml_profile_workspace_bytes": (_sz, [_i, _i64, _i64, _i64]),
    "ml_steric_local_profile": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _d, _i64, _i64, _i64,
                                     _vp, _vp, _vp, _vp, _sz, _vp]),
    "ml_region_profile_workspace_bytes": (_sz, [_i, _i, _i64, _i64, _i64]),
    "ml_steric_local_region_profile": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _d, _i64,
                                            _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ml_zonal_profile_workspace_bytes": (_sz, [_i, _i64, _i64, _i64, _i64]),
    "ml_steric_local_zonal_profile": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _d, _i64, _i64,
                                           _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ml_delta_rho": (_i, [_i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _i64, _i64, _i64, _vp, _vp]),
    "ml_delta_rho_annual": (_i, [_i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "ml_steric_local_selfref": (_i, [_i, _i, _vp, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _d, _i64, _i64, _i64, _vp, _vp, _vp,
                                     _vp, _sz, _vp]),
    "ml_steric_local_variants": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _d, _i64, _i64, _i64, _vp, _vp,
                                      _vp, _vp, _vp, _vp, _sz, _vp]),
    "ml_calc_masso": (_i, [_i, _vp, _i, _vp, _i64, _i64, _vp, _vp, _sz, _vp]),
    "ml_mean_state_bytes": (_sz, [_i64, _i64]),
    "ml_mean_state_accumulate": (_i, [_i, _vp, _vp, _vp, _i, _vp, _i64, _i64, _i64, _vp, _sz, _i, _vp, _vp, _vp, _vp]),
    "ml_steric_global": (_i, [_i, _i, _vp, _vp, _i, _i, _vp, _i, _vp, _i64, _i64, _i64, _vp, _vp, _sz, _vp]),
    "ml_steric_global_variants": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp,
                                       _sz, _vp]),
    "ml_host_stream_begin": (_i, [_i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i64, _i64, _i64, _i,
                                  ctypes.POINTER(ctypes.c_void_p)]),
    "ml_host_stream_push": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "ml_host_stream_finish": (_i, [_vp, _vp, _vp]),
    "ml_host_stream_abort": (_i, [_vp]),
    "ml_host_release": (_i, []),
    "ml_host_set_packing": (_i, [_i, _i]),
    "ml_host_last_packed_fraction": (_d, []),
    "ml_host_last_pack_threads": (_i, []),
    "ml_host_last_h2d_bytes": (ctypes.c_uint64, []),
    "ml_host_last_timings": (_i, [_vp]),
    "ml_host_tuner_share_selftest": (_i, [ctypes.c_char_p, _i, _i, _i64, _i64, _vp, _vp, _i]),
    "ml_pack_index_rows": (ctypes.c_uint64, [_vp, _i64, _i64, _vp, _vp, _vp]),
    "ml_pack_rows": (None, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "ml_pack_rows_cached": (None, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "ml_pack_simd": (_i, []),
    "ml_calc_n2": (_i, [_i, _i, _vp, _vp, _vp, _d, _d, _i, _i, _i64, _i64, _i64, _vp, _vp]),
    "ml_adjust_negative_n2": (_i, [_vp, _i, _i64, _i64, _i64, _vp, _vp]),
    "ml_stability_angle": (_i, [_i, _i, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "ml_wave_speed": (_i, [_vp, _vp, _i, _i64, _i64, _i64, _vp, _vp]),
    "ml_steric_global_host": (_i, [_i, _i, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i, _vp]),
    "ml_steric_local_variants_host": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i64, _i64, _i64, _i, _vp, _vp, _vp, _vp,
                                           _vp]),
    "ml_steric_local_host": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i64, _i64, _i64, _i, _vp, _vp, _vp]),
}


class MLError(RuntimeError):
    """Non-zero return from libmomlevel_b200 (negative: argument error, positive: cudaError_t)."""

    def __init__(self, code, message):
        super().__init__(f"libmomlevel_b200 error {code}: {message}")
        self.code = code


_LIB = None


def library_path():
    return pathlib.Path(os.environ.get("MOMLEVEL_B200_LIB", str(_build.LIB)))


def lib():
    """Load (building first if the sources are newer and nvcc is present) and return the CDLL."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if "MOMLEVEL_B200_LIB" not in os.environ:
        try:
            _build.build()
        except RuntimeError:
            if not path.exists():
                raise
    if not path.exists():
        raise MLError(-8, f"{path} is missing: run `python -m momlevel_b200._build`; there is no CPU fallback")
    handle = ctypes.CDLL(str(path))
    for name, (res, args) in EXPORTS.items():
        fn = getattr(handle, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if handle.ml_version() != 1:
        raise MLError(-8, f"ABI version {handle.ml_version()} != 1")
    _LIB = handle
    return handle


def check(code):
    if code != 0:
        raise MLError(code, lib().ml_last_error().decode("utf-8", "replace"))
