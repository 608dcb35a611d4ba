"""ctypes binding of libastrild_pk.so (C ABI in include/astrild_pk.h).

The library is the product: there is no CPU or PyTorch fallback.  If the shared object is
missing the import of this module raises, loudly.
"""
from __future__ import annotations

import ctypes as ct
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ASTRILD_PK_LIB: path of another build of the same library (kernel A/B measurements)
LIB_PATH = os.environ.get("ASTRILD_PK_LIB") or os.path.join(_HERE, "lib", "libastrild_pk.so")

APK_F32, APK_F64 = 0, 1
APK_AOS, APK_SOA = 0, 1
APK_NGP, APK_CIC, APK_TSC = 1, 2, 3
APK_DEPOSIT_AUTO, APK_DEPOSIT_ATOMIC, APK_DEPOSIT_SORTED = 0, 1, 2

RESAMPLERS = {"nearest": APK_NGP, "ngp": APK_NGP, "nnb": APK_NGP, "cic": APK_CIC, "linear": APK_CIC,
              "tsc": APK_TSC, "quadratic": APK_TSC}
DEPOSIT_METHODS = {"auto": APK_DEPOSIT_AUTO, "atomic": APK_DEPOSIT_ATOMIC, "sorted": APK_DEPOSIT_SORTED}


class AstrildPkError(RuntimeError):
    """A libastrild_pk.so call returned a non-zero status."""


_vp, _i, _i64, _d, _sz = ct.c_void_p, ct.c_int, ct.c_int64, ct.c_double, ct.c_size_t

# name -> argtypes; every function returns int status unless noted
SIGNATURES = {
    "apk_plan_create": [ct.POINTER(_vp), _i, _d, _i, _i, _i],
    "apk_plan_destroy": [_vp],
    "apk_plan_mesh_elems": [_vp, ct.POINTER(_i64)],
    "apk_plan_workspace_bytes": [_vp, _i64, _i, _i, ct.POINTER(_sz)],
    "apk_plan_set_workspace": [_vp, _vp, _sz],
    "apk_plan_ghost_planes": [_vp, ct.POINTER(_i), ct.POINTER(_i)],
    "apk_plan_enable_timing": [_vp, _i],
    "apk_plan_last_deposit_ms": [_vp, ct.POINTER(ct.c_float)],
    "apk_binning_last_ms": [_vp, ct.POINTER(ct.c_float)],
    "apk_deposit": [_vp, _vp, _vp, _vp, _i, _i, _d, _vp, _i, _i64, _i, _d, _i, _i, _vp, _vp],
    "apk_route_particles": [_vp, _vp, _vp, _vp, _i, _i, _d, _vp, _i, _i64, _i, _vp, _i64, _vp, _vp, _vp],
    "apk_mesh_accumulate": [_vp, _vp, _vp, _i64, _vp],
    "apk_slab_transpose_p2p": [_vp, _vp, _vp, _i64, _i, _vp],
    "apk_deposit_interlaced": [_vp, _vp, _vp, _vp, _i, _i, _d, _vp, _i, _i64, _i, _i, _i, _vp, _vp, _vp],
    "apk_mesh_sum": [_vp, _vp, _i, _vp, _vp],
    "apk_padded_mesh_sum": [_vp, _vp, _vp, _vp],
    "apk_load_mesh": [_vp, _vp, _i, _d, _vp, _vp],
    "apk_store_mesh": [_vp, _vp, _d, _vp, _vp],
    "apk_fft_r2c": [_vp, _vp, _vp],
    "apk_fft_r2c_2d": [_vp, _vp, _vp],
    "apk_fft_c2c_1d": [_vp, _vp, _i, _vp],
    "apk_plan_prepare_fft1d": [_vp, _i],
    "apk_plan_prepare_fft2d": [_vp],
    "apk_plan_set_first_mesh_event": [_vp, _vp],
    "apk_binning_create": [ct.POINTER(_vp), _vp, _i, _i, _i] + [_vp] * 5 + [_i] + [_vp] * 6 + [_i, _i],
    "apk_binning_destroy": [_vp],
    "apk_bin_power": [_vp] * 9 + [_vp],
    "apk_kmu_create": [ct.POINTER(_vp), _vp, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, _i, _vp] + [_vp] * 6 + [_i, _i],
    "apk_kmu_destroy": [_vp],
    "apk_kmu_bin": [_vp] * 11,
    "apk_bispec_create": [ct.POINTER(_vp), _vp, _d, _d, _d, _i, _i, _i],
    "apk_bispec_destroy": [_vp],
    "apk_bispec_triples": [_vp, _vp, _i, ct.POINTER(_i)],
    "apk_bispec_scratch_bytes": [_vp, ct.POINTER(_sz)],
    "apk_bispec_count": [_vp, _vp, _sz, _vp, ct.POINTER(_d), _vp],
    "apk_bispec_measure": [_vp, _vp, _vp, _vp, _sz, _vp, _vp],
    "apk_bispec_last_ms": [_vp, ct.POINTER(ct.c_float)],
    "apk_xi_create": [ct.POINTER(_vp), _vp, _d, _d, _d, _i, _vp, _i, _vp, _i, _i],
    "apk_xi_destroy": [_vp],
    "apk_xi_edges": [_vp, _vp, _i, ct.POINTER(_i)],
    "apk_xi_scratch_bytes": [_vp, ct.POINTER(_sz)],
    "apk_xi_grid_scale": [_vp, ct.POINTER(_d)],
    "apk_xi_measure": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp],
    "apk_xi_last_ms": [_vp, ct.POINTER(ct.c_float)],
    "apk_tf_create": [ct.POINTER(_vp), _vp, _i],
    "apk_tf_destroy": [_vp],
    "apk_tf_scratch_bytes": [_vp, _i, ct.POINTER(_sz)],
    "apk_tf_field": [_vp, _vp, _vp, _vp, _i, _i, _d, _vp, _i, _i64, _i, _vp, _sz, _vp, _vp],
    "apk_tf_last_ms": [_vp, ct.POINTER(ct.c_float)],
    "apk_tables_r_axis": [_i, _d, _vp],
    "apk_tables_r_edges": [_i, _d, _d, _d, _d, _vp, _i, ct.POINTER(_i)],
    "apk_assign_grid": [_vp, _vp, _vp, _vp, _i, _vp, _i, _i64, _vp, _vp, _vp, _vp],
    "apk_gather_records": [_vp, _vp, _i64, _vp, _i, _vp],
    "apk_tables_k_axis": [_i, _d, _i, _vp],
    "apk_tables_k_edges": [_i, _d, _d, _d, _d, _vp, _i, ct.POINTER(_i)],
    "apk_tables_hermitian_weights": [_i, _vp],
    "apk_tables_compensation": [_i, _i, _i, _vp],
    "apk_tables_interlace_phase": [_i, _d, _vp],
    "apk_power_scratch_elems": [_vp, _i, _i, ct.POINTER(_i64)],
    "apk_power_from_particles": [_vp, _vp, _vp, _vp, _i, _i, _d, _vp, _i, _i64, _i, _i, _i, _i, _d, _d, _d, _vp, _vp, _vp, _vp,
                                 _i, ct.POINTER(_i), ct.POINTER(_d), _vp],
    "apk_power_from_mesh": [_vp, _vp, _vp, _i, _d, _d, _d, _vp, _vp, _vp, _vp, _i, ct.POINTER(_i), _vp],
}

_lib = None


def load() -> ct.CDLL:
    """Load the shared library once; raise if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AstrildPkError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C astrild_b200/csrc` (there is no CPU fallback)")
        lib = ct.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = ct.c_int
        lib.apk_version.restype = ct.c_int
        lib.apk_version.argtypes = []
        lib.apk_last_error.restype = ct.c_char_p
        lib.apk_last_error.argtypes = []
        _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().apk_last_error()
        raise AstrildPkError(f"{what} failed ({status}): {msg.decode() if msg else 'no message'}")


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)
