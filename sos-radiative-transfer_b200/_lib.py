"""ctypes binding of libsos_b200.so (the C ABI declared in include/sos_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, the
package raises.  Build the library with `python -c "import __graft_entry__ as g; g.build()"`
(or `make -C sos-radiative-transfer_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SOS_B200_LIB") or os.path.join(_HERE, "libsos_b200.so")   # (SOS_B200_LIB: an experimental build of the same ABI)


class SosError(RuntimeError):
    pass


class SosRetry(SosError):
    """sos_solve returned SOS_ERR_RETRY: the plan left its fused order kernel; restore the inputs and solve again."""


class sos_grid(C.Structure):
    _fields_ = [
        ("nb_layers", C.c_int),
        ("nb_angles", C.c_int),
        ("n_scenarios", C.c_int),
        ("n_regions", C.c_int),
        ("region_start", C.c_int * 4),
        ("surface", C.c_int),
        ("ld", C.c_int),
        ("chunk_rows", C.c_int),
    ]


class sos_scenario(C.Structure):
    _fields_ = [
        ("mu0", C.c_double),
        ("grd_alb", C.c_double),
        ("tauStar_tot", C.c_double),
        ("coef_atm", C.c_double),
        ("coef_mix_atm", C.c_double),
        ("coef_mix_aer", C.c_double),
        ("threshold", C.c_double),
        ("phase_atm", C.c_int),
        ("phase_aer", C.c_int),
        ("extrap_width", C.c_int * 3),
        ("order_cap", C.c_int),
    ]


# the same 80 bytes as a NumPy record: whole batches are marshalled without a Python loop (engine.scenario_table)
SCENARIO_DTYPE = np.dtype([("mu0", "f8"), ("grd_alb", "f8"), ("tauStar_tot", "f8"), ("coef_atm", "f8"), ("coef_mix_atm", "f8"),
                           ("coef_mix_aer", "f8"), ("threshold", "f8"), ("phase_atm", "i4"), ("phase_aer", "i4"),
                           ("extrap_width", "i4", 3), ("order_cap", "i4")])
assert SCENARIO_DTYPE.itemsize == C.sizeof(sos_scenario)


# one entry of sos_single_scatter_correction (sos_ss_entry): 104 bytes, marshalled as a NumPy record array
SS_ENTRY_DTYPE = np.dtype([("scenario", "i4"), ("geo", "i4"), ("family", "i4", 2), ("series", "i4", 2), ("tab_off", "i4", 2),
                           ("tab_n", "i4", 2), ("g", "f8", 2), ("norm", "f8", 2), ("w", "f8", 4)])
assert SS_ENTRY_DTYPE.itemsize == 104


class sos_result(C.Structure):
    _fields_ = [
        ("ratio_toa", C.c_double),
        ("ratio_surf", C.c_double),
        ("n_orders", C.c_int),
        ("active", C.c_int),
        ("status", C.c_uint),
        ("reserved", C.c_int),
    ]


SURFACE_NONE, SURFACE_SPECULAR, SURFACE_LAMBERT, SURFACE_LAMBERT_README, SURFACE_LAMBERT_DIFFUSE = 0, 1, 2, 3, 4
SURFACE_ROSSLI, SURFACE_OCEAN = 5, 6
QUERY_FUSED_ORDER, QUERY_GENERATED_SOURCE, QUERY_FOLDED, QUERY_DEVICE = 0, 1, 2, 3
STATUS_BLEND_OVERRUN, STATUS_NONFINITE, STATUS_MAX_ORDERS = 1, 2, 4

_dp = C.POINTER(C.c_double)
_vp = C.c_void_p

# name -> (restype, argtypes); must list every symbol of include/sos_b200.h
SIGNATURES = {
    "sos_abi_version": (C.c_int, []),
    "sos_strerror": (C.c_char_p, [C.c_int]),
    "sos_last_cuda_error": (C.c_char_p, []),
    "sos_plan_create": (C.c_int, [C.POINTER(_vp), C.POINTER(sos_grid), _vp, _vp, C.POINTER(sos_scenario), _vp, C.c_int]),
    "sos_plan_destroy": (C.c_int, [_vp]),
    "sos_plan_update": (C.c_int, [_vp, _vp, C.POINTER(sos_scenario), _vp]),
    "sos_extrap_layout": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sos_build_contraction": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    "sos_build_phase": (C.c_int, [_vp, C.c_int, C.c_double, C.c_double, _vp, _vp, _vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp]),
    "sos_build_phase_modes": (C.c_int, [_vp, C.c_int, C.c_double, C.c_double, C.c_int, _vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp,
                                        C.c_int, C.c_size_t, _vp, _vp]),
    "sos_build_brdf_modes": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp, C.c_int, C.c_size_t, _vp]),
    "sos_plan_set_brdf": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.c_int, C.c_int]),
    "sos_plan_set_brdf_scenarios": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "sos_build_glint_modes": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_double, C.c_double, _vp, C.c_int, C.c_size_t, _vp]),
    "sos_glint_correction": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp]),
    "sos_single_scatter_correction": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, C.c_int,
                                                C.c_int, _vp, _vp]),
    "sos_azimuth_synthesis": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp]),
    "sos_plan_set_phase": (C.c_int, [_vp, C.POINTER(_vp), C.c_int, C.c_int]),
    "sos_fold_layout": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sos_build_folded": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.POINTER(C.c_double), _vp]),
    "sos_plan_set_folded": (C.c_int, [_vp, C.POINTER(_vp), C.c_int, C.c_int]),
    "sos_plan_set_lowrank": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int), C.c_int, C.c_int]),
    "sos_lowrank_layout": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sos_build_lowrank_mu2": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int), _vp]),
    "sos_first_order": (C.c_int, [_vp, _vp, _vp, _vp]),
    "sos_first_order2": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "sos_first_order_tab": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "sos_source": (C.c_int, [_vp, _vp, _vp, _vp]),
    "sos_source_rows": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    "sos_source_peers": (C.c_int, [_vp, C.POINTER(_vp), C.c_int, C.POINTER(C.c_int), _vp, _vp]),
    "sos_ipc_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp), C.c_char_p]),
    "sos_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(_vp)]),
    "sos_ipc_close": (C.c_int, [_vp]),
    "sos_ipc_free": (C.c_int, [_vp]),
    "sos_copy_d2d": (C.c_int, [_vp, _vp, C.c_size_t, _vp]),
    "sos_sweeps": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "sos_converge": (C.c_int, [_vp, C.c_int, _vp]),
    "sos_solve": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.POINTER(sos_result), _vp]),
    "sos_get_results": (C.c_int, [_vp, C.POINTER(sos_result), _vp]),
    "sos_reset": (C.c_int, [_vp, _vp, _vp]),
    "sos_quadratures": (C.c_int, [_vp, _vp, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sos_launch_count": (C.c_longlong, [_vp]),
    "sos_plan_query": (C.c_int, [_vp, C.c_int]),
    "sos_plan_set_columns": (C.c_int, [_vp, C.c_int, C.c_int]),
    "sos_layer_mailbox_bytes": (C.c_int, [_vp, C.POINTER(C.c_size_t)]),
    "sos_plan_set_layers": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sos_state_ratios": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "sos_set_profiling": (C.c_int, [_vp, C.c_int]),
    "sos_get_profile": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_longlong), _vp]),
    "sos_fp64_peak": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
}

_lib = None


def load():
    """Load libsos_b200.so (once) and attach the prototypes.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise SosError(
            f"{LIB_PATH} not found: the CUDA library has not been built "
            "(run __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.sos_abi_version() != 1:
        raise SosError("libsos_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(code: int, what: str = ""):
    if code == 0:
        return
    if code == -6:
        raise SosRetry(f"{what or 'libsos_b200'}: solve must be repeated with the plan's general kernels")
    lib = load()
    msg = lib.sos_strerror(code).decode()
    extra = lib.sos_last_cuda_error().decode()
    raise SosError(f"{what or 'libsos_b200'}: {msg} ({code})" + (f": {extra}" if extra and code == -2 else ""))
