"""ctypes binding of libocmps.so (the C ABI declared in include/ocmps.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is present when a
context is created, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libocmps.so")

# every symbol include/ocmps.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "ocmps_last_error", "ocmps_version", "ocmps_launch_count", "ocmps_profile_enable", "ocmps_profile_read",
    "ocmps_ctx_create", "ocmps_ctx_destroy", "ocmps_ctx_synchronize", "ocmps_ctx_trim", "ocmps_timer_start", "ocmps_timer_stop",
    "ocmps_mps_create", "ocmps_mps_destroy", "ocmps_mps_upload", "ocmps_mps_sizes", "ocmps_mps_download",
    "ocmps_mps_bond_dims", "ocmps_mps_copy", "ocmps_mps_position1", "ocmps_mps_norm", "ocmps_overlap", "ocmps_overlap_K",
    "ocmps_stepper_create", "ocmps_stepper_destroy", "ocmps_stepper_set_tstep", "ocmps_stepper_get_tstep",
    "ocmps_step", "ocmps_apply_K", "ocmps_ground_state", "ocmps_ground_state_dmrg", "ocmps_stepper_schedule", "ocmps_stepper_gate",
    "ocmps_store_create", "ocmps_store_destroy", "ocmps_store_get", "ocmps_store_put", "ocmps_store_bond_dims",
    "ocmps_forward_sweep", "ocmps_backward_sweep", "ocmps_sweep_pair", "ocmps_sweep_batch", "ocmps_backward_sweep_divT",
    "ocmps_store_overlaps", "ocmps_store_divT", "ocmps_store_apply_K", "ocmps_hessian_rows", "ocmps_hessian_eval",
    "ocmps_store_site_expectations", "ocmps_store_entanglement_entropy", "ocmps_store_correlations",
    "ocmps_store_energy_moments",
]


class OcmpsError(RuntimeError):
    pass


_lib = None


def load():
    """Load libocmps.so (built by ``make`` / ``__graft_entry__.build()``); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OcmpsError(f"{LIB_PATH} not found: build it with `make` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i, d = C.c_void_p, C.c_int, C.c_double
    pi, pd, pvp = C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_void_p)
    pll = C.POINTER(C.c_longlong)
    sig = {
        "ocmps_last_error": (C.c_char_p, []),
        "ocmps_version": (i, []),
        "ocmps_launch_count": (C.c_longlong, []),
        "ocmps_profile_enable": (i, [i]),
        "ocmps_profile_read": (i, [pd]),
        "ocmps_ctx_create": (i, [i, pvp]),
        "ocmps_ctx_destroy": (i, [vp]),
        "ocmps_ctx_synchronize": (i, [vp]),
        "ocmps_ctx_trim": (i, [vp]),
        "ocmps_timer_start": (i, [vp]),
        "ocmps_timer_stop": (i, [vp, pd]),
        "ocmps_mps_create": (i, [vp, i, i, i, pvp]),
        "ocmps_mps_destroy": (i, [vp]),
        "ocmps_mps_upload": (i, [vp, pi, pi, pd, i, i]),
        "ocmps_mps_sizes": (i, [vp, pll, pll]),
        "ocmps_mps_download": (i, [vp, pi, pi, pd, pi, pi]),
        "ocmps_mps_position1": (i, [vp]),
        "ocmps_mps_bond_dims": (i, [vp, pi]),
        "ocmps_mps_copy": (i, [vp, vp]),
        "ocmps_mps_norm": (i, [vp, pd]),
        "ocmps_overlap": (i, [vp, vp, pd]),
        "ocmps_overlap_K": (i, [vp, vp, pd]),
        "ocmps_stepper_create": (i, [vp, i, i, d, d, d, i, i, i, pvp]),
        "ocmps_stepper_destroy": (i, [vp]),
        "ocmps_stepper_set_tstep": (i, [vp, d]),
        "ocmps_stepper_get_tstep": (d, [vp]),
        "ocmps_step": (i, [vp, vp, d, d, i]),
        "ocmps_apply_K": (i, [vp, vp, vp]),
        "ocmps_stepper_schedule": (i, [vp, pi, i]),
        "ocmps_stepper_gate": (i, [vp, i, pd]),
        "ocmps_store_create": (i, [vp, i, i, i, i, pvp]),
        "ocmps_store_destroy": (i, [vp]),
        "ocmps_store_get": (i, [vp, i, vp]),
        "ocmps_store_put": (i, [vp, i, vp]),
        "ocmps_store_bond_dims": (i, [vp, pi]),
        "ocmps_forward_sweep": (i, [vp, vp, pd, i, vp]),
        "ocmps_backward_sweep": (i, [vp, vp, pd, i, vp]),
        "ocmps_sweep_pair": (i, [vp, vp, vp, pd, i, vp, vp]),
        "ocmps_sweep_batch": (i, [vp, i, pvp, pi, pd, i, pvp]),
        "ocmps_backward_sweep_divT": (i, [vp, vp, pd, i, vp, pd]),
        "ocmps_store_overlaps": (i, [vp, vp, i, pd]),
        "ocmps_store_divT": (i, [vp, vp, i, pd]),
        "ocmps_store_apply_K": (i, [vp, vp, i, vp]),
        "ocmps_hessian_rows": (i, [vp, vp, vp, pd, i, pi, i, i, pd, pd]),
        "ocmps_hessian_eval": (i, [vp, vp, vp, pd, i, vp, vp, vp, pi, i, i, i, i, pd, pd, pd, pd]),
        "ocmps_store_site_expectations": (i, [vp, i, i, pd, i, pd, pd]),
        "ocmps_store_entanglement_entropy": (i, [vp, i, i, pd]),
        "ocmps_store_correlations": (i, [vp, i, pd, i, pi, i, pd]),
        "ocmps_store_energy_moments": (i, [vp, i, i, d, pd, pd, i, pd]),
        "ocmps_ground_state": (i, [vp, i, i, i, d, d, i, d, d, vp, pd, pi]),
        "ocmps_ground_state_dmrg": (i, [vp, i, i, i, d, d, i, d, i, vp, pd, pd]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().ocmps_last_error()
        raise OcmpsError(f"libocmps error {rc}: {msg.decode() if msg else ''}")
