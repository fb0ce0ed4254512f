"""ctypes loader of the CUDA library ``libusim.so`` (C ABI of include/usim.h).

There is no CPU fallback: if the library is missing or cannot be loaded the
import of this module's :func:`lib` raises.
"""
from __future__ import annotations

import ctypes as C
import os

from .abi import UsimConfig, UsimModel

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("USIM_LIB") or os.path.join(_HERE, "libusim.so")  # USIM_LIB: developer override (kernel variants)

_vp = C.c_void_p
_lib = None

# every symbol include/usim.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "usim_create": (C.c_int, [C.POINTER(UsimModel), C.POINTER(UsimConfig), C.c_int, C.POINTER(_vp)]),
    "usim_destroy": (C.c_int, [_vp]),
    "usim_reset": (C.c_int, [_vp, _vp, _vp, _vp]),
    "usim_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "usim_step_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int]),
    "usim_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "usim_get_state": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "usim_set_state": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "usim_get_contacts": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "usim_get_diag": (C.c_int, [_vp, _vp, _vp]),
    "usim_set_contact_record": (C.c_int, [_vp, C.c_int]),
    "usim_get_contact_forces": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "usim_get_arm_record": (C.c_int, [_vp, _vp, _vp]),
    "usim_num_envs": (C.c_int, [_vp]),
    "usim_nq": (C.c_int, [_vp]),
    "usim_nv": (C.c_int, [_vp]),
    "usim_action_dim": (C.c_int, [_vp]),
    "usim_launch_count": (C.c_int64, [_vp]),
    "usim_divergence_count": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "usim_contact_overflow_count": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "usim_substeps": (C.c_int, [_vp]),
    "usim_set_timing": (C.c_int, [_vp, C.c_int]),
    "usim_kernel_time": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "usim_last_error": (C.c_char_p, []),
    "usim_abi_version": (C.c_int, []),
    "usim_sizeof_model": (C.c_size_t, []),
    "usim_sizeof_config": (C.c_size_t, []),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the Ultrasound env step)"
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


class UsimError(RuntimeError):
    pass


def check(rc: int):
    if rc != 0:
        raise UsimError(lib().usim_last_error().decode())
