"""ctypes binding of libiic_b200.so (the C ABI declared in include/iic_b200.h).

There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libiic_b200.so")

ABI_VERSION = 10
FLAG_NAN_LOSS = 1
FLAG_NOT_SIMPLEX = 2
FLAG_BAD_LABEL = 4
FLAG_XCHG_TIMEOUT = 8
ITEM_LOCAL = 0
ITEM_GLOBAL_ROWS = 1
ITEM_GLOBAL_LOGITS = 2
UNSUPPORTED = 3
FLIP_H = 1      # axis 1 of a (C, H, W) sample
FLIP_W = 2      # axis 2

_p = C.c_void_p
_ll = C.c_longlong
_i = C.c_int
_d = C.c_double
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors include/iic_b200.h one to one
PROTOTYPES = {
    "iic_b200_abi_version": (_i, []),
    "iic_b200_last_error": (C.c_char_p, []),
    "iic_b200_sm_count": (_i, [_i]),
    "iic_b200_set_option": (_i, [C.c_char_p, _i]),
    "iic_b200_get_option": (_i, [C.c_char_p]),
    "iic_simplex_check": (_i, [_p, _ll, _i, _ll, _ll, _ll, _p, _p]),
    "iic_local_num_patches": (_i, [_i] * 6),
    "iic_local_joint_workspace_bytes": (_sz, [_i] * 10),
    "iic_local_joint": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll,
                             _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _sz, _p, _p]),
    "iic_local_coeff_floats": (_sz, [_i, _i, _i]),
    "iic_local_epilogue_workspace_bytes": (_sz, [_i, _i, _i]),
    "iic_local_epilogue": (_i, [_p, _i, _i, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p]),
    "iic_local_backward": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll,
                                _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _ll, _ll, _p]),
    "iic_local_joint_from_logits": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i, C.c_float,
                                         _p, _p, _sz, _p, _p]),
    "iic_local_joint_partials": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll,
                                      _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p, _p, _p]),
    "iic_finish_workspace_bytes": (_sz, []),
    "iic_finish": (_i, [_p, _i, _p, _ll, _p, _p, _p, _i, _i, _ll, _i, _p]),
    "iic_local_backward_from_logits": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i, C.c_float,
                                            _p, _p, _p, _p, _p, _ll, _ll, _p]),
    "iic_local_logit_stats_floats": (_sz, [_i, _i, _i]),
    "iic_local_joint_from_logits_workspace_bytes": (_sz, [_i] * 6),
    "iic_local_from_logits_covered": (_i, [_i, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i]),
    "iic_local_joint_from_logits_stats": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i, C.c_float, _p,
                                               _p, _p, _sz, _p, _p]),
    "iic_local_backward_from_logits_stats": (_i, [_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i, C.c_float,
                                                  _p, _p, _p, _p, _p, _p, _ll, _ll, _p]),
    "iic_global_joint_workspace_bytes": (_sz, [_i, _ll, _i]),
    "iic_global_joint": (_i, [_p, _ll, _p, _ll, _ll, _i, _p, _p, _sz, _p, _p]),
    "iic_global_epilogue": (_i, [_p, _i, _d, _i, _p, _p, _p, _p]),
    "iic_global_backward": (_i, [_p, _ll, _p, _ll, _ll, _i, _p, _d, _i, _p, _p, _p, _p, _p, _ll, _ll, _p]),
    "iic_global_backward_from_logits": (_i, [_p, _ll, _p, _ll, _ll, _i, _p, _d, _i, C.c_float, _p, _p, _p, _p, _p, _ll,
                                             _ll, _p]),
    "iic_uda_workspace_bytes": (_sz, [_i]),
    "iic_uda_forward": (_i, [_p, _p, _ll, _i, _ll, _i, _d, _p, _i, _p, _p, _i, _p, _p]),
    "iic_uda_backward": (_i, [_p, _p, _ll, _i, _ll, _i, _d, _p, _i, _p, _p, _p]),
    "iic_sup_workspace_bytes": (_sz, [_i, _ll]),
    "iic_sup_forward": (_i, [_p, _p, _ll, _i, _ll, _d, _p, _p, _p, _p, _p, _p]),
    "iic_sup_backward": (_i, [_p, _p, _ll, _i, _ll, _d, _p, _p, _p, _p]),
    "iic_sup_forward_ignore": (_i, [_p, _p, _ll, _i, _ll, _d, _p, _ll, _p, _p, _p, _p, _p, _p]),
    "iic_sup_backward_ignore": (_i, [_p, _p, _ll, _i, _ll, _d, _p, _ll, _p, _p, _p, _p]),
    "iic_flip_batch": (_i, [_p, _p, _p, _ll, _i, _i, _i, _p]),
    "iic_uda_flip_workspace_bytes": (_sz, [_i, _ll]),
    "iic_uda_flip_forward": (_i, [_p, _p, _p, _ll, _i, _i, _i, _i, _d, _i, _p, _p, _p, _p]),
    "iic_uda_flip_backward": (_i, [_p, _p, _p, _ll, _i, _i, _i, _i, _d, _i, _p, _p, _p]),
    "iic_xchg_buffer_bytes": (_sz, [_i, _ll]),
    "iic_xchg_create": (_i, [_i, _ll, _p]),
    "iic_xchg_export": (_i, [_p, _p]),
    "iic_xchg_import": (_i, [_p, _p]),
    "iic_xchg_release": (_i, [_p, _i]),
    "iic_xchg_allreduce": (_i, [_p, _ll, _ll, _p, _i, _i, _p, _p]),
}



class SlotInfo(C.Structure):
    """iic_slot_info (include/iic_b200.h)."""
    _fields_ = [("layout", _i), ("n_slots", _i), ("slot_stride", _ll), ("nb", _i)]


class FinishItem(C.Structure):
    """iic_finish_item (include/iic_b200.h); field order and types mirror the C struct."""
    _fields_ = [("kind", _i), ("K", _i), ("lamda", _d),
                ("slots", _p), ("layout", _i), ("n_slots", _i), ("nb", _i), ("slot_stride", _ll),
                ("pad", _i), ("n_patches", _i), ("epilogue_workspace", _p),
                ("x", _p), ("x_sn", _ll), ("y", _p), ("y_sn", _ll), ("N", _ll),
                ("symmetric", _i), ("check_simplex", _i),
                ("loss_out", _p), ("Wx", _p), ("Wy", _p), ("P_out", _p), ("inv_temperature", C.c_float)]


_lib = None


class IICLibraryError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises if the CUDA library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IICLibraryError(
            f"{LIB_PATH} is missing. Build it with `python {os.path.join(HERE, 'build.py')}` "
            "(needs nvcc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    got = lib.iic_b200_abi_version()
    if got != ABI_VERSION:
        raise IICLibraryError(f"libiic_b200.so ABI {got} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def set_option(name: str, value: int) -> int:
    """Change a dispatch switch of the library (include/iic_b200.h: iic_b200_set_option); returns the old value."""
    lib = load()
    old = lib.iic_b200_get_option(name.encode())
    check(lib.iic_b200_set_option(name.encode(), int(value)), f"iic_b200_set_option({name})")
    return old


def check(rc: int, what: str):
    if rc != 0:
        msg = load().iic_b200_last_error()
        raise IICLibraryError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
