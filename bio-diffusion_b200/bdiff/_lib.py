"""ctypes binding of libbdiff_sm100.so (the C ABI in include/bdiff.h).

There is NO fallback: if the shared library is missing or cannot be loaded this module raises, and every
product entry point that needs the GPU raises with it.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbdiff_sm100.so")

MODE_PARITY_FP32 = 0
MODE_TENSOR = 1


class BdiffError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("num_h", C.c_int32), ("num_context", C.c_int32), ("num_layers", C.c_int32),
                ("h_hidden", C.c_int32), ("chi_hidden", C.c_int32), ("e_hidden", C.c_int32),
                ("xi_hidden", C.c_int32), ("mode", C.c_int32)]


# name -> (restype, argtypes): exactly the symbols include/bdiff.h declares
PROTOTYPES = {
    "bdiff_abi_version": (C.c_int32, []),
    "bdiff_create": (C.c_int32, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "bdiff_destroy": (None, [C.c_void_p]),
    "bdiff_last_error": (C.c_char_p, [C.c_void_p]),
    "bdiff_set_weight": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "bdiff_weights_missing": (C.c_int32, [C.c_void_p]),
    "bdiff_prepare": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bdiff_selftest_split": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bdiff_selftest_pair": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bdiff_tc_edge_stream_layout": (C.c_int32, [C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "bdiff_plan_topology": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_int64)]),
    "bdiff_edge_index": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bdiff_denoise_forward": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bdiff_profile_forward": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_float)]),
    "bdiff_debug_tap": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64),
                                    C.POINTER(C.c_int64)]),
    "bdiff_reverse_step": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "bdiff_decode_z0": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    "bdiff_center_noise": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bdiff_check": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bdiff_check_stability": (C.c_int32, [C.c_void_p] * 4 + [C.c_int32, C.c_int32] + [C.c_void_p] * 3 + [C.c_float] * 3 +
                              [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bdiff_bond_orders": (C.c_int32, [C.c_void_p] * 5 + [C.c_int32, C.c_int32] + [C.c_void_p] * 3 + [C.c_float] * 3 +
                          [C.c_int32, C.c_void_p]),
    "bdiff_collate_count": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "bdiff_collate_packed": (C.c_int32, [C.c_void_p] * 6 + [C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 4),
    "bdiff_prepare_context": (C.c_int32, [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_int32, C.c_void_p]),
    "bdiff_optimizer_chunk": (C.c_int32, []),
    "bdiff_optimizer_step": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                         C.c_void_p]),
    "bdiff_param_floats": (C.c_int64, [C.c_void_p]),
    "bdiff_param_layout": (C.c_int32, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bdiff_train_precision": (C.c_int32, [C.c_void_p, C.c_int32]),
    "bdiff_train_variant": (C.c_int32, [C.c_void_p, C.c_int32]),
    "bdiff_train_timing": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_char_p, C.c_int64]),
    "bdiff_train_forward": (C.c_int32, [C.c_void_p] * 7),
    "bdiff_train_backward": (C.c_int32, [C.c_void_p] * 4),
    "bdiff_nan_guard_count": (C.c_int32, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "bdiff_launch_count": (C.c_int64, [C.c_void_p]),
}

_lib = None


def load():
    """Load the shared library (once) and attach prototypes.  Raises BdiffError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BdiffError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C bio-diffusion_b200/csrc`).  There is no CPU / PyTorch fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise BdiffError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError = a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.bdiff_abi_version() != 1:
        raise BdiffError("libbdiff_sm100.so ABI version mismatch")
    _lib = lib
    return lib


def check(handle, rc, what):
    if rc != 0:
        lib = load()
        msg = lib.bdiff_last_error(handle)
        raise BdiffError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")
