"""ctypes binding of libdiffpose_b200.so (the C ABI declared in include/diffpose_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdiffpose_b200.so")

ENGINE_AUTO, ENGINE_FP32, ENGINE_TCX, ENGINE_TCG = 0, 1, 2, 3
ENGINE_NAMES = {ENGINE_FP32: "fp32", ENGINE_TCX: "tcx", ENGINE_TCG: "tcg"}


class DpStep(ctypes.Structure):
    _fields_ = [("t", ctypes.c_float), ("sqrt_at", ctypes.c_float), ("sqrt_1m_at", ctypes.c_float),
                ("sqrt_an", ctypes.c_float), ("c1", ctypes.c_float), ("c2", ctypes.c_float)]


class DpMmaOp(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint) for n in ("a_off", "a_lbo", "a_sbo", "b_off", "b_lbo", "b_sbo", "idesc", "tmem_col", "accumulate")]


class DpNoiseKey(ctypes.Structure):
    """dp_noise_key: the keyed noise stream of one call (include/diffpose_b200.h)."""
    _fields_ = [("seed", ctypes.c_ulonglong), ("pose_offset", ctypes.c_long), ("step_offset", ctypes.c_int)]


def noise_key(seed, pose_offset=0, step_offset=0):
    """A DpNoiseKey for a Python int seed (taken modulo 2^64, so negative seeds are valid too)."""
    return DpNoiseKey(int(seed) & 0xFFFFFFFFFFFFFFFF, int(pose_offset), int(step_offset))


# name -> (restype, argtypes); kept in one table so tests can check every header symbol is exported
_P, _I, _L = ctypes.c_void_p, ctypes.c_int, ctypes.c_long
SIGNATURES = {
    "dp_create": (_I, [ctypes.POINTER(_P), _I, _I, _I, _I, _I, _I, _I]),
    "dp_param_count": (_L, [_P]),
    "dp_pack": (_I, [_P, _P, _L, _P, _P]),
    "dp_set_engine": (_I, [_P, _I]),
    "dp_get_engine": (_I, [_P]),
    "dp_get_forward_engine": (_I, [_P]),
    "dp_device": (_I, [_P]),
    "dp_lift": (_I, [_P, _P, _P, _P, _L, _P]),
    "dp_forward": (_I, [_P, _P, _P, _P, _P, _L, _P]),
    "dp_sample": (_I, [_P, _P, _I, _P, _L, _I, ctypes.POINTER(DpStep), _I, _P, ctypes.POINTER(DpNoiseKey), _P, _I, _P, _P, _P]),
    "dp_noise_fill": (_I, [ctypes.POINTER(DpNoiseKey), _I, _L, _I, _I, _I, _P, _P]),
    "dp_hstream_create": (_I, [ctypes.POINTER(_P), _P, _L, _I, _I, _I]),
    "dp_hstream_submit": (_I, [_P, _P, _P, _P, _L, ctypes.POINTER(DpStep), _I, _P, ctypes.POINTER(DpNoiseKey), _P, _P, _P,
                               ctypes.POINTER(_I)]),
    "dp_hstream_wait": (_I, [_P, _I]),
    "dp_hstream_destroy": (None, [_P]),
    "dp_metrics": (_I, [_P, _I, _I, _P, _L, _I, _P, _P, _P]),
    "dp_selftest_umma": (_I, [_P, _I, _P, _I, _P, _I, _P]),
    "dp_selftest_umma_ts": (_I, [_P, _I, _P, _I, _I, _P, _I, _P, _I, _P]),
    "dp_selftest_cycles": (_I, [ctypes.POINTER(ctypes.c_longlong)]),
    "dp_set_trace": (_I, [_P, _P, _I]),
    "dp_launch_count": (_L, []),
    "dp_last_launch_info": (_I, [_P, ctypes.POINTER(_L)]),
    "dp_last_error": (ctypes.c_char_p, []),
    "dp_version": (ctypes.c_char_p, []),
    "dp_destroy": (None, [_P]),
}

_lib = None


def load():
    """Load the shared library once; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C diffpose_nw_b200/csrc`). diffpose_nw_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().dp_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (status {rc}): {msg}")


def launch_count():
    return int(load().dp_launch_count())
