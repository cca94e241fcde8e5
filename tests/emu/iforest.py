"""ctypes binding of tests/emu/cyg_emu_iforest.cpp: the device detector fit compiled for the host (TEST INFRASTRUCTURE).

Not a product path: cygym_b200 never imports this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from cygym_b200._capi import DET_WORDS

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_SO = os.path.join(_HERE, "_build", "libcyg_emu_iforest.so")
_SRCS = [os.path.join(_HERE, "cyg_emu_iforest.cpp"), os.path.join(_ROOT, "cygym_b200", "csrc", "cyg_iforest.cuh"),
         os.path.join(_ROOT, "cygym_b200", "csrc", "cyg_core.cuh"), os.path.join(_ROOT, "include", "cygym_b200.h")]


def build(force=False):
    if not force and os.path.exists(_SO) and all(os.path.getmtime(_SO) >= os.path.getmtime(s) for s in _SRCS):
        return _SO
    os.makedirs(os.path.dirname(_SO), exist_ok=True)
    subprocess.run(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _SO, _SRCS[0]],
                   check=True, capture_output=True, text=True)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.emu_fit_detector.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        L.emu_np_stream.argtypes = [C.c_uint32, C.c_void_p, C.c_int, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def fit_detector(ring, n_logs, seed):
    """The device fit of one env on the host: hop-log ring (record i at i % len(ring)), n_logs records in all, seed of
    numpy's global stream -> detector slot (uint32[CYG_DET_WORDS])."""
    ring = np.ascontiguousarray(ring, np.uint32)
    slot = np.zeros(DET_WORDS, np.uint32)
    if lib().emu_fit_detector(_p(ring), len(ring), int(n_logs), int(seed) & 0xFFFFFFFF, _p(slot)) != 0:
        raise ValueError("no records, or fewer ring records than the fit reads")
    return slot


def np_stream(seed, ops):
    """numpy's legacy RandomState(seed) as the device restates it.  ops: list of ("uniform", None), ("bounded", r) (an
    integer in [0, r], i.e. randint(0, r + 1)) or ("permutation", n) -> float64 array of all outputs in order."""
    kinds = {"uniform": 0, "bounded": 1, "permutation": 2}
    a = np.array([(kinds[k], 0 if v is None else int(v)) for k, v in ops], np.int64).reshape(-1, 2)
    out = np.zeros(sum(int(v) if k == "permutation" else 1 for k, v in ops), np.float64)
    n = lib().emu_np_stream(int(seed) & 0xFFFFFFFF, _p(a), len(a), _p(out))
    return out[:n]
