"""ctypes binding of tests/host_emul/encode_emul.cpp (TEST INFRASTRUCTURE): the host emulation of tests/host_emul/emul.py with
the network-input encoder (`EmulEnv.encode`, the logic of gcb_env_encode / BatchedChessEnv.encode) and, through
tests/host_emul/clone_emul.py, the per-env clone."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.host_emul import clone_emul, emul

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhost_emul_encode.so")
_lib = None
_DTYPES = {np.dtype(np.float32): 0, np.dtype(np.uint16): 1, np.dtype(np.uint8): 2}  # uint16 = bf16 bit patterns


def build(force=False):
    srcs = [os.path.join(_HERE, "encode_emul.cpp"), os.path.join(_HERE, "host_emul.cpp"),
            os.path.join(emul._CSRC, "chess_core.cuh"), os.path.join(emul._CSRC, "env_core.cuh")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _SO, srcs[0]])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.emul_env_encode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _lib = L
    return _lib


class EmulEnv(clone_emul.EmulEnv):
    """clone_emul.EmulEnv + encode.  (All emulation libraries compile the same EmulEnv struct from host_emul.cpp and allocate
    with the C library's malloc, so an env made by one is a valid argument of the others.)"""

    def encode(self, dtype=np.uint8):
        """-> (planes [N, 19, 64] of dtype float32, uint16 (bf16 bit patterns) or uint8, rep uint8 [N])"""
        planes = np.full((self.N, 19, 64), 7, dtype)  # (a value no plane holds: every element must be written)
        rep = np.full(self.N, 0xEE, np.uint8)
        lib().emul_env_encode(self._h, planes.ctypes.data, _DTYPES[np.dtype(dtype)], rep.ctypes.data)
        return planes, rep

    def repetition_count(self):
        rep = np.full(self.N, 0xEE, np.uint8)
        lib().emul_env_encode(self._h, None, 0, rep.ctypes.data)
        return rep
