"""ctypes binding of tests/host_emul/policy_emul.cpp (TEST INFRASTRUCTURE): the host emulation of tests/host_emul/emul.py
with policy sampling (`EmulEnv.sample_policy`, the logic of gcb_env_sample_policy / BatchedChessEnv.sample_policy)."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.host_emul import emul

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhost_emul_policy.so")
_lib = None


def build(force=False):
    srcs = [os.path.join(_HERE, "policy_emul.cpp"), os.path.join(_HERE, "host_emul.cpp"),
            os.path.join(emul._CSRC, "chess_core.cuh"), os.path.join(emul._CSRC, "env_core.cuh")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _SO, srcs[0]])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.emul_env_sample_policy.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_void_p, C.c_void_p,
                                             C.c_void_p]
        _lib = L
    return _lib


class EmulEnv(emul.EmulEnv):
    """emul.EmulEnv + sample_policy.  (Both libraries compile the same EmulEnv struct from host_emul.cpp and allocate with the
    C library's malloc, so an env made by one is a valid argument of the other.)"""

    def sample_policy(self, logits, temperature=1.0, u32=None):
        """logits: float32 [N, >= 4101], or uint16 [N, >= 4101] holding bf16 bit patterns (numpy rows may be padded: the row
        stride is taken from the array).  -> (actions int32[N], logp float32[N])"""
        assert logits.ndim == 2 and logits.shape[0] == self.N and logits.shape[1] >= 4101 and logits.strides[1] == logits.itemsize
        dtype = {np.dtype(np.float32): 0, np.dtype(np.uint16): 1}[logits.dtype]
        words = None if u32 is None else np.ascontiguousarray(np.asarray(u32).astype(np.uint32).reshape(self.N))
        act, logp = np.zeros(self.N, np.int32), np.zeros(self.N, np.float32)
        lib().emul_env_sample_policy(self._h, logits.ctypes.data, dtype, logits.strides[0] // logits.itemsize, float(temperature),
                                     None if words is None else words.ctypes.data, act.ctypes.data, logp.ctypes.data)
        return act, logp
