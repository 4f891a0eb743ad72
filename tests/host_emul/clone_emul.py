"""ctypes binding of tests/host_emul/clone_emul.cpp (TEST INFRASTRUCTURE): the host emulation of tests/host_emul/emul.py
with the per-env clone (`EmulEnv.clone_from`, the logic of gcb_env_clone / BatchedChessEnv.clone_from)."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.host_emul import emul

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhost_emul_clone.so")
_lib = None


def build(force=False):
    srcs = [os.path.join(_HERE, "clone_emul.cpp"), os.path.join(_HERE, "host_emul.cpp"),
            os.path.join(emul._CSRC, "chess_core.cuh"), os.path.join(emul._CSRC, "env_core.cuh")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _SO, srcs[0]])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.emul_env_clone.argtypes = [C.c_void_p] * 3
        _lib = L
    return _lib


class EmulEnv(emul.EmulEnv):
    """emul.EmulEnv + clone_from.  (Both libraries compile the same EmulEnv struct from host_emul.cpp and allocate with the C
    library's malloc, so an env made by one is a valid argument of the other.)"""

    def __init__(self, num_envs, **kw):
        super().__init__(num_envs, **kw)
        self.cfg = dict(kw, num_envs=num_envs)

    def clone_from(self, source, index):
        """env j becomes env index[j] of `source` for 0 <= index[j] < source.N; index < 0 leaves row j alone"""
        same = ("history_cap", "opponent", "player_color", "moves_max")
        assert all(self.cfg.get(k) == source.cfg.get(k) for k in same), "configuration mismatch"
        idx = np.ascontiguousarray(np.asarray(index, np.int32).reshape(self.N))
        lib().emul_env_clone(self._h, source._h, idx.ctypes.data)
