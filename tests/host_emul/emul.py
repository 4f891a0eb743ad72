"""ctypes binding of tests/host_emul/host_emul.cpp (TEST INFRASTRUCTURE: the device rules compiled with g++).

Lets `pytest -m "not gpu"` check the bitboard / step logic of gym_chess_b200/csrc/*.cuh against the oracle
without a GPU, and the per-env clone, policy sampling and the network-input encoder (EmulEnv.clone_from, sample_policy,
encode: the logic of gcb_env_clone, gcb_env_sample_policy and gcb_env_encode).  Never imported by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhost_emul.so")
_CSRC = os.path.join(_HERE, "..", "..", "gym_chess_b200", "csrc")
_lib = None
_ENCODE_DTYPES = {np.dtype(np.float32): 0, np.dtype(np.uint16): 1, np.dtype(np.uint8): 2}  # uint16 = bf16 bit patterns


def build(force=False):
    srcs = [os.path.join(_HERE, "host_emul.cpp"), os.path.join(_CSRC, "chess_core.cuh"), os.path.join(_CSRC, "env_core.cuh")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _SO, srcs[0]])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        vp = C.c_void_p
        L.emul_movegen.argtypes = [C.c_int, vp, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp, vp]
        L.emul_next_state.argtypes = [C.c_int] + [vp] * 9
        L.emul_update_state.argtypes = [C.c_int] + [vp] * 4
        L.emul_philox.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.emul_philox.restype = C.c_uint32
        L.emul_nth_target_check.argtypes = [C.c_uint64, C.c_int]
        L.emul_nth_target_check.restype = C.c_long
        L.emul_env_create.argtypes = [C.c_int, C.c_uint32, C.c_uint64] + [C.c_int] * 7 + [vp]
        L.emul_env_create.restype = vp
        L.emul_env_destroy.argtypes = [vp]
        L.emul_env_step.argtypes = [vp, C.c_int] + [vp] * 6
        L.emul_env_export.argtypes = [vp, vp, vp, vp, C.c_int]
        L.emul_env_import.argtypes = [vp] * 6
        L.emul_env_stats.argtypes = [vp, vp]
        L.emul_env_piece_slots.argtypes = [vp]
        L.emul_env_clone.argtypes = [vp] * 3
        L.emul_env_sample_policy.argtypes = [vp, vp, C.c_int, C.c_longlong, C.c_float, vp, vp, vp]
        L.emul_env_encode.argtypes = [vp, vp, C.c_int, vp]
        L.emul_pack_result.argtypes = [C.c_int, C.c_int, C.c_uint32]
        L.emul_pack_result.restype = C.c_uint16
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data


def movegen(boards, players, rights, attack=False, castles_only=False, stride=256):
    boards = np.ascontiguousarray(np.asarray(boards, np.int8).reshape(-1, 64))
    n = len(boards)
    players = np.ascontiguousarray(np.broadcast_to(np.asarray(players, np.int8), (n,)))
    rights = np.ascontiguousarray(np.broadcast_to(np.asarray(rights, np.uint8), (n, 4)))
    out = np.zeros((n, stride), np.uint16)
    cnt = np.zeros(n, np.int32)
    chk = np.zeros(n, np.uint8)
    lib().emul_movegen(n, _p(boards), _p(players), _p(rights), int(attack), int(castles_only), _p(out), stride, _p(cnt), _p(chk))
    return out, cnt, chk


def next_state(boards, players, rights, actions):
    boards = np.ascontiguousarray(np.asarray(boards, np.int8).reshape(-1, 64))
    n = len(boards)
    players = np.ascontiguousarray(np.broadcast_to(np.asarray(players, np.int8), (n,)))
    rights = np.ascontiguousarray(np.broadcast_to(np.asarray(rights, np.uint8), (n, 4)))
    actions = np.ascontiguousarray(np.asarray(actions, np.int32))
    ob, orr, oc = np.zeros((n, 64), np.int8), np.zeros((n, 4), np.uint8), np.zeros((n, 2), np.uint8)
    rew, st = np.zeros(n, np.int32), np.zeros(n, np.int8)
    lib().emul_next_state(n, _p(boards), _p(players), _p(rights), _p(actions), _p(ob), _p(orr), _p(oc), _p(rew), _p(st))
    return ob, orr, oc, rew, st


def update_state(boards, rights):
    boards = np.ascontiguousarray(np.asarray(boards, np.int8).reshape(-1, 64))
    n = len(boards)
    rights = np.ascontiguousarray(np.broadcast_to(np.asarray(rights, np.uint8), (n, 4)))
    orr, oc = np.zeros((n, 4), np.uint8), np.zeros((n, 2), np.uint8)
    lib().emul_update_state(n, _p(boards), _p(rights), _p(orr), _p(oc))
    return orr, oc


class EmulEnv:
    """Host emulation of the batched env with the interface subset the tests need (mirrors BatchedChessEnv)."""

    def __init__(self, num_envs, opponent="none", player_color="WHITE", seed=0, auto_reset=True, env_id_offset=0,
                 legal_stride=144, history_cap=512, moves_max=149, initial_boards=None):
        tb, nt = None, 0
        if initial_boards is not None:
            tb = np.ascontiguousarray(np.asarray(initial_boards, np.int8).reshape(-1, 64))
            nt = len(tb)
        self._tb = tb
        self.N, self.stride = num_envs, legal_stride
        self.opponent, self.player_color, self.history_cap, self.moves_max = opponent, player_color, history_cap, moves_max
        self._h = lib().emul_env_create(num_envs, env_id_offset, seed, {"none": 0, "random": 1, "external": 2}[opponent],
                                        int(player_color == "BLACK"), int(auto_reset), 0, history_cap, moves_max, nt, _p(tb))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().emul_env_destroy(self._h)
            self._h = None

    def _step(self, mode, inp, record=False):
        N = self.N
        r, d, f = np.zeros(N, np.int32), np.zeros(N, np.uint8), np.zeros(N, np.uint8)
        a, b = np.full(N, -1, np.int32), np.full(N, -1, np.int32)
        lib().emul_env_step(self._h, mode, _p(inp), _p(r), _p(d), _p(f), _p(a), _p(b))
        return r, d, f, a, b

    def step(self, actions):
        return self._step(0, np.ascontiguousarray(np.asarray(actions, np.int32)))

    def step_index(self, u32):
        return self._step(1, np.ascontiguousarray(np.asarray(u32, np.uint32)))

    def step_sampled(self):
        return self._step(2, None)

    def bot_ply(self, bot_actions):
        return self._step(4, np.ascontiguousarray(np.asarray(bot_actions, np.int32)))

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(np.asarray(mask, np.uint8))
        lib().emul_env_step(self._h, 3, _p(m), None, None, None, None, None)

    def set_state(self, boards, players, rights, move_count=None, mask=None):
        b = np.ascontiguousarray(np.asarray(boards, np.int8).reshape(self.N, 64))
        p = np.ascontiguousarray(np.asarray(players, np.int8).reshape(self.N))
        r = np.ascontiguousarray(np.asarray(rights, np.uint8).reshape(self.N, 4))
        mc = None if move_count is None else np.ascontiguousarray(np.asarray(move_count, np.int32))
        m = None if mask is None else np.ascontiguousarray(np.asarray(mask, np.uint8))
        lib().emul_env_import(self._h, _p(b), _p(p), _p(r), _p(mc), _p(m))

    def export(self):
        boards = np.zeros((self.N, 64), np.int8)
        info = np.zeros((self.N, 16), np.int32)
        legal = np.zeros((self.N, self.stride), np.uint16)
        lib().emul_env_export(self._h, _p(boards), _p(info), _p(legal), self.stride)
        return boards, info, legal

    def stats(self):
        s = np.zeros(16, np.uint64)
        lib().emul_env_stats(self._h, _p(s))
        return s

    def clone_from(self, source, index):
        """env j becomes env index[j] of `source` for 0 <= index[j] < source.N; index < 0 leaves row j alone"""
        mine, theirs = [(e.history_cap, e.opponent, e.player_color, e.moves_max, lib().emul_env_piece_slots(e._h))
                        for e in (self, source)]
        assert mine == theirs, "configuration mismatch: %r here, %r in the source" % (mine, theirs)
        idx = np.ascontiguousarray(np.asarray(index, np.int32).reshape(self.N))
        lib().emul_env_clone(self._h, source._h, idx.ctypes.data)

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

    def encode(self, dtype=np.uint8):
        """-> (planes [N, 19, 64] of dtype float32, uint16 (bf16 bit patterns) or uint8, rep uint8 [N])"""
        planes = np.full((self.N, 19, 64), 7, dtype)  # (a value no plane holds: every element must be written)
        rep = np.full(self.N, 0xEE, np.uint8)
        lib().emul_env_encode(self._h, planes.ctypes.data, _ENCODE_DTYPES[np.dtype(dtype)], rep.ctypes.data)
        return planes, rep

    def repetition_count(self):
        rep = np.full(self.N, 0xEE, np.uint8)
        lib().emul_env_encode(self._h, None, 0, rep.ctypes.data)
        return rep
