"""NumPy reference of the network-input encoder (gcb_env_encode / BatchedChessEnv.encode), shared by the host-emulation test
(tests/test_encode_host.py) and the GPU test (tests/test_encode_gpu.py).

The planes come from an oracle env's view() (board, current_player, wk..bq); the repetition count is the number of rows of
the oracle's saved_boards history (every pre-move board of the episode, chess_v2.py:404-407) equal to the current board,
saturated at 2.  The history is read through the gco_env struct layout kept in tests/clone_helpers.py.  Envs with an
external opponent are modelled by tests/external_helpers.py, whose model keeps the same history.
"""
import ctypes as C

import numpy as np

from tests import clone_helpers as ch

N_PLANES = 19


def planes_ref(board, current_player, rights, rep):
    """uint8 [19, 64] of one env: board int8 [64] (wire codes), current_player +1 / -1, rights (wk, wq, bk, bq), rep 0..2"""
    b = np.asarray(board, np.int8).reshape(64)
    p = np.zeros((N_PLANES, 64), np.uint8)
    for k in range(6):  # K Q R B N P = wire codes 1..6
        p[k] = b == k + 1
        p[6 + k] = b == -(k + 1)
    p[12] = current_player < 0
    for k in range(4):
        p[13 + k] = bool(rights[k])
    p[17], p[18] = rep >= 1, rep >= 2
    return p


def rep_count(board, history):
    """occurrences of `board` among the rows of `history` [n, 64], saturated at 2"""
    h = np.asarray(history, np.int8).reshape(-1, 64)
    return min(2, int((h == np.asarray(board, np.int8).reshape(1, 64)).all(1).sum()))


def oracle_history(o):
    """the pre-move boards of the oracle env's episode, int8 [hist_n, 64]"""
    e = ch._raw(o)
    if e.hist_n == 0:
        return np.zeros((0, 64), np.int8)
    return np.frombuffer((C.c_int8 * (64 * e.hist_n)).from_address(e.hist), np.int8).reshape(e.hist_n, 64).copy()


def oracle_reference(oracles):
    """(planes uint8 [N, 19, 64], rep uint8 [N]) of a list of OracleEnv"""
    planes, reps = [], []
    for o in oracles:
        v = o.view()
        r = rep_count(v["board"], oracle_history(o))
        planes.append(planes_ref(v["board"], v["current_player"], [v[k] for k in ("wk", "wq", "bk", "bq")], r))
        reps.append(r)
    return np.stack(planes), np.array(reps, np.uint8)


def model_reference(models):
    """(planes, rep) of a list of external_helpers.ExternalModel: the position export() must show, and the model's history"""
    planes, reps = [], []
    for m in models:
        v = m.view()
        r = rep_count(v["board"], m.hist) if m.hist else 0
        planes.append(planes_ref(v["board"], int(v["info"][0]), v["info"][1:5], r))
        reps.append(r)
    return np.stack(planes), np.array(reps, np.uint8)


def assert_planes(planes, rep, ref_planes, ref_rep, tag=""):
    """byte-for-byte: planes [N, 19, 64] (any dtype holding 0 / 1, compared as uint8 values) and rep [N] against the reference"""
    got = np.asarray(planes).reshape(len(ref_rep), N_PLANES, 64)
    assert got.dtype == np.uint8, got.dtype
    bad = np.nonzero((got != ref_planes).any(2))
    if len(bad[0]):
        e, c = int(bad[0][0]), int(bad[1][0])
        raise AssertionError("%sencode differs at %d (env, plane) pairs; first: env %d plane %d got %s expected %s"
                             % (tag, len(bad[0]), e, c, got[e, c].tolist(), ref_planes[e, c].tolist()))
    bad = np.nonzero(np.asarray(rep) != ref_rep)[0]
    assert len(bad) == 0, "%srepetition count differs at envs %s: got %s expected %s" % (
        tag, bad[:10].tolist(), np.asarray(rep)[bad[:10]].tolist(), ref_rep[bad[:10]].tolist())


def bf16_as_u8(bits):
    """bf16 bit patterns of 0.0 / 1.0 (0x0000 / 0x3F80) -> uint8 0 / 1; any other pattern -> 255"""
    b = np.asarray(bits).view(np.uint16)
    return np.where(b == 0, 0, np.where(b == 0x3F80, 1, 255)).astype(np.uint8)


def f32_as_u8(x):
    """float32 0.0 / 1.0 -> uint8 0 / 1; any other value (-0.0 included) -> 255"""
    u = np.asarray(x, np.float32).view(np.uint32)
    return np.where(u == 0, 0, np.where(u == 0x3F800000, 1, 255)).astype(np.uint8)
