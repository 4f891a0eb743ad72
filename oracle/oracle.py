"""ctypes binding of the CPU ORACLE (oracle/gc_oracle.c).

TEST INFRASTRUCTURE ONLY -- see oracle/gc_oracle.h.  Imported by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs, never by
the product package gym_chess_b200/.

`OracleEngine` mirrors the reference's PyO3 class `ChessEngine`
(/root/reference/src/lib.rs:1412-1512): same 4 methods, same dict/str wire format, so the
reference's own chess_v2.py shell and test-suite can run on top of it unmodified
(tests/golden/make_golden.py).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgc_oracle.so")

WHITE, BLACK = "WHITE", "BLACK"
CASTLE_NAMES = {
    4096: "CASTLE_KING_SIDE_WHITE",
    4097: "CASTLE_QUEEN_SIDE_WHITE",
    4098: "CASTLE_KING_SIDE_BLACK",
    4099: "CASTLE_QUEEN_SIDE_BLACK",
}
CASTLE_CODES = {v: k for k, v in CASTLE_NAMES.items()}
MAX_MOVES = 2048


def build(force=False):
    """Compile oracle/libgc_oracle.so with gcc (oracle/Makefile)."""
    src = os.path.join(_HERE, "gc_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(
        os.path.getmtime(src), os.path.getmtime(os.path.join(_HERE, "gc_oracle.h"))
    ):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return _SO


class _State(C.Structure):
    _fields_ = [
        ("board", C.c_int8 * 64),
        ("current_player", C.c_int8),
        ("white_king_on_board", C.c_uint8),
        ("black_king_on_board", C.c_uint8),
        ("wk", C.c_uint8),
        ("wq", C.c_uint8),
        ("bk", C.c_uint8),
        ("bq", C.c_uint8),
        ("wchk", C.c_uint8),
        ("bchk", C.c_uint8),
    ]


class Stats(C.Structure):
    _fields_ = [
        (k, C.c_uint64)
        for k in ("steps", "plies", "episodes", "mates", "repetitions", "caps", "wedged", "invalid")
    ] + [("reward_sum", C.c_int64), ("legal_sum", C.c_uint64), ("in_check", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        P = C.POINTER
        L.gco_state_new.argtypes = [P(_State), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.gco_get_possible_moves.argtypes = [P(_State), C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.gco_get_castle_moves.argtypes = [P(_State), C.c_int, C.c_void_p, C.c_int]
        L.gco_next_state.argtypes = [P(_State), C.c_int, C.c_int, P(_State), P(C.c_int), P(C.c_int)]
        L.gco_update_state.argtypes = [P(_State)]
        L.gco_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.gco_draw_u32.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.gco_draw_u32.restype = C.c_uint32
        L.gco_env_new.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_uint32]
        L.gco_env_new.restype = C.c_void_p
        L.gco_env_delete.argtypes = [C.c_void_p]
        L.gco_env_reset.argtypes = [C.c_void_p]
        L.gco_env_step.argtypes = [C.c_void_p, C.c_int, P(C.c_int), P(C.c_int)]
        L.gco_env_pick.argtypes = [C.c_void_p, C.c_uint32]
        L.gco_env_view.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gco_env_set_episode.argtypes = [C.c_void_p, C.c_uint32]
        L.gco_env_set_moves_max.argtypes = [C.c_void_p, C.c_int]
        L.gco_env_import.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 6
        L.gco_env_force_bot.argtypes = [C.c_void_p, C.c_int]
        L.gco_selfplay.argtypes = [C.c_void_p, C.c_uint64, P(Stats)]
        L.gco_selfplay_mt.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, P(Stats)]
        L.gco_movegen_batch.argtypes = [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.gco_movegen_batch_mt.argtypes = L.gco_movegen_batch.argtypes + [C.c_int]
        L.gco_next_state_batch.argtypes = [C.c_int] + [C.c_void_p] * 9
        L.gco_update_state_batch.argtypes = [C.c_int] + [C.c_void_p] * 4
        L.gco_harvest.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int] + [C.c_void_p] * 3 + [C.c_int]
        L.gco_default_board.restype = C.POINTER(C.c_int8 * 64)
        _lib = L
    return _lib


def default_board():
    return np.array(lib().gco_default_board().contents, dtype=np.int8).reshape(8, 8)


# ----------------------------------------------------------------------------- codec (host helpers)
def action_to_str(a):
    """action code -> the engine's move string (lib.rs:1278-1290 / CASTLE_* literals)."""
    a = int(a)
    if a >= 4096:
        return CASTLE_NAMES[a]
    f, t = divmod(a, 64)
    return "abcdefgh"[f % 8] + str(8 - f // 8) + "abcdefgh"[t % 8] + str(8 - t // 8)


def str_to_action(m):
    """engine move string -> action code (lib.rs:1311-1373)."""
    if m in CASTLE_CODES:
        return CASTLE_CODES[m]
    f = (8 - int(m[1])) * 8 + "abcdefgh".index(m[0])
    t = (8 - int(m[3])) * 8 + "abcdefgh".index(m[2])
    return f * 64 + t


def _player_int(p):
    # lib.rs:424-441: anything but "BLACK" ends up White (an exception is set but White is used)
    return -1 if p == BLACK else 1


def _mk_state(state, player_field=None):
    b = np.ascontiguousarray(np.asarray(state["board"], dtype=np.int8).reshape(64))
    s = _State()
    lib().gco_state_new(
        C.byref(s),
        b.ctypes.data,
        _player_int(state["current_player"] if player_field is None else player_field),
        int(bool(state["white_king_castle_is_possible"])),
        int(bool(state["white_queen_castle_is_possible"])),
        int(bool(state["black_king_castle_is_possible"])),
        int(bool(state["black_queen_castle_is_possible"])),
    )
    return s


def _state_to_dict(s):
    # State::to_py_object, lib.rs:355-395
    return dict(
        white_king_castle_is_possible=bool(s.wk),
        white_queen_castle_is_possible=bool(s.wq),
        black_king_castle_is_possible=bool(s.bk),
        black_queen_castle_is_possible=bool(s.bq),
        white_king_is_checked=bool(s.wchk),
        black_king_is_checked=bool(s.bchk),
        board=[[int(s.board[r * 8 + c]) for c in range(8)] for r in range(8)],
        current_player=WHITE if s.current_player == 1 else BLACK,
    )


class OracleEngine:
    """Drop-in for `gym_chess.gym_chess.ChessEngine` backed by the C oracle."""

    def next_state(self, state, player, move):
        s = _mk_state(state)
        out = _State()
        rew, both = C.c_int(0), C.c_int(0)
        rc = lib().gco_next_state(C.byref(s), _player_int(player), str_to_action(move), C.byref(out), C.byref(rew), C.byref(both))
        if rc == -1:
            raise RuntimeError("Bad move - piece is empty !")  # reference: Rust panic -> PanicException
        if rc:
            raise ValueError("bad move %r" % (move,))
        return _state_to_dict(out), int(rew.value)

    def get_possible_moves(self, state, player, attack=False):
        s = _mk_state(state)
        buf = (C.c_uint16 * MAX_MOVES)()
        n = lib().gco_get_possible_moves(C.byref(s), _player_int(player), int(bool(attack)), buf, MAX_MOVES)
        return [action_to_str(buf[i]) for i in range(n)]

    def get_castle_moves(self, state, player):
        s = _mk_state(state)
        buf = (C.c_uint16 * 4)()
        n = lib().gco_get_castle_moves(C.byref(s), _player_int(player), buf, 4)
        return [action_to_str(buf[i]) for i in range(n)]

    def update_state(self, state):
        s = _mk_state(state)
        lib().gco_update_state(C.byref(s))
        return _state_to_dict(s)


# ----------------------------------------------------------------------------- env level
class OracleEnv:
    """One env of the C restatement of chess_v2.py:183-294 (step / reset / random bot)."""

    def __init__(self, initial_board=None, player_color=WHITE, opponent="none", seed=0, env_id=0, first_bot_action=-1,
                 moves_max=149):
        ib = None
        if initial_board is not None:
            self._ib = np.ascontiguousarray(np.asarray(initial_board, dtype=np.int8).reshape(64))
            ib = self._ib.ctypes.data
        self._h = lib().gco_env_new(ib, int(player_color == BLACK), {"none": 0, "random": 1}[opponent], seed, env_id)
        if moves_max != 149:
            lib().gco_env_set_moves_max(self._h, int(moves_max))
        if first_bot_action >= 0:  # replay: the reset inside gco_env_new already drew; redo it with the forced move
            lib().gco_env_force_bot(self._h, first_bot_action)
            lib().gco_env_reset(self._h)
            lib().gco_env_force_bot(self._h, -1)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gco_env_delete(self._h)
            self._h = None

    def reset(self, episode=None):
        if episode is not None:
            lib().gco_env_set_episode(self._h, episode)
        lib().gco_env_reset(self._h)

    def import_state(self, board, player, rights, move_count=0, episode=None):
        """new episode from an arbitrary position (board int8[64], player +1/-1, rights (wk, wq, bk, bq))"""
        if episode is not None:
            lib().gco_env_set_episode(self._h, episode)
        b = np.ascontiguousarray(np.asarray(board, np.int8).reshape(64))
        lib().gco_env_import(self._h, b.ctypes.data, int(player), *[int(x) for x in rights], int(move_count))

    def step(self, action, bot_action=-1):
        """-> (reward, done, raised).  bot_action >= 0 forces the bot's reply (replay of a recorded game)."""
        r, d = C.c_int(0), C.c_int(0)
        lib().gco_env_force_bot(self._h, int(bot_action))
        raised = lib().gco_env_step(self._h, int(action), C.byref(r), C.byref(d))
        lib().gco_env_force_bot(self._h, -1)
        return int(r.value), bool(d.value), bool(raised)

    def pick(self, u32):
        return int(lib().gco_env_pick(self._h, int(u32)))

    def view(self):
        board = np.zeros(64, np.int8)
        info = np.zeros(16, np.int32)
        legal = np.zeros(MAX_MOVES, np.uint16)
        lib().gco_env_view(self._h, board.ctypes.data, info.ctypes.data, legal.ctypes.data, MAX_MOVES)
        keys = ("current_player wk wq bk bq wchk bchk done move_count n_legal episode step_in_episode "
                "last_bot_action wedged_bot hist_n").split()
        d = {k: int(info[i]) for i, k in enumerate(keys)}
        d["board"] = board
        d["legal"] = legal[: d["n_legal"]].copy()
        return d

    def selfplay(self, nsteps):
        st = Stats()
        lib().gco_selfplay(self._h, nsteps, C.byref(st))
        return st.as_dict()


def selfplay_mt(seed, env_lo, env_hi, nsteps_per_env, threads):
    st = Stats()
    lib().gco_selfplay_mt(seed, env_lo, env_hi, nsteps_per_env, threads, C.byref(st))
    return st.as_dict()


class SelfplayPool:
    """persistent envs with global ids [env_lo, env_hi) on the host threads: the CPU arm of bench.py (self-play from the
    default board) and, configured like a BatchedChessEnv, the reference of a whole device batch.  Env id g starts from
    initial_boards[g % T] (int8 [T,8,8] / [T,64], None: the default board)."""

    def __init__(self, seed, env_lo, env_hi, *, opponent="none", player_color=WHITE, moves_max=149, initial_boards=None):
        L = lib()
        L.gco_pool_new_cfg.restype = C.c_void_p
        L.gco_pool_new_cfg.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.gco_pool_run.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(Stats)]
        L.gco_pool_free.argtypes = [C.c_void_p]
        L.gco_pool_run_staggered.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(Stats)]
        L.gco_pool_reset.argtypes = [C.c_void_p, C.c_void_p]
        L.gco_pool_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self.n = int(env_hi) - int(env_lo)
        tb, nt = None, 0
        if initial_boards is not None:
            tb = np.ascontiguousarray(np.asarray(initial_boards, dtype=np.int8).reshape(-1, 64))
            nt = len(tb)
        self._h = L.gco_pool_new_cfg(seed, env_lo, env_hi, {"none": 0, "random": 1}[opponent], int(player_color == BLACK),
                                     int(moves_max), nt, None if tb is None else tb.ctypes.data)

    def run(self, nsteps_per_env, threads, stagger=0):
        """every env plays nsteps_per_env more steps (+ env index % stagger with stagger > 0: spreads the episode phases)"""
        st = Stats()
        lib().gco_pool_run_staggered(self._h, nsteps_per_env, stagger, threads, C.byref(st))
        return st.as_dict()

    def reset(self, mask):
        """ChessEnvV2.reset of the envs with mask[i] != 0 (a new episode each, like BatchedChessEnv.reset(mask))"""
        m = np.ascontiguousarray(np.asarray(mask).reshape(self.n) != 0, dtype=np.uint8)
        lib().gco_pool_reset(self._h, m.ctypes.data)

    def export(self, stride=256):
        """-> (boards int8 [n,64], info int32 [n,16], legal uint16 [n,stride]): OracleEnv.view() of every env, info in the
        column order of OracleEnv.view(); the first min(n_legal, stride) entries of a legal row are the list, the rest 0"""
        boards = np.zeros((self.n, 64), np.int8)
        info = np.zeros((self.n, 16), np.int32)
        legal = np.zeros((self.n, stride), np.uint16)
        lib().gco_pool_export(self._h, boards.ctypes.data, info.ctypes.data, legal.ctypes.data, int(stride))
        return boards, info, legal

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gco_pool_free(self._h)
            self._h = None


def harvest(seed, env_lo, env_hi, nsteps, every, threads=1):
    """positions of sampled self-play games of envs [env_lo, env_hi), uniform over the ply index
    -> (boards int8[n,64], players int8[n], rights uint8[n,4]); deterministic (independent of `threads`)"""
    from concurrent.futures import ThreadPoolExecutor

    L = lib()
    per = -(-int(nsteps) // int(every)) + 1

    def run(lo, hi):
        cap = (hi - lo) * per
        b, p, r = np.zeros((cap, 64), np.int8), np.zeros(cap, np.int8), np.zeros((cap, 4), np.uint8)
        n = L.gco_harvest(seed, lo, hi, nsteps, every, b.ctypes.data, p.ctypes.data, r.ctypes.data, cap)
        return b[:n], p[:n], r[:n]

    threads = max(1, min(int(threads), env_hi - env_lo))
    cuts = [env_lo + (env_hi - env_lo) * t // threads for t in range(threads + 1)]
    with ThreadPoolExecutor(threads) as ex:  # ctypes releases the GIL during the call
        parts = list(ex.map(lambda k: run(cuts[k], cuts[k + 1]), range(threads)))
    return tuple(np.concatenate([q[i] for q in parts]) for i in range(3))


def draw_u32(seed, env_id, episode, step, purpose):
    return int(lib().gco_draw_u32(seed, env_id, episode, step, purpose))


def philox4x32_10(ctr, key):
    c = np.asarray(ctr, np.uint32)
    k = np.asarray(key, np.uint32)
    o = np.zeros(4, np.uint32)
    lib().gco_philox4x32_10(c.ctypes.data, k.ctypes.data, o.ctypes.data)
    return o


# ----------------------------------------------------------------------------- batch level
def _prep(boards, players, rights):
    boards = np.ascontiguousarray(np.asarray(boards, np.int8).reshape(-1, 64))
    n = boards.shape[0]
    players = np.ascontiguousarray(np.broadcast_to(np.asarray(players, np.int8), (n,)))
    rights = np.ascontiguousarray(np.broadcast_to(np.asarray(rights, np.uint8), (n, 4)))
    return n, boards, players, rights


def movegen_batch(boards, players, rights, attack=False, stride=256, threads=1):
    """-> (actions uint16[n,stride], counts int32[n]) in reference order."""
    n, boards, players, rights = _prep(boards, players, rights)
    out = np.zeros((n, stride), np.uint16)
    counts = np.zeros(n, np.int32)
    lib().gco_movegen_batch_mt(n, boards.ctypes.data, players.ctypes.data, rights.ctypes.data, int(bool(attack)),
                               out.ctypes.data, stride, counts.ctypes.data, threads)
    return out, counts


def next_state_batch(boards, players, rights, actions):
    n, boards, players, rights = _prep(boards, players, rights)
    actions = np.ascontiguousarray(np.asarray(actions, np.int32))
    ob = np.zeros((n, 64), np.int8)
    orr = np.zeros((n, 4), np.uint8)
    oc = np.zeros((n, 2), np.uint8)
    rew = np.zeros(n, np.int32)
    status = np.zeros(n, np.int8)
    lib().gco_next_state_batch(n, boards.ctypes.data, players.ctypes.data, rights.ctypes.data, actions.ctypes.data,
                               ob.ctypes.data, orr.ctypes.data, oc.ctypes.data, rew.ctypes.data, status.ctypes.data)
    return ob, orr, oc, rew, status


def update_state_batch(boards, rights):
    n, boards, _, rights = _prep(boards, 1, rights)
    orr = np.zeros((n, 4), np.uint8)
    oc = np.zeros((n, 2), np.uint8)
    lib().gco_update_state_batch(n, boards.ctypes.data, rights.ctypes.data, orr.ctypes.data, oc.ctypes.data)
    return orr, oc
