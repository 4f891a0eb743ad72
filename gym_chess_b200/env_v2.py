"""`ChessEnvV2` -- single-env, gym-style compat class with the reference's surface
(gym_chess/envs/chess_v2.py:132-602): constructor, reset/step/render/render_moves, `state`, `possible_moves`,
`possible_actions`, `info`, flags, codec helpers, `get_possible_moves(state, player, attack)`, `get_castle_moves`.

It is a thin host-side view of a `BatchedChessEnv` with one env: `step()` is one launch of the fused CUDA step
kernel (two when an opponent replies), `get_possible_moves(state=...)` one launch of the batched movegen kernel.
Opponents run on the HOST exactly like the reference's (`opponent(env) -> move`, chess_v2.py:116-127, 171-179): the
device env is created with opponent "external", its step stops where the bot would move, the policy is called with
this object (state after the agent's ply, `possible_moves` = the bot's) and its move is applied without a membership
test (gcb_env_bot_ply) -- for "random" that policy is the reference's `np.random.choice` over `possible_moves` (the
GLOBAL numpy generator, Q18), so a seeded `np.random` replays the same games as the reference.  WHITE and BLACK agents.
gym itself is not needed (and not installed in this image); `observation_space` / `action_space` are minimal stand-ins
with `contains` / `sample`; `highlight` restates gym.utils.colorize (gym/utils/colorize.py of the pinned gym<1).
"""
import sys
from io import StringIO

import numpy as np

from . import codec
from .batched_env import F_BOT_PENDING, F_CAP, F_INVALID, F_REPETITION, BatchedChessEnv
from .codec import (CASTLE_KING_SIDE_BLACK, CASTLE_KING_SIDE_WHITE, CASTLE_MOVES, CASTLE_QUEEN_SIDE_BLACK,
                    CASTLE_QUEEN_SIDE_WHITE, RESIGN)
from .engine import ChessEngine

WHITE, BLACK = "WHITE", "BLACK"
KING_ID, QUEEN_ID, ROOK_ID, BISHOP_ID, KNIGHT_ID, PAWN_ID = 1, 2, 3, 4, 5, 6
DEFAULT_BOARD = [
    [-3, -5, -4, -2, -1, -4, -5, -3],
    [-6] * 8, [0] * 8, [0] * 8, [0] * 8, [0] * 8,
    [6] * 8,
    [3, 5, 4, 2, 1, 4, 5, 3],
]
# chess_v2.py:64-84
ID_TO_ICON = {-6: "♙", -5: "♘", -4: "♗", -3: "♖", -2: "♕", -1: "♔", 0: ".", 1: "♚", 2: "♛", 3: "♜", 4: "♝", 5: "♞", 6: "♟"}
ID_TO_DESC = {-6: "", -5: "N", -4: "B", -3: "R", -2: "Q", -1: "K", 0: "", 1: "K", 2: "Q", 3: "R", 4: "B", 5: "N", 6: ""}


class _Discrete:
    def __init__(self, n):
        self.n = n

    def contains(self, x):
        try:
            return 0 <= int(x) < self.n and int(x) == x
        except (TypeError, ValueError):
            return False

    def sample(self):
        return int(np.random.randint(self.n))


class _Box:
    def __init__(self, low, high, shape):
        self.low, self.high, self.shape = low, high, shape

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == tuple(self.shape) and bool((x >= self.low).all() and (x <= self.high).all())


_COLOR2NUM = dict(gray=30, red=31, green=32, yellow=33, blue=34, magenta=35, cyan=36, white=37, crimson=38)


def _colorize(string, color, bold=False, highlight=False):
    # gym.utils.colorize: SGR code = colour number (+10 as a background), ";1" when bold
    attrs = ";".join([str(_COLOR2NUM[color] + (10 if highlight else 0))] + (["1"] if bold else []))
    return "\x1b[%sm%s\x1b[0m" % (attrs, string)


def highlight(string, background="white", color="gray"):
    # chess_v2.py:110-111: colorize(colorize(string, color), background, highlight=True)
    return _colorize(_colorize(string, color), background, highlight=True)


def make_random_policy(np_random, bot_player):
    """chess_v2.py:116-127: a uniform index into env.possible_moves drawn from the GLOBAL numpy generator (the
    `np_random` argument is ignored there too, Q18); "resign" when there is no move (-> TypeError downstream, Q9)"""

    def random_policy(env):
        moves = env.possible_moves
        if len(moves) == 0:
            return "resign"
        return moves[np.random.choice(np.arange(len(moves)))]

    return random_policy


class ChessEnvV2:
    def __init__(self, player_color=WHITE, opponent="random", log=True, initial_board=DEFAULT_BOARD, seed=0, device=0):
        self.moves_max = 149
        self.log = log
        self.initial_board = initial_board
        self.engine = ChessEngine()
        self.observation_space = _Box(-6, 6, (8, 8))
        self.action_space = _Discrete(64 * 64 + 4 + 1)
        self.player = player_color
        self.player_2 = self.get_other_player(player_color)
        self.opponent = opponent
        self._seed, self._device = seed, device
        if isinstance(opponent, str):
            if opponent == "random":
                self.opponent_policy = make_random_policy(None, self.player_2)
            elif opponent == "none":
                self.opponent_policy = None
            else:
                raise ValueError(f"Unrecognized opponent policy {opponent}")  # gym.error.Error in the reference
        else:
            self.opponent_policy = opponent
        if player_color == BLACK and self.opponent_policy is None:
            raise TypeError("'NoneType' object is not callable")  # what the reference does (Q23, chess_v2.py:208-209)
        self._env = BatchedChessEnv(1, opponent="none" if self.opponent_policy is None else "external", player_color=player_color,
                                    seed=seed, device=device, auto_reset=False, initial_boards=np.asarray(initial_board, np.int8))
        self._first = True
        self.reset()

    def seed(self, seed=None):
        self._seed = 0 if seed is None else seed
        return [seed]

    # ------------------------------------------------------------------ state mirror
    def _pull(self):
        boards, info, legal = self._env.export_numpy()
        r = info[0]
        self.board = boards[0].reshape(8, 8).tolist()
        self.current_player = WHITE if r[0] > 0 else BLACK
        self.white_king_castle_is_possible, self.white_queen_castle_is_possible = bool(r[1]), bool(r[2])
        self.black_king_castle_is_possible, self.black_queen_castle_is_possible = bool(r[3]), bool(r[4])
        self.white_king_is_checked, self.black_king_is_checked = bool(r[5]), bool(r[6])
        self.done, self.move_count = bool(r[7]), int(r[8])
        self._possible_moves = [codec.ACTION_TO_MOVE[a] for a in legal[0, : r[9]]]
        self._possible_actions = [int(a) for a in legal[0, : r[9]]]

    def _log_ply(self, move):
        # player_move's log (chess_v2.py:409-411): the mover and the move on the PRE-move board
        print(" " * 10, ">" * 10, self.current_player)
        self.render_moves([move], mode="human")

    def _bot_ply(self):
        """the opponent's ply: policy(env) -> move -> player_move without a membership test (chess_v2.py:277-283, 208-213).
        -> (reward to add, done)"""
        move = self.opponent_policy(self)
        action = self.move_to_action(move)
        if action is None or not isinstance(action, (int, np.integer)):
            # "resign" (make_random_policy without moves, Q9) or anything else move_to_action does not know
            raise TypeError("'>=' not supported between instances of 'NoneType' and 'int'")
        if action < 4096 and self.board[(action >> 6) >> 3][(action >> 6) & 7] == 0:
            raise RuntimeError("Bad move - piece is empty !")  # the reference's engine panics (lib.rs:693-695)
        r, d, f = self._env.bot_ply(np.array([action], np.int32))
        r, d, f = int(r[0]), bool(d[0]), int(f[0])
        if self.log and not (f & F_REPETITION):
            self._log_ply(self.action_to_move(action))
        self._pull()
        return r, d

    def reset(self):
        """chess_v2.py:183-217"""
        if not self._first:
            self._env.reset()
        self._first = False
        self._pull()
        self.white_king_on_the_board = self.piece_is_on_board(self.board, KING_ID)    # set here only (Q8)
        self.black_king_on_the_board = self.piece_is_on_board(self.board, -KING_ID)
        if self.player == BLACK:  # the opponent opens for White (chess_v2.py:208-216)
            self._bot_ply()
        return self.state

    def step(self, action):
        """chess_v2.py:219-294"""
        assert self.action_space.contains(action), "ACTION ERROR {}".format(action)
        was_done, capped = self.done, self.move_count > self.moves_max
        r, d, f = self._env.step_host(np.array([action], np.int32))
        reward, done, flags = int(r[0]), bool(d[0]), int(f[0])
        played = not (flags & F_INVALID) and not was_done and not capped
        if not (flags & F_INVALID) and (was_done or capped):
            reward = 0.0  # the two float literals of chess_v2.py:248,255
        if played and self.log and not (flags & F_REPETITION):
            self._log_ply(self.action_to_move(action))
        self._pull()
        if flags & F_BOT_PENDING and not flags & F_INVALID:  # chess_v2.py:277-288 (a refused step plays no ply: no reply)
            r2, done = self._bot_ply()
            reward += r2
        return self.state, reward, done, self.info

    # ------------------------------------------------------------------ properties (chess_v2.py:301-391)
    @property
    def state(self):
        return dict(
            board=self.board, current_player=self.current_player,
            white_king_castle_is_possible=self.white_king_castle_is_possible,
            white_queen_castle_is_possible=self.white_queen_castle_is_possible,
            black_king_castle_is_possible=self.black_king_castle_is_possible,
            black_queen_castle_is_possible=self.black_queen_castle_is_possible,
            white_king_is_checked=self.white_king_is_checked, black_king_is_checked=self.black_king_is_checked)

    @state.setter
    def state(self, state):
        """chess_v2.py:315-323 assigns the board and the six flags and nothing else (possible_moves, saved_boards and the
        side to move keep their old values).  Here the assignment starts a new episode from that position for the side
        currently to move: flags are re-derived by update_state, possible_moves is regenerated and the repetition window
        is emptied (gcb_env_import) -- the consistent form of what the reference's callers do by hand."""
        board = np.asarray(state.get("board"), np.int8).reshape(1, 64)
        rights = np.array([[bool(state.get(k)) for k in ("white_king_castle_is_possible", "white_queen_castle_is_possible",
                                                         "black_king_castle_is_possible", "black_queen_castle_is_possible")]], np.uint8)
        player = np.array([1 if state.get("current_player", self.current_player) == WHITE else -1], np.int8)
        self._env.set_state(board, player, rights, np.array([self.move_count], np.int32))
        self._pull()

    @property
    def possible_moves(self):
        return self._possible_moves

    @property
    def possible_actions(self):
        return list(self._possible_actions)

    @property
    def info(self):
        return dict(
            move_count=self.move_count, current_player=self.current_player, possible_moves=self.possible_moves,
            white_king_castle_is_possible=self.white_king_castle_is_possible,
            white_queen_castle_is_possible=self.white_queen_castle_is_possible,
            black_king_castle_is_possible=self.black_king_castle_is_possible,
            black_queen_castle_is_possible=self.black_queen_castle_is_possible,
            white_king_is_checked=self.white_king_is_checked, black_king_is_checked=self.black_king_is_checked,
            white_king_on_the_board=self.white_king_on_the_board, black_king_on_the_board=self.black_king_on_the_board)

    @property
    def opponent_player(self):
        return BLACK if self.current_player == WHITE else WHITE

    @property
    def current_player_is_white(self):
        return self.current_player == WHITE

    @property
    def current_player_is_black(self):
        return not self.current_player_is_white

    def king_is_checked(self, player):
        return self.white_king_is_checked if player == WHITE else self.black_king_is_checked

    def piece_is_on_board(self, board, piece_id):
        return any(sq == piece_id for row in board for sq in row)

    def player_can_castle(self, player):
        if player == WHITE:
            return self.white_king_castle_is_possible and self.white_queen_castle_is_possible
        return self.black_king_castle_is_possible and self.black_queen_castle_is_possible

    def get_other_player(self, player):
        return BLACK if player == WHITE else WHITE

    # ------------------------------------------------------------------ engine queries (chess_v2.py:414-420, 569-593)
    def next_state(self, state, player, move):
        if state is None:
            state = self.state
        return self.engine.next_state(state, player, self.move_to_str_code(move))

    def get_possible_actions(self):
        return [self.move_to_action(m) for m in self.get_possible_moves(player=self.current_player)]

    def get_possible_moves(self, state=None, player=None, attack=False):
        state = self.state if state is None else state
        player = self.current_player if player is None else player
        return [self.rust_move_to_coords(m) for m in self.engine.get_possible_moves(state, player, attack)]

    def get_castle_moves(self, state=None, player=None):
        state = self.state if state is None else state
        player = self.current_player if player is None else player
        return [self.rust_move_to_coords(m) for m in self.engine.get_castle_moves(state, player)]

    def is_resignation(self, action):
        return False

    def encode_board(self):
        mapping = "0ABCDEFfedcba"
        return "".join(mapping[val] for row in self.board for val in row)

    # ------------------------------------------------------------------ codec (chess_v2.py:492-567)
    def move_to_action(self, move):
        return codec.move_to_action(move)

    def action_to_move(self, action):
        return codec.action_to_move(action)

    def action_to_move_str(self, action):
        # the reference raises NameError here (Q17, chess_v2.py:532); return the intended string instead
        return codec.ACTION_TO_STR[int(action)]

    def move_to_str_code(self, move):
        return codec.move_to_str_code(move)

    def rust_move_to_coords(self, move):
        return codec.str_code_to_move(move)

    def move_to_string(self, move):
        if move in (CASTLE_KING_SIDE_WHITE, CASTLE_KING_SIDE_BLACK):
            return "O-O"
        if move in (CASTLE_QUEEN_SIDE_WHITE, CASTLE_QUEEN_SIDE_BLACK):
            return "O-O-O"
        _from, _to = move
        rows, cols = list(reversed("12345678")), "abcdefgh"
        desc = ID_TO_DESC[self.board[_from[0]][_from[1]]]
        capture = self.board[_to[0]][_to[1]] != 0
        return f"{desc}{cols[_from[1]]}{rows[_from[0]]}{'x' if capture else ''}{cols[_to[1]]}{rows[_to[0]]}"

    # ------------------------------------------------------------------ render (chess_v2.py:422-490)
    def board_to_grid(self):
        return [[f" {ID_TO_ICON[sq]} " for sq in row] for row in self.board]

    def render_grid(self, grid, mode="human"):
        outfile = sys.stdout if mode == "human" else StringIO()
        outfile.write("    " + "-" * 25 + "\n")
        rows = "87654321"
        for i, row in enumerate(grid):
            outfile.write(f" {rows[i]} | " + "".join(row) + "|\n")
        outfile.write("    " + "-" * 25 + "\n      a  b  c  d  e  f  g  h \n")
        if mode == "string":
            return outfile.getvalue()
        if mode != "human":
            return outfile

    def render(self, mode="human"):
        return self.render_grid(self.board_to_grid(), mode=mode)

    def render_moves(self, moves, mode="human"):
        grid = self.board_to_grid()
        for move in moves:
            if type(move) is str and move in CASTLE_MOVES:
                row = 7 if move in (CASTLE_QUEEN_SIDE_WHITE, CASTLE_KING_SIDE_WHITE) else 0
                if move in (CASTLE_QUEEN_SIDE_WHITE, CASTLE_QUEEN_SIDE_BLACK):
                    grid[row][0] = highlight(grid[row][0], background="white")
                    grid[row][1] = highlight(" >>", background="green")
                    grid[row][2] = highlight("> <", background="green")
                    grid[row][3] = highlight("<< ", background="green")
                    grid[row][4] = highlight(grid[row][4], background="white")
                else:
                    grid[row][4] = highlight(grid[row][4], background="white")
                    grid[row][5] = highlight(" >>", background="green")
                    grid[row][6] = highlight("<< ", background="green")
                    grid[row][7] = highlight(grid[row][7], background="white")
                continue
            (x0, y0), (x1, y1) = move
            if len(grid[x0][y0]) < 4:
                grid[x0][y0] = highlight(grid[x0][y0], background="white")
            if len(grid[x1][y1]) < 4:
                grid[x1][y1] = highlight(grid[x1][y1], background="red" if self.board[x1][y1] else "green")
        return self.render_grid(grid, mode=mode)

    def close(self):
        self._env.close()


# the two modes the reference registers with gym (gym_chess/__init__.py:32-42)
REGISTRY = {"ChessVsRandomBot-v2": dict(opponent="random"), "ChessVsSelf-v2": dict(opponent="none")}


def make(env_id, **kwargs):
    """gym.make stand-in for the v2 ids"""
    kw = dict(REGISTRY[env_id])
    kw.update(kwargs)
    return ChessEnvV2(**kw)
