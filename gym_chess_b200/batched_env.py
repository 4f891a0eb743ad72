"""BatchedChessEnv -- N gym-chess v2 envs resident in B200 HBM, advanced by the fused step kernel.

Host-side mirror of the reference's env interface (`ChessEnvV2`, gym_chess/envs/chess_v2.py:132-294) with a
leading batch dimension: same constructor vocabulary (`player_color`, `opponent`, `initial_board`), same
`reset` / `step` / `possible_actions` / `state` / `info` notions, same action encoding, rewards and done rules
(including the reference's quirks, SURVEY.md section 9).  All compute happens in libgymchess_b200.so
(hand-written sm_100a kernels behind the C ABI of include/gymchess_b200.h); torch is only used for device
buffers and streams.  There is no CPU fallback.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import EnvConfig, Positions, check

WHITE, BLACK = "WHITE", "BLACK"

F_INVALID, F_MATE, F_REPETITION, F_CAP, F_WEDGED, F_RESET, F_BOT_PENDING = 1, 2, 4, 8, 16, 32, 64
_OPPONENTS = {"none": 0, "random": 1, "external": 2}
STAT_NAMES = ("steps", "plies", "episodes", "mates", "repetitions", "caps", "wedged", "invalid", "reward_sum",
              "legal_sum", "in_check", "hist_overflow", "slot_overflow", "hist_scanned", "hist_window")
INFO_NAMES = ("current_player", "white_king_castle_is_possible", "white_queen_castle_is_possible",
              "black_king_castle_is_possible", "black_queen_castle_is_possible", "white_king_is_checked",
              "black_king_is_checked", "done", "move_count", "n_legal", "episode", "step_in_episode", "hist_len", "castles", "bot_pending")
# the 19 planes of encode(), in order
OBS_PLANE_NAMES = ("white_king", "white_queen", "white_rook", "white_bishop", "white_knight", "white_pawn",
                   "black_king", "black_queen", "black_rook", "black_bishop", "black_knight", "black_pawn", "black_to_move",
                   "white_king_castle_is_possible", "white_queen_castle_is_possible", "black_king_castle_is_possible",
                   "black_queen_castle_is_possible", "repeated_once", "repeated_twice")
_ENCODE_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.uint8: 2}  # GCB_DT_F32 / GCB_DT_BF16 / GCB_DT_U8


class _DevArray:
    """zero-copy view of library-owned device memory through __cuda_array_interface__"""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False), version=2)


def _stream_ptr(stream=None, device=None):
    """cudaStream_t of `stream`, or of the current torch stream of `device` (default: the current device)"""
    return C.c_void_p((torch.cuda.current_stream(device) if stream is None else stream).cuda_stream)


def _host_ptr(buf):
    """address of a host buffer: numpy array, CPU torch tensor, ctypes pointer / int, or None"""
    if buf is None or isinstance(buf, (int, C.c_void_p)):
        return buf
    if isinstance(buf, torch.Tensor):
        return C.c_void_p(buf.data_ptr())
    return C.c_void_p(buf.ctypes.data)


class BatchedChessEnv:
    def __init__(self, num_envs, opponent="random", player_color=WHITE, seed=0, device=0, auto_reset=True,
                 initial_boards=None, env_id_offset=0, legal_stride=144, history_cap=512, moves_max=149, piece_slots=0):
        """
        opponent      "random" (the bot replies inside step, chess_v2.py:277-288; drawn on the device), "none" (self-play)
                      or "external" (a callable opponent, chess_v2.py:171-179: step() stops with F_BOT_PENDING where the
                      bot would move and the caller supplies its ply with bot_ply())
        player_color  "WHITE" | "BLACK" (BLACK needs a bot to open for White, opponent "random" or "external", like the
                      reference: Q23)
        initial_boards  None (DEFAULT_BOARD) or int8 [T,8,8] / [8,8]; env with global id g starts from board g % T
        env_id_offset   global id of local env 0 -- shards of one job use disjoint id ranges so that the
                        Philox draws (counter = global env id, episode, step) do not depend on the sharding
        """
        _lib.require_gpu()
        if opponent not in _OPPONENTS:
            raise ValueError("opponent must be 'random', 'none' or 'external' (callables: see gym_chess_b200.ChessEnvV2)")
        self.num_envs, self.opponent, self.player_color = int(num_envs), opponent, player_color
        self.device = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        self.auto_reset, self.seed, self.env_id_offset = bool(auto_reset), int(seed), int(env_id_offset)
        self.legal_stride = int(legal_stride)
        self.history_cap = int(history_cap) or 512  # (resolved like gcb_env_create does)
        self.moves_max = 149 if moves_max < 0 else int(moves_max)
        cfg = EnvConfig()
        cfg.num_envs, cfg.env_id_offset, cfg.seed = self.num_envs, self.env_id_offset, self.seed
        cfg.opponent, cfg.agent_black, cfg.auto_reset = _OPPONENTS[opponent], int(player_color == BLACK), int(auto_reset)
        cfg.piece_slots, cfg.history_cap, cfg.moves_max = piece_slots, history_cap, moves_max
        self._templates = None
        if initial_boards is not None:
            tb = np.ascontiguousarray(np.asarray(initial_boards, dtype=np.int8).reshape(-1, 64))
            self._templates = tb
            cfg.n_templates, cfg.template_boards = len(tb), tb.ctypes.data
        cfg.device = self.device.index or 0
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_create(C.byref(cfg), C.byref(self._h)))
            N = self.num_envs
            self.reward = torch.zeros(N, dtype=torch.int32, device=self.device)
            self.done = torch.zeros(N, dtype=torch.uint8, device=self.device)
            self.flags = torch.zeros(N, dtype=torch.uint8, device=self.device)
        self.observation_shape, self.num_actions = (8, 8), 64 * 64 + 4 + 1  # Box(-6,6,(8,8)), Discrete(4101)

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._h = C.c_void_p()
            try:
                _lib.lib().gcb_env_destroy(h)
            except Exception:  # noqa: BLE001  (interpreter shutdown: module globals may already be gone)
                pass

    __del__ = close

    # ------------------------------------------------------------------ stepping (device tensors)
    def reset(self, mask=None):
        """ChessEnvV2.reset for all envs (or those with mask != 0); returns the board observation."""
        with torch.cuda.device(self.device):
            m = None
            if mask is not None:
                m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            check(_lib.lib().gcb_env_reset(self._h, C.c_void_p(m.data_ptr()) if m is not None else None, _stream_ptr()))
        return self.observe()

    def set_state(self, boards, players, rights, move_count=None, mask=None):
        """State import (the reference's `state` setter, chess_v2.py:315-323, for many envs): a new episode of the selected
        envs from arbitrary positions.  boards int8 [N,8,8] or [N,64]; players int8 [N] (+1 WHITE / -1 BLACK); rights
        uint8 [N,4] (wk, wq, bk, bq); move_count int32 [N] or None; mask [N] or None (all)."""
        dev = self.device
        b = torch.as_tensor(boards, device=dev).to(torch.int8).reshape(self.num_envs, 64).contiguous()
        p = torch.as_tensor(players, device=dev).to(torch.int8).reshape(self.num_envs).contiguous()
        r = torch.as_tensor(rights, device=dev).to(torch.uint8).reshape(self.num_envs, 4).contiguous()
        mc = None if move_count is None else torch.as_tensor(move_count, device=dev).to(torch.int32).contiguous()
        m = None if mask is None else torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
        with torch.cuda.device(dev):
            check(_lib.lib().gcb_env_import(self._h, C.c_void_p(b.data_ptr()), C.c_void_p(p.data_ptr()), C.c_void_p(r.data_ptr()),
                                            C.c_void_p(mc.data_ptr()) if mc is not None else None,
                                            C.c_void_p(m.data_ptr()) if m is not None else None, _stream_ptr()))

    def clone_from(self, source, index):
        """Per-env clone (branching a game mid-episode: search rollouts, lookahead, duplicating games): env j becomes env
        index[j] of `source` (a BatchedChessEnv, possibly self) for every j with 0 <= index[j] < source.num_envs; rows with
        index[j] < 0 are left untouched, repeated indices fan one source env out.  index int [num_envs] (tensor or array).
        Unlike set_state the clone continues the source's episode: board, counters, done, an owed bot ply and the repetition
        window (a clone scores a 3-fold repetition exactly as its source would).  Env j keeps its global id, seed, templates and
        statistics; its episode counter advances by one, so its random draws differ from the source's and from an earlier clone
        into the same row.  Both envs must agree in history_cap, piece slots, opponent, player_color and moves_max.  With
        source = self, no selected row may also be the source of a selected row."""
        if not isinstance(source, BatchedChessEnv):
            raise ValueError("clone_from: source must be a BatchedChessEnv")
        if source.device != self.device:
            raise ValueError("clone_from: source lives on %s, this env on %s" % (source.device, self.device))
        for name, mine, theirs in (("history_cap", self.history_cap, source.history_cap),
                                   ("piece slots", self._n_slots(), source._n_slots()), ("opponent", self.opponent, source.opponent),
                                   ("player_color", self.player_color, source.player_color),
                                   ("moves_max", self.moves_max, source.moves_max)):
            if mine != theirs:
                raise ValueError("clone_from: %s differs (%r here, %r in the source)" % (name, mine, theirs))
        idx = torch.as_tensor(index, device=self.device)
        if tuple(idx.shape) != (self.num_envs,):
            raise ValueError("clone_from: index must have shape [%d], got %s" % (self.num_envs, list(idx.shape)))
        if idx.dtype.is_floating_point or idx.dtype == torch.bool:
            raise ValueError("clone_from: index must be an integer tensor")
        idx = idx.to(torch.int32).contiguous()
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_clone(self._h, source._h, C.c_void_p(idx.data_ptr()), _stream_ptr()))

    def _n_slots(self):
        n = C.c_int32()
        check(_lib.lib().gcb_env_piece_slots(self._h, None, C.byref(n)))
        return n.value

    def _outs(self):
        return C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()), C.c_void_p(self.flags.data_ptr())

    def step(self, actions):
        """actions: int32 [N] cuda tensor.  -> (reward int32[N], done uint8[N], flags uint8[N]) (reused buffers).
        opponent="external": F_BOT_PENDING marks the envs that owe the bot a ply when the call returns (see bot_ply)."""
        a = torch.as_tensor(actions, device=self.device).to(torch.int32).contiguous()
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_step(self._h, C.c_void_p(a.data_ptr()), *self._outs(), _stream_ptr()))
        return self.reward, self.done, self.flags

    def bot_ply(self, bot_actions):
        """opponent="external": the bot's ply of every env that owes one, applied like the reference applies
        opponent_policy(env) (no membership test).  An env owes a ply exactly when the last step / bot_ply output of its row
        carried F_BOT_PENDING (and after reset() with player_color BLACK; info column bot_pending): the reply to the agent's
        ply, or White's opening of a new BLACK-agent episode.  -> (reward, done, flags), written only for the envs that owed a ply:
        for a reply the reward is to be ADDED to that of the agent's half; the opening reports 0, not done, no flags (the
        reference's reset discards it).  flags carry F_BOT_PENDING again when an auto-reset started a BLACK-agent episode.
        Envs that owe nothing are left alone, their output rows untouched.  A step() of an env that owes a ply is refused:
        reward -10, F_INVALID | F_BOT_PENDING, state unchanged."""
        a = torch.as_tensor(bot_actions, device=self.device).to(torch.int32).contiguous()
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_bot_ply(self._h, C.c_void_p(a.data_ptr()), *self._outs(), _stream_ptr()))
        return self.reward, self.done, self.flags

    def step_index(self, u32):
        """env i plays legal[i][(u32[i] * n_legal[i]) >> 32]: make_random_policy's uniform draw with caller words."""
        u = torch.as_tensor(u32, device=self.device)
        if u.dtype not in (torch.int32, torch.uint32):
            u = u.to(torch.int64).to(torch.int32)
        u = u.contiguous()
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_step_index(self._h, C.c_void_p(u.data_ptr()), *self._outs(), _stream_ptr()))
        return self.reward, self.done, self.flags

    def step_sampled(self, nsteps=1, record=False):
        """`nsteps` self-play / vs-bot steps with on-device Philox draws.  record=True also returns the actions
        taken, int32 [nsteps, N] (agent) and [nsteps, N] (bot, -1 = none)."""
        acts = bots = None
        with torch.cuda.device(self.device):
            if record:
                acts = torch.empty((nsteps, self.num_envs), dtype=torch.int32, device=self.device)
                bots = torch.empty((nsteps, self.num_envs), dtype=torch.int32, device=self.device)
            check(_lib.lib().gcb_env_step_sampled(
                self._h, int(nsteps), *self._outs(), C.c_void_p(acts.data_ptr()) if record else None,
                C.c_void_p(bots.data_ptr()) if record else None, _stream_ptr()))
        if record:
            return self.reward, self.done, self.flags, acts, bots
        return self.reward, self.done, self.flags

    def dephase(self, groups=43, period=301):
        """Spread the episode phases of a batch that was reset together.  Three random self-play episodes in four end at the
        150-move cap after exactly `period` = 301 steps (chess_v2.py:252-258), so such a batch moves through the game in
        lockstep for good -- every later window sees one narrow band of plies.  Group g (global env id % groups) is reset
        again after (g + 1) * (period // groups) sampled steps, which leaves the groups period // groups steps apart."""
        ids = torch.arange(self.num_envs, device=self.device) + self.env_id_offset
        for g in range(groups):
            self.step_sampled(max(1, period // groups))
            self.reset(ids % groups == g)

    def sample_policy(self, logits, temperature=1.0, u32=None):
        """Act from a learned policy: for every env, a legal action of the side to move drawn from `logits` (cuda float32 or
        bfloat16 [N, >= 4101] on this env's device, last-dim stride 1; only the entries of legal actions are read).
        -> (actions int32[N], logp float32[N]).  temperature T > 0 samples softmax(logits / T) restricted to the legal set,
        logp is the log-probability of the sampled action under it; T = 0 takes the argmax (ties to the lowest action code,
        logp 0).  No legal move, or no finite legal logit: RESIGN (4100), logp 0.  The draw walks the legal set in ascending
        action code, not in the order of legal_actions().  u32: optional int32 / uint32 [N] random words; by default Philox on
        the env's key (counter: global env id, episode, step in episode, 3 + side to move is black), so sharding is invisible
        and a clone draws differently from its source.  A pure read: no state, statistic or mask output changes.  With
        opponent="external" it samples for the bot too once a step has left F_BOT_PENDING (feed the result to bot_ply)."""
        N = self.num_envs
        if not isinstance(logits, torch.Tensor) or not logits.is_cuda or logits.device != self.device:
            raise ValueError("sample_policy: logits must be a cuda tensor on %s" % self.device)
        if logits.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("sample_policy: logits must be float32 or bfloat16, got %s" % logits.dtype)
        if logits.dim() != 2 or logits.shape[0] != N or logits.shape[1] < self.num_actions:
            raise ValueError("sample_policy: logits must have shape [%d, >= %d], got %s" % (N, self.num_actions, list(logits.shape)))
        row_stride = logits.stride(0) if N > 1 else max(logits.stride(0), logits.shape[1])
        if logits.stride(1) != 1 or row_stride < self.num_actions:
            raise ValueError("sample_policy: logits need last-dim stride 1 and a row stride >= %d, got strides %s"
                             % (self.num_actions, list(logits.stride())))
        temperature = float(temperature)
        if not (0.0 <= temperature < float("inf")):
            raise ValueError("sample_policy: temperature must be finite and >= 0, got %r" % temperature)
        dtype = 0 if logits.dtype == torch.float32 else 1  # GCB_DT_F32 / GCB_DT_BF16
        u = None
        if u32 is not None:
            u = torch.as_tensor(u32, device=self.device)
            if tuple(u.shape) != (N,):
                raise ValueError("sample_policy: u32 must have shape [%d], got %s" % (N, list(u.shape)))
            if u.dtype not in (torch.int32, torch.uint32):
                u = u.to(torch.int64).to(torch.int32)
            u = u.contiguous()
        with torch.cuda.device(self.device):
            actions = torch.empty(N, dtype=torch.int32, device=self.device)
            logp = torch.empty(N, dtype=torch.float32, device=self.device)
            check(_lib.lib().gcb_env_sample_policy(self._h, C.c_void_p(logits.data_ptr()), dtype, row_stride, temperature,
                                                   C.c_void_p(u.data_ptr()) if u is not None else None,
                                                   C.c_void_p(actions.data_ptr()), C.c_void_p(logp.data_ptr()), _stream_ptr()))
        return actions, logp

    def step_policy(self, logits, temperature=1.0):
        """sample_policy(logits, temperature) followed by step() of the sampled actions on the same stream, with no host
        synchronisation in between.  -> (actions, logp, reward, done, flags)"""
        actions, logp = self.sample_policy(logits, temperature)
        reward, done, flags = self.step(actions)
        return actions, logp, reward, done, flags

    # ------------------------------------------------------------------ stepping (host buffers, copies inside)
    def step_host(self, actions, reward=None, done=None, flags=None):
        """numpy in / numpy out through gcb_env_step_host (H2D + kernel + D2H inside the call)."""
        a = np.ascontiguousarray(actions, dtype=np.int32)
        return self._host_call(_lib.lib().gcb_env_step_host, a, reward, done, flags)

    def step_index_host(self, u32, reward=None, done=None, flags=None):
        u = np.ascontiguousarray(u32, dtype=np.uint32)
        return self._host_call(_lib.lib().gcb_env_step_index_host, u, reward, done, flags)

    # asynchronous host-buffer steps (page-locked numpy / torch buffers only): enqueue on the current torch stream and return;
    # results are valid after wait().  Two env objects (shards of one device) stepped alternately on two streams keep the
    # device busy while the host reads one shard's results and writes its next actions.
    def step_host_async(self, actions, reward, done, flags, stream=None):
        return self._host_async(_lib.lib().gcb_env_step_host_async, actions, reward, done, flags, stream)

    def step_index_host_async(self, u32, reward, done, flags, stream=None):
        return self._host_async(_lib.lib().gcb_env_step_index_host_async, u32, reward, done, flags, stream)

    def _host_async(self, fn, inp, reward, done, flags, stream):
        check(fn(self._h, _host_ptr(inp), _host_ptr(reward), _host_ptr(done), _host_ptr(flags), _stream_ptr(stream)))

    # packed 16-bit records (2 bytes in, 2 bytes out per env): uint16 actions / random words, uint16 results (bits 0-7 reward
    # as int8, bits 8-14 the flags F_INVALID .. F_BOT_PENDING, bit 15 done); buffers are cuda tensors or page-locked host
    # tensors / arrays; asynchronous like the calls above
    def step_packed(self, actions16, result16, stream=None):
        check(_lib.lib().gcb_env_step_packed(self._h, _host_ptr(actions16), _host_ptr(result16), _stream_ptr(stream)))

    def step_index_packed(self, u16, result16, stream=None):
        check(_lib.lib().gcb_env_step_index_packed(self._h, _host_ptr(u16), _host_ptr(result16), _stream_ptr(stream)))

    @staticmethod
    def unpack_result(result16):
        """uint16 records -> (reward int32, done uint8, flags uint8); numpy array or torch tensor (viewed as int16/int32)"""
        r = np.asarray(result16).view(np.uint16) if not isinstance(result16, torch.Tensor) else result16.cpu().numpy().view(np.uint16)
        return (r & 0xFF).astype(np.uint8).view(np.int8).astype(np.int32), (r >> 15).astype(np.uint8), ((r >> 8) & 127).astype(np.uint8)

    def wait(self, stream=None):
        """block until the steps enqueued on `stream` (default: the current torch stream) have finished"""
        check(_lib.lib().gcb_env_wait(self._h, _stream_ptr(stream)))

    def _host_call(self, fn, inp, reward, done, flags):
        N = self.num_envs
        assert inp.shape == (N,)
        reward = np.empty(N, np.int32) if reward is None else reward
        done = np.empty(N, np.uint8) if done is None else done
        flags = np.empty(N, np.uint8) if flags is None else flags
        # (no torch.cuda.device(...) context here: the library selects and restores the device itself, and this is the hot
        # synchronous path -- the context manager alone costs more than the launch)
        check(fn(self._h, inp.ctypes.data, reward.ctypes.data, done.ctypes.data, flags.ctypes.data, _stream_ptr(None, self.device)))
        return reward, done, flags

    # ------------------------------------------------------------------ observation / state
    def observe(self):
        """`state["board"]` for every env: int8 [N,8,8] (the Box(-6,6,(8,8)) observation, chess_v2.py:156)."""
        with torch.cuda.device(self.device):
            b = torch.empty((self.num_envs, 8, 8), dtype=torch.int8, device=self.device)
            check(_lib.lib().gcb_env_export(self._h, C.c_void_p(b.data_ptr()), None, _stream_ptr()))
        return b

    def info_tensor(self):
        """int32 [N,16]: columns INFO_NAMES (current_player is +1 WHITE / -1 BLACK)."""
        with torch.cuda.device(self.device):
            t = torch.empty((self.num_envs, 16), dtype=torch.int32, device=self.device)
            check(_lib.lib().gcb_env_export(self._h, None, C.c_void_p(t.data_ptr()), _stream_ptr()))
        return t

    def encode(self, dtype=torch.float32, out=None):
        """The network input of every env: [N, 19, 8, 8] binary planes (OBS_PLANE_NAMES) in float32, bfloat16 or uint8,
        square [row, col] with row 0 = rank 8 (the orientation of observe() and of the action codes, not mirrored for the
        side to move).  Planes 0-5 White K Q R B N P, 6-11 Black K Q R B N P, 12 Black to move, 13-16 the castle flags
        wk wq bk bq (info_tensor() columns 1-4), 17 the board has occurred at least once and 18 at least twice as the pre-move
        board of a ply of this episode -- with 18 set, the next ply ends the episode with F_REPETITION.  The count comes from
        the env's repetition table, so it misses a repetition exactly where the step does (a window beyond history_cap, a
        64-bit key collision).  out: a contiguous, 16-byte aligned tensor of this shape and dtype on the env's device (e.g.
        buf[t] of a [T, N, 19, 8, 8] rollout buffer), written in place and returned.  A pure read of the env: no state,
        statistic or mask output changes."""
        if dtype not in _ENCODE_DTYPES:
            raise ValueError("encode: dtype must be torch.float32, torch.bfloat16 or torch.uint8, got %r" % (dtype,))
        shape = (self.num_envs, 19, 8, 8)
        if out is None:
            with torch.cuda.device(self.device):
                out = torch.empty(shape, dtype=dtype, device=self.device)
        elif not isinstance(out, torch.Tensor) or not out.is_cuda or out.device != self.device:
            raise ValueError("encode: out must be a cuda tensor on %s" % self.device)
        elif out.dtype != dtype or tuple(out.shape) != shape:
            raise ValueError("encode: out must be %s %s, got %s %s" % (dtype, list(shape), out.dtype, list(out.shape)))
        elif not out.is_contiguous() or out.data_ptr() % 16:
            raise ValueError("encode: out must be contiguous and 16-byte aligned")
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_encode(self._h, C.c_void_p(out.data_ptr()), _ENCODE_DTYPES[dtype], None, _stream_ptr()))
        return out

    def repetition_count(self):
        """uint8 [N]: how often the current board has occurred as the pre-move board of a ply of this episode, saturated at
        2 (= planes 17 + 18 of encode(); 2: the next ply ends the episode with F_REPETITION).  A pure read."""
        with torch.cuda.device(self.device):
            rep = torch.empty(self.num_envs, dtype=torch.uint8, device=self.device)
            check(_lib.lib().gcb_env_encode(self._h, None, 0, C.c_void_p(rep.data_ptr()), _stream_ptr()))
        return rep

    def legal_actions(self, stride=None):
        """(legal int16-viewed uint16 [N, stride], n_legal int32 [N]) = possible_actions in the reference's order,
        decoded on access from the resident piece slots (like the reference's property, chess_v2.py:333-335)."""
        stride = int(stride or self.legal_stride)
        with torch.cuda.device(self.device):
            out = torch.zeros((self.num_envs, stride), dtype=torch.int16, device=self.device)
            cnt = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            check(_lib.lib().gcb_env_legal_actions(self._h, C.c_void_p(out.data_ptr()), stride, C.c_void_p(cnt.data_ptr()),
                                                   _stream_ptr()))
        return out, cnt

    def piece_slots(self):
        """zero-copy int64 [S, N] view of the resident legal set (slot r = legal targets of the r-th own piece)."""
        ptr, n = C.c_void_p(), C.c_int32()
        check(_lib.lib().gcb_env_piece_slots(self._h, C.byref(ptr), C.byref(n)))
        with torch.cuda.device(self.device):
            return torch.as_tensor(_DevArray(ptr.value, (n.value, self.num_envs), "<i8"), device=self.device)

    def legal_mask(self):
        """uint8 [N, 4101] mask of possible_actions."""
        with torch.cuda.device(self.device):
            m = torch.empty((self.num_envs, 4101), dtype=torch.uint8, device=self.device)
            check(_lib.lib().gcb_env_legal_mask(self._h, C.c_void_p(m.data_ptr()), _stream_ptr()))
        return m

    def legal_bitmask(self, out=None):
        """int64 [N, 65] bit mask of possible_actions: bit (a & 63) of word (a >> 6); word `from` = the legal targets of the
        piece on that square, word 64 = castles (actions 4096..4099 in bits 0..3).  520 B per env: the per-step form."""
        with torch.cuda.device(self.device):
            m = torch.empty((self.num_envs, 65), dtype=torch.int64, device=self.device) if out is None else out
            check(_lib.lib().gcb_env_legal_bitmask(self._h, C.c_void_p(m.data_ptr()), int(m.stride(0)), _stream_ptr()))
        return m

    def set_mask_output(self, bits=None):
        """Register (or, with None, remove) a cuda int64 [N, W >= 65] buffer that EVERY later step call fills with the bit mask
        of possible_actions of the state the step leaves behind (layout of legal_bitmask) -- written by the step kernel
        itself while the legal set sits in shared memory.  An even W (66) lets the rows be written as 16-byte stores."""
        if bits is not None:
            assert bits.is_cuda and bits.dtype == torch.int64 and bits.dim() == 2 and bits.shape[0] == self.num_envs and bits.stride(1) == 1
        self._mask_out = bits  # keeps the buffer alive
        check(_lib.lib().gcb_env_step_mask_output(self._h, None if bits is None else C.c_void_p(bits.data_ptr()),
                                                  0 if bits is None else int(bits.stride(0))))

    @staticmethod
    def unpack_bitmask(bits):
        """int64 [N, 65] bit mask -> bool [N, 4101] (torch ops; for tests and small batches)"""
        sh = torch.arange(64, device=bits.device, dtype=torch.int64)
        full = ((bits[:, :, None] >> sh) & 1).to(torch.bool).reshape(bits.shape[0], 65 * 64)
        return full[:, :4101]

    def export_numpy(self):
        """(boards int8[N,64], info int32[N,16], legal uint16[N,stride]) on the host -- test / debug helper."""
        boards = self.observe().reshape(self.num_envs, 64).cpu().numpy()
        info = self.info_tensor().cpu().numpy()
        legal = self.legal_actions()[0].cpu().numpy().view(np.uint16)
        return boards, info, legal

    def state(self, i):
        """The reference's state dict (chess_v2.py:301-313) of env i."""
        boards, info, _ = self.export_numpy()
        r = info[i]
        return dict(board=boards[i].reshape(8, 8).tolist(), current_player=WHITE if r[0] > 0 else BLACK,
                    white_king_castle_is_possible=bool(r[1]), white_queen_castle_is_possible=bool(r[2]),
                    black_king_castle_is_possible=bool(r[3]), black_queen_castle_is_possible=bool(r[4]),
                    white_king_is_checked=bool(r[5]), black_king_is_checked=bool(r[6]))

    # ------------------------------------------------------------------ checkpoint / resume
    def snapshot(self):
        """-> (uint8 cuda tensor, tick): the whole resident state; `restore` resumes bit-identically (torch.save-able)."""
        n, tick = C.c_uint64(), C.c_uint64()
        check(_lib.lib().gcb_env_snapshot_bytes(self._h, C.byref(n)))
        with torch.cuda.device(self.device):
            buf = torch.empty(n.value, dtype=torch.uint8, device=self.device)
            check(_lib.lib().gcb_env_snapshot(self._h, C.c_void_p(buf.data_ptr()), C.byref(tick), _stream_ptr()))
        return buf, int(tick.value)

    def restore(self, snap):
        buf, tick = snap
        n = C.c_uint64()
        check(_lib.lib().gcb_env_snapshot_bytes(self._h, C.byref(n)))
        if buf.numel() != n.value or buf.dtype != torch.uint8:
            raise ValueError("snapshot does not belong to an env of this configuration")
        with torch.cuda.device(self.device):
            buf = buf.to(self.device).contiguous()
            check(_lib.lib().gcb_env_restore(self._h, C.c_void_p(buf.data_ptr()), C.c_uint64(tick), _stream_ptr()))

    # ------------------------------------------------------------------ statistics
    def stats(self):
        out = np.zeros(16, np.uint64)
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_stats(self._h, out.ctypes.data, _stream_ptr()))
        d = {k: int(out[i]) for i, k in enumerate(STAT_NAMES)}
        d["reward_sum"] = int(out[8:9].view(np.int64)[0])
        return d

    def stats_tensor(self):
        """zero-copy int64 [16] view of the device counters (for an NCCL reduce)."""
        ptr = C.c_void_p()
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_stats_ptr(self._h, C.byref(ptr), _stream_ptr()))
            return torch.as_tensor(_DevArray(ptr.value, (16,), "<i8"), device=self.device)

    def reset_stats(self):
        with torch.cuda.device(self.device):
            check(_lib.lib().gcb_env_stats_reset(self._h, _stream_ptr()))

    def positions(self):
        p = Positions()
        check(_lib.lib().gcb_env_positions(self._h, C.byref(p)))
        return p

    def planes(self):
        """zero-copy views of the resident board: (int64 [N, 2] bit-planes t0 | t1, int64 [N, 2] bit-plane t2 | colour plane
        white) -- piece code (t2 t1 t0) = the reference id: K=001 Q=010 R=011 B=100 N=101 P=110; square = row * 8 + col, row 0 =
        rank 8.  This is the observation a learner can read without any export kernel (32 B per env)."""
        p = self.positions()
        with torch.cuda.device(self.device):
            return (torch.as_tensor(_DevArray(p.bb01, (self.num_envs, 2), "<i8"), device=self.device),
                    torch.as_tensor(_DevArray(p.bb23, (self.num_envs, 2), "<i8"), device=self.device))
