"""opponent="external" on the GPU (gcb_env_step / _step_index / host / packed forms + gcb_env_bot_ply): against the reference
model of tests/external_helpers.py at a few hundred envs; at scale against the random-bot kernels (oracle-checked in
test_gpu_parity.py) fed with their own recorded moves; and the packed records' F_BOT_PENDING bit."""
import numpy as np
import pytest

from gym_chess_b200.boards import DEFAULT_BOARD, endgame_boards
from tests import external_helpers as xh

pytestmark = pytest.mark.gpu
F_BOT_PENDING, F_RESET, F_WEDGED = xh.F_BOT_PENDING, xh.F_RESET, xh.F_WEDGED


def _np(res):
    return tuple(x.cpu().numpy() for x in res[:3])


class GpuExternal:
    """BatchedChessEnv(opponent="external") with the adapter interface of external_helpers: every step form of the library"""

    def __init__(self, N, **kw):
        import torch

        from gym_chess_b200 import BatchedChessEnv

        self.torch, self.N = torch, N
        self.env = BatchedChessEnv(N, opponent="external", legal_stride=256, **kw)
        self.res16 = torch.empty(N, dtype=torch.int16, device=self.env.device)
        self.in16_host = torch.empty(N, dtype=torch.int16).pin_memory()
        self.res16_host = torch.empty(N, dtype=torch.int16).pin_memory()

    def call(self, form, inp):
        torch, env = self.torch, self.env
        if form == "step":
            return _np(env.step(torch.from_numpy(inp).cuda())) + (None,)
        if form == "index":
            return _np(env.step_index(torch.from_numpy(inp.view(np.int32)).cuda())) + (None,)
        if form == "host":
            return env.step_host(inp) + (None,)
        if form == "index_host":
            return env.step_index_host(inp) + (None,)
        if form == "packed":  # device buffers
            env.step_packed(torch.from_numpy(inp.astype(np.uint16).view(np.int16)).cuda(), self.res16)
            env.wait()
            return env.unpack_result(self.res16) + (None,)
        assert form == "index_packed"  # page-locked host buffers, read and written in place
        self.in16_host.numpy()[:] = inp.view(np.int16)
        env.step_index_packed(self.in16_host, self.res16_host)
        env.wait()
        return env.unpack_result(self.res16_host) + (None,)

    def bot_ply(self, acts):
        env = self.env
        env.reward.fill_(xh.SENTINEL[0]), env.done.fill_(xh.SENTINEL[1]), env.flags.fill_(xh.SENTINEL[2])
        return _np(env.bot_ply(self.torch.from_numpy(np.ascontiguousarray(acts, np.int32)).cuda()))

    def reset(self, mask=None):
        self.env.reset(None if mask is None else self.torch.from_numpy(np.asarray(mask, np.uint8)).cuda())

    def export(self):
        return self.env.export_numpy()

    def stats(self):
        from gym_chess_b200.batched_env import STAT_NAMES

        s = self.env.stats()
        return np.array([s[k] for k in STAT_NAMES], np.int64)


FORMS = ("step", "index", "host", "index_host", "packed", "index_packed")


@pytest.mark.parametrize("color,auto_reset,boards,moves_max", [("WHITE", True, "default", 12), ("BLACK", True, "endgame", 149),
                                                               ("BLACK", False, "default", 149), ("WHITE", False, "endgame", 12),
                                                               ("BLACK", True, "default", 12)])
def test_external_opponent_vs_model_gpu(color, auto_reset, boards, moves_max):
    N, seed = 301, 9  # (not a multiple of the block size: the last block is ragged)
    tb = endgame_boards() if boards == "endgame" else None
    env = GpuExternal(N, player_color=color, seed=seed, auto_reset=auto_reset, moves_max=moves_max, initial_boards=tb)
    models = xh.make_models(N, color, seed, auto_reset, moves_max, tb)
    xh.cmp_export(env, models, "create")
    rng = np.random.RandomState(len(color) * 7 + int(auto_reset) * 3 + moves_max)
    tot = xh.run_external(env, models, rng, 140, forms=FORMS, compare_every=10, p_reset=0.02 if auto_reset else 0.05)
    xh.check_totals(env, tot)
    assert tot[xh.ST_INVALID] > 0 and tot[xh.ST_PLIES] > 0


def _opening_actions(boards, rows):
    """White's opening from the default start position, read off the boards after it: the two squares it changed"""
    start = np.asarray(DEFAULT_BOARD, np.int8)
    b = boards[rows]
    changed = b != start[None]
    assert (changed.sum(1) == 2).all()
    frm = np.argmax(changed & (b == 0), axis=1)
    to = np.argmax(changed & (b != 0), axis=1)
    assert (start[frm] > 0).all()
    return (frm * 64 + to).astype(np.int32)


@pytest.mark.parametrize("color", ["WHITE", "BLACK"])
def test_external_replays_the_random_bot_at_scale(color):
    """N = 262,147 envs: a "random" env steps with on-device draws; an "external" env of the same seed gets the recorded agent
    move through step() and the recorded bot reply through bot_ply(), White's openings (read off the random env's board)
    through a further bot_ply().  Rewards (agent half + bot half), done, flags and exports agree every step; all statistics
    counters agree at the end (hist_scanned too: both envs make the same repetition-table operations in the same order),
    once the envs whose bot had no move (the random env reports F_WEDGED and resets; the external env owes a ply that cannot
    be played and gets a masked reset) and the openings played at creation are accounted for."""
    import torch

    from gym_chess_b200 import BatchedChessEnv
    from gym_chess_b200.batched_env import STAT_NAMES

    N, seed, steps = 262147, 31, 160
    R = BatchedChessEnv(N, opponent="random", player_color=color, seed=seed)
    X = BatchedChessEnv(N, opponent="external", player_color=color, seed=seed)
    black = color == "BLACK"

    def sentinel_bot_ply(acts):
        X.reward.fill_(xh.SENTINEL[0]), X.done.fill_(xh.SENTINEL[1]), X.flags.fill_(xh.SENTINEL[2])
        return _np(X.bot_ply(torch.from_numpy(acts).cuda()))

    def openings(rows):
        """X owes exactly `rows` their opening: play the one R played"""
        info = X.info_tensor()[:, 14].cpu().numpy()
        assert (np.nonzero(info)[0] == rows).all() and len(rows) == int(info.sum())
        if not len(rows):
            return
        acts = np.zeros(N, np.int32)
        acts[rows] = _opening_actions(R.observe().reshape(N, 64).cpu().numpy(), rows)
        r, d, f = sentinel_bot_ply(acts)
        owed = np.zeros(N, bool)
        owed[rows] = True
        assert (r[owed] == 0).all() and (d[owed] == 0).all() and (f[owed] == 0).all()
        assert (r[~owed] == xh.SENTINEL[0]).all() and (d[~owed] == xh.SENTINEL[1]).all() and (f[~owed] == xh.SENTINEL[2]).all()

    def compare_exports(t, full):
        for a, b, what in ((R.observe(), X.observe(), "boards"), (R.info_tensor(), X.info_tensor(), "info")) + (
                ((R.legal_bitmask(), X.legal_bitmask(), "legal"),) if full else ()):
            bad = (a != b).reshape(N, -1).any(1)
            assert not bool(bad.any()), ("step %d: %s differ in %d envs, first %d" % (t, what, int(bad.sum()), int(bad.nonzero()[0, 0])))

    openings(np.arange(N) if black else np.zeros(0, np.int64))
    compare_exports(-1, True)
    botless_total = 0
    for t in range(steps):
        r, d, f, acts, bots = R.step_sampled(1, record=True)
        r, d, f, bots = r.cpu().numpy(), d.cpu().numpy(), f.cpu().numpy(), bots[0].cpu().numpy()
        rx, dx, fx = _np(X.step(acts[0]))
        owes = ((fx & F_BOT_PENDING) != 0) & ((fx & F_RESET) == 0)  # a reply is owed (not the opening of a new episode)
        botless = owes & (bots < 0)  # the bot had no move: R reports F_WEDGED (and resets), X owes a ply it cannot play
        replied = owes & ~botless
        assert (bots[~owes] == -1).all()
        assert ((f[botless] & (255 ^ F_RESET)) == F_WEDGED).all() and (r[botless] == rx[botless]).all() and not d[botless].any()
        botless_total += int(botless.sum())
        if botless.any():  # reset X's side of those envs (R has reset them already)
            X.reset(torch.from_numpy(botless.astype(np.uint8)).cuda())
        # one bot ply: the replies, and with a BLACK agent the openings of the episodes R began in this step so far (the
        # agent's ply ended the game, or the bot had no move) -- R played them already
        opening = black & ((((fx & F_RESET) != 0) & ~replied) | botless)
        bacts = np.where(replied, bots, 0).astype(np.int32)
        if opening.any():
            bacts[opening] = _opening_actions(R.observe().reshape(N, 64).cpu().numpy(), np.nonzero(opening)[0])
        rb, db, fb = sentinel_bot_ply(bacts)
        plied = replied | opening
        assert (rb[~plied] == xh.SENTINEL[0]).all() and (db[~plied] == xh.SENTINEL[1]).all() and (fb[~plied] == xh.SENTINEL[2]).all()
        assert (rb[opening] == 0).all() and (db[opening] == 0).all() and (fb[opening] == 0).all()
        # R's step = X's step + X's bot ply
        rr, dd, ff = rx.copy(), dx.copy(), fx.copy()
        rr[replied] += rb[replied]
        dd[replied], ff[replied] = db[replied], fb[replied]
        ok = ~botless
        assert (rr[ok] == r[ok]).all(), "step %d: rewards differ in %d envs" % (t, int((rr[ok] != r[ok]).sum()))
        assert (dd[ok] == d[ok]).all() and ((ff[ok] & (255 ^ F_BOT_PENDING)) == (f[ok] & (255 ^ F_BOT_PENDING))).all(), t
        # F_BOT_PENDING after the last call of the step = a BLACK-agent episode began (the opening is owed)
        assert (((ff[ok] & F_BOT_PENDING) != 0) == (black & ((f[ok] & F_RESET) != 0))).all(), t
        openings(np.nonzero(black & ((fb & F_RESET) != 0) & replied)[0])  # the bot's ply ended the game
        compare_exports(t, t % 8 == 7 or t == steps - 1)
    sr, sx = R.stats(), X.stats()
    assert sr["steps"] == N * steps and sr["invalid"] == 0
    # R's wedged steps of bot-less envs end an episode, X's end nothing; R's creation plays the N openings of a BLACK agent
    # inside the reset, which counts no ply, while X's come through bot_ply, which counts its ply
    shift = dict(wedged=-botless_total, episodes=-botless_total, plies=N if black else 0)
    for k in STAT_NAMES:
        assert sx[k] == sr[k] + shift.get(k, 0), (k, sx[k], sr[k], shift, sx, sr)
    assert sr["mates"] > 0 and sr["repetitions"] > 0 and sr["wedged"] > 0 and botless_total > 0


def test_packed_records_carry_bot_pending():
    """the packed step forms of an external env: bit 14 of every record is F_BOT_PENDING, and the records equal the wide
    outputs of a twin env stepped through gcb_env_step / gcb_env_step_index with the same inputs"""
    import torch

    from gym_chess_b200 import BatchedChessEnv

    N = 4099
    A = BatchedChessEnv(N, opponent="external", player_color="BLACK", seed=3, legal_stride=256)
    B = BatchedChessEnv(N, opponent="external", player_color="BLACK", seed=3, legal_stride=256)
    rng = np.random.RandomState(2)
    res16 = torch.empty(N, dtype=torch.int16, device="cuda")
    seen_pending = 0
    for t in range(40):
        legal, n = A.legal_actions()
        legal, n = legal.cpu().numpy().view(np.uint16), n.cpu().numpy()
        w = rng.randint(0, 2 ** 16, size=N).astype(np.uint16)
        pick = np.where(n > 0, legal[np.arange(N), (w.astype(np.int64) * n) >> 16], 4100).astype(np.int32)
        if rng.rand() < 0.35:  # a bot ply for both (rows that owe nothing are left alone)
            ra, da, fa = _np(A.bot_ply(torch.from_numpy(pick).cuda()))
            rb, db, fb = _np(B.bot_ply(torch.from_numpy(pick).cuda()))
            assert (ra == rb).all() and (da == db).all() and (fa == fb).all()
            continue
        if t % 2:
            ra, da, fa = _np(A.step(torch.from_numpy(pick).cuda()))
            B.step_packed(torch.from_numpy(pick.astype(np.int16)).cuda(), res16)
        else:
            ra, da, fa = _np(A.step_index(torch.from_numpy((w.astype(np.uint32) << 16).view(np.int32)).cuda()))
            B.step_index_packed(torch.from_numpy(w.view(np.int16)).cuda(), res16)
        B.wait()
        rec = res16.cpu().numpy().view(np.uint16)
        assert (((rec >> 14) & 1) == ((fa >> 6) & 1)).all(), t
        rb, db, fb = B.unpack_result(rec)
        assert (rb == ra).all() and (db == da).all() and (fb == fa).all(), t
        seen_pending += int(((rec >> 14) & 1).sum())
    for x, y in zip(A.export_numpy(), B.export_numpy()):
        assert (x == y).all()
    assert seen_pending > N  # the bit was set (refused steps, replies owed, openings owed)
