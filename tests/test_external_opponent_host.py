"""opponent="external" (the caller supplies the bot's plies: callable opponents, a learner against its own policy) on the host
emulation of the device rules: the whole interplay of step / step_index / bot_ply / masked resets against the reference
model of tests/external_helpers.py, and the regressions of the owed opening ply, its outputs, F_BOT_PENDING and the packed
record layout."""
import numpy as np
import pytest

from gym_chess_b200.boards import endgame_boards
from oracle import oracle as orc
from tests import external_helpers as xh
from tests.host_emul import emul

E2E4, E7E5, D2D4 = orc.str_to_action("e2e4"), orc.str_to_action("e7e5"), orc.str_to_action("d2d4")


class EmulExternal:
    """the host emulation with the adapter interface of external_helpers (forms "step" and "index")"""

    def __init__(self, N, **kw):
        self.N = N
        self.e = emul.EmulEnv(N, opponent="external", legal_stride=256, **kw)

    def _outs(self, fill):
        N = self.N
        return np.full(N, fill[0], np.int32), np.full(N, fill[1], np.uint8), np.full(N, fill[2], np.uint8)

    def call(self, form, inp):
        r, d, f = self._outs((0, 0, 0))
        a, b = np.full(self.N, -1, np.int32), np.full(self.N, -1, np.int32)
        mode, inp = {"step": (0, np.int32), "index": (1, np.uint32)}[form][0], np.ascontiguousarray(inp)
        emul.lib().emul_env_step(self.e._h, mode, emul._p(inp), emul._p(r), emul._p(d), emul._p(f), emul._p(a), emul._p(b))
        assert (b == -1).all()  # the device never draws a move for an external bot
        return r, d, f, a

    def bot_ply(self, acts, fill=xh.SENTINEL):
        r, d, f = self._outs(fill)
        a = np.ascontiguousarray(acts, np.int32)
        emul.lib().emul_env_step(self.e._h, 4, emul._p(a), emul._p(r), emul._p(d), emul._p(f), None, None)
        return r, d, f

    def reset(self, mask=None):
        self.e.reset(mask)

    def export(self):
        return self.e.export()

    def stats(self):
        return self.e.stats()


CASES = [(color, auto_reset, boards, mm) for color in ("WHITE", "BLACK") for auto_reset in (True, False)
         for boards in ("default", "endgame") for mm in (149, 12)]


@pytest.mark.parametrize("color,auto_reset,boards,moves_max", CASES)
def test_external_opponent_vs_model(color, auto_reset, boards, moves_max):
    N, seed = 28, 5
    tb = endgame_boards() if boards == "endgame" else None
    env = EmulExternal(N, player_color=color, seed=seed, auto_reset=auto_reset, moves_max=moves_max, initial_boards=tb)
    models = xh.make_models(N, color, seed, auto_reset, moves_max, tb)
    xh.cmp_export(env, models, "create")
    rng = np.random.RandomState(100 + CASES.index((color, auto_reset, boards, moves_max)))
    tot = xh.run_external(env, models, rng, 300, forms=("step", "index"), p_reset=0.02 if auto_reset else 0.05)
    xh.check_totals(env, tot)
    assert tot[xh.ST_INVALID] > 0 and tot[xh.ST_PLIES] > 0
    if boards == "endgame":
        assert tot[xh.ST_EPISODES] > 0 and (tot[xh.ST_REPS] > 0 or not auto_reset)  # repetitions happen on these boards
    if moves_max == 12 and color == "WHITE":
        assert tot[xh.ST_CAPS] > 0  # (a BLACK agent's move_count stays 1: chess_v2.py:291-292 counts after White's plies)


def test_refused_steps_then_the_opening_ply():
    """a step refused because the opening is owed leaves the env alone; the opening is then applied as the opening
    (move_count 1, like the reference's reset) however many steps were refused before it"""
    for refused in (0, 1, 3):
        env = EmulExternal(1, player_color="BLACK", auto_reset=False)
        for _ in range(refused):
            r, d, f, _ = env.call("step", np.array([E7E5], np.int32))
            assert (int(r[0]), int(d[0]), int(f[0])) == (-10, 0, xh.F_INVALID | xh.F_BOT_PENDING)
            info = env.export()[1][0]
            assert (info[8], info[11], info[14]) == (0, 0, 1)  # move_count, step_in_episode, bot_pending untouched
        r, d, f = env.bot_ply(np.array([E2E4], np.int32))
        assert (int(r[0]), int(d[0]), int(f[0])) == (0, 0, 0)
        board, info = (x[0] for x in env.export()[:2])
        assert (info[0], info[8], info[11], info[14]) == (-1, 1, 0, 0), (refused, info)
        o = orc.OracleEnv(None, "BLACK", "random", 0, 0, first_bot_action=E2E4)
        assert (board == o.view()["board"]).all() and o.view()["move_count"] == 1
        r, d, f, _ = env.call("step", np.array([E7E5], np.int32))
        assert (int(r[0]), int(d[0]), int(f[0])) == (-10, 0, xh.F_BOT_PENDING)  # the agent's ply, the reply is owed
        st = env.stats()
        assert (st[0], st[1], st[7]) == (refused + 1, 2, refused)  # steps, plies, invalid


def test_opening_ply_writes_its_outputs_and_leaves_other_rows_alone():
    """the opening's outputs are written over whatever the buffers held (reward 0, done 0, flags 0), through the library
    call itself; a bot ply for envs that owe nothing writes nothing and changes nothing"""
    L, p = emul.lib(), emul._p
    e = emul.EmulEnv(3, opponent="external", player_color="BLACK", auto_reset=True)
    r, d, f = np.full(3, 55, np.int32), np.full(3, 7, np.uint8), np.full(3, 99, np.uint8)
    L.emul_env_step(e._h, 4, p(np.array([E2E4, D2D4, E2E4], np.int32)), p(r), p(d), p(f), None, None)
    assert r.tolist() == [0, 0, 0] and d.tolist() == [0, 0, 0] and f.tolist() == [0, 0, 0]
    before = e.export()
    r, d, f = np.full(3, 55, np.int32), np.full(3, 7, np.uint8), np.full(3, 99, np.uint8)
    L.emul_env_step(e._h, 4, p(np.array([E7E5, E7E5, E7E5], np.int32)), p(r), p(d), p(f), None, None)
    assert r.tolist() == [55] * 3 and d.tolist() == [7] * 3 and f.tolist() == [99] * 3
    after = e.export()
    assert all((x == y).all() for x, y in zip(before, after))
    assert e.stats()[1] == 3  # the three openings are the only plies


def test_bot_pending_after_a_reset_into_a_black_episode():
    """a terminal step with auto-reset into a BLACK-agent episode reports F_BOT_PENDING with F_RESET: the opening is owed"""
    b = np.zeros(64, np.int8)
    b[56], b[42], b[33] = 1, -1, -2  # white Ka1; black Kc3, Qb4 to move: Qb2 mates
    env = EmulExternal(2, player_color="BLACK", auto_reset=True)
    env.bot_ply(np.array([E2E4, E2E4], np.int32))
    env.e.set_state(np.stack([b, b]), np.array([-1, -1], np.int8), np.zeros((2, 4), np.uint8), None, np.array([1, 0], np.uint8))
    r, d, f, _ = env.call("step", np.array([orc.str_to_action("b4b2"), E7E5], np.int32))
    assert (int(r[0]), int(d[0]), int(f[0])) == (90, 1, xh.F_MATE | xh.F_RESET | xh.F_BOT_PENDING)
    assert (int(r[1]), int(d[1]), int(f[1])) == (-10, 0, xh.F_BOT_PENDING)  # env 1: e7e5 played, the reply is owed
    info = env.export()[1]
    assert info[:, 14].tolist() == [1, 1] and info[0, 8] == 0 and info[0, 0] == 1
    r, d, f = env.bot_ply(np.array([D2D4, D2D4], np.int32))
    assert (int(r[0]), int(d[0]), int(f[0])) == (0, 0, 0)  # env 0: the new episode's opening
    assert (int(r[1]), int(d[1]), int(f[1])) == (0, 0, 0)  # env 1: the reply
    assert env.export()[1][:, 14].tolist() == [0, 0]


def test_packed_record_carries_every_flag():
    """the 16-bit record of the packed step forms (pack_result as compiled for the device, unpacked by
    BatchedChessEnv.unpack_result): reward bits 0-7 as int8, the seven flags in bits 8-14, done in bit 15"""
    from gym_chess_b200.batched_env import BatchedChessEnv

    L = emul.lib()
    rewards = np.array([-120, -110, -10, -1, 0, 1, 10, 90, 100], np.int32)
    recs, exp = [], []
    for flags in range(128):
        for done in (0, 1):
            for rw in rewards:
                recs.append(L.emul_pack_result(int(rw), done, flags))
                exp.append((int(rw), done, flags))
    recs = np.array(recs, np.uint16)
    assert ((recs >> 8) & 127).tolist() == [e[2] for e in exp]
    r, d, f = BatchedChessEnv.unpack_result(recs)
    assert list(zip(r.tolist(), d.tolist(), f.tolist())) == exp
    assert L.emul_pack_result(0, 0, xh.F_BOT_PENDING) == 1 << 14
