"""Network-input encoder (gcb_env_encode / BatchedChessEnv.encode) on the host emulation: env_encode_one of env_core.cuh
compiled with g++ (tests/host_emul/encode_emul.cpp), compared byte for byte with the NumPy reference of
tests/encode_helpers.py (planes from the oracle's view, the repetition count from the oracle's saved_boards history) in
self-play from the default board (with takebacks) and sampled from the endgame templates, against the random bot with either
colour, with an external opponent while a bot ply is owed, after state imports, for clones and for done envs without
auto-reset.  The same checks on the GPU are in test_encode_gpu.py."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests import encode_helpers as eh
from tests import external_helpers as xh
from tests import parity_helpers as ph
from tests.host_emul import encode_emul as ee
from tests.test_external_opponent_host import EmulExternal

F_REPETITION = 4
NF3, NF6, NG1, NG8 = 62 * 64 + 45, 6 * 64 + 21, 45 * 64 + 62, 21 * 64 + 6
SHUFFLE = [NF3, NF6, NG1, NG8] * 2 + [NF3]
DTYPES = (np.float32, np.uint16, np.uint8)  # (uint16: bf16 bit patterns)


def _as_u8(planes):
    if planes.dtype == np.float32:
        return eh.f32_as_u8(planes)
    return eh.bf16_as_u8(planes) if planes.dtype == np.uint16 else planes


def _check(E, ref, tag, dtypes=DTYPES):
    for dt in dtypes:
        planes, rep = E.encode(dt)
        eh.assert_planes(_as_u8(planes), rep, ref[0], ref[1], "%s%s: " % (tag, np.dtype(dt)))
    assert (E.repetition_count() == ref[1]).all(), tag
    return np.bincount(ref[1], minlength=3)


def _oracles(N, tb, color, opponent, seed, moves_max=149):
    return [orc.OracleEnv(None if tb is None else tb[i % len(tb)], color, opponent, seed, i, moves_max=moves_max) for i in range(N)]


def _run_takebacks(E, O, rng, tag):
    """one self-play step through step(actions): every env plays, with probability 1/2, the move that takes back its side's
    previous move when that is legal, otherwise a uniform entry of the oracle's legal list -- the default board then sees
    repetitions as often as the endgame templates do"""
    acts = np.zeros(E.N, np.int32)
    for i, o in enumerate(O):
        v, last = o.view(), o.last_move[int(o.view()["current_player"] < 0)]
        back = None if last is None or last >= 4096 else (last & 63) * 64 + (last >> 6)
        acts[i] = back if back in set(int(x) for x in v["legal"]) and rng.rand() < 0.5 else int(v["legal"][rng.randint(v["n_legal"])])
    r, d, f = E.step(acts)[:3]
    for i, o in enumerate(O):
        side = int(o.view()["current_player"] < 0)
        rr, dd, _ = o.step(int(acts[i]))
        assert (rr, dd) == (int(r[i]), bool(d[i])), (tag, i, int(acts[i]))
        o.last_move[side] = int(acts[i])
        v2 = o.view()
        if dd or v2["n_legal"] == 0:
            o.reset(v2["episode"] + 1)
            o.last_move = [None, None]


@pytest.mark.parametrize("opponent,color,boards,driver,steps,min_counts", [
    ("none", "WHITE", "default", "takebacks", 200, (1500, 150)),
    ("none", "WHITE", "endgames", "sampled", 250, (1500, 100)),
    ("random", "WHITE", "endgames", "sampled", 250, (1000, 50)),
    ("random", "BLACK", "endgames", "sampled", 250, (1000, 50)),
])
def test_encode_matches_reference_in_self_play_and_against_the_bot(opponent, color, boards, driver, steps, min_counts):
    N, seed = 128, 13
    tb = ph.endgame_boards() if boards == "endgames" else None
    E = ee.EmulEnv(N, opponent=opponent, player_color=color, seed=seed, initial_boards=tb)
    O = _oracles(N, tb, color, opponent, seed)
    for o in O:
        o.last_move = [None, None]
    rng = np.random.RandomState(4)
    seen, tot = np.zeros(3, np.int64), dict(steps=0, reward_sum=0, episodes=0)
    seen += _check(E, eh.oracle_reference(O), "reset ")
    for t in range(steps):
        if driver == "sampled":
            ph._run_sampled(E, O, seed, 1, tot, tag="step %d " % t)
        else:
            _run_takebacks(E, O, rng, "step %d " % t)
        seen += _check(E, eh.oracle_reference(O), "step %d " % t, DTYPES if t % 8 == 0 else (np.uint8,))
    # both repetition planes are exercised: count 1 and count 2 occur many times
    assert seen[1] >= min_counts[0] and seen[2] >= min_counts[1], seen


class EncodeExternal(EmulExternal):
    """the external-opponent adapter of test_external_opponent_host.py on an emulation env that also encodes"""

    def __init__(self, N, **kw):
        self.N = N
        self.e = ee.EmulEnv(N, opponent="external", legal_stride=256, **kw)


@pytest.mark.parametrize("color", ["WHITE", "BLACK"])
def test_encode_external_opponent_while_a_bot_ply_is_owed(color):
    """the env encodes the side to move: the bot while a ply is owed (after the agent's ply), the agent otherwise"""
    N, seed = 128, 5
    tb = ph.endgame_boards()
    env = EncodeExternal(N, player_color=color, seed=seed, auto_reset=True, moves_max=149, initial_boards=tb)
    models = xh.make_models(N, color, seed, True, 149, tb)
    rng = np.random.RandomState(17 + len(color))
    seen, owed_rows = np.zeros(3, np.int64), 0
    bot_black = color == "WHITE"
    for c in range(200):
        xh.run_external(env, models, rng, 1, forms=("step", "index"), p_bot=0.45, p_garbage_bot=0.0, p_reset=0.0)
        ref = eh.model_reference(models)
        seen += _check(env.e, ref, "call %d " % c, DTYPES if c % 8 == 0 else (np.uint8,))
        owed = np.array([m.owed is not None for m in models])
        planes = env.e.encode(np.uint8)[0]
        assert (planes[owed, 12] == int(bot_black)).all()  # while a ply is owed, the bot is the side to move
        owed_rows += int(owed.sum())
    assert owed_rows >= 5000 and seen[1] >= 500 and seen[2] >= 25, (owed_rows, seen)


def test_encode_after_state_import_starts_with_count_zero():
    N, seed = 64, 7
    rng = np.random.RandomState(3)
    E = ee.EmulEnv(N, opponent="none", seed=seed)
    O = _oracles(N, None, "WHITE", "none", seed)
    tot = dict(steps=0, reward_sum=0, episodes=0)
    ph._run_sampled(E, O, seed, 60, tot)
    hb, hp, _ = ph.harvest_positions(n_envs=24, steps=300, seed=9)
    for rnd in range(3):
        pick = rng.randint(0, len(hb), size=N)
        boards, players = hb[pick], hp[pick] * rng.choice([-1, 1], size=N).astype(np.int8)
        rights = rng.randint(0, 2, size=(N, 4)).astype(np.uint8)
        mask = (rng.rand(N) < 0.5).astype(np.uint8)
        E.set_state(boards, players, rights, None, mask)
        for i, o in enumerate(O):
            if mask[i]:
                o.import_state(boards[i], int(players[i]), rights[i], 0, episode=o.view()["episode"] + 1)
        ref = eh.oracle_reference(O)
        _check(E, ref, "import %d " % rnd)
        assert (ref[1][mask == 1] == 0).all() and (ref[0][mask == 1, 17:] == 0).all()
        assert (ref[0][mask == 1, 12] != 0).any() and (ref[0][mask == 1, 13:17] != 0).any()
        for t in range(30):
            ph._run_sampled(E, O, seed, 1, tot, tag="after import %d " % rnd)
            _check(E, eh.oracle_reference(O), "after import %d step %d " % (rnd, t), (np.uint8,))


def test_encode_done_envs_without_auto_reset():
    """auto_reset off: an env that ended (mate, repetition, wedged) keeps its last position and is encoded as it stands"""
    N, seed = 96, 19
    tb = ph.endgame_boards()
    E = ee.EmulEnv(N, opponent="none", seed=seed, initial_boards=tb, auto_reset=False)
    O = _oracles(N, tb, "WHITE", "none", seed)
    tot, done_rows = dict(steps=0, reward_sum=0, episodes=0), 0
    for t in range(150):
        ph._run_sampled(E, O, seed, 1, tot, auto_reset=False, tag="step %d " % t)
        _check(E, eh.oracle_reference(O), "step %d " % t, DTYPES if t % 10 == 0 else (np.uint8,))
        done_rows += int((E.export()[1][:, 7] == 1).sum())
    assert done_rows >= 1000, done_rows


def test_clone_encodes_like_its_source():
    rng = np.random.RandomState(21)
    N = 128
    kw = dict(opponent="none", auto_reset=False, history_cap=64, moves_max=250, initial_boards=ph.endgame_boards())
    S = ee.EmulEnv(N, seed=3, **kw)
    for rnd in range(3):
        for _ in range(40):
            S.step_index(rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32))
        S.reset((rng.rand(N) < 0.2).astype(np.uint8))
    for _ in range(25):
        S.step_index(rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32))
    D = ee.EmulEnv(N, seed=4, env_id_offset=7000, **kw)
    idx = rng.randint(0, N, size=N).astype(np.int32)
    idx[::5] = -1
    before = D.encode(np.uint8)
    D.clone_from(S, idx)
    sel = idx >= 0
    for dt in DTYPES:
        (ps, rs), (pd, rd) = S.encode(dt), D.encode(dt)
        assert (pd[sel] == ps[idx[sel]]).all() and (rd[sel] == rs[idx[sel]]).all(), dt
    pd, rd = D.encode(np.uint8)
    assert (pd[~sel] == before[0][~sel]).all() and (rd[~sel] == before[1][~sel]).all()
    rs = S.repetition_count()[idx[sel]]
    assert (rs == 1).sum() >= 5 and (rs == 2).sum() >= 1, np.bincount(rs, minlength=3)


def test_knight_shuffle_sets_plane_17_after_4_plies_and_plane_18_after_8():
    E = ee.EmulEnv(1, opponent="none", auto_reset=False, seed=1)
    expected = [0, 0, 0, 0, 1, 1, 1, 1, 2]  # the count of the board each ply is played FROM
    for k, a in enumerate(SHUFFLE):
        planes, rep = E.encode(np.uint8)
        assert int(rep[0]) == expected[k], (k, int(rep[0]))
        assert (planes[0, 17] == int(expected[k] >= 1)).all() and (planes[0, 18] == int(expected[k] >= 2)).all()
        r, d, f = E.step(np.array([a], np.int32))[:3]
        assert bool(f[0] & F_REPETITION) == (k == 8) and bool(d[0]) == (k == 8), (k, int(f[0]))


def test_encode_is_a_pure_read():
    E = ee.EmulEnv(64, opponent="random", seed=12, initial_boards=ph.endgame_boards())
    for _ in range(30):
        E.step_sampled()
    before = E.export(), E.stats()
    a = [E.encode(dt) for dt in DTYPES]
    b = [E.encode(dt) for dt in DTYPES]
    assert all((x[0] == y[0]).all() and (x[1] == y[1]).all() for x, y in zip(a, b))
    after = E.export(), E.stats()
    assert all((p == q).all() for p, q in zip(before[0], after[0])) and (before[1] == after[1]).all()
    # the three dtypes hold the same values
    assert (a[0][0] == a[2][0]).all() and (eh.bf16_as_u8(a[1][0]) == a[2][0]).all()
