"""Per-env clone (gcb_env_clone / BatchedChessEnv.clone_from) on the host emulation: the GCB_HD code of env_core.cuh that
k_env_clone runs, compiled with g++ (tests/host_emul/host_emul.cpp) and checked against the oracle and against the
source envs themselves.  The same checks on the GPU are in test_clone_gpu.py."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests import clone_helpers as ch
from tests import parity_helpers as ph
from tests.host_emul import emul

F_REPETITION = 4

# SURVEY.md section 9.5 vector 5: Nf3 Nf6 Ng1 Ng8 x2, then Nf3 -- the start position is the pre-move board for the 3rd time
NF3, NF6, NG1, NG8 = 62 * 64 + 45, 6 * 64 + 21, 45 * 64 + 62, 21 * 64 + 6
SHUFFLE = [NF3, NF6, NG1, NG8] * 2 + [NF3]


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_clone_vs_oracle(opponent, color):
    ch.check_clone_vs_oracle(emul.EmulEnv, opponent, color, 192, np.random.RandomState(5))


def test_clone_external_opponent_continues_like_its_source():
    """opponent "external" (the oracle has no such mode): clones taken while a bot ply is owed and between full steps
    continue exactly like their sources"""
    rng = np.random.RandomState(6)
    kw = dict(opponent="external", player_color="BLACK", auto_reset=False)
    S = emul.EmulEnv(96, seed=1, **kw)
    ch.drive_pair(S, S, np.full(96, -1, np.int32), 30, rng, external=True)  # (plays the source only)
    D = emul.EmulEnv(96, seed=2, env_id_offset=500, **kw)
    S.step_index(rng.randint(0, 2 ** 32, size=96, dtype=np.uint64).astype(np.uint32))   # now a bot ply is owed
    assert (S.export()[1][:, 14] == 1).any()
    idx = rng.permutation(96).astype(np.int32)
    D.clone_from(S, idx)
    ch.assert_same_rows(S.export(), D.export(), idx)
    owed = D.export()[1][:, 14] == 1
    bot = S.export()[2][:, 0].astype(np.int32)
    rs, ds, fs = [np.array(x) for x in S.bot_ply(bot)[:3]]
    rd, dd, fd = [np.array(x) for x in D.bot_ply(bot[idx])[:3]]
    assert (rs[idx][owed] == rd[owed]).all() and (ds[idx][owed] == dd[owed]).all() and (fs[idx][owed] == fd[owed]).all()
    ch.drive_pair(S, D, idx, 120, rng, external=True, tag="external ")


def _shuffle_env(cls, **kw):
    return cls(1, opponent="none", auto_reset=False, **kw)


def test_repetition_window_is_carried_across_the_clone():
    """5 plies of the knight shuffle, clone, 4 more plies on the clone: the 3-fold repetition fires at ply 9 as it does on
    the source.  A state import of the same board starts a new episode with an empty window and does NOT fire: this is
    why the clone exists."""
    S = _shuffle_env(emul.EmulEnv, seed=1)
    for a in SHUFFLE[:5]:
        r, d, f = S.step(np.array([a], np.int32))[:3]
        assert not d[0] and not f[0] & F_REPETITION
    D = _shuffle_env(emul.EmulEnv, seed=77, env_id_offset=9)
    D.clone_from(S, np.array([0], np.int32))
    boards, info, _ = S.export()
    I = _shuffle_env(emul.EmulEnv, seed=1)
    I.set_state(boards, info[:, 0].astype(np.int8), info[:, 1:5].astype(np.uint8), info[:, 8].astype(np.int32))
    for k, a in enumerate(SHUFFLE[5:]):
        last = k == len(SHUFFLE) - 6
        for env, fires in ((S, last), (D, last), (I, False)):
            r, d, f = env.step(np.array([a], np.int32))[:3]
            assert bool(d[0]) == fires and bool(f[0] & F_REPETITION) == fires, (k, env is I)
    assert D.export()[1][0, 7] == 1 and I.export()[1][0, 7] == 0


@pytest.mark.parametrize("boards,history_cap,moves_max,in_object", [
    ("endgames", 8, 250, False),       # 16-slot tables: windows far beyond them (overflow replacement)
    ("endgames", 512, 250, False),
    ("endgames", 512, 250, True),      # in-object, disjoint: rows [0, N/2) -> [N/2, N)
    ("default", 64, 149, False),
])
def test_clone_continues_exactly_like_its_source(boards, history_cap, moves_max, in_object):
    rng = np.random.RandomState(history_cap + moves_max + in_object)
    N = 128
    kw = dict(opponent="none", auto_reset=False, history_cap=history_cap, moves_max=moves_max,
              initial_boards=ph.endgame_boards() if boards == "endgames" else None)
    S = emul.EmulEnv(N, seed=3, **kw)
    # long windows: up to 180 steps before the clone, rows staggered by resets
    for rnd in range(3):
        for _ in range(60):
            S.step_index(rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32))
        S.reset((rng.rand(N) < 0.2).astype(np.uint8))
    if in_object:
        D = S
        idx = np.full(N, -1, np.int32)
        idx[N // 2:] = np.arange(N // 2)
    else:
        D = emul.EmulEnv(N, seed=4, env_id_offset=7000, **kw)
        idx = rng.permutation(N).astype(np.int32)
    assert S.export()[1][:, 12].max() > (8 if history_cap == 8 else 20)  # non-trivial windows are being cloned
    st_s, st_d = S.stats(), D.stats()
    D.clone_from(S, idx)
    ch.assert_same_rows(S.export(), D.export(), idx, "after clone: ")
    ch.drive_pair(S, D, idx, 250, rng, tag="continue ")
    if not in_object:
        assert ch.stats_delta(S.stats(), st_s) == ch.stats_delta(D.stats(), st_d)
        d_s, d_d = np.asarray(S.stats()) - np.asarray(st_s), np.asarray(D.stats()) - np.asarray(st_d)
        assert (d_s[:15] == d_d[:15]).all(), (d_s, d_d)  # repetitions, hist_overflow, probes: every counter


def test_clone_leaves_unselected_and_out_of_range_rows_alone():
    rng = np.random.RandomState(9)
    S = emul.EmulEnv(40, opponent="none", seed=3)
    D = emul.EmulEnv(50, opponent="none", seed=4)
    for _ in range(20):
        S.step_sampled()
        D.step_sampled()
    before = D.export()
    idx = rng.randint(0, 40, size=50).astype(np.int32)
    idx[::3] = -1
    idx[1::7] = 40 + rng.randint(0, 1000, size=len(idx[1::7]))   # out of range
    D.clone_from(S, idx)
    after = D.export()
    keep = (idx < 0) | (idx >= 40)
    for a, b in zip(before, after):
        assert (a[keep] == b[keep]).all()
    sel = np.where(keep, -1, idx)
    ch.assert_same_rows(S.export(), after, sel)


def test_oracle_clone_helper_copies_the_history():
    """the oracle side of the clone (tests/clone_helpers.oracle_clone) reproduces the repetition of the shuffle"""
    src, dst = orc.OracleEnv(seed=1, env_id=0), orc.OracleEnv(seed=5, env_id=3)
    for a in SHUFFLE[:5]:
        src.step(a)
    ch.oracle_clone(dst, src)
    assert dst.view()["hist_n"] == 5 and dst.view()["episode"] == 1
    dones = [dst.step(a)[1] for a in SHUFFLE[5:]]
    assert dones == [False, False, False, True]
