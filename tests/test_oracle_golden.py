"""Pins the CPU oracle (oracle/gc_oracle.c) to the fixtures produced from the reference's REAL chess_v2.py and its own
v2 test-suite (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests import parity_helpers as ph


def test_reference_v2_suite_passed_against_oracle(golden):
    rep = golden["reference_tests"]
    assert len(rep) == 24
    failed = [r for r in rep if not r["passed"] and r["module"] != "test_benchmark"]  # benchmark = wall-clock assert only
    assert not failed, failed
    assert sum(len(r.get("calls", [])) for r in rep) >= 23


def test_oracle_engine_replays_reference_test_calls(golden):
    assert ph.check_reference_test_calls(orc.OracleEngine(), golden["reference_tests"]) >= 23


def test_oracle_movegen_matches_reference_shell_positions(golden):
    def mg(boards, player, rights, attack):
        return orc.movegen_batch(boards, player, rights, attack, stride=256)

    ph.check_positions(mg, orc.update_state_batch, golden["positions"])


def test_oracle_env_replays_real_chess_v2_trajectories(golden):
    """rewards, dones, boards, flags, move_count and ordered legal lists of 91 recorded games of the real chess_v2.py
    (self-play, WHITE/BLACK agent vs bot, edge boards, invalid actions, steps after done)"""
    nsteps = 0
    for t in golden["trajectories"]:
        e = orc.OracleEnv(np.array(t["initial_board"], np.int8), t["player_color"], t["opponent"],
                          first_bot_action=t["reset"]["bot_action"])

        def cmp(s, where):
            v = e.view()
            assert [int(x) for x in v["board"]] == s["board"], where
            assert [v[k] for k in "wk wq bk bq wchk bchk".split()] == s["flags"], where
            assert v["move_count"] == s["move_count"], where
            assert [int(x) for x in v["legal"]] == s["legal"], where
            assert v["current_player"] == (1 if s["current_player"] == "WHITE" else -1), where

        cmp(t["reset"], (t["name"], "reset"))
        for i, s in enumerate(t["steps"]):
            r, d, raised = e.step(s["action"], s["bot_action"])
            nsteps += 1
            if s["raised"]:
                assert raised  # bot without moves: the reference raises TypeError (Q9)
                break
            assert not raised and r == s["reward"] and d == s["done"], (t["name"], t["seed"], i)
            cmp(s, (t["name"], t["seed"], i))
    assert nsteps > 15000


def test_survey_golden_vectors():
    """SURVEY.md section 9.5"""
    K, Q, R, B, N, P = 1, 2, 3, 4, 5, 6

    def board(**pc):
        b = np.zeros((8, 8), np.int8)
        for sq, v in pc.items():
            b[8 - int(sq[1]), "abcdefgh".index(sq[0])] = v
        return b

    # 1. start position: 20 moves in this order
    e = orc.OracleEnv()
    assert [int(x) for x in e.view()["legal"]] == [3112, 3104, 3177, 3169, 3242, 3234, 3307, 3299, 3372, 3364, 3437, 3429,
                                                   3502, 3494, 3567, 3559, 3688, 3690, 4013, 4015]
    # 2. king may retreat along the checking ray and is then captured (Q6, Q7)
    e = orc.OracleEnv(board(e2=K, e8=-R, a8=-K))
    v = e.view()
    assert v["wchk"] == 1
    assert [((a >> 6) // 8, (a >> 6) % 8, (a & 63) // 8, (a & 63) % 8)[2:] for a in v["legal"]] == \
        [(7, 4), (6, 5), (6, 3), (7, 5), (7, 3), (5, 5), (5, 3)]
    r, d, _ = e.step(orc.str_to_action("e2e1"))
    assert orc.str_to_action("e8e1") in e.view()["legal"]
    r, d, _ = e.step(orc.str_to_action("e8e1"))
    v = e.view()
    assert (r, d, v["n_legal"], v["wchk"]) == (-10, False, 0, 0)
    # 3. black never castles (Q3)
    eng = orc.OracleEngine()
    st = dict(board=board(e8=-K, a8=-R, h8=-R, e1=K).tolist(), current_player="BLACK", white_king_castle_is_possible=True,
              white_queen_castle_is_possible=True, black_king_castle_is_possible=True, black_queen_castle_is_possible=True)
    assert eng.get_castle_moves(st, "BLACK") == []
    st["board"] = board(e8=K, h8=R, a1=-K).tolist()
    assert eng.get_castle_moves(st, "BLACK") == []
    # 4. OR-ed castle rights (Q4) and column-only rights update (Q5)
    e = orc.OracleEnv(board(e1=K, a1=R, h1=R, c8=-K, h7=-P))
    for m in ("a1a2", "c8d8", "a2a1", "d8c8"):
        e.step(orc.str_to_action(m))
    v = e.view()
    assert (v["wk"], v["wq"]) == (1, 0) and [int(x) for x in v["legal"][-2:]] == [4097, 4096]
    for m in ("h1h2", "c8d8", "h2h1", "d8c8"):
        e.step(orc.str_to_action(m))
    v = e.view()
    assert (v["wk"], v["wq"]) == (0, 0) and all(a < 4096 for a in v["legal"])
    e = orc.OracleEnv(board(e1=K, h1=R, a5=R, c8=-K))
    e.step(orc.str_to_action("a5b5"))
    assert e.view()["wq"] == 0
    # 5. knight shuffle: done on ply 9, reward -10, move_count 4 (Q11)
    e = orc.OracleEnv()
    out = [e.step(orc.str_to_action(m)) for m in ["g1f3", "g8f6", "f3g1", "f6g8"] * 2 + ["g1f3"]]
    assert [o[1] for o in out] == [False] * 8 + [True] and out[-1][0] == -10 and e.view()["move_count"] == 4
    # 6. dead promotion (Q1)
    e = orc.OracleEnv(board(a7=P, e1=K, h8=-K))
    r, d, _ = e.step(orc.str_to_action("a7a8"))
    assert r == -10 and e.view()["board"][0] == 6
    ns, rew = eng.next_state(dict(st, board=board(a2=P, e1=K, h8=-K).tolist(), current_player="WHITE"), "WHITE", "a2a1")
    assert ns["board"][7][0] == 2 and rew == 10
    # 7. stalemate is not terminal (Q9), mate is, invalid action is evaluated before done (Q16)
    e = orc.OracleEnv(board(a8=-K, b5=Q, c6=K))
    r, d, _ = e.step(orc.str_to_action("b5b6"))
    v = e.view()
    assert (r, d, v["n_legal"], v["bchk"]) == (-10, False, 0, 0)
    assert e.step(0)[:2] == (-10, False)
    e = orc.OracleEnv(board(a8=-K, b5=Q, c6=K))
    assert e.step(orc.str_to_action("b5b7"))[:2] == (90, True)
    assert e.step(0)[:2] == (-10, True)
    # 8. pawn double step jumps over a piece (Q13)
    e = orc.OracleEnv(board(a2=P, a3=-N, e1=K, e8=-K))
    assert [a for a in e.view()["legal"] if (a >> 6) == 48] == [48 * 64 + 32]


def test_philox_known_answers():
    """Random123 kat_vectors for philox4x32-10"""
    assert [hex(x) for x in orc.philox4x32_10([0, 0, 0, 0], [0, 0])] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    assert [hex(x) for x in orc.philox4x32_10([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2)] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]
    assert [hex(x) for x in orc.philox4x32_10([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0])] == \
        ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_selfplay_statistics_shape():
    """SURVEY 9.5 #9 orientation: mean legal moves ~23, most games end at the move cap"""
    st = orc.selfplay_mt(0, 0, 32, 3000, 4)
    assert st["steps"] == 32 * 3000
    assert 20 < st["legal_sum"] / st["steps"] < 27
    assert st["caps"] > st["mates"] > 0 and st["episodes"] == st["mates"] + st["repetitions"] + st["caps"] + st["wedged"]


def test_oracle_matches_move_sets_of_the_reference_pure_python_env(golden):
    """second, independent pin: the reference's own chess_v1.py (pure Python, shares no code with lib.rs or the oracle)
    produced these move sets in the build container (tests/golden/make_golden_v1.py)"""
    def mg(boards, players, rights, attack):
        return orc.movegen_batch(boards, players, rights, attack, stride=256)

    assert len(golden["v1_move_sets"]) > 800
    assert ph.check_v1_move_sets(mg, golden["v1_move_sets"]) > 15000


def test_next_states_of_the_reference_pure_python_env(golden):
    assert ph.check_v1_next_states(orc.next_state_batch, golden["v1_next_states"]) > 3500


def test_v1_castle_through_attack_vector():
    def fn(b, p):
        out, cnt = orc.movegen_batch(b[None], p, np.ones((1, 4), np.uint8), False)
        return [int(a) for a in out[0, : cnt[0]] if a >= 4096]
    ph.check_v1_castle_through_attack_vector(fn)


POOL_CONFIGS = {  # opponent, player_color, moves_max, templates
    "selfplay": ("none", orc.WHITE, 149, None),
    "random-white": ("random", orc.WHITE, 149, None),
    "random-black": ("random", orc.BLACK, 149, None),
    "endgames": ("none", orc.WHITE, 250, "endgames"),
}


@pytest.mark.parametrize("config", list(POOL_CONFIGS))
def test_pool_matches_the_per_env_driver(config):
    """SelfplayPool (the host threads' reference of whole device batches) against OracleEnvs driven one sampled step at a
    time by the driver of the device parity tests (parity_helpers.oracle_sampled_step): 64 envs with global ids from 1001,
    self-play, the random bot for either agent colour and the endgame templates (env g starts from template g % 7), with a
    masked reset in mid-game.  The exports and the pool's steps / reward_sum / episodes must be the driver's."""
    opponent, color, moves_max, templates = POOL_CONFIGS[config]
    boards = ph.endgame_boards() if templates else None
    n, lo, seed = 64, 1001, 5
    pool = orc.SelfplayPool(seed, lo, lo + n, opponent=opponent, player_color=color, moves_max=moves_max, initial_boards=boards)
    O = [orc.OracleEnv(None if boards is None else boards[(lo + i) % len(boards)], color, opponent, seed, lo + i,
                       moves_max=moves_max) for i in range(n)]
    ph.check_export_arrays(pool.export(), ph.oracle_views(O), lo, "reset: ")
    tot = dict(steps=0, reward_sum=0, episodes=0)
    got = dict(steps=0, reward_sum=0, episodes=0)

    def run(k, tag):
        st = pool.run(k, 4)
        for key in got:
            got[key] += st[key]
        for _ in range(k):
            for i, o in enumerate(O):
                ph.oracle_sampled_step(o, seed, lo + i, tot)
        ph.check_export_arrays(pool.export(), ph.oracle_views(O), lo, tag)
        assert got == tot, (tag, got, tot)

    run(1, "1 step: ")
    run(159, "160 steps: ")
    mask = np.random.RandomState(3).rand(n) < 0.4
    pool.reset(mask)
    for i in np.nonzero(mask)[0]:
        O[i].reset(O[i].view()["episode"] + 1)
    ph.check_export_arrays(pool.export(), ph.oracle_views(O), lo, "masked reset: ")
    run(160, "320 steps: ")
    assert tot["episodes"] > 0
