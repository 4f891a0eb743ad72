"""The device rules (gym_chess_b200/csrc/chess_core.cuh, env_core.cuh) compiled with g++ (tests/host_emul) and
checked against the fixtures and the oracle: a LOGIC test for boxes without a GPU.  The parity tests proper, through
the C ABI on the GPU, are in test_gpu_parity.py."""
import numpy as np
import pytest

from oracle import oracle as orc
from tests import parity_helpers as ph
from tests.host_emul import emul


def _mg(boards, players, rights, attack):
    return emul.movegen(boards, players, rights, attack)


def test_golden_positions(golden):
    ph.check_positions(_mg, emul.update_state, golden["positions"])


def test_movegen_selfplay_positions_vs_oracle():
    b, p, r = ph.harvest_positions(n_envs=48, steps=330, seed=1)
    assert len(b) > 5000
    total = ph.check_movegen_vs_oracle(_mg, b, p, r, attack=False)
    assert total > 100000
    ph.check_movegen_vs_oracle(_mg, b, p, r, attack=True)
    ph.check_movegen_vs_oracle(_mg, b, -p, r, attack=False)  # the side NOT to move as well


def test_movegen_and_next_state_crafted_vs_oracle():
    rng = np.random.RandomState(3)
    b, p, r = ph.crafted_positions(rng, 6000)
    ph.check_movegen_vs_oracle(_mg, b, p, r, attack=False)
    ph.check_movegen_vs_oracle(_mg, b, p, r, attack=True)
    out, cnt, _ = emul.movegen(b, p, r)
    ph.check_next_state_vs_oracle(emul.next_state, out, cnt, b, p, r, rng)
    hb, hp, hr = ph.harvest_positions(n_envs=16, steps=300, seed=5)
    out, cnt, _ = emul.movegen(hb, hp, hr)
    ph.check_next_state_vs_oracle(emul.next_state, out, cnt, hb, hp, hr, rng)


def test_castle_only_lists():
    rng = np.random.RandomState(9)
    b, p, r = ph.crafted_positions(rng, 3000)
    out, cnt, _ = emul.movegen(b, p, r, castles_only=True)
    full, fcnt = orc.movegen_batch(b, p, r, False)
    n_castles = 0
    for i in range(len(b)):
        exp = [int(a) for a in full[i, : fcnt[i]] if a >= 4096]
        assert [int(a) for a in out[i, : cnt[i]]] == exp
        n_castles += len(exp)
    assert n_castles > 100


def test_philox_matches_oracle():
    for args in [(0, 0, 0, 0, 0), (123456789012345, 77, 3, 250, 1), (2 ** 64 - 1, 2 ** 32 - 1, 9, 1, 2)]:
        assert emul.lib().emul_philox(*args) == orc.draw_u32(*args)


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_env_sampled_vs_oracle(opponent, color):
    env = emul.EmulEnv(12, opponent=opponent, player_color=color, seed=21, auto_reset=True)
    st = ph.check_sampled_vs_oracle(env, opponent, color, 21, 650)
    assert st[2] > 0  # episodes ended (cap / mate / repetition / wedge all occur in 650 steps x 12 envs)


def test_env_index_mode_and_offset_vs_oracle():
    env = emul.EmulEnv(8, opponent="none", seed=5, auto_reset=True, env_id_offset=1000)
    ph.check_sampled_vs_oracle(env, "none", "WHITE", 5, 200, env_id_offset=1000, mode="index", rng=np.random.RandomState(1))


def test_env_edge_templates_vs_oracle(golden):
    boards = []
    for t in golden["trajectories"]:
        if t["name"].startswith("selfplay_") and t["initial_board"] not in boards:
            boards.append(t["initial_board"])
    boards = np.array(boards, np.int8)
    assert len(boards) >= 15
    for opponent, color in (("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")):
        env = emul.EmulEnv(len(boards) * 2, opponent=opponent, player_color=color, seed=8, auto_reset=True, initial_boards=boards)
        ph.check_sampled_vs_oracle(env, opponent, color, 8, 260, boards=boards)


def test_env_no_autoreset_wedge_and_done_behaviour():
    # stalemate wedge: every further action is invalid (-10, done False); after mate: invalid (-10, True) first (Q16)
    K, Q = 1, 2
    b = np.zeros((8, 8), np.int8)
    b[0, 0], b[3, 1], b[2, 2] = -K, Q, K
    env = emul.EmulEnv(1, opponent="none", auto_reset=False, initial_boards=b)
    r, d, f, _, _ = env.step([orc.str_to_action("b5b6")])
    assert (r[0], d[0], f[0] & 16) == (-10, 0, 16)
    r, d, f, _, _ = env.step([0])
    assert (r[0], d[0], f[0] & 1) == (-10, 0, 1)
    env = emul.EmulEnv(1, opponent="none", auto_reset=False, initial_boards=b)
    r, d, f, _, _ = env.step([orc.str_to_action("b5b7")])
    assert (r[0], d[0], f[0] & 2) == (90, 1, 2)
    r, d, f, _, _ = env.step([0])
    assert (r[0], d[0]) == (-10, 1)


def test_env_replays_real_chess_v2_selfplay_games(golden):
    n = 0
    for t in golden["trajectories"]:
        if t["opponent"] != "none":
            continue
        n += ph.check_trajectory_replay(lambda ib: emul.EmulEnv(1, opponent="none", auto_reset=False, initial_boards=ib), t)
    assert n > 5000


def test_external_opponent_replays_real_chess_v2_bot_games(golden):
    """opponent="external" (callable opponents, chess_v2.py:171-179): the recorded WHITE- and BLACK-agent games of the real
    chess_v2.py against its callable bot, the bot's plies supplied from outside"""
    n = 0
    for t in golden["trajectories"]:
        if t["opponent"] != "random":
            continue
        n += ph.check_external_bot_replay(
            lambda ib, color: emul.EmulEnv(1, opponent="external", player_color=color, auto_reset=False, initial_boards=ib), t)
    assert n > 4000


def test_many_piece_templates_use_more_slots():
    """initial boards with more than 16 pieces of one colour: more piece slots, uncounted-slot path of the ordered pick"""
    rng = np.random.RandomState(4)
    boards = np.zeros((6, 64), np.int8)
    for i in range(6):
        sq = rng.permutation(64)
        boards[i, sq[:22]] = rng.choice([2, 3, 4, 5, 6], size=22)
        boards[i, sq[22:40]] = -rng.choice([2, 3, 4, 5, 6], size=18)
        boards[i, sq[40]], boards[i, sq[41]] = 1, -1
    for opponent, color in (("none", "WHITE"), ("random", "BLACK")):
        env = emul.EmulEnv(12, opponent=opponent, player_color=color, seed=11, auto_reset=True, initial_boards=boards)
        ph.check_sampled_vs_oracle(env, opponent, color, 11, 150, boards=boards, compare_every=10)


def test_more_than_255_legal_moves():
    """queen-heavy initial boards: more than 255 legal moves, beyond the byte-wise prefix sums of the ordered pick
    (the pick then scans the count bytes one by one)"""
    boards = ph.queen_heavy_boards()
    n_max = max(orc.OracleEnv(b, "WHITE", "none", 1, 0).view()["n_legal"] for b in boards)
    assert n_max > 255
    env = emul.EmulEnv(8, opponent="none", seed=21, auto_reset=True, initial_boards=boards, legal_stride=512)
    ph.check_sampled_vs_oracle(env, "none", "WHITE", 21, 60, boards=boards, compare_every=5)


def test_endgames_with_long_repetition_windows():
    """BASELINE.json configs[4]: repetition-heavy endgames, move cap lifted, 512-slot ring: the Bloom-gated ring scan
    must find every 3-fold the reference's dict finds (windows grow to hundreds of plies here)"""
    boards = ph.endgame_boards()
    env = emul.EmulEnv(21, opponent="none", seed=17, auto_reset=True, initial_boards=boards, moves_max=250, history_cap=512)
    st = ph.check_sampled_vs_oracle(env, "none", "WHITE", 17, 900, boards=boards, compare_every=50, moves_max=250)
    assert st[4] > 20 and st[11] == 0  # repetitions happened, no ring overflow
    assert st[14] / st[1] > 20         # mean window far above random play's ~6
    env = emul.EmulEnv(14, opponent="random", player_color="BLACK", seed=18, auto_reset=True, initial_boards=boards, history_cap=512)
    ph.check_sampled_vs_oracle(env, "random", "BLACK", 18, 500, boards=boards, compare_every=50)  # BLACK agent: no cap (Q12)


def test_move_sets_of_the_reference_pure_python_env(golden):
    assert ph.check_v1_move_sets(_mg, golden["v1_move_sets"]) > 15000


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_state_import_vs_oracle(opponent, color):
    env = emul.EmulEnv(16, opponent=opponent, player_color=color, seed=41, auto_reset=True)
    ph.check_state_import_vs_oracle(env, opponent, color, 41, np.random.RandomState(6))


@pytest.mark.parametrize("opponent,color,auto_reset", [("none", "WHITE", True), ("random", "WHITE", True), ("random", "BLACK", True),
                                                         ("none", "WHITE", False), ("random", "WHITE", False)])
def test_external_actions_incl_invalid_vs_oracle(opponent, color, auto_reset):
    env = emul.EmulEnv(10, opponent=opponent, player_color=color, seed=77, auto_reset=auto_reset)
    st = ph.check_external_actions_vs_oracle(env, opponent, color, 77, 420, np.random.RandomState(8), auto_reset)
    assert st[7] > 0  # invalid actions occurred


def test_next_state_reports_both_kings_in_check():
    """Q19 (lib.rs:1442-1446): a move after which BOTH kings are in check is applied, and flagged with status 1"""
    b = np.zeros(64, np.int8)
    b[60], b[56], b[28], b[7] = 1, 3, -3, -1          # Ke1, Ra1; black Re5 (checks e1), Kh8
    a = 56 * 64 + 0                                    # Ra1-a8+: the white king stays in check, the black king is checked
    for fn in (orc.next_state_batch, emul.next_state):
        ob, orr, oc, rew, st = fn(b[None], 1, np.ones((1, 4), np.uint8), [a])
        assert st[0] == 1 and list(oc[0]) == [1, 1] and ob[0, 0] == 3 and ob[0, 56] == 0
    ob, orr, oc, rew, st = emul.next_state(b[None], 1, np.ones((1, 4), np.uint8), [56 * 64 + 57])   # Ra1-b1: only White in check
    assert st[0] == 0 and list(oc[0]) == [1, 0]


def test_hypothesis_random_boards_movegen_and_next_state():
    """SURVEY.md 8(c)(iii): hypothesis-driven differential test on arbitrary boards (illegal, kingless, many pieces of a
    kind, pawns anywhere): ordered legal / attack lists, update_state and next_state of the device rules == the oracle"""
    from hypothesis import given, settings, strategies as hs

    piece = hs.sampled_from([0, 0, 0, 0, 1, -1, 2, -2, 3, -3, 4, -4, 5, -5, 6, -6])

    @settings(max_examples=300, deadline=None)
    @given(hs.lists(piece, min_size=64, max_size=64), hs.sampled_from([1, -1]), hs.lists(hs.booleans(), min_size=4, max_size=4),
           hs.integers(0, 4100))
    def check(cells, player, rights, action):
        b = np.array(cells, np.int8)[None]
        r = np.array(rights, np.uint8)[None]
        for attack in (False, True):
            out, cnt, _ = emul.movegen(b, player, r, attack)
            exp, ecnt = orc.movegen_batch(b, player, r, attack, stride=out.shape[1])
            assert cnt[0] == ecnt[0] and (out[0, : cnt[0]] == exp[0, : cnt[0]]).all()
        assert all((x == y).all() for x, y in zip(emul.update_state(b, r), orc.update_state_batch(b, r)))
        out, cnt, _ = emul.movegen(b, player, r, False)
        a = int(out[0, action % cnt[0]]) if cnt[0] and action % 3 else action
        assert all((np.asarray(x) == np.asarray(y)).all() for x, y in zip(emul.next_state(b, player, r, [a]), orc.next_state_batch(b, player, r, [a])))

    check()


def test_next_states_of_the_reference_pure_python_env(golden):
    assert ph.check_v1_next_states(emul.next_state, golden["v1_next_states"]) > 3500


def test_v1_castle_through_attack_vector():
    def fn(b, p):
        out, cnt, _ = emul.movegen(b[None], p, np.ones((1, 4), np.uint8), False, castles_only=True)
        return [int(a) for a in out[0, : cnt[0]]]
    ph.check_v1_castle_through_attack_vector(fn)


def test_ordered_pick_equals_the_walk_over_the_directions():
    """nth_target (search over the cumulative direction masks) == the idx-th move emit_piece_moves lists, for every piece
    class, colour, from-square, the class's full reach and 24 random subsets of it, every index."""
    n = emul.lib().emul_nth_target_check(20260101, 24)
    assert n > 40000, n  # (a negative value is -(1 + index of the first mismatching case))
