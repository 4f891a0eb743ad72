"""Policy sampling (gcb_env_sample_policy / BatchedChessEnv.sample_policy) on the host emulation: env_policy_sample_one of
env_core.cuh compiled with g++ (tests/host_emul/host_emul.cpp), checked against the float64 reference of
tests/policy_helpers.py on oracle self-play, golden and crafted positions.  The same checks on the GPU are in
test_policy_gpu.py."""
import numpy as np
import pytest

from tests import parity_helpers as ph
from tests import policy_helpers as ph_pol
from tests.host_emul import emul

RESIGN = 4100


def _imported(boards, players, rights, seed=3, **kw):
    E = emul.EmulEnv(len(boards), opponent="none", seed=seed, auto_reset=False, **kw)
    E.set_state(boards, players, rights)
    return E


def _golden_env():
    pos = ph.load_golden()["positions"]
    boards = np.array([p["board"] for p in pos], np.int8)
    rights = np.array([p["rights"] for p in pos], np.uint8)
    players = np.where(np.arange(len(pos)) % 2 == 0, 1, -1).astype(np.int8)
    return _imported(boards, players, rights)


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_policy_matches_reference_on_selfplay(opponent, color):
    E = emul.EmulEnv(256, opponent=opponent, player_color=color, seed=11, env_id_offset=1000)
    rng = np.random.RandomState(2)
    for k in range(6):  # positions from several phases, both sides to move (the step count varies per env)
        for _ in range(int(rng.randint(3, 25))):
            E.step_sampled()
        exc = ph_pol.check_env(E, 11, 1000, rng, tag="step block %d: " % k)
        assert exc <= 3


def test_policy_matches_reference_on_golden_positions():
    E = _golden_env()
    info = E.export()[1]
    assert (info[:, 0] == -1).any() and (info[:, 0] == 1).any() and (info[:, 13] != 0).any()  # both colours, castles
    ph_pol.check_env(E, 3, 0, np.random.RandomState(4))


def test_policy_matches_reference_with_more_than_16_pieces():
    """crafted boards with 24 and 28 white pieces (more than 255 legal moves): slots beyond 16, many rounds of 32"""
    boards = ph.queen_heavy_boards()
    E = emul.EmulEnv(8, opponent="none", seed=5, initial_boards=boards, auto_reset=False)
    info = E.export()[1]
    assert (info[:, 9] > 255).all()
    ph_pol.check_env(E, 5, 0, np.random.RandomState(6))


def test_greedy_takes_the_argmax_and_the_lowest_code_of_a_tie():
    E = _golden_env()
    boards, info, _ = E.export()
    codes, cnt = ph_pol.legal_codes(boards, info)
    N = len(cnt)
    rng = np.random.RandomState(7)
    x = rng.standard_normal((N, 4101)).astype(np.float32) - 10
    # force a tie of the top value on two legal entries (bf16 makes ties common): the lower code must win
    for e in np.nonzero(cnt >= 2)[0]:
        i, j = sorted(rng.choice(cnt[e], 2, replace=False))
        x[e, codes[e, i]] = x[e, codes[e, j]] = 5.0
    bits = ph_pol.bf16_bits(x)
    for inp in (x, bits):
        act, logp = E.sample_policy(inp, 0.0)
        xv = x if inp is x else ph_pol.bf16_values(bits)
        ph_pol.compare(act, logp, xv, codes, cnt, 0.0, None)
        top = np.where(cnt >= 2)[0]
        assert all(xv[e, act[e]] == 5.0 for e in top)
        assert (logp == 0).all()


def test_minus_inf_is_never_chosen_and_all_minus_inf_resigns():
    E = _golden_env()
    boards, info, _ = E.export()
    codes, cnt = ph_pol.legal_codes(boards, info)
    N = len(cnt)
    rng = np.random.RandomState(8)
    x = (rng.standard_normal((N, 4101)) * 3).astype(np.float32)
    masked = np.zeros((N, 4101), bool)
    for e in range(N):  # -inf on all legal entries but one (or all of them for every 5th env)
        keep = -1 if e % 5 == 0 or cnt[e] == 0 else codes[e, rng.randint(cnt[e])]
        for a in codes[e, : cnt[e]]:
            if a != keep:
                masked[e, a] = True
    x[masked] = -np.inf
    words = rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32)
    for T in (0.0, 1.0):
        act, logp = E.sample_policy(x, T, words)
        ph_pol.compare(act, logp, x, codes, cnt, T, words)
        all_masked = (np.arange(N) % 5 == 0) | (cnt == 0)
        assert (act[all_masked] == RESIGN).all() and (logp[all_masked] == 0).all()
        assert not masked[np.arange(N)[~all_masked], act[~all_masked]].any()
        if T:
            assert np.abs(logp[~all_masked]).max() < 1e-5  # a single finite entry: probability 1


def test_no_legal_move_resigns():
    """mate and stalemate positions: RESIGN with logp 0, at every temperature"""
    K, k, Q = 1, -1, 2
    mate = np.zeros(64, np.int8)
    mate[0], mate[9], mate[17] = k, Q, K   # black king a8, white queen b7 guarded by the king on b6: mate
    stale = np.zeros(64, np.int8)
    stale[0], stale[10], stale[17] = k, Q, K   # black king a8, white queen c7, king b6: stalemate
    E = _imported(np.stack([mate, stale]), np.array([-1, -1], np.int8), np.zeros((2, 4), np.uint8))
    assert (E.export()[1][:, 9] == 0).all()
    for T in (0.0, 0.5, 1.0):
        act, logp = E.sample_policy(np.zeros((2, 4101), np.float32), T)
        assert (act == RESIGN).all() and (logp == 0).all()


def test_only_legal_entries_are_read():
    """NaN / +inf / 1e30 written into every illegal entry leaves the outputs bit-identical"""
    E = _golden_env()
    boards, info, _ = E.export()
    codes, cnt = ph_pol.legal_codes(boards, info)
    N = len(cnt)
    rng = np.random.RandomState(9)
    x = (rng.standard_normal((N, 4101)) * 3).astype(np.float32)
    legal = np.zeros((N, 4101), bool)
    for e in range(N):
        legal[e, codes[e, : cnt[e]]] = True
    words = rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32)
    for junk in (np.nan, np.inf, 1e30):
        y = x.copy()
        y[~legal] = junk
        for T in (0.0, 0.5, 1.0):
            for w in (words, None):
                a0, l0 = E.sample_policy(x, T, w)
                a1, l1 = E.sample_policy(y, T, w)
                assert (a0 == a1).all() and (l0.view(np.uint32) == l1.view(np.uint32)).all(), (junk, T)
                b0 = E.sample_policy(ph_pol.bf16_bits(x), T, w)
                b1 = E.sample_policy(ph_pol.bf16_bits(y), T, w)
                assert (b0[0] == b1[0]).all() and (b0[1].view(np.uint32) == b1[1].view(np.uint32)).all(), (junk, T)


def test_bf16_is_the_fp32_result_on_the_rounded_values():
    E = _golden_env()
    rng = np.random.RandomState(10)
    x = (rng.standard_normal((E.N, 4101)) * 3).astype(np.float32)
    bits = ph_pol.bf16_bits(x)
    words = rng.randint(0, 2 ** 32, size=E.N, dtype=np.uint64).astype(np.uint32)
    for T in (0.0, 0.5, 1.0, 2.0):
        for w in (words, None):
            a0, l0 = E.sample_policy(bits, T, w)
            a1, l1 = E.sample_policy(ph_pol.bf16_values(bits), T, w)
            assert (a0 == a1).all() and (l0.view(np.uint32) == l1.view(np.uint32)).all()


def test_padded_row_stride():
    E = _golden_env()
    rng = np.random.RandomState(11)
    x = (rng.standard_normal((E.N, 4101)) * 3).astype(np.float32)
    pad = np.full((E.N, 4160), np.nan, np.float32)
    pad[:, :4101] = x
    words = rng.randint(0, 2 ** 32, size=E.N, dtype=np.uint64).astype(np.uint32)
    for T in (0.0, 1.0):
        a0, l0 = E.sample_policy(x, T, words)
        a1, l1 = E.sample_policy(pad, T, words)
        assert (a0 == a1).all() and (l0.view(np.uint32) == l1.view(np.uint32)).all()
        pb = np.zeros((E.N, 4160), np.uint16)
        pb[:, :4101] = ph_pol.bf16_bits(x)
        assert (E.sample_policy(pb, T, words)[0] == E.sample_policy(ph_pol.bf16_bits(x), T, words)[0]).all()


def test_sampling_is_a_pure_read():
    E = emul.EmulEnv(64, opponent="random", seed=12)
    for _ in range(9):
        E.step_sampled()
    before = E.export(), E.stats()
    x = (np.random.RandomState(12).standard_normal((64, 4101)) * 3).astype(np.float32)
    a0, l0 = E.sample_policy(x, 1.0)
    a1, l1 = E.sample_policy(x, 1.0)
    assert (a0 == a1).all() and (l0 == l1).all()
    after = E.export(), E.stats()
    assert all((p == q).all() for p, q in zip(before[0], after[0])) and (before[1] == after[1]).all()
