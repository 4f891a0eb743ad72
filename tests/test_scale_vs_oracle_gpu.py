"""Benchmark-scale sampled runs against the C oracle, env by env.

`bench.py` times `step_sampled(64)` on phase-spread batches: the multi-step tile kernel, split into two env ranges on two
internal streams, with the statistics counters reduced per warp in packed bit fields.  Here 131,149 envs (two ranges for
runs of more than 64 steps; a partial last warp and block) are spread like `BatchedChessEnv.dephase` spreads them and then
stepped through every kernel variant of `gcb_env_step_sampled`.  The same global env ids run on the host threads in
`oracle.SelfplayPool` with the device's Philox draws and auto-reset.  After each segment every env's exported state and
the statistics counters must equal the oracle's exactly.
"""
import os
import time

import numpy as np
import pytest

from oracle import oracle as orc
from tests import parity_helpers as ph

pytestmark = pytest.mark.gpu

N = 131_149  # >= 2 * 65536: runs of more than 64 steps split into two env ranges; N % 32 != 0: a partial last warp
STRIDE = 256  # legal-list columns compared (no position of these games has more legal moves; asserted)
THREADS = os.cpu_count() or 1
ALL_COUNTERS = ("steps", "plies", "episodes", "mates", "repetitions", "caps", "wedged", "invalid", "reward_sum",
                "legal_sum", "in_check")
# in bot modes the device counts the bot's opening ply of an auto-reset inside the step and the oracle does not, so
# plies and the episode-end categories are held to the external-opponent model instead (test_external_opponent_gpu.py)
BOT_COUNTERS = ("steps", "episodes", "invalid", "reward_sum", "legal_sum", "in_check")


class ScalePair:
    """a device batch and the oracle pool of the same global env ids, stepped and reset together"""

    def __init__(self, seed, opponent="none", color="WHITE", env_id_offset=0, boards=None, moves_max=149, history_cap=512):
        from gym_chess_b200 import BatchedChessEnv

        self.env = BatchedChessEnv(N, opponent=opponent, player_color=color, seed=seed, env_id_offset=env_id_offset,
                                   initial_boards=boards, legal_stride=STRIDE, history_cap=history_cap, moves_max=moves_max)
        self.pool = orc.SelfplayPool(seed, env_id_offset, env_id_offset + N, opponent=opponent, player_color=color,
                                     moves_max=moves_max, initial_boards=boards)
        self.offset = env_id_offset
        self.ref = dict.fromkeys(ALL_COUNTERS, 0)
        self.oracle_s = 0.0

    def oracle_run(self, k):
        t0 = time.perf_counter()
        st = self.pool.run(k, THREADS)
        self.oracle_s += time.perf_counter() - t0
        for key in self.ref:
            self.ref[key] += st[key]

    def dephase(self, groups=43, period=301):
        """BatchedChessEnv.dephase on the device (the launches are queued first, so the GPU runs while the host threads
        replay it on the pool)"""
        self.env.dephase(groups, period)
        ids = np.arange(N) + self.offset
        for g in range(groups):
            self.oracle_run(max(1, period // groups))
            self.pool.reset(ids % groups == g)

    def segment(self, k, tag):
        self.env.step_sampled(k)
        self.oracle_run(k)
        self.compare(tag)

    def compare(self, tag):
        ref = self.pool.export(STRIDE)
        assert int(ref[1][:, 9].max()) <= STRIDE, "a legal list is longer than the compared stride"
        ph.check_export_arrays(self.env.export_numpy(), ref, self.offset, tag)
        return ref

    def check_counters(self, names, tag):
        st = self.env.stats()
        diff = {k: (st[k], self.ref[k]) for k in names if st[k] != self.ref[k]}
        assert not diff, "%scounters differ (device, oracle): %s" % (tag, diff)
        assert st["slot_overflow"] == 0 and st["hist_overflow"] == 0, (tag, st)
        assert st["episodes"] == st["mates"] + st["repetitions"] + st["caps"] + st["wedged"], (tag, st)
        return st


def expected_bits(legal, n_legal):
    """the legal_bitmask rows [n, 65] of reference legal lists: bit (a & 63) of word (a >> 6) for every listed action"""
    bits = np.zeros((len(legal), 65), np.uint64)
    rows = np.arange(len(legal))
    for k in range(legal.shape[1]):
        sel = k < n_legal
        if not sel.any():
            break
        a = legal[sel, k].astype(np.int64)
        bits[rows[sel], a >> 6] |= np.left_shift(np.uint64(1), (a & 63).astype(np.uint64))
    return bits


def run_segments(p, counters, long_run=150):
    """Every kernel variant of gcb_env_step_sampled, each followed by a full comparison with the pool:
    1 and 3 steps without a mask output (generic kernel, TILE 0), 2 steps with a registered mask output (TILE 2; the mask
    must equal the reference legal lists), 7 steps (multi-step tile kernel, TILE 1, one launch) and `long_run` steps (more
    than 64: several launches per env range, two ranges)."""
    import torch

    p.check_counters(counters, "after dephase: ")
    p.segment(1, "1 step: ")
    p.segment(3, "3 steps: ")
    bits = torch.full((N, 66), -1, dtype=torch.int64, device=p.env.device)
    p.env.set_mask_output(bits)
    try:
        p.env.step_sampled(2)
        p.oracle_run(2)
        ref = p.compare("2 steps with a mask output: ")
    finally:
        p.env.set_mask_output(None)
    got = bits[:, :65].cpu().numpy().view(np.uint64)
    bad = (got != expected_bits(ref[2], ref[1][:, 9])).any(1)
    assert not bad.any(), "mask output differs from the reference legal lists at env ids %s" % (np.nonzero(bad)[0][:8] + p.offset).tolist()
    p.check_counters(counters, "after 6 steps: ")
    p.segment(7, "7 steps: ")
    p.segment(long_run, "%d steps: " % long_run)
    return p.check_counters(counters, "end: ")


@pytest.mark.parametrize("env_id_offset", [0, 1_000_003])
def test_selfplay_benchmark_workload_matches_oracle(env_id_offset):
    """the bench.py workload: self-play from the default board, seed 2, dephase(); every env and all 11 counters"""
    p = ScalePair(2, env_id_offset=env_id_offset)
    p.dephase()
    st = run_segments(p, ALL_COUNTERS)
    if env_id_offset == 0:
        assert min(st["mates"], st["repetitions"], st["caps"], st["wedged"]) > 0, st
    print("oracle %.1f s, %d threads" % (p.oracle_s, THREADS))


@pytest.mark.parametrize("color", ["WHITE", "BLACK"])
def test_random_bot_matches_oracle(color):
    """the random-bot figures of bench.py: dephase(period=151), the bot drawing on the device"""
    p = ScalePair(2, opponent="random", color=color)
    p.dephase(period=151)
    st = run_segments(p, BOT_COUNTERS)
    assert st["episodes"] > 0, st
    print("oracle %.1f s, %d threads" % (p.oracle_s, THREADS))


def test_endgames_match_oracle():
    """repetition-heavy endgame templates (env g starts from template g % 7), moves_max 250: windows stay below
    history_cap, so the repetition table must see every repetition the oracle's saved boards see"""
    p = ScalePair(5, boards=ph.endgame_boards(), moves_max=250, history_cap=512)
    p.dephase(groups=16, period=256)
    st = run_segments(p, ALL_COUNTERS)
    assert st["repetitions"] > N // 8, st
    print("oracle %.1f s, %d threads" % (p.oracle_s, THREADS))


def test_done_envs_without_auto_reset_match_the_driver():
    """Without auto-reset a done env stays done, and every further step of it ends an episode again with no other event
    (no mate, repetition, cap, wedge or invalid action).  Such a step is the one case in which the warp's rare-event
    counters see only the episodes bit, so this is where a dropped episode would show.  1,031 endgame envs (a partial
    last warp) run 70 steps in two launches of the multi-step tile kernel; OracleEnvs driven step by step with the same
    draws must give the same final state and the same steps / reward_sum / episodes (the tallies the single-step parity
    tests already hold without auto-reset)."""
    from gym_chess_b200 import BatchedChessEnv

    n, seed, boards = 1031, 5, ph.endgame_boards()
    env = BatchedChessEnv(n, opponent="none", seed=seed, auto_reset=False, initial_boards=boards, legal_stride=STRIDE,
                          moves_max=250)
    O = [orc.OracleEnv(boards[i % len(boards)], "WHITE", "none", seed, i, moves_max=250) for i in range(n)]
    env.step_sampled(70)
    tot = dict(steps=0, reward_sum=0, episodes=0)
    for _ in range(70):
        for i, o in enumerate(O):
            ph.oracle_sampled_step(o, seed, i, tot, auto_reset=False)
    ref = ph.oracle_views(O, STRIDE)
    ph.check_export_arrays(env.export_numpy(), ref, 0, "70 steps without auto-reset: ")
    st = env.stats()
    assert {k: st[k] for k in tot} == tot, (st, tot)
    assert (ref[1][:, 7] == 1).sum() > n // 20 and tot["episodes"] > 10 * n // 20, tot
