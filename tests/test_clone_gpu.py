"""Per-env clone on the GPU (gcb_env_clone / BatchedChessEnv.clone_from, kernel k_env_clone): against the oracle, at full
size against the source envs themselves, in-object, with a registered mask output, argument checks, and the memory-safety
net (guard regions, CHECKED build) in a subprocess."""
import numpy as np
import pytest

from tests import clone_helpers as ch
from tests import memsafety_exercise as mx

pytestmark = pytest.mark.gpu
CHK_CLONE_INDEX, CHK_CLONE_ALIAS = 6, 7


class GpuEnv:
    """numpy-facing adapter of BatchedChessEnv (the interface of the host emulation)"""

    def __init__(self, N, **kw):
        from gym_chess_b200 import BatchedChessEnv

        self.N = N
        self.env = BatchedChessEnv(N, **kw)

    @staticmethod
    def _np(res):
        return tuple(x.cpu().numpy() for x in res[:3])

    def step(self, a):
        return self._np(self.env.step(np.asarray(a, np.int32))) + (None, None)

    def step_index(self, u):
        import torch

        return self._np(self.env.step_index(torch.from_numpy(np.asarray(u, np.uint32).view(np.int32)).cuda())) + (None, None)

    def step_sampled(self):
        r, d, f, a, b = self.env.step_sampled(1, record=True)
        return self._np((r, d, f)) + (a[-1].cpu().numpy(), b[-1].cpu().numpy())

    def bot_ply(self, a):
        return self._np(self.env.bot_ply(np.asarray(a, np.int32)))

    def reset(self, mask=None):
        self.env.reset(mask)

    def export(self):
        return self.env.export_numpy()

    def stats(self):
        from gym_chess_b200.batched_env import STAT_NAMES

        s = self.env.stats()
        return np.array([np.int64(s[k]).astype(np.uint64) if k == "reward_sum" else s[k] for k in STAT_NAMES] + [0], np.uint64)

    def clone_from(self, source, index):
        self.env.clone_from(source.env, index)


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_clone_vs_oracle(opponent, color):
    ch.check_clone_vs_oracle(GpuEnv, opponent, color, 2048, np.random.RandomState(5))


def test_clone_external_opponent_continues_like_its_source():
    rng = np.random.RandomState(6)
    kw = dict(opponent="external", player_color="BLACK", auto_reset=False)
    S = GpuEnv(3000, seed=1, **kw)
    ch.drive_pair(S, S, np.full(3000, -1, np.int32), 30, rng, external=True)
    S.step_index(rng.randint(0, 2 ** 32, size=3000, dtype=np.uint64).astype(np.uint32))  # a bot ply is owed now
    D = GpuEnv(3000, seed=2, env_id_offset=5000, **kw)
    idx = rng.permutation(3000).astype(np.int32)
    D.clone_from(S, idx)
    ch.assert_same_rows(S.export(), D.export(), idx)
    ch.drive_pair(S, D, idx, 100, rng, external=True, tag="external ")


def _drive_full(S, D, idx, steps, seed):
    """the same step_index words, gathered by idx, to source rows and clone rows (D may be S): outputs equal at every step"""
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    idx_t = torch.as_tensor(idx, device="cuda").long()
    sel = idx_t >= 0
    src_rows = idx_t[sel]
    for t in range(steps):
        w = torch.randint(-2 ** 31, 2 ** 31 - 1, (S.num_envs,), generator=g, device="cuda", dtype=torch.int64).to(torch.int32)
        if D is S:
            w[sel] = w[src_rows]
            r, d, f = [x.clone() for x in S.step_index(w)]
            outs = ((r, r), (d, d), (f, f))
        else:
            wd = torch.randint(-2 ** 31, 2 ** 31 - 1, (D.num_envs,), generator=g, device="cuda", dtype=torch.int64).to(torch.int32)
            wd[sel] = w[src_rows]
            rs, ds, fs = [x.clone() for x in S.step_index(w)]
            rd, dd, fd = D.step_index(wd)
            outs = ((rs, rd), (ds, dd), (fs, fd))
        for (a, b), name in zip(outs, ("reward", "done", "flags")):
            assert torch.equal(a[src_rows], b[sel]), "step %d: %s differ" % (t, name)
    ch.assert_same_rows(S.export_numpy(), D.export_numpy(), np.asarray(idx))


@pytest.mark.parametrize("fan_out", [False, True])
def test_clone_at_full_size_continues_like_its_source(fan_out):
    import torch
    from gym_chess_b200 import BatchedChessEnv

    N = 524288
    S = BatchedChessEnv(N, opponent="none", seed=1)
    S.dephase()
    D = BatchedChessEnv(N, opponent="none", seed=2, env_id_offset=N)
    if fan_out:  # 4096 roots x 128 clones
        roots = torch.randperm(N, generator=torch.Generator().manual_seed(3))[:4096].to(torch.int32)
        idx = roots.repeat_interleave(128).numpy()
    else:
        idx = np.arange(N, dtype=np.int32)
    assert int(S.info_tensor()[:, 12].max()) > 20
    D.clone_from(S, idx)
    _drive_full(S, D, idx, 300, seed=4)
    _sampled_rows_vs_oracle(D, seed=2, env_id_offset=N)


def _sampled_rows_vs_oracle(D, seed, env_id_offset, rows=64, steps=12):
    """step_sampled on the clone (its own Philox draws) for a sample of rows whose repetition window is empty -- there the
    oracle can take the row over through a state import plus the counters -- against the oracle"""
    from oracle import oracle as orc

    b, info, _ = D.export_numpy()
    pick = np.nonzero((info[:, 12] == 0) & (info[:, 7] == 0) & (info[:, 9] > 0))[0]
    pick = pick[np.linspace(0, len(pick) - 1, rows).astype(np.int64)]
    O = []
    for j in pick:
        o = orc.OracleEnv(seed=seed, env_id=env_id_offset + int(j))
        o.import_state(b[j], int(info[j, 0]), info[j, 1:5], int(info[j, 8]), episode=int(info[j, 10]))
        ch._raw(o).step_in_episode = int(info[j, 11])
        O.append(o)
    for t in range(steps):
        r, d, f = [x.cpu().numpy() for x in D.step_sampled(1)]
        for o, j in zip(O, pick):
            v = o.view()
            rr, dd, _ = o.step(o.pick(orc.draw_u32(seed, env_id_offset + int(j), v["episode"], v["step_in_episode"], 0)))
            assert (rr, dd) == (int(r[j]), bool(d[j])), (t, int(j))
            if dd or o.view()["n_legal"] == 0:
                o.reset(v["episode"] + 1)
    b, info, _ = D.export_numpy()
    for o, j in zip(O, pick):
        v = o.view()
        assert (b[j] == v["board"]).all() and (int(info[j, 10]), int(info[j, 11])) == (v["episode"], v["step_in_episode"]), int(j)


def test_in_object_disjoint_gather_continues_like_its_source():
    from gym_chess_b200 import BatchedChessEnv

    N = 262144
    E = BatchedChessEnv(N, opponent="none", seed=5)
    E.dephase()
    idx = np.full(N, -1, np.int32)
    idx[N // 2:] = np.arange(N // 2)
    E.clone_from(E, idx)
    _drive_full(E, E, idx, 300, seed=6)


def test_registered_mask_output_is_current_after_a_clone():
    import torch
    from gym_chess_b200 import BatchedChessEnv

    S = BatchedChessEnv(5000, opponent="none", seed=1)
    D = BatchedChessEnv(5000, opponent="none", seed=2)
    S.step_sampled(37)
    D.step_sampled(5)
    bits = torch.zeros((5000, 66), dtype=torch.int64, device="cuda")
    D.set_mask_output(bits)
    D.clone_from(S, np.random.RandomState(1).randint(-1, 5000, size=5000))
    assert torch.equal(bits[:, :65], D.legal_bitmask())
    D.set_mask_output(None)


def test_configuration_mismatch_raises_value_error():
    from gym_chess_b200 import BatchedChessEnv
    from gym_chess_b200.boards import endgame_boards

    base = dict(opponent="random", player_color="WHITE", history_cap=512, moves_max=149)
    S = BatchedChessEnv(8, **base)
    for change in (dict(history_cap=256), dict(piece_slots=20), dict(opponent="external"), dict(player_color="BLACK"),
                   dict(moves_max=250)):
        D = BatchedChessEnv(8, **dict(base, **change))
        with pytest.raises(ValueError):
            D.clone_from(S, np.arange(8))
    D = BatchedChessEnv(8, **dict(base, seed=9, env_id_offset=3, auto_reset=False, initial_boards=endgame_boards()[:1]))
    D.clone_from(S, np.arange(8))  # seed, offset, auto_reset and templates may differ
    with pytest.raises(ValueError):
        D.clone_from(S, np.arange(7))
    with pytest.raises(ValueError):
        D.clone_from(S, np.arange(16).reshape(2, 8))


def test_clone_guard_regions_stay_intact():
    res = mx.run()["clone_valid"]
    assert res["guard_bad_bytes"] == 0 and res["violations"] == 0, res


def test_checked_build_reports_no_violation_for_valid_clones():
    res = mx.run("checked")["clone_valid"]
    assert res["checked"] == 1 and res["violations"] == 0 and res["guard_bad_bytes"] == 0, res


def test_checked_build_flags_an_out_of_range_index_and_leaves_the_row():
    res = mx.run("checked")["clone_out_of_range"]
    assert res["checked"] == 1 and res["violations"] == 1 << CHK_CLONE_INDEX and res["untouched"], res
    assert res["guard_bad_bytes"] == 0


def test_checked_build_flags_aliasing():
    res = mx.run("checked")["clone_alias"]
    assert res["checked"] == 1 and res["violations"] == 1 << CHK_CLONE_ALIAS and res["guard_bad_bytes"] == 0, res
