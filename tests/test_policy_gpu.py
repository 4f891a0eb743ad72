"""Policy sampling on the GPU (gcb_env_sample_policy / BatchedChessEnv.sample_policy / step_policy, kernel
k_env_policy_sample): against the float64 reference of tests/policy_helpers.py at ~100k envs (self-play, random bot with
either agent colour, external opponent for both the agent and the owed bot ply), determinism and sharding invariance,
step_policy against sample_policy + step, the sampled distribution at 1,048,576 draws, argument errors, a registered mask
output, and the memory-safety net (guard regions, CHECKED build) in a subprocess."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import policy_helpers as pp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_BIG = 100_003
F_BOT_PENDING = 64


def _torch_logits(x):
    import torch

    if x.dtype == np.uint16:
        return torch.from_numpy(x.view(np.int16)).cuda().view(torch.bfloat16)
    return torch.from_numpy(x).cuda()


class GpuEnv:
    """numpy-facing adapter of BatchedChessEnv for tests/policy_helpers.py"""

    def __init__(self, env):
        self.env, self.N = env, env.num_envs

    def export(self):
        return self.env.export_numpy()

    def sample_policy(self, x, T, u32=None):
        import torch

        u = None if u32 is None else torch.from_numpy(np.asarray(u32, np.uint32).view(np.int32)).cuda()
        a, lp = self.env.sample_policy(_torch_logits(x), T, u)
        return a.cpu().numpy(), lp.cpu().numpy()


def _randn(seed):
    import torch

    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return lambda n: torch.randn(n, 4101, generator=g, device="cuda").cpu().numpy()


def _env(N, **kw):
    from gym_chess_b200 import BatchedChessEnv

    return BatchedChessEnv(N, **kw)


def test_policy_matches_reference_phase_spread_selfplay():
    env = _env(N_BIG, opponent="none", seed=21, env_id_offset=7)
    env.dephase(groups=13, period=130)
    exc = pp.check_env(GpuEnv(env), 21, 7, np.random.RandomState(1), randn=_randn(1))
    assert exc <= N_BIG // 1000


@pytest.mark.parametrize("color", ["WHITE", "BLACK"])
def test_policy_matches_reference_vs_random_bot(color):
    env = _env(N_BIG, opponent="random", player_color=color, seed=22)
    env.step_sampled(37)
    pp.check_env(GpuEnv(env), 22, 0, np.random.RandomState(2), temperatures=(1.0,), randn=_randn(2))


def _check_once(E, seed, T, rng, randn):
    boards, info, _ = E.export()
    codes, cnt = pp.legal_codes(boards, info)
    x = randn(E.N) * np.float32(3)
    act, logp = E.sample_policy(x, T)
    pp.compare(act, logp, x, codes, cnt, T, pp.philox_words(seed, 0, info))
    return act, info


@pytest.mark.parametrize("color", ["WHITE", "BLACK"])
def test_policy_serves_agent_and_external_bot(color):
    """opponent "external": while most envs owe a bot ply the sample is the bot's (the side to move) and goes to bot_ply,
    otherwise it is the agent's and goes to step; every draw is checked against the reference"""
    import torch

    env = _env(N_BIG, opponent="external", player_color=color, seed=23)
    E, rng, randn = GpuEnv(env), np.random.RandomState(3), _randn(3)
    bot_side = 1 if color == "BLACK" else -1
    plies = {"agent": 0, "bot": 0}
    for k in range(12):
        act, info = _check_once(E, 23, (1.0, 0.5, 0.0)[k % 3], rng, randn)
        owed = info[:, 14] == 1
        assert (info[owed, 0] == bot_side).all() and (info[~owed, 0] == -bot_side).all()
        if owed.mean() > 0.5:
            env.bot_ply(torch.from_numpy(act).cuda())  # (rows that owe nothing are left alone)
            plies["bot"] += 1
        else:
            env.step(torch.from_numpy(act).cuda())
            plies["agent"] += 1
    assert plies["agent"] >= 5 and plies["bot"] >= 5, plies


def test_policy_is_deterministic_and_sharding_invariant():
    import torch

    N = 65_536
    x = torch.randn(N, 4101, device="cuda") * 3
    a = _env(N, opponent="random", seed=24)
    b1, b2 = _env(N // 2, opponent="random", seed=24), _env(N // 2, opponent="random", seed=24, env_id_offset=N // 2)
    for e in (a, b1, b2):
        e.step_sampled(25)
    for T in (0.0, 0.5, 1.0):
        r1, r2 = a.sample_policy(x, T), a.sample_policy(x, T)
        assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1].view(torch.int32), r2[1].view(torch.int32))
        s1, s2 = b1.sample_policy(x[: N // 2], T), b2.sample_policy(x[N // 2:], T)
        assert torch.equal(torch.cat([s1[0], s2[0]]), r1[0])
        assert torch.equal(torch.cat([s1[1], s2[1]]).view(torch.int32), r1[1].view(torch.int32))


def test_step_policy_equals_sample_then_step():
    import torch

    N = 65_536
    src = _env(N, opponent="random", seed=25)
    src.step_sampled(40)
    c1, c2 = _env(N, opponent="random", seed=26), _env(N, opponent="random", seed=26)
    idx = torch.arange(N, device="cuda", dtype=torch.int32)
    c1.clone_from(src, idx)
    c2.clone_from(src, idx)
    for k in range(5):
        x = (torch.randn(N, 4101, device="cuda") * 2).to(torch.bfloat16 if k % 2 else torch.float32)
        a1, l1, r1, d1, f1 = c1.step_policy(x, 1.0)
        a2, l2 = c2.sample_policy(x, 1.0)
        r2, d2, f2 = c2.step(a2)
        assert torch.equal(a1, a2) and torch.equal(l1.view(torch.int32), l2.view(torch.int32))
        assert torch.equal(r1, r2) and torch.equal(d1, d2) and torch.equal(f1, f2)
        assert all((p == q).all() for p, q in zip(c1.export_numpy(), c2.export_numpy()))


@pytest.mark.parametrize("T", [1.0, 0.5])
def test_sampled_distribution_is_the_softmax(T):
    """one position fanned out to 1,048,576 rows (each row its own env id, so its own Philox words), one draw per row:
    chi-square against the softmax over the legal set"""
    import torch
    from scipy import stats

    src = _env(1, opponent="none", seed=27, history_cap=8)
    src.step_sampled(9)
    N = 1 << 20
    fan = _env(N, opponent="none", seed=28, history_cap=8)
    fan.clone_from(src, torch.zeros(N, dtype=torch.int32, device="cuda"))
    boards, info, _ = src.export_numpy()
    codes, cnt = pp.legal_codes(boards, info)
    L = codes[0, : cnt[0]]
    assert len(L) >= 10
    g = torch.Generator(device="cuda")
    g.manual_seed(29)
    row = torch.randn(4101, generator=g, device="cuda")
    x = row.expand(N, 4101).contiguous()
    act, _ = fan.sample_policy(x, T)
    counts = torch.bincount(act.long(), minlength=4101).cpu().numpy()
    assert counts.sum() == N and counts[L].sum() == N
    z = row.cpu().numpy().astype(np.float64)[L] / T
    p = np.exp(z - z.max())
    p /= p.sum()
    exp = p * N
    keep = exp >= 5
    obs = np.append(counts[L][keep], counts[L][~keep].sum())
    e = np.append(exp[keep], exp[~keep].sum())
    if e[-1] == 0:
        obs, e = obs[:-1], e[:-1]
    assert stats.chisquare(obs, e).pvalue > 1e-3


def test_argument_errors():
    import torch

    from gym_chess_b200 import _lib

    N = 64
    env = _env(N, opponent="none", seed=30)
    good = torch.randn(N, 4101, device="cuda")
    bad = [torch.randn(N + 1, 4101, device="cuda"), torch.randn(N, 4100, device="cuda"), torch.randn(N, 4101, 1, device="cuda"),
           torch.randn(N, 4101, device="cuda").half(), torch.zeros(N, 4101, dtype=torch.int32, device="cuda"),
           torch.randn(N, 4101), torch.randn(N, 8202, device="cuda")[:, ::2], torch.randn(4101, N, device="cuda").t(),
           good.cpu().numpy()]
    for x in bad:
        with pytest.raises(ValueError):
            env.sample_policy(x)
    for T in (-1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            env.sample_policy(good, T)
    with pytest.raises(ValueError):
        env.sample_policy(good, 1.0, torch.zeros(N + 1, dtype=torch.int32, device="cuda"))
    a = torch.empty(N, dtype=torch.int32, device="cuda")
    L, p = _lib.lib(), C.c_void_p(good.data_ptr())
    GCB_E_ARG = -2
    assert L.gcb_env_sample_policy(env._h, p, 2, 4101, 1.0, None, C.c_void_p(a.data_ptr()), None, None) == GCB_E_ARG
    assert L.gcb_env_sample_policy(env._h, p, 0, 4100, 1.0, None, C.c_void_p(a.data_ptr()), None, None) == GCB_E_ARG
    assert L.gcb_env_sample_policy(env._h, p, 0, 4101, -0.5, None, C.c_void_p(a.data_ptr()), None, None) == GCB_E_ARG
    assert L.gcb_env_sample_policy(env._h, p, 0, 4101, float("inf"), None, C.c_void_p(a.data_ptr()), None, None) == GCB_E_ARG
    assert L.gcb_env_sample_policy(env._h, p, 0, 4101, 1.0, None, None, None, None) == GCB_E_ARG
    assert L.gcb_env_sample_policy(env._h, p, 0, 4101, 1.0, None, C.c_void_p(a.data_ptr()), None, None) == 0  # logp may be NULL
    torch.cuda.synchronize()
    assert ((a >= 0) & (a <= 4100)).all()


def test_sample_is_a_pure_read_of_state_statistics_and_mask_output():
    import torch

    N = 4099
    env = _env(N, opponent="random", seed=31)
    bits = torch.zeros(N, 66, dtype=torch.int64, device="cuda")
    env.set_mask_output(bits)
    env.step_sampled(12)
    before, mask, stats = env.export_numpy(), bits.clone(), env.stats()
    for T in (0.0, 1.0):
        env.sample_policy(torch.randn(N, 4101, device="cuda"), T)
    torch.cuda.synchronize()
    assert torch.equal(bits, mask) and env.stats() == stats
    assert all((p == q).all() for p, q in zip(before, env.export_numpy()))


def _memsafety(variant=None):
    from gym_chess_b200 import _lib

    env = dict(os.environ)
    if variant:
        env["GYMCHESS_B200_LIB"] = _lib.build(variant=variant)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "policy_memsafety.py")], env=env,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_policy_guard_regions_stay_intact():
    res = _memsafety()
    assert res["guard_bad_bytes"] == 0 and res["out_guard_bad"] == 0 and res["violations"] == 0, res


def test_checked_build_reports_no_violation_for_policy_samples():
    res = _memsafety("checked")
    assert res["checked"] == 1 and res["violations"] == 0 and res["guard_bad_bytes"] == 0 and res["out_guard_bad"] == 0, res
