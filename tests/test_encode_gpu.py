"""Network-input encoder on the GPU (gcb_env_encode / BatchedChessEnv.encode / repetition_count, kernel k_env_encode): all
three dtypes against the host emulation stepped with the same draws at 100,003 envs (self-play, random bot with either colour,
external opponent), against the NumPy reference of tests/encode_helpers.py at 301 envs in every opponent mode, the repetition
invariant (plane 18 <=> the next ply reports F_REPETITION) over 524,288 envs, the pure-read guarantee, out= into a slice of a
rollout buffer, clones, argument errors and the memory-safety net (guard regions, CHECKED build) in a subprocess."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import encode_helpers as eh
from tests import external_helpers as xh
from tests import parity_helpers as ph
from tests.host_emul import encode_emul as ee
from tests.test_clone_gpu import GpuEnv
from tests.test_external_opponent_gpu import GpuExternal

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_BIG = 100_003
F_REPETITION, F_CAP = 4, 8
GCB_E_ARG = -2


def _encode_all(env):
    """encode() in all three dtypes; asserts that they hold the same values, bit for bit, and that repetition_count() is
    planes 17 + 18.  -> (uint8 numpy [N, 19, 64], rep numpy [N])"""
    import torch

    N = env.num_envs
    u8, f32, bf = env.encode(torch.uint8), env.encode(torch.float32), env.encode(torch.bfloat16)
    assert tuple(u8.shape) == (N, 19, 8, 8) and int(u8.max()) <= 1
    assert torch.equal(f32, bf.float()) and torch.equal(f32, u8.float())
    assert torch.equal(f32.view(torch.int32), u8.to(torch.int32) * 0x3F800000)  # (no -0.0)
    assert torch.equal(bf.view(torch.int16), u8.to(torch.int16) * 0x3F80)
    rep = env.repetition_count()
    flat = u8.reshape(N, 19, 64)
    assert torch.equal(rep, flat[:, 17, 0] + flat[:, 18, 0])
    assert (flat[:, 12:] == flat[:, 12:, :1]).all()  # planes 12-18 are constant per env
    return flat.cpu().numpy(), rep.cpu().numpy()


class _Pair:
    """a GPU env and its host emulation, driven with the same inputs"""

    def __init__(self, N, **kw):
        from gym_chess_b200 import BatchedChessEnv

        self.g = BatchedChessEnv(N, legal_stride=256, **kw)
        self.h = ee.EmulEnv(N, legal_stride=256, **kw)
        self.N = N

    def compare(self, tag):
        planes, rep = _encode_all(self.g)
        hp, hr = self.h.encode(np.uint8)
        assert (rep == hr).all(), tag
        bad = np.nonzero((planes != hp).any(2))
        assert len(bad[0]) == 0, "%s: %d (env, plane) pairs differ, first %s" % (tag, len(bad[0]), (bad[0][0], bad[1][0]))
        return np.bincount(rep, minlength=3)


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_encode_matches_host_emulation_at_scale(opponent, color):
    P = _Pair(N_BIG, opponent=opponent, player_color=color, seed=41, initial_boards=ph.endgame_boards())
    seen = P.compare("reset")
    done = 0
    for block in (5, 25, 50, 80):
        for _ in range(block):
            P.h.step_sampled()
        P.g.step_sampled(block)
        done += block
        seen += P.compare("after %d steps" % done)
    assert seen[1] >= 5000 and seen[2] >= 300, seen


def test_encode_matches_host_emulation_external_opponent():
    import torch

    P = _Pair(N_BIG, opponent="external", player_color="BLACK", seed=42, initial_boards=ph.endgame_boards())
    rng = np.random.RandomState(42)
    seen = P.compare("reset")
    for c in range(60):
        # the owed bot plies (White's openings at first), then the agent's step from caller words
        _, info, legal = P.h.export()
        acts = legal[np.arange(P.N), rng.randint(0, 1 << 30, size=P.N) % np.maximum(info[:, 9], 1)].astype(np.int32)
        P.h.bot_ply(acts)
        P.g.bot_ply(torch.from_numpy(acts).cuda())
        if c % 10 == 0:
            seen += P.compare("call %d bot ply" % c)
        words = rng.randint(0, 2 ** 32, size=P.N, dtype=np.uint64).astype(np.uint32)
        P.h.step_index(words)
        P.g.step_index(torch.from_numpy(words.view(np.int32)).cuda())
        if c % 10 == 0 or c == 59:
            assert (P.h.export()[1][:, 14] == 1).mean() > 0.5  # most envs owe the bot a ply while they are encoded
            seen += P.compare("call %d step" % c)
    assert seen[1] >= 5000 and seen[2] >= 100, seen


@pytest.mark.parametrize("opponent,color", [("none", "WHITE"), ("random", "WHITE"), ("random", "BLACK")])
def test_encode_matches_reference_301_envs(opponent, color):
    from oracle import oracle as orc

    N, seed = 301, 43
    tb = ph.endgame_boards()
    E = GpuEnv(N, opponent=opponent, player_color=color, seed=seed, initial_boards=tb)
    O = [orc.OracleEnv(tb[i % len(tb)], color, opponent, seed, i) for i in range(N)]
    tot, seen = dict(steps=0, reward_sum=0, episodes=0), np.zeros(3, np.int64)
    for t in range(120):
        ph._run_sampled(E, O, seed, 1, tot, compare_every=20, tag="step %d " % t)
        planes, rep = _encode_all(E.env)
        ref = eh.oracle_reference(O)
        eh.assert_planes(planes, rep, ref[0], ref[1], "step %d: " % t)
        seen += np.bincount(rep, minlength=3)
    assert seen[1] >= 300 and seen[2] >= 20, seen


@pytest.mark.parametrize("color", ["WHITE", "BLACK"])
def test_encode_matches_reference_301_envs_external(color):
    N, seed = 301, 44
    tb = ph.endgame_boards()
    env = GpuExternal(N, player_color=color, seed=seed, auto_reset=True, moves_max=149, initial_boards=tb)
    models = xh.make_models(N, color, seed, True, 149, tb)
    rng = np.random.RandomState(44 + len(color))
    seen, owed_rows = np.zeros(3, np.int64), 0
    for c in range(100):
        xh.run_external(env, models, rng, 1, forms=("step", "index"), compare_every=10, p_bot=0.45, p_reset=0.0)
        planes, rep = _encode_all(env.env)
        ref = eh.model_reference(models)
        eh.assert_planes(planes, rep, ref[0], ref[1], "call %d: " % c)
        owed_rows += sum(m.owed is not None for m in models)
        seen += np.bincount(rep, minlength=3)
    assert owed_rows >= 5000 and seen[1] >= 300 and seen[2] >= 10, (owed_rows, seen)


def test_plane_18_predicts_the_repetition_at_scale():
    """524,288 self-play envs from the endgame templates, auto-reset on: for every step that did not stop at the move cap,
    the step reports F_REPETITION exactly when plane 18 was set before it"""
    import torch

    from gym_chess_b200 import BatchedChessEnv

    N = 524_288
    env = BatchedChessEnv(N, opponent="none", seed=45, initial_boards=ph.endgame_boards())
    buf = torch.empty(N, 19, 8, 8, dtype=torch.uint8, device="cuda")
    mismatch = torch.zeros((), dtype=torch.int64, device="cuda")
    reps = torch.zeros((), dtype=torch.int64, device="cuda")
    for t in range(240):
        p18 = env.encode(torch.uint8, out=buf)[:, 18, 0, 0] != 0
        _, _, f = env.step_sampled(1)
        live = (f & F_CAP) == 0
        rep = (f & F_REPETITION) != 0
        mismatch += ((rep != p18) & live).sum()
        reps += rep.sum()
    assert int(mismatch) == 0 and int(reps) >= 5000, (int(mismatch), int(reps))


def test_encode_is_a_pure_read():
    import torch

    from gym_chess_b200 import BatchedChessEnv

    N = 4099
    kw = dict(opponent="random", seed=46, initial_boards=ph.endgame_boards())
    env, twin = BatchedChessEnv(N, **kw), BatchedChessEnv(N, **kw)
    bits = torch.zeros(N, 66, dtype=torch.int64, device="cuda")
    env.set_mask_output(bits)
    env.step_sampled(30)
    twin.step_sampled(30)
    before, mask, stats = env.export_numpy(), bits.clone(), env.stats()
    first = [env.encode(dt) for dt in (torch.float32, torch.bfloat16, torch.uint8)] + [env.repetition_count()]
    second = [env.encode(dt) for dt in (torch.float32, torch.bfloat16, torch.uint8)] + [env.repetition_count()]
    torch.cuda.synchronize()
    assert all(torch.equal(a.view(torch.uint8), b.view(torch.uint8)) for a, b in zip(first, second))
    assert torch.equal(bits, mask) and env.stats() == stats
    assert all((p == q).all() for p, q in zip(before, env.export_numpy()))
    # the next sampled step (Philox counters included) is that of a twin that never encoded
    for _ in range(3):
        a = [x.clone() for x in env.step_sampled(1, record=True)]
        b = [x.clone() for x in twin.step_sampled(1, record=True)]
        assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("dtype_name", ["float32", "bfloat16", "uint8"])
def test_encode_into_a_slice_of_a_rollout_buffer(dtype_name):
    import torch

    from gym_chess_b200 import BatchedChessEnv

    dt = getattr(torch, dtype_name)
    N = 4097
    env = BatchedChessEnv(N, opponent="none", seed=47, initial_boards=ph.endgame_boards())
    env.step_sampled(50)
    buf = torch.full((3, N, 19, 8, 8), 7, dtype=dt, device="cuda")
    sentinel = buf[0].clone()
    for t in range(3):
        res = env.encode(dt, out=buf[1])
        assert res.data_ptr() == buf[1].data_ptr()
        assert torch.equal(buf[0], sentinel) and torch.equal(buf[2], sentinel)
        assert torch.equal(buf[1], env.encode(dt))
        env.step_sampled(5)


def test_clone_encodes_like_its_source():
    import torch

    from gym_chess_b200 import BatchedChessEnv

    kw = dict(opponent="none", seed=48, initial_boards=ph.endgame_boards(), history_cap=64, moves_max=250)
    src = BatchedChessEnv(4096, **kw)
    for rnd in range(3):
        src.step_sampled(40)
        src.reset(torch.rand(4096, device="cuda") < 0.2)
    src.step_sampled(20)
    child = BatchedChessEnv(65_536, **dict(kw, seed=49, env_id_offset=10_000))
    idx = torch.randint(0, 4096, (65_536,), dtype=torch.int32, device="cuda")
    child.clone_from(src, idx)
    for dt in (torch.float32, torch.bfloat16, torch.uint8):
        assert torch.equal(child.encode(dt), src.encode(dt)[idx.long()])
    rep = child.repetition_count()
    assert torch.equal(rep, src.repetition_count()[idx.long()])
    assert int((rep == 1).sum()) >= 100 and int((rep == 2).sum()) >= 1


def test_argument_errors():
    import torch

    from gym_chess_b200 import BatchedChessEnv, _lib

    N = 64
    env = BatchedChessEnv(N, opponent="none", seed=50)
    for dt in (torch.float16, torch.int32, torch.float64, "float32", None):
        with pytest.raises(ValueError):
            env.encode(dt)
    raw = torch.empty(N * 19 * 64 * 4 + 64, dtype=torch.uint8, device="cuda")
    bad = [torch.empty(N, 19, 8, 8, dtype=torch.bfloat16, device="cuda"),            # dtype differs from the argument
           torch.empty(N + 1, 19, 8, 8, device="cuda"), torch.empty(N, 19, 64, device="cuda"),
           torch.empty(N, 18, 8, 8, device="cuda"), torch.empty(N, 19, 8, 8),       # host memory
           torch.empty(N, 19, 8, 16, device="cuda")[..., ::2],                        # not contiguous
           torch.empty(19, N, 8, 8, device="cuda").transpose(0, 1),
           raw[4:4 + N * 19 * 64 * 4].view(torch.float32).view(N, 19, 8, 8),          # 4-byte but not 16-byte aligned
           np.zeros((N, 19, 8, 8), np.float32)]
    for out in bad:
        with pytest.raises(ValueError):
            env.encode(torch.float32, out=out)
    with pytest.raises(ValueError):
        env.encode(torch.uint8, out=raw[1:1 + N * 19 * 64].view(N, 19, 8, 8))
    L, s = _lib.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)
    good = torch.empty(N, 19, 8, 8, device="cuda")
    rep = torch.empty(N, dtype=torch.uint8, device="cuda")
    p, r = C.c_void_p(good.data_ptr()), C.c_void_p(rep.data_ptr())
    for dt in (-1, 3, 7):
        assert L.gcb_env_encode(env._h, p, dt, r, s) == GCB_E_ARG
    assert L.gcb_env_encode(env._h, None, 0, None, s) == GCB_E_ARG
    for off in (1, 4, 8):
        assert L.gcb_env_encode(env._h, C.c_void_p(raw.data_ptr() + off), 0, None, s) == GCB_E_ARG
    assert L.gcb_env_encode(env._h, p, 0, None, s) == 0 and L.gcb_env_encode(env._h, None, 2, r, s) == 0
    torch.cuda.synchronize()
    assert torch.equal(good, env.encode()) and torch.equal(rep, env.repetition_count())


def _memsafety(variant=None):
    from gym_chess_b200 import _lib

    env = dict(os.environ)
    if variant:
        env["GYMCHESS_B200_LIB"] = _lib.build(variant=variant)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "encode_memsafety.py")], env=env,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_encode_guard_regions_stay_intact():
    res = _memsafety()
    assert res["guard_bad_bytes"] == 0 and res["out_guard_bad"] == 0 and res["violations"] == 0, res


def test_checked_build_reports_no_violation_for_encodes():
    res = _memsafety("checked")
    assert res["checked"] == 1 and res["violations"] == 0 and res["guard_bad_bytes"] == 0 and res["out_guard_bad"] == 0, res
