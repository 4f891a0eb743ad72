"""The memory-safety net of the env API (DESIGN.md section 3.8): named scenarios drive the env kernels on awkward env counts
with guard regions around every env array (GCB_GUARD_BYTES) and -- when GYMCHESS_B200_LIB points at the CHECKED build --
index checks compiled into the kernels.

`python tests/memsafety_exercise.py <scenario> ...` runs the scenarios one after the other in one process and prints one
JSON object keyed by scenario: {"checked": 0|1, "violations": bit set of failed index checks, "guard_bad_bytes": n, ...the
scenario's own fields}.  run(variant) does that in a subprocess for the scenarios of one build, once per test session; the
GPU tests (test_memory_safety.py, test_clone_gpu.py, test_policy_gpu.py, test_encode_gpu.py) assert on its entries."""
import ctypes as C
import functools
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gym_chess_b200 import BatchedChessEnv, _lib  # noqa: E402
from gym_chess_b200.boards import endgame_boards  # noqa: E402

# the scenarios of each build: None = the product library, otherwise a gym_chess_b200._lib.VARIANTS build
BUILDS = {
    None: ("steps", "clone_valid", "policy", "encode"),
    "checked": ("steps", "clone_valid", "policy", "encode", "clone_out_of_range", "clone_alias"),
    "checked_selftest": ("steps_quick",),
}


@functools.lru_cache(maxsize=None)
def run(variant=None):
    """the scenarios of BUILDS[variant] in one subprocess on that build -> {scenario: its result}"""
    env = dict(os.environ)
    if variant:
        env["GYMCHESS_B200_LIB"] = _lib.build(variant=variant)
    out = subprocess.run([sys.executable, os.path.abspath(__file__)] + list(BUILDS[variant]), env=env, capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def _guarded(n, dtype, guard, fill):
    """an output vector of n elements between two guard regions of `guard` elements, all filled with `fill`
    -> (the whole buffer, the vector, a function counting the guard elements that changed)"""
    buf = torch.full((n + 2 * guard,), fill, dtype=dtype, device="cuda")
    return buf, buf[guard:guard + n], lambda: int((buf[:guard] != fill).sum() + (buf[guard + n:] != fill).sum())


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _steps(envs, sizes, quick=False):
    """every step form, the exports, masks, resets, imports and snapshots in all five opponent / colour / template
    configurations (quick: self-play only)"""
    rng = np.random.RandomState(1)
    for N in sizes:
        for kw in (dict(opponent="none"), dict(opponent="random"), dict(opponent="random", player_color="BLACK"),
                   dict(opponent="external", player_color="BLACK"),
                   dict(opponent="none", initial_boards=endgame_boards(), history_cap=8, moves_max=250)):
            if quick and kw.get("opponent") != "none":
                continue
            env = BatchedChessEnv(N, seed=3, **kw)
            envs.append(env)
            if kw["opponent"] == "external":
                env.bot_ply(torch.full((N,), 3364, dtype=torch.int32))          # e2e4 for every env
                legal, cnt = env.legal_actions()
                env.step(legal[:, 0].to(torch.int32) & 0xFFFF)
                env.bot_ply(torch.full((N,), 3299, dtype=torch.int32))          # d2d4
            else:
                env.step_sampled(1)
                env.step_sampled(70)                                             # two launches, multi-step kernel
                legal, cnt = env.legal_actions()
                acts = (legal[:, 0].to(torch.int32) & 0xFFFF)
                acts[::7] = 4100                                                 # some invalid actions
                env.step(acts)
                env.step_index(torch.from_numpy(rng.randint(0, 2 ** 31, size=N).astype(np.int32)).cuda())
                env.step_index_host(rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32))   # pageable: staged chunks
                pin16 = torch.zeros(N, dtype=torch.int16).pin_memory()
                out16 = torch.zeros(N, dtype=torch.int16).pin_memory()
                env.step_index_packed(pin16, out16)
                env.wait()
            env.observe(), env.info_tensor(), env.legal_bitmask(), env.legal_actions()
            if N <= 70001:
                env.legal_mask()
            m = (torch.arange(N, device="cuda") % 3 == 0).to(torch.uint8)
            env.reset(m)
            b = env.observe().reshape(N, 64)
            info = env.info_tensor()
            env.set_state(b, info[:, 0].to(torch.int8), info[:, 1:5].to(torch.uint8), None, m)
            snap = env.snapshot()
            env.step_sampled(3) if kw["opponent"] != "external" else None
            env.restore(snap)
            env.stats()


# the configurations of the clone, policy and encode scenarios, each at 1, 33 and 4097 envs
FEATURE_CONFIGS = (dict(opponent="none"), dict(opponent="random", player_color="BLACK"),
                   dict(opponent="none", initial_boards=endgame_boards(), history_cap=8, moves_max=250))


def _clone_valid(envs):
    """cross-object clones (identity, fan-out, -1 rows, another env count) and an in-object disjoint gather, each followed by
    steps"""
    rng = np.random.RandomState(1)
    for N in (1, 33, 4097):
        for kw in FEATURE_CONFIGS:
            S = BatchedChessEnv(N, seed=3, **kw)
            S.step_sampled(40)
            for M in (N, 2 * N + 1):
                D = BatchedChessEnv(M, seed=4, env_id_offset=N, **kw)
                D.clone_from(S, np.arange(M) % N)
                idx = rng.randint(-1, N, size=M)
                D.clone_from(S, idx)
                D.step_sampled(5)
                envs.append(D)
            idx = np.full(N, -1)
            idx[N // 2 + N % 2:] = np.arange(N // 2)
            S.clone_from(S, idx)
            S.step_sampled(3)
            envs.append(S)


def _clone_source(envs):
    """4097 self-play envs 20 steps into their games"""
    S =BatchedChessEnv(4097, opponent="none", seed=3)
    envs.append(S)
    S.step_sampled(20)
    S.export_numpy()
    return S


def _clone_out_of_range(envs):
    """one index >= the source's env count: that row must be left untouched (CHK_CLONE_INDEX in the checked build)"""
    S = _clone_source(envs)
    N = S.num_envs
    D = BatchedChessEnv(N, opponent="none", seed=4)
    envs.append(D)
    D.step_sampled(7)
    before = D.export_numpy()
    idx = np.full(N, -1)
    idx[100] = N + 5
    D.clone_from(S, idx)
    after = D.export_numpy()
    return dict(untouched=all(bool((a == b).all()) for a, b in zip(before, after)))


def _clone_alias(envs):
    """an in-object index vector whose destination rows are also source rows (CHK_CLONE_ALIAS in the checked build)"""
    S = _clone_source(envs)
    idx = np.full(S.num_envs, -1)
    idx[10], idx[20] = 20, 30  # row 20 is a destination and the source of row 10
    S.clone_from(S, idx)


def _policy(envs):
    """fp32 and bf16 logits with padded rows, every temperature form, caller and Philox words, guard regions around the
    caller's output vectors"""
    L, G, out_bad = _lib.lib(), 1024, 0
    torch.manual_seed(1)
    for N in (1, 33, 4097):
        for kw in FEATURE_CONFIGS:
            env = BatchedChessEnv(N, seed=3, **kw)
            envs.append(env)
            env.step_sampled(30)
            for dt in (torch.float32, torch.bfloat16):
                x = torch.randn(N, 4160, device="cuda").mul_(3).to(dt)[:, :4101]
                words = torch.randint(0, 2 ** 31, (N,), dtype=torch.int32, device="cuda")
                for T in (0.0, 0.5, 1.0):
                    for w in (words, None):
                        _, act, act_bad = _guarded(N, torch.int32, G, 0x5A5A5A5A)
                        _, logp, logp_bad = _guarded(N, torch.float32, G, 7.25)
                        _lib.check(L.gcb_env_sample_policy(env._h, _ptr(x), int(dt == torch.bfloat16), 4160, T,
                                                           None if w is None else _ptr(w), _ptr(act), _ptr(logp), _stream()))
                        out_bad += act_bad() + logp_bad() + int(((act < 0) | (act > 4100)).sum())
            env.step_policy(torch.randn(N, 4101, device="cuda"))
    return dict(out_guard_bad=out_bad)


def _encode(envs):
    """every dtype, planes and repetition counts together and alone, guard regions around the caller's output vectors (a
    multiple of 16 bytes: the planes stay aligned)"""
    L, G, out_bad = _lib.lib(), 4096, 0
    for N in (1, 33, 4097):
        for kw in FEATURE_CONFIGS:
            env = BatchedChessEnv(N, seed=3, **kw)
            envs.append(env)
            env.step_sampled(40)
            for dt, size in ((0, 4), (1, 2), (2, 1)):
                for with_planes, with_rep in ((True, True), (True, False), (False, True)):
                    planes_buf, planes, planes_bad = _guarded(N * 19 * 64 * size, torch.uint8, G, 0xA5)
                    rep_buf, rep, rep_bad = _guarded(N, torch.uint8, G, 0xA5)
                    _lib.check(L.gcb_env_encode(env._h, _ptr(planes) if with_planes else None, dt,
                                                _ptr(rep) if with_rep else None, _stream()))
                    out_bad += planes_bad() + rep_bad()
                    if not with_planes:
                        out_bad += int((planes_buf != 0xA5).sum())
                    if not with_rep:
                        out_bad += int((rep_buf != 0xA5).sum())
                    if with_rep:
                        out_bad += int((rep > 2).sum())
            env.encode(torch.bfloat16)
            env.repetition_count()
    return dict(out_guard_bad=out_bad)


SCENARIOS = {
    "steps": lambda envs: _steps(envs, [1, 33, 64, 160, 3000, 70001, 131149]),
    "steps_quick": lambda envs: _steps(envs, [64, 160], quick=True),
    "clone_valid": _clone_valid,
    "clone_out_of_range": _clone_out_of_range,
    "clone_alias": _clone_alias,
    "policy": _policy,
    "encode": _encode,
}


def exercise(name):
    """one scenario between a reset of the violation word and a check of the guard bytes of every env it created"""
    L = _lib.lib()
    _lib.check(L.gcb_debug_violations(C.byref(C.c_uint64()), 1))
    envs = []
    extra = SCENARIOS[name](envs) or {}
    torch.cuda.synchronize()
    bad = 0
    for env in envs:
        n = C.c_uint64()
        _lib.check(L.gcb_env_check_guards(env._h, C.byref(n)))
        if n.value:
            print("%s: guard damage N=%d: %s" % (name, env.num_envs, L.gcb_last_error().decode()), file=sys.stderr)
        bad += n.value
    v = C.c_uint64()
    _lib.check(L.gcb_debug_violations(C.byref(v), 1))
    for env in envs:
        env.close()
    return dict(checked=int(L.gcb_build_is_checked()), violations=int(v.value), guard_bad_bytes=int(bad), **extra)


if __name__ == "__main__":
    os.environ["GCB_GUARD_BYTES"] = "4096"
    print(json.dumps({name: exercise(name) for name in sys.argv[1:]}))
