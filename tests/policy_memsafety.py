"""Memory-safety net of policy sampling, run as a subprocess by tests/test_policy_gpu.py (GYMCHESS_B200_LIB selects the
CHECKED build).  Guard regions around every env array (GCB_GUARD_BYTES) and around the caller's output buffers, at awkward
sizes (1, 33, 4097 envs), fp32 and bf16 logits with padded rows, every temperature form, caller and Philox words; prints one
JSON line {"checked": 0|1, "violations": bit set, "guard_bad_bytes": n, "out_guard_bad": n}."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

G = 1024  # guard elements on each side of an output buffer


def run():
    os.environ["GCB_GUARD_BYTES"] = "4096"
    import torch

    from gym_chess_b200 import BatchedChessEnv, _lib
    from gym_chess_b200.boards import endgame_boards

    L = _lib.lib()
    _lib.check(L.gcb_debug_violations(C.byref(C.c_uint64()), 1))
    envs, out_bad = [], 0
    torch.manual_seed(1)
    for N in (1, 33, 4097):
        for kw in (dict(opponent="none"), dict(opponent="random", player_color="BLACK"),
                   dict(opponent="none", initial_boards=endgame_boards(), history_cap=8, moves_max=250)):
            env = BatchedChessEnv(N, seed=3, **kw)
            env.step_sampled(30)
            for dt in (torch.float32, torch.bfloat16):
                x = torch.randn(N, 4160, device="cuda").mul_(3).to(dt)[:, :4101]
                words = torch.randint(0, 2 ** 31, (N,), dtype=torch.int32, device="cuda")
                for T in (0.0, 0.5, 1.0):
                    for w in (words, None):
                        act = torch.full((N + 2 * G,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
                        logp = torch.full((N + 2 * G,), 7.25, dtype=torch.float32, device="cuda")
                        _lib.check(L.gcb_env_sample_policy(env._h, C.c_void_p(x.data_ptr()), int(dt == torch.bfloat16), 4160,
                                                           T, None if w is None else C.c_void_p(w.data_ptr()),
                                                           C.c_void_p(act[G:].data_ptr()), C.c_void_p(logp[G:].data_ptr()),
                                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
                        out_bad += int((act[:G] != 0x5A5A5A5A).sum() + (act[G + N:] != 0x5A5A5A5A).sum())
                        out_bad += int((logp[:G] != 7.25).sum() + (logp[G + N:] != 7.25).sum())
                        a = act[G:G + N]
                        out_bad += int(((a < 0) | (a > 4100)).sum())
            env.step_policy(torch.randn(N, 4101, device="cuda"))
            envs.append(env)
    torch.cuda.synchronize()
    bad = 0
    for e in envs:
        n = C.c_uint64()
        _lib.check(L.gcb_env_check_guards(e._h, C.byref(n)))
        bad += n.value
    v = C.c_uint64()
    _lib.check(L.gcb_debug_violations(C.byref(v), 1))
    return dict(checked=int(L.gcb_build_is_checked()), violations=int(v.value), guard_bad_bytes=int(bad), out_guard_bad=int(out_bad))


if __name__ == "__main__":
    print(json.dumps(run()))
