"""Memory-safety net of the network-input encoder, run as a subprocess by tests/test_encode_gpu.py (GYMCHESS_B200_LIB selects
the CHECKED build).  Guard regions around every env array (GCB_GUARD_BYTES) and around the caller's output buffers, at awkward
sizes (1, 33, 4097 envs), every dtype, planes and repetition counts together and alone, in self-play, against the bot and from
the endgame templates; prints one JSON line {"checked": 0|1, "violations": bit set, "guard_bad_bytes": n, "out_guard_bad": n}."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

G = 4096  # guard bytes on each side of an output buffer (a multiple of 16: the planes stay aligned)


def run():
    os.environ["GCB_GUARD_BYTES"] = "4096"
    import torch

    from gym_chess_b200 import BatchedChessEnv, _lib
    from gym_chess_b200.boards import endgame_boards

    L = _lib.lib()
    _lib.check(L.gcb_debug_violations(C.byref(C.c_uint64()), 1))
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    envs, out_bad = [], 0
    for N in (1, 33, 4097):
        for kw in (dict(opponent="none"), dict(opponent="random", player_color="BLACK"),
                   dict(opponent="none", initial_boards=endgame_boards(), history_cap=8, moves_max=250)):
            env = BatchedChessEnv(N, seed=3, **kw)
            env.step_sampled(40)
            for dt, size in ((0, 4), (1, 2), (2, 1)):
                nbytes = N * 19 * 64 * size
                for with_planes, with_rep in ((True, True), (True, False), (False, True)):
                    planes = torch.full((nbytes + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
                    rep = torch.full((N + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
                    _lib.check(L.gcb_env_encode(env._h, C.c_void_p(planes[G:].data_ptr()) if with_planes else None, dt,
                                                C.c_void_p(rep[G:].data_ptr()) if with_rep else None, stream()))
                    out_bad += int((planes[:G] != 0xA5).sum() + (planes[G + nbytes:] != 0xA5).sum())
                    out_bad += int((rep[:G] != 0xA5).sum() + (rep[G + N:] != 0xA5).sum())
                    if not with_planes:
                        out_bad += int((planes != 0xA5).sum())
                    if not with_rep:
                        out_bad += int((rep != 0xA5).sum())
                    if with_rep:
                        out_bad += int((rep[G:G + N] > 2).sum())
            env.encode(torch.bfloat16)
            env.repetition_count()
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
