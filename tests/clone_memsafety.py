"""Memory-safety net of the per-env clone, run as a subprocess by tests/test_clone_gpu.py (GYMCHESS_B200_LIB selects the
CHECKED build).  Guard regions around every env array (GCB_GUARD_BYTES); prints one JSON line
{"checked": 0|1, "violations": bit set, "guard_bad_bytes": n, "untouched": bool}.
  valid         cross-object clones (identity, fan-out, -1 rows, another env count) and an in-object disjoint gather at
                awkward sizes (1, 33, 4097 envs), each followed by steps
  out_of_range  one index >= the source's env count: that row must be left untouched (CHK_CLONE_INDEX in the checked build)
  alias         an in-object index vector whose destination rows are also source rows (CHK_CLONE_ALIAS in the checked build)
"""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def run(mode):
    os.environ["GCB_GUARD_BYTES"] = "4096"
    import numpy as np
    import torch

    from gym_chess_b200 import BatchedChessEnv, _lib
    from gym_chess_b200.boards import endgame_boards

    L = _lib.lib()
    _lib.check(L.gcb_debug_violations(C.byref(C.c_uint64()), 1))
    envs, untouched = [], True
    rng = np.random.RandomState(1)
    if mode == "valid":
        for N in (1, 33, 4097):
            for kw in (dict(opponent="none"), dict(opponent="random", player_color="BLACK"),
                       dict(opponent="none", initial_boards=endgame_boards(), history_cap=8, moves_max=250)):
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
    else:
        N = 4097
        S = BatchedChessEnv(N, opponent="none", seed=3)
        S.step_sampled(20)
        before = S.export_numpy()
        if mode == "out_of_range":
            D = BatchedChessEnv(N, opponent="none", seed=4)
            D.step_sampled(7)
            before = D.export_numpy()
            idx = np.full(N, -1)
            idx[100] = N + 5
            D.clone_from(S, idx)
            after = D.export_numpy()
            untouched = all((a == b).all() for a, b in zip(before, after))
            envs += [S, D]
        else:
            idx = np.full(N, -1)
            idx[10], idx[20] = 20, 30  # row 20 is a destination and the source of row 10
            S.clone_from(S, idx)
            envs.append(S)
    torch.cuda.synchronize()
    bad = 0
    for e in envs:
        n = C.c_uint64()
        _lib.check(L.gcb_env_check_guards(e._h, C.byref(n)))
        bad += n.value
    v = C.c_uint64()
    _lib.check(L.gcb_debug_violations(C.byref(v), 1))
    return dict(checked=int(L.gcb_build_is_checked()), violations=int(v.value), guard_bad_bytes=int(bad), untouched=bool(untouched))


if __name__ == "__main__":
    print(json.dumps(run(sys.argv[1] if len(sys.argv) > 1 else "valid")))
