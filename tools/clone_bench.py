"""Per-env clone throughput on one GPU (gcb_env_clone, kernel k_env_clone) -> one JSON document (stdout, and --out).

W1 fan-out: 4096 phase-spread self-play roots (a source object of 4096 envs) cloned 128 times each into 524,288
           destination rows of another object, at history_cap 512 and 64.
W2 full fork: identity clone of 524,288 phase-spread rows into an object of the same configuration, alternated in the same
           run with snapshot() + restore() of the source (into a preallocated buffer) -- the only way to fork a batch
           without the clone.
Timing: CUDA events around each call after a warm-up, median of --repeats bracketed repeats.
Algorithmic bytes per cloned row: 2 x (72 + 8 * slots) + 12 B of state and index, plus, where the source's window is
non-empty, 32 * history_cap B of table read and 16 B per live entry written (live entries <= hist_len, info column 12,
taken as hist_len) -- computed from the sources' actual hist_len before timing.  Share of peak = GB/s over the HBM peak
bench.py uses (bench.peaks()).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, sm = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, sm_max_clock=sm)
    except Exception as e:  # noqa: BLE001
        return dict(name=None, error=str(e))


def alg_bytes(src_hist, idx, slots, history_cap):
    import numpy as np

    h = src_hist[idx[idx >= 0]].astype(np.int64)
    state = (2 * (72 + 8 * slots) + 12) * len(h)
    table = int((h > 0).sum()) * 32 * history_cap + 16 * int(h.sum())
    return state + table, dict(rows=int(len(h)), nonempty_windows=int((h > 0).sum()), mean_hist_len=float(h.mean()))


def timed(fn, warmup, repeats):
    import torch

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def median(xs):
    return sorted(xs)[len(xs) // 2]


def report(name, ms, nbytes, rows, peak_gbs, extra):
    us = median(ms) * 1e3
    gbs = nbytes / (us * 1e-6) / 1e9
    return dict(workload=name, us_per_call=round(us, 1), clones_per_s=rows / (us * 1e-6), algorithmic_bytes=nbytes,
                gb_per_s=round(gbs, 1), share_of_hbm_peak=round(gbs / peak_gbs, 3), repeat_ms=[round(x, 4) for x in ms], **extra)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=524288)
    ap.add_argument("--roots", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch

    import bench
    from gym_chess_b200 import BatchedChessEnv, _lib

    _lib.require_gpu()
    peak_gbs, peak_src = bench.peaks()
    N, R = args.envs, args.roots
    out = dict(tool="tools/clone_bench.py", card=card(), hbm_peak_gbs=peak_gbs, hbm_peak_source=peak_src, envs=N, results=[])

    # W1: fan-out, cross-object
    for H in (512, 64):
        S = BatchedChessEnv(R, opponent="none", seed=1, history_cap=H)
        S.dephase()
        D = BatchedChessEnv(N, opponent="none", seed=2, env_id_offset=R, history_cap=H)
        idx = torch.arange(N, device="cuda", dtype=torch.int32) // (N // R)
        hist = S.info_tensor()[:, 12].cpu().numpy()
        nbytes, shape = alg_bytes(hist, idx.cpu().numpy(), S._n_slots(), H)
        ms = timed(lambda: D.clone_from(S, idx), args.warmup, args.repeats)
        out["results"].append(report("W1 fan-out %d roots x %d, history_cap %d" % (R, N // R, H), ms, nbytes, N, peak_gbs,
                                     dict(history_cap=H, **shape)))
        del S, D
        torch.cuda.empty_cache()

    # W2: full fork vs snapshot + restore, alternated
    H = 512
    S = BatchedChessEnv(N, opponent="none", seed=1, history_cap=H)
    S.dephase()
    D = BatchedChessEnv(N, opponent="none", seed=2, env_id_offset=N, history_cap=H)
    idx = torch.arange(N, device="cuda", dtype=torch.int32)
    hist = S.info_tensor()[:, 12].cpu().numpy()
    nbytes, shape = alg_bytes(hist, idx.cpu().numpy(), S._n_slots(), H)
    nsnap = C.c_uint64()
    _lib.check(_lib.lib().gcb_env_snapshot_bytes(S._h, C.byref(nsnap)))
    buf = torch.empty(nsnap.value, dtype=torch.uint8, device="cuda")
    tick = C.c_uint64()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def snap_restore():
        _lib.check(_lib.lib().gcb_env_snapshot(S._h, C.c_void_p(buf.data_ptr()), C.byref(tick), stream))
        _lib.check(_lib.lib().gcb_env_restore(S._h, C.c_void_p(buf.data_ptr()), tick.value, stream))

    clone_ms, snap_ms = [], []
    for _ in range(args.repeats):
        clone_ms += timed(lambda: D.clone_from(S, idx), 1, 1)
        snap_ms += timed(snap_restore, 1, 1)
    w2 = report("W2 full fork %d rows, history_cap %d" % (N, H), clone_ms, nbytes, N, peak_gbs, dict(history_cap=H, **shape))
    sr_us = median(snap_ms) * 1e3
    w2.update(snapshot_restore_us=round(sr_us, 1), snapshot_bytes=int(nsnap.value),
              snapshot_restore_traffic_gb_per_s=round(4 * nsnap.value / (sr_us * 1e-6) / 1e9, 1),
              snapshot_restore_repeat_ms=[round(x, 4) for x in snap_ms], speedup_vs_snapshot_restore=round(sr_us / w2["us_per_call"], 2))
    out["results"].append(w2)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
