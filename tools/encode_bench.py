"""Network-input encoder throughput on one GPU (gcb_env_encode, kernel k_env_encode) -> one JSON document (stdout, and --out).

Workloads: 524,288 and 65,536 phase-spread self-play envs (dephase), and 524,288 self-play envs from the endgame templates
(boards.endgame_boards(), played --endgame-steps sampled steps first, so that many repetition windows are live).  For each
workload and dtype (float32, bfloat16, uint8):
  kernel     encode(dtype, out=buf) into a preallocated [N, 19, 8, 8] buffer: median of --repeats CUDA-event-bracketed calls
             after a warm-up.
  torch      planes 0-16 built in torch from observe() + info_tensor() (one-hot compares, broadcasts, cat, .to(dtype)), in the
             same dtype, alternated with the kernel in the same run.  It cannot build planes 17-18: the repetition count lives
             only in the env's table.
  loop       encode(out=buf) + step_policy(bf16 logits) against step_policy alone, alternated: the encoder's share of an act step.
Algorithmic bytes per call (computed here from info_tensor()): the planes written (N x 19 x 64 x element size), 32 B of board
and 8 B of meta per env, and for every env with a non-empty repetition window (info column hist_len != 0) 8 B of key, 4 B of
window generation and one 32-B sector of its table.  Share of peak = those bytes over kernel time over the HBM peak bench.py
uses (bench.peaks()).  A row whose output fits the 126 MB L2 is marked so: consecutive calls overwrite L2-resident lines.
"""
import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from clone_bench import card, median, timed  # noqa: E402

L2_BYTES = 126e6


def alg_bytes(info, elsize):
    N = info.shape[0]
    live = int((info[:, 12] != 0).sum())
    return N * 19 * 64 * elsize + 40 * N + (8 + 4 + 32) * live, live


def torch_encoder(env, dtype):
    """planes 0-16 from the exported board and info columns, in torch"""
    import torch

    N = env.num_envs
    codes = torch.arange(1, 7, dtype=torch.int8, device=env.device).view(1, 6, 1)

    def run():
        b = env.observe().reshape(N, 1, 64)
        info = env.info_tensor()
        side = (info[:, 0] < 0).view(N, 1, 1).expand(N, 1, 64)
        rights = (info[:, 1:5] != 0).view(N, 4, 1).expand(N, 4, 64)
        return torch.cat([b == codes, b == -codes, side, rights], 1).to(dtype).view(N, 17, 8, 8)

    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[524288, 65536])
    ap.add_argument("--endgame-envs", type=int, default=524288)
    ap.add_argument("--endgame-steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import bench
    from gym_chess_b200 import BatchedChessEnv, _lib
    from gym_chess_b200.boards import endgame_boards

    _lib.require_gpu()
    peak_gbs, peak_src = bench.peaks()
    out = dict(tool="tools/encode_bench.py", card=card(), library=_lib.SO_PATH, hbm_peak_gbs=peak_gbs, hbm_peak_source=peak_src,
               results=[])
    workloads = [("phase-spread self-play", N, None) for N in args.envs]
    if args.endgame_envs:
        workloads.append(("endgame templates", args.endgame_envs, endgame_boards()))
    for name, N, boards in workloads:
        env = BatchedChessEnv(N, opponent="none", seed=1, initial_boards=boards)
        if boards is None:
            env.dephase()
        else:
            env.step_sampled(args.endgame_steps)
        info = env.info_tensor().cpu().numpy()
        rep = env.repetition_count()
        counts = torch.bincount(rep.long(), minlength=3).tolist()
        bufs = {}
        for dt in (torch.float32, torch.bfloat16, torch.uint8):
            buf = bufs[dt] = torch.empty(N, 19, 8, 8, dtype=dt, device="cuda")
            nbytes, live = alg_bytes(info, buf.element_size())
            kern = lambda: env.encode(dt, out=buf)  # noqa: E731
            tenc = torch_encoder(env, dt)
            assert torch.equal(tenc(), kern()[:, :17])  # the baseline computes the same planes 0-16
            for f in (kern, tenc):
                timed(f, args.warmup, 1)
            ms, tms = [], []
            for _ in range(args.repeats):
                ms += timed(kern, 0, 1)
                tms += timed(tenc, 0, 1)
            us = median(ms) * 1e3
            gbs = nbytes / (us * 1e-6) / 1e9
            planes_bytes = N * 19 * 64 * buf.element_size()
            out["results"].append(dict(
                workload=name, envs=N, dtype=str(dt).replace("torch.", ""), planes_bytes=planes_bytes,
                output_fits_l2=planes_bytes < L2_BYTES, nonempty_windows=live, repetition_counts=counts, algorithmic_bytes=nbytes,
                us_per_call=round(us, 1), envs_per_s=N / (us * 1e-6), gb_per_s=round(gbs, 1), share_of_hbm_peak=round(gbs / peak_gbs, 3),
                at_peak_us=round(nbytes / (peak_gbs * 1e9) * 1e6, 1), repeat_ms=[round(t, 4) for t in ms],
                torch_planes_0_16_us=round(median(tms) * 1e3, 1), torch_repeat_ms=[round(t, 4) for t in tms],
                speedup_vs_torch=round(median(tms) * 1e3 / us, 1)))
            torch.cuda.empty_cache()
        # the act step of a learner's loop: observation -> (network) -> logits -> step_policy
        logits = torch.randn(N, 4101, device="cuda", dtype=torch.bfloat16)
        for dt, buf in bufs.items():
            loop = lambda: (env.encode(dt, out=buf), env.step_policy(logits))  # noqa: E731
            act = lambda: env.step_policy(logits)  # noqa: E731
            for f in (loop, act):
                timed(f, args.warmup, 1)
            lms, ams = [], []
            for _ in range(args.repeats):
                lms += timed(loop, 0, 1)
                ams += timed(act, 0, 1)
            row = next(r for r in out["results"] if r["workload"] == name and r["envs"] == N and r["dtype"] == str(dt).replace("torch.", ""))
            row.update(encode_plus_step_policy_us=round(median(lms) * 1e3, 1), step_policy_us=round(median(ams) * 1e3, 1),
                       loop_repeat_ms=[round(t, 4) for t in lms], step_policy_repeat_ms=[round(t, 4) for t in ams])
        del logits, bufs, env
        torch.cuda.empty_cache()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
