"""Policy sampling throughput on one GPU (gcb_env_sample_policy, kernel k_env_policy_sample) -> one JSON document (stdout,
and --out).

For --envs (default 524,288 and 65,536) phase-spread self-play envs and fp32 / bf16 logits from torch.randn (524,288 x 4101
fp32 = 8.6 GB, far beyond L2):
  kernel     sample_policy(logits, T=1) with Philox words: median of --repeats CUDA-event-bracketed calls after a warm-up.
  torch      the pipeline a learner needs without it, alternated with the kernel in the same run: legal_bitmask ->
             unpack_bitmask -> masked_fill(-inf) -> log_softmax -> multinomial -> gather of the log-prob.
  step       step_policy(logits) against step(actions) with given actions, alternated.
Touched bytes per env (computed on the host from a legal_bitmask export, by the code below): the distinct 32-B sectors of
the logit row that hold a legal entry, plus the state the kernel reads (board 32 B, meta 8 B, episode 4 B, 8 B per staged
piece slot of the side to move) and the outputs (action 4 B, logp 4 B).  Share of peak = those bytes over kernel time, over
the HBM peak bench.py uses (bench.peaks()).  One full pass over the logits (N x 4101 x element size) at that peak is
reported beside it, as the bound the torch pipeline cannot beat.
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


def touched_bytes(bits, boards, info, elsize, row_stride, chunk=32768):
    """distinct 32-B logit sectors of every env's legal set + state + output bytes (see the module docstring)"""
    import numpy as np

    N = bits.shape[0]
    sectors = 0
    for lo in range(0, N, chunk):
        b = np.ascontiguousarray(bits[lo:lo + chunk]).view(np.uint8)
        legal = np.unpackbits(b, axis=1, bitorder="little")[:, :4101]
        e, a = np.nonzero(legal)
        sec = ((e.astype(np.int64) + lo) * row_stride + a) * elsize // 32
        sectors += len(np.unique(sec))
    own = np.where(info[:, :1] > 0, boards > 0, boards < 0).sum(1)
    state = int((32 + 8 + 4 + 8 * np.minimum(own, 16) + 8).sum())
    return 32 * sectors + state, dict(logit_sectors=int(sectors), mean_legal=float(info[:, 9].mean()),
                                      state_and_output_bytes=state)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[524288, 65536])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=9)
    ap.add_argument("--kernel-only", action="store_true", help="skip the torch pipeline and the step comparison")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import bench
    from gym_chess_b200 import BatchedChessEnv, _lib

    _lib.require_gpu()
    peak_gbs, peak_src = bench.peaks()
    out = dict(tool="tools/policy_bench.py", card=card(), library=_lib.SO_PATH, hbm_peak_gbs=peak_gbs, hbm_peak_source=peak_src,
               temperature=1.0, results=[])
    for N in args.envs:
        env = BatchedChessEnv(N, opponent="none", seed=1)
        env.dephase()
        bits = env.legal_bitmask().cpu().numpy()
        boards, info, _ = env.export_numpy()
        for dt in (torch.float32, torch.bfloat16):
            x = torch.randn(N, 4101, device="cuda", dtype=dt)
            nbytes, shape = touched_bytes(bits, boards, info, x.element_size(), x.stride(0))
            full_pass_us = N * 4101 * x.element_size() / (peak_gbs * 1e9) * 1e6
            kern = lambda: env.sample_policy(x, 1.0)  # noqa: E731
            res = dict(envs=N, dtype=str(dt).replace("torch.", ""), touched_bytes=nbytes, **shape,
                       one_logit_pass_at_peak_us=round(full_pass_us, 1))
            if args.kernel_only:
                ms = timed(kern, args.warmup, args.repeats)
            else:
                bitsbuf = torch.empty(N, 65, dtype=torch.int64, device="cuda")

                def torch_pipeline():
                    mask = BatchedChessEnv.unpack_bitmask(env.legal_bitmask(out=bitsbuf))
                    mask[:, 4100] |= ~mask.any(1)  # no legal move: RESIGN, as the kernel does
                    lp = torch.log_softmax(x.float().masked_fill(~mask, float("-inf")), dim=1)
                    a = torch.multinomial(lp.exp(), 1)
                    return a.squeeze(1), lp.gather(1, a).squeeze(1)

                for f in (kern, torch_pipeline):
                    timed(f, args.warmup, 1)
                ms, tms = [], []
                for _ in range(args.repeats):
                    ms += timed(kern, 0, 1)
                    tms += timed(torch_pipeline, 0, 1)
                torch.cuda.empty_cache()
                acts = env.sample_policy(x, 1.0)[0]
                sp = lambda: env.step_policy(x, 1.0)  # noqa: E731
                st = lambda: env.step(acts)  # noqa: E731
                for f in (sp, st):
                    timed(f, args.warmup, 1)
                sp_ms, st_ms = [], []
                for _ in range(args.repeats):
                    sp_ms += timed(sp, 0, 1)
                    st_ms += timed(st, 0, 1)
                res.update(torch_pipeline_us=round(median(tms) * 1e3, 1), torch_repeat_ms=[round(t, 4) for t in tms],
                           step_policy_us=round(median(sp_ms) * 1e3, 1), step_given_actions_us=round(median(st_ms) * 1e3, 1))
            us = median(ms) * 1e3
            gbs = nbytes / (us * 1e-6) / 1e9
            res.update(us_per_call=round(us, 1), samples_per_s=N / (us * 1e-6), touched_gb_per_s=round(gbs, 1),
                       share_of_hbm_peak=round(gbs / peak_gbs, 3), repeat_ms=[round(t, 4) for t in ms])
            if "torch_pipeline_us" in res:
                res["speedup_vs_torch"] = round(res["torch_pipeline_us"] / us, 1)
            out["results"].append(res)
            del x
            torch.cuda.empty_cache()
        del env
        torch.cuda.empty_cache()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
