#!/usr/bin/env python
"""bench.py -- env steps/s (and legal-movegen positions/s) of the batched gym-chess v2 env on B200.

    python bench.py [--gpus N --steps K --warmup W]                 our CUDA path (default N=1)
    python bench.py --impl reference [--gpus N --steps K --warmup W]  the reference algorithm on the host cores
    torchrun ... bench.py --gpus N ...                              one rank per GPU, weak scaling

Workload (BASELINE.json configs[3] "4M envs sharded across 8xB200", per-GPU shard): 524,288 envs per GPU, random
self-play (opponent "none"), uniformly random legal action per ply drawn on the device (Philox4x32-10), auto-reset.
A "step" is one ChessEnvV2.step() of every env of the rank; the fused step kernel runs up to 64 consecutive steps per
launch.  Before anything is timed the episode phases of the batch are SPREAD (BatchedChessEnv.dephase): three episodes
in four end at the 150-move cap after exactly 301 steps, so a batch reset together would stay in lockstep and a short
timed window would see one narrow band of plies -- not the workload.

`value` = env steps of all ranks / max-over-ranks device time of EXACTLY K steps, state resident in HBM; the K-step block
is repeated (--repeats, default 5), every repeat bracketed by barrier + synchronize on both sides, and the MEDIAN repeat
is reported (all of them are in `repeat_ms`).  `e2e` = the same metric through the host-buffer C ABI calls (what a binding
of the reference env would call): per step the caller's 16-bit words cross PCIe host->device from pinned memory and a
16-bit result record per env device->host, inside the timed region (the kernel reads / writes the page-locked buffers in
place); the rank's envs are stepped as two shards (PipelinedChessEnv), one in flight while the host handles the other.
`e2e.full_*` are the same loop carrying what step() returns to a learner: + the observation (32 B of bit-planes per env)
and + the 528-byte legal-action bit mask per env.

--dump-outputs DIR writes what the timed call (step_sampled) returned for its last step as float32 .npy files, so that two
builds can be compared output for output: reward.npy, done.npy, flags.npy [N] (a seeded sample of DUMP_MAX_ENVS envs when
N is larger) and observation.npy [DUMP_OBS_ENVS, 64], the board each env of a seeded sample was left with.  The envs,
seeds and step counts depend only on the arguments, so the same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree, which may be read-only

ENVS_PER_GPU = 524288
METRIC = "env_steps_per_sec"
UNIT = "env steps/s"
WORKLOAD = ("random self-play, opponent=none, auto-reset, on-device Philox action draw; %d envs per GPU "
            "(BASELINE.json configs[3]: 4M envs over 8xB200, per-GPU shard)")
CPU_SAMPLE_ENVS = 65536     # the CPU arm's bounded sample of the same workload
PUBLISHED = {"steps_per_sec": 3205, "source": "gym_chess/test/v2/test_benchmark.py:46-50 (1851 steps in 0.5776 s, 1 thread, unspecified CPU)"}
DUMP_MAX_ENVS = 1 << 20     # --dump-outputs: reward / done / flags of at most this many envs (12 MB of float32)
DUMP_OBS_ENVS = 16384       # ... and the observation of this many (4 MB)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def dump_outputs(out_dir, env):
    """--dump-outputs: reward / done / flags of the last step of the timed step_sampled call (the env's output buffers hold
    them until it is stepped again) and the board observation that step left behind, as float32 out_dir/<name>.npy"""
    import numpy as np

    N = env.num_envs

    def sample(k, seed):
        return np.arange(N) if N <= k else np.sort(np.random.RandomState(seed).choice(N, k, replace=False))

    idx = sample(DUMP_MAX_ENVS, 1)
    arrays = {name: t.cpu().numpy()[idx] for name, t in (("reward", env.reward), ("done", env.done), ("flags", env.flags))}
    arrays["observation"] = env.observe().reshape(N, 64).cpu().numpy()[sample(DUMP_OBS_ENVS, 2)]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region"""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
        except OSError:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i] == "Active" for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_arm(steps, warmup, min_region_s=1.5, max_blocks=40):
    """The reference algorithm (oracle/gc_oracle.c: C restatement of src/lib.rs + chess_v2.py; kind "port" because the Rust
    engine cannot be built here) on all host threads, on a bounded sample of the GPU arm's workload: a persistent pool of
    CPU_SAMPLE_ENVS self-play envs, episode phases spread (env i burns in 300 + i % 301 steps), `warmup` steps, then blocks
    of exactly `steps` steps of every env until the timed blocks cover at least `min_region_s` seconds; the MEDIAN block is
    reported per step.  Threads are created inside each block (16 pthread_create per >= 30 ms block: < 0.1 %)."""
    from oracle import oracle as orc

    threads = os.cpu_count() or 1
    pool = orc.SelfplayPool(0, 0, CPU_SAMPLE_ENVS)
    t0 = time.time()
    pool.run(300, threads, stagger=301)
    pool.run(max(1, warmup), threads)
    burn_s = time.time() - t0
    blocks, total = [], 0.0
    while (total < min_region_s or len(blocks) < 3) and len(blocks) < max_blocks:
        t0 = time.perf_counter()
        st = pool.run(steps, threads)
        dt = time.perf_counter() - t0
        assert st["steps"] == CPU_SAMPLE_ENVS * steps
        blocks.append(dt)
        total += dt
    dt = median(blocks)
    return dict(value=CPU_SAMPLE_ENVS * steps / dt, block_s=dt, blocks=len(blocks), timed_region_s=total, burn_in_s=burn_s,
                threads=threads, spread=(max(blocks) - min(blocks)) / dt)


def cpu_sample_text(r, steps):
    return ("%d envs x %d steps per block, median of %d blocks (%.2f s timed, block spread %.0f %%) after a phase-spreading "
            "burn-in of 300 + (env %% 301) steps; C oracle (restates src/lib.rs + chess_v2.py; the Rust engine is unbuildable "
            "here), %d pthreads" % (CPU_SAMPLE_ENVS, steps, r["blocks"], r["timed_region_s"], 100 * r["spread"], r["threads"]))


def run_reference(args, rank, world):
    if rank != 0:
        return
    r = cpu_arm(args.steps, args.warmup)
    v = r["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["block_s"] / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": WORKLOAD % ENVS_PER_GPU, "sample": cpu_sample_text(r, args.steps)},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": cpu_sample_text(r, args.steps)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "timed_region_s": r["timed_region_s"], "blocks": r["blocks"],
        "published_reference": PUBLISHED,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5, help="the K-step block is timed this many times; the median is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--burn-in", type=int, default=600, help="untimed steps after the phases have been spread")
    ap.add_argument("--no-extras", action="store_true", help="skip the movegen / small-config / cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(3, args.warmup)  # timing rule: at least 3 warm-up steps (the JSON reports the value used)
    args.steps = max(1, args.steps)
    args.repeats = max(1, args.repeats)
    # stdout carries exactly ONE JSON line: anything a library prints meanwhile (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist

    from gym_chess_b200 import BatchedChessEnv, PipelinedChessEnv, _lib, sharding

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    N, K, R = args.envs_per_gpu, args.steps, args.repeats
    off, _ = sharding.shard_of(rank, world, N)
    L = _lib.lib()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        return sharding.max_over_ranks(ms, device=dev)

    def timed_repeats(fn, repeats, stream=None, wall=False):
        """`repeats` x [barrier + sync, fn(), barrier + sync]: device time of fn (CUDA events on the launching stream), or the
        slower of device and host wall time (wall=True: loops the host takes part in); max over ranks of every repeat"""
        out = []
        for _ in range(repeats):
            barrier()
            ev0.record(stream)
            t0 = time.perf_counter()
            fn()
            t1 = time.perf_counter()
            ev1.record(stream)
            barrier()
            ms = ev0.elapsed_time(ev1)
            out.append(max_over_ranks(max(ms, (t1 - t0) * 1e3) if wall else ms))
        return out

    # ---- the envs: phases spread, burn-in, warm-up
    env = BatchedChessEnv(N, opponent="none", seed=2, device=local_rank, auto_reset=True, env_id_offset=off)
    env.dephase()
    env.step_sampled(args.burn_in)
    env.reset_stats()
    env.step_sampled(301)            # one full episode period: the workload's steady-state mix (untimed)
    steady = env.stats()
    env.step_sampled(args.warmup)
    env.reset_stats()
    # ---- timed region 1: kernel-only, state resident in HBM.  Working set (72 B state + 128 B piece slots + 16 KB
    # repetition table per env = 8.7 GB at 524,288 envs) is far larger than the 126 MB L2: no flush needed.
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = L.gcb_launch_count()
    rep_ms = timed_repeats(lambda: env.step_sampled(K), R)
    launches = (L.gcb_launch_count() - launches0) // R
    ms = median(rep_ms)
    st = env.stats()
    assert st["steps"] == N * K * R, (st["steps"], N, K, R)   # every repeat stepped every env exactly K times
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env)
    value = world * N * K / (ms * 1e-3)

    # ---- final NCCL reduce of the episode statistics (the only collective of the job)
    tot = sharding.reduce_stats(env.stats_tensor()).cpu().numpy()

    # ---- timed region 2: end to end through the host-buffer C ABI calls, pinned host memory (see the module docstring)
    e2e_steps = max(10, min(K, 602))
    words = torch.empty((8, N), dtype=torch.int32).pin_memory()
    words.random_(-2 ** 31, 2 ** 31 - 1)
    h_r = torch.empty(N, dtype=torch.int32).pin_memory()
    h_d = torch.empty(N, dtype=torch.uint8).pin_memory()
    h_f = torch.empty(N, dtype=torch.uint8).pin_memory()
    wn, rn, dn, fn = words.numpy().view(np.uint32), h_r.numpy(), h_d.numpy(), h_f.numpy()
    for i in range(3):
        env.step_index_host(wn[i % 8], rn, dn, fn)
    sync_ms = median(timed_repeats(lambda: [env.step_index_host(wn[i % 8], rn, dn, fn) for i in range(e2e_steps)], R, wall=True))
    sync_value = world * N * e2e_steps / (sync_ms * 1e-3)

    H = N // 2
    words16 = torch.empty((8, 2, H), dtype=torch.int16).pin_memory()   # this rank's inputs of 8 steps, page-locked
    words16.random_(-2 ** 15, 2 ** 15 - 1)
    src16 = [[words16[j, k] for k in range(2)] for j in range(8)]

    def pipelined(observe, mask, shards=2):
        """the rank's envs as two shards stepped alternately through PipelinedChessEnv.send_words / recv: uint16 words in,
        uint16 records out (+ observation planes / + bit mask, copied device -> host behind each step); shards=1: one
        synchronous send + recv per step"""
        pipe = PipelinedChessEnv(N, shards=shards, device=local_rank, env_id_offset=off, opponent="none", seed=2, auto_reset=True,
                                 observe=observe, mask=mask)
        pipe.burn_in(args.burn_in, dephase=True)
        src1 = [words16[j].reshape(-1) for j in range(8)]

        def loop(steps):
            if shards == 1:
                for i in range(steps):
                    pipe.send_words(0, src=src1[i % 8])
                    pipe.recv(0)
                return
            pipe.send_words(0, src=src16[0][0])
            for i in range(steps):
                pipe.send_words(1, src=src16[i % 8][1])
                pipe.recv(0)   # shard 0's results of step i are in host memory
                if i + 1 < steps:
                    pipe.send_words(0, src=src16[(i + 1) % 8][0])
                pipe.recv(1)   # shard 1's results of step i are in host memory

        loop(3)
        t = median(timed_repeats(lambda: loop(e2e_steps), R, stream=pipe.streams[0], wall=True))
        pipe.close()
        return world * N * e2e_steps / (t * 1e-3)

    e2e_value = pipelined(False, False)
    clk = clocks.stop() if rank == 0 else None  # sampled over the timed regions (kernel-only and end-to-end)
    sync_packed_value = pipelined(False, False, shards=1)
    full_obs_value = pipelined(True, False)
    full_mask_value = pipelined(True, True) if not args.no_extras else None

    # ---- the other modes of the step (SURVEY.md 8(f)2): the random bot replies inside the step (two plies per step)
    modes = {}
    for name, color in (("vs_random_bot_white_agent", "WHITE"), ("vs_random_bot_black_agent", "BLACK")):
        bot = BatchedChessEnv(N, opponent="random", player_color=color, seed=2, device=local_rank, env_id_offset=off)
        bot.dephase(period=151)
        bot.step_sampled(300)
        bot.reset_stats()
        t = median(timed_repeats(lambda: bot.step_sampled(K), 3))
        bs = bot.stats()
        modes[name] = {"value": world * N * K / (t * 1e-3), "unit": UNIT, "plies_per_step": bs["plies"] / max(1, bs["steps"])}
        bot.close()

    # ---- roofline of the dominant kernel (k_env_step<sampled>): algorithmic bytes per env step, SURVEY.md 8(d):
    # 40 B state read + 40 B state write + 4 B action + 4 B reward + 1 B done + 8 B history append + 8 B x W scanned
    # W = mean repetition window (plies since the last pawn move / capture) the algorithm has to cover; the kernel
    # reads about one hash-table entry per ply instead -- the algorithmic figure stays the survey's.
    W = st["hist_window"] / max(1, st["plies"])
    W_steady = steady["hist_window"] / max(1, steady["plies"])
    bytes_per_step = 97.0 + 8.0 * W
    # the step kernel is the only kernel in the timed region; one launch runs up to 64 consecutive steps
    # (gcb_env_step_sampled), so bytes per launch = N * steps-per-launch * bytes_per_step and
    # achieved = bytes per launch / average launch duration = N * bytes_per_step / (ms per step)
    kernel_ms = ms / K
    steps_per_launch = K / max(1, launches)
    achieved = bytes_per_step * N / (kernel_ms * 1e-3) / 1e9
    peak, peak_src = peaks()
    traffic, traffic_src = None, None   # dram bytes per launch from the committed ncu --set full capture: a PROFILE CITATION
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        if tj.get("envs") == N:  # per launch like `achieved`: a launch of the sampled kernel runs up to 64 steps
            traffic = tj["dram_bytes_per_step"] * K / max(1, launches)
            traffic_src = "profile, not measured in this run: " + tj["source"]
    pipes = None  # what actually bounds the kernel (integer pipe), from the committed ncu capture
    pp = os.path.join(ROOT, "profiles", "pipes.json")
    if os.path.exists(pp):
        with open(pp) as f:
            pipes = json.load(f)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "repeats": R, "repeat_ms": rep_ms,
        "config": {"workload": WORKLOAD % N, "envs_per_gpu": N, "total_envs": world * N, "burn_in_steps": args.burn_in,
                   "phases": "spread before timing (43 groups reset 7 steps apart, then %d burn-in steps)" % args.burn_in,
                   "l2": "inputs larger than L2 (8.7 GB resident state per GPU vs 126 MB L2), no flush"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * N, "d2h_bytes_per_step": 2 * N,
                "steps": e2e_steps, "launches": 2 * e2e_steps,
                "api": "PipelinedChessEnv.send_words / recv (gcb_env_step_index_packed + gcb_env_wait): uint16 random words "
                       "in, uint16 result records (reward int8 | flags | done) out, page-locked host buffers read / written in "
                       "place by the step kernel; the rank's envs as two shards stepped alternately (one in flight while the "
                       "host handles the other)",
                "full_obs_value": full_obs_value,
                "full_obs_bytes": {"h2d_bytes_per_step": 2 * N, "d2h_bytes_per_step": 34 * N},
                "full_obs_api": "the same loop with PipelinedChessEnv(observe=True): + the observation of every env device -> "
                                "host behind each step (32 B of bit-planes per env, the resident form of state['board'])",
                "full_obs_mask_value": full_mask_value,
                "full_obs_mask_bytes": {"h2d_bytes_per_step": 2 * N, "d2h_bytes_per_step": (34 + 528) * N},
                "full_obs_mask_api": "PipelinedChessEnv(observe=True, mask=True): + the 66-word legal-action bit mask per env "
                                     "(written by the step kernel, gcb_env_step_mask_output); PCIe-bound",
                "sync_call_value": sync_value,
                "sync_call_api": "gcb_env_step_index_host: one synchronous call per step for all envs of the rank (4 + 6 bytes per env "
                                 "step across PCIe: 5.2 MB per step of 524,288 envs -- the link, not the kernel, bounds it)",
                "sync_packed_value": sync_packed_value,
                "sync_packed_api": "one synchronous send + recv per step with the 16-bit records (PipelinedChessEnv with one shard)"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "k_env_step<MODE_SAMPLED, TILE 1, SELFPLAY>",
                     "bytes_per_unit": bytes_per_step, "mean_hist_window": W, "mean_hist_window_steady_state": W_steady,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": bytes_per_step * N * steps_per_launch, "steps_per_launch": steps_per_launch,
                     "launch_ms": ms / max(1, launches),
                     "note": "integer-pipe (ALU) bound, not HBM bound: see DESIGN.md section 3 and profiles/",
                     "pipes_from_profile": pipes},
        "other_modes": modes,
        "episode_stats_all_ranks": {k: int(tot[i]) for i, k in enumerate(
            ("steps", "plies", "episodes", "mates", "repetitions", "caps", "wedged", "invalid", "reward_sum", "legal_sum",
             "in_check", "hist_overflow", "slot_overflow", "hist_scanned", "hist_window"))},
    }
    if clk is not None:
        line["clocks"] = clk

    if rank == 0 and world == 1 and not args.no_extras:  # the secondary configs and the CPU baseline: single-GPU runs only
        line.update(extras(args, env, dev, local_rank, peak, timed_repeats, ev0, ev1))
    env.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)


def extras(args, env, dev, local_rank, peak, timed_repeats, ev0, ev1):
    import numpy as np
    import torch

    from gym_chess_b200 import BatchedChessEnv, _lib
    from gym_chess_b200._lib import Positions, check

    L = _lib.lib()
    N, K = args.envs_per_gpu, args.steps
    out = {}

    def loop_ms(fn, reps):
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps

    # ---- legal-movegen positions/s on the FIXED 1,048,576-position set of BASELINE.json configs[1] (tests/golden/
    # make_positions_1m.py: ~92 % seeded self-play uniform over the ply index, ~8 % crafted castle / check / promotion-row /
    # kingless ... boards, both sides; SHA-256 committed).  Its self-play share is regenerated here by the CUDA env -- the
    # oracle is not involved on this side; tests/test_gpu_parity.py byte-compares every list of this set with the oracle.
    from tests.golden import make_positions_1m as mp

    boards, players, rights = mp.build(lambda *a: mp.harvest_gpu(*a, device=local_rank))
    M = len(boards)
    d_b, d_p, d_r = (torch.from_numpy(x).to(dev) for x in (boards, players, rights))
    bb01 = torch.empty((M, 2), dtype=torch.int64, device=dev)
    bb23 = torch.empty((M, 2), dtype=torch.int64, device=dev)
    pl, rt = torch.empty(M, dtype=torch.uint8, device=dev), torch.empty(M, dtype=torch.uint8, device=dev)
    pos = Positions(bb01.data_ptr(), bb23.data_ptr(), pl.data_ptr(), rt.data_ptr())
    check(L.gcb_pack(M, d_b.data_ptr(), d_p.data_ptr(), d_r.data_ptr(), pos, None))
    lst = torch.empty((M, 144), dtype=torch.int16, device=dev)
    cnt = torch.empty(M, dtype=torch.int32, device=dev)
    mg = {"metric": "legal_movegen_positions_per_sec", "positions": M, "set": "fixed (tests/golden/make_positions_1m.py)",
          "sha256_matches_committed": mp.digest(boards, players, rights) == mp.committed_digest()}
    for attack, key in ((0, "legal"), (1, "attack")):
        call = lambda: check(L.gcb_get_possible_moves(M, pos, attack, 0, lst.data_ptr(), 144, cnt.data_ptr(), None, None))
        for _ in range(3):
            call()
        ms = loop_ms(call, 20)
        nl = float(cnt.float().mean().item())
        byt = 40 + 2 + 2 * nl
        mg[key] = {"value": M / (ms * 1e-3), "ms_per_launch": ms, "mean_moves": nl, "bytes_per_position": byt,
                   "hbm_frac": byt * M / (ms * 1e-3) / 1e9 / peak, "kernel": "k_movegen<%s>" % ("true" if attack else "false")}
    mg["value"] = mg["legal"]["value"]
    out["movegen"] = mg
    del d_b, d_p, d_r, bb01, bb23, pl, rt, lst, cnt

    # ---- the learner-facing outputs of a step (SURVEY.md 8(f)1).  Observation: the resident bit-planes (32 B per env,
    # BatchedChessEnv.planes(): zero-copy).  Legal set: the reference-ordered uint16 list (k_env_legal_list), or the 66-word
    # bit mask -- written by the step kernel itself (gcb_env_step_mask_output) or by the stand-alone mask kernel.
    words = torch.randint(-2 ** 31, 2 ** 31 - 1, (8, N), dtype=torch.int32, device=dev)
    ksteps = max(10, min(K, 100))
    i = [0]

    def step_index():
        env.step_index(words[i[0] % 8])
        i[0] += 1

    lstN = torch.empty((N, 144), dtype=torch.int16, device=dev)
    cntN = torch.empty(N, dtype=torch.int32, device=dev)
    bits = torch.empty((N, 66), dtype=torch.int64, device=dev)
    for _ in range(3):
        step_index()
    t_step = loop_ms(step_index, ksteps)
    out["single_step"] = {"value": N / (t_step * 1e-3), "unit": UNIT, "us_per_step": t_step * 1e3,
                          "note": "gcb_env_step_index (caller's random words, device buffers), one step per launch"}
    t = loop_ms(lambda: (step_index(), check(L.gcb_env_legal_actions(env._h, lstN.data_ptr(), 144, cntN.data_ptr(), None))), ksteps)
    out["step_plus_action_list"] = {"value": N / (t * 1e-3), "unit": UNIT,
                                    "note": "k_env_step + k_env_legal_list (uint16[N][144] list + count) per step"}
    bits65 = torch.empty((N, 65), dtype=torch.int64, device=dev)   # the stand-alone kernel's best layout: 65-word rows
    bm_ms = loop_ms(lambda: check(L.gcb_env_legal_bitmask(env._h, bits65.data_ptr(), 65, None)), 20)
    own_pieces = float(((env.observe().reshape(N, 64) != 0).sum(1).float().mean() / 2).item())
    bm_bytes = 520 + 40 + 8 * own_pieces
    out["legal_bitmask"] = {"kernel": "k_env_legal_bits", "envs": N, "ms_per_launch": bm_ms, "bytes_per_env": bm_bytes,
                            "achieved_gbs": bm_bytes * N / (bm_ms * 1e-3) / 1e9, "peak_gbs": peak,
                            "hbm_frac": bm_bytes * N / (bm_ms * 1e-3) / 1e9 / peak,
                            "note": "bound: hbm; every other kernel of the path is integer-pipe bound"}
    t2 = loop_ms(lambda: (step_index(), check(L.gcb_env_legal_bitmask(env._h, bits65.data_ptr(), 65, None))), ksteps)
    env.set_mask_output(bits)
    t1 = loop_ms(step_index, ksteps)
    env.set_mask_output(None)
    out["step_plus_bitmask"] = {"value": N / (t1 * 1e-3), "unit": UNIT, "two_kernels_value": N / (t2 * 1e-3),
                                "note": "one launch per step: the step kernel writes the uint64[N][66] mask itself "
                                        "(gcb_env_step_mask_output); two_kernels_value = k_env_step + k_env_legal_bits"}
    # the same with the envs as two halves on two streams (what PipelinedChessEnv does): the mask stores of one half run under
    # the integer work of the other
    halves = [BatchedChessEnv(N // 2, opponent="none", seed=2, device=local_rank, env_id_offset=k * (N // 2)) for k in range(2)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    hb = [torch.empty((N // 2, 66), dtype=torch.int64, device=dev) for _ in range(2)]
    for k in range(2):
        with torch.cuda.stream(streams[k]):
            halves[k].dephase()
            halves[k].step_sampled(args.burn_in)
            halves[k].set_mask_output(hb[k])
    torch.cuda.synchronize()

    def two_streams():
        for k in range(2):
            with torch.cuda.stream(streams[k]):
                halves[k].step_index(words[i[0] % 8, k * (N // 2):(k + 1) * (N // 2)])
        i[0] += 1

    for _ in range(3):
        two_streams()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(ksteps):
        two_streams()
    torch.cuda.synchronize()
    out["step_plus_bitmask"]["two_streams_value"] = N * ksteps / (time.perf_counter() - t0)
    for h in halves:
        h.close()
    del bits, bits65, lstN, cntN, hb

    # ---- BASELINE.json configs[2]: 65,536 envs on one GPU
    small = BatchedChessEnv(65536, opponent="none", seed=2, device=local_rank)
    small.dephase()
    small.step_sampled(args.burn_in)
    t = median(timed_repeats(lambda: small.step_sampled(max(K, 64)), 3))
    out["config_65536_envs"] = {"value": 65536 * max(K, 64) / (t * 1e-3), "unit": UNIT, "steps": max(K, 64),
                                "note": "2,048 warps on a device that holds 2,960: 69 % of the resident capacity"}
    small.close()
    # ---- BASELINE.json configs[4]: repetition / promotion-heavy endgames, 512-slot Zobrist-hash history, 1M envs (the
    # regime in which the repetition windows are long: mean window ~80 plies)
    from gym_chess_b200.boards import endgame_boards
    eg = BatchedChessEnv(1 << 20, opponent="none", seed=5, device=local_rank, initial_boards=endgame_boards(), moves_max=250,
                         history_cap=512)
    eg.step_sampled(600)
    eg.reset_stats()
    t = loop_ms(lambda: eg.step_sampled(200), 1)
    egs = eg.stats()
    out["config_endgames_1M_envs"] = {"value": (1 << 20) * 200 / (t * 1e-3), "unit": UNIT,
                                      "mean_hist_window": egs["hist_window"] / max(1, egs["plies"]),
                                      "extra_table_probes_per_ply": egs["hist_scanned"] / max(1, egs["plies"]),
                                      "repetitions": egs["repetitions"], "history_cap": 512}
    eg.close()
    # ---- BASELINE.json configs[0]: the reference's own CPU-runnable case -- a single env, random-vs-random self-play,
    # ~1k games -- on ONE host thread (the reference is single-threaded), plus legal-movegen positions/s of the same
    # code on one thread and on all of them (a 65,536-position sample of the fixed set).  The engine is the oracle port.
    from oracle import oracle as orc
    t0 = time.time()
    s1 = orc.selfplay_mt(0, 0, 1, 270000, 1)
    dt1 = time.time() - t0
    nthreads = os.cpu_count() or 1
    t0 = time.time()
    orc.movegen_batch(boards[:16384], players[:16384], rights[:16384], False, stride=144, threads=1)
    dtm1 = time.time() - t0
    t0 = time.time()
    orc.movegen_batch(boards[:262144], players[:262144], rights[:262144], False, stride=144, threads=nthreads)
    dtma = time.time() - t0
    out["config_1_cpu"] = {
        "workload": "single env, random self-play (opponent none), 270,000 steps = %d games, 1 thread" % s1["episodes"],
        "env_steps_per_sec_1_thread": s1["steps"] / dt1, "movegen_positions_per_sec_1_thread": 16384 / dtm1,
        "movegen_positions_per_sec_all_threads": 262144 / dtma, "threads": nthreads, "kind": "port",
        "reference_published": {"env_steps_per_sec": 3205, "movegen_positions_per_sec": 4167,
                                "source": "gym_chess/test/v2/test_benchmark.py:46-50, README.md:372-374 (1 thread, unspecified CPU)"}}
    # ---- CPU baseline on this box's host cores: the same procedure as `--impl reference`
    r = cpu_arm(K, args.warmup)
    out["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                           "sample": cpu_sample_text(r, K) + "; reference's published single-thread figure: 3.2e3 steps/s"}
    return out


if __name__ == "__main__":
    main()
