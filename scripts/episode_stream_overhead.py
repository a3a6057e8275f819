"""What does drawing episodes on the device cost?  (GPU) The bench's rollout configuration (L-DGN, N = 50, B = 32768,
bf16, captured CUDA graph, L2 flushed between rounds), once restarting finished episodes from the host-built tuple
pool and once from the device episode stream (EpisodeStream), in the same process, alternating; then the same for
env-only rounds (fixed random actions, no network).

Per workload: median round time over the repetitions (CUDA events, one per round), the spread of the per-repetition
medians, and the episode restarts per round; then a torch.profiler kernel breakdown of a few rounds of each source.

    python scripts/episode_stream_overhead.py [--reps 15] [--steps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from melissa_b200 import _lib
from melissa_b200.batched_env import BatchedGraphEnv, EpisodeStream, ResetTuplesDevice
from melissa_b200.networks import NETWORKS
from melissa_b200.rollout import Rollout

N, B, G = 50, 32768, 1024
PREROLL = 30              # untimed rounds after start: episodes spread over their lifetimes, restarts at steady state


def make(source, with_net, dev, pool):
    env = BatchedGraphEnv(B, N, pool, device=dev)
    net = None
    if with_net:
        torch.manual_seed(9)
        net = NETWORKS["l_dgn"](5, 128, 2, 4, N, dueling_param=({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]}),
                                device=str(dev)).to(dev)
        net.set_precision("bf16")
    ro = Rollout(env, net, eps=0.05, seed=9)
    ro.start(source)
    if net is None:
        g = torch.Generator(device=dev)
        g.manual_seed(9)
        ro.act.copy_(torch.randint(0, 2, ro.act.shape, device=dev, dtype=torch.int8, generator=g))
    for _ in range(PREROLL - 2):
        ro.round()
    ro.capture(warmup_rounds=2)
    torch.cuda.synchronize()
    return ro


def timed(ro, steps, flush):
    """Per-round device times of `steps` captured rounds (L2 flushed before each, outside the events) and the restarts."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    r0 = int(ro.env.episode[:, _lib.MLS_EP_N_RESETS].sum())
    torch.cuda.synchronize()
    for a, b in evs:
        flush.zero_()
        a.record()
        ro.round()
        b.record()
    torch.cuda.synchronize()
    restarts = int(ro.env.episode[:, _lib.MLS_EP_N_RESETS].sum()) - r0
    return [a.elapsed_time(b) for a, b in evs], restarts


def kernel_breakdown(ro, rounds):
    """Device time per kernel name over `rounds` captured rounds (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    warnings.filterwarnings("ignore", message=".*Profiler clears events")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(rounds):
            ro.round()
        torch.cuda.synchronize()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and e.count > 0:
            rows.append((e.key, e.count, t / rounds))
    rows.sort(key=lambda r: -r[2])
    return [{"kernel": k[:110], "launches_per_round": round(c / rounds, 2), "us_per_round": round(t, 2)} for k, c, t in rows[:12]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--profile-rounds", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("episode_stream_overhead.py needs a GPU")
    dev = torch.device("cuda")
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    print(json.dumps({"card": torch.cuda.get_device_name(), "power_limit": power, "N": N, "B": B, "graphs": G,
                      "reps": args.reps, "steps_per_rep": args.steps, "preroll_rounds": PREROLL,
                      "l2": "flushed before every round (256 MiB memset outside the events)"}), flush=True)
    pool = bench.load_pool(N, G)
    gi, src, inter, scr = bench.load_tuples(N, G, 2 * B)
    tuples = ResetTuplesDevice(gi, src, inter, scr, N, dev, pool_size=G)
    stream = EpisodeStream(N, G, seed=9)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for workload, with_net in (("rollout_l_dgn_bf16", True), ("env_only", False)):
        ros = {"pool": make(tuples, with_net, dev, pool), "stream": make(stream, with_net, dev, pool)}
        for name in ros:                                      # warm-up of the timing loop itself
            timed(ros[name], 3, flush)
        per_rep = {k: [] for k in ros}
        restarts = {k: 0 for k in ros}
        rounds = {k: 0 for k in ros}
        for i in range(args.reps):
            for name in (("pool", "stream") if i % 2 == 0 else ("stream", "pool")):
                ms, r = timed(ros[name], args.steps, flush)
                per_rep[name].append(float(np.median(ms)))
                restarts[name] += r
                rounds[name] += args.steps
        med = {k: float(np.median(v)) for k, v in per_rep.items()}
        out = {"workload": workload,
               "round_ms_median": {k: round(v, 4) for k, v in med.items()},
               "round_ms_rep_medians_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in per_rep.items()},
               "stream_over_pool": round(med["stream"] / med["pool"] - 1.0, 4),
               "restarts_per_round": {k: round(restarts[k] / rounds[k], 1) for k in ros}}
        print(json.dumps(out), flush=True)
        for name, ro in ros.items():
            print(json.dumps({"workload": workload, "source": name,
                              "kernels": kernel_breakdown(ro, args.profile_rounds)}), flush=True)
        del ros
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
