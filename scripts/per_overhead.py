"""What does prioritized replay cost?  (GPU) At the bench's training configuration (L-DGN, N = 50, B = 32768, bf16
rollout, DQNPolicy n_step 4 / gamma 0.99 / target_update_freq 500, Adam lr 1e-3, M = 4096 sampled transitions):

* DQNPolicy.update with the uniform ring and with the prioritized ring (alpha 0.6, beta 0.4), in the same process,
  alternating, at ring 8 (the bench's) and ring 64 -- both rings hold the same rounds (one collector feeds both);
* CUDA event times of the three prioritized-replay kernels: round build (rotating over the ring's slots), sample and
  update at M = 4096.

    python scripts/per_overhead.py [--pairs 30]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from melissa_b200 import _lib
from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
from melissa_b200.data_parallel import FlatParameters, FusedAdam
from melissa_b200.networks import NETWORKS
from melissa_b200.policy import BatchedCollector, DQNPolicy
from melissa_b200.replay import DevicePrioritizedReplay, DeviceReplay

N, B, G, M = 50, 32768, 1024, 4096
ROUND_MS = 2.72            # bench rollout round, L-DGN N = 50 B = 32768 (DESIGN section 3)


class Both:
    """Stores every round in two rings (the collector's ``buffer`` only needs begin_round / end_round)."""

    def __init__(self, *rings):
        self.rings = rings

    def begin_round(self, obs, active):
        for r in self.rings:
            r.begin_round(obs, active)

    def end_round(self, act, reward, terminated):
        for r in self.rings:
            r.end_round(act, reward, terminated)


def event_ms(fn, reps):
    """Mean device time of fn() over reps calls, bracketed by one event pair."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run(ring, pairs, pool, tuples, dev):
    torch.manual_seed(9)
    net = NETWORKS["l_dgn"](5, 128, 2, 4, N, dueling_param=({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]}),
                            device="cuda").to(dev)
    net.set_precision("bf16")
    pol = DQNPolicy(net, FusedAdam(FlatParameters(net), lr=1e-3), discount_factor=0.99, estimation_step=4,
                    target_update_freq=500, eps=0.05)
    env = BatchedGraphEnv(B, N, pool, device=dev, want_info=True)
    uni = DeviceReplay(B, N, ring, device=dev)
    per = DevicePrioritizedReplay(B, N, ring, alpha=0.6, beta=0.4, device=dev)
    gi, src, inter, scr = tuples
    col = BatchedCollector(agents_num=N, policy=pol, env=env, buffer=Both(uni, per), exploration_noise=True,
                           tuples=ResetTuplesDevice(gi, src, inter, scr, N, dev, pool_size=G))
    for _ in range(ring):
        col.iterate(0.05)
    for _ in range(10):                          # warm up both paths (cuBLAS variants for the sampled row counts)
        pol.update(M, uni)
        pol.update(M, per)
    times = {"uniform": [], "prioritized": []}
    for i in range(pairs):
        order = [("uniform", uni), ("prioritized", per)]
        for name, rep in (order if i % 2 == 0 else order[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            pol.update(M, rep)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
    med = {k: float(np.median(v)) for k, v in times.items()}
    # the three kernels on their own
    L, st = per.lib, _lib.current_stream_ptr()
    build_ms = event_ms(lambda i=0: _lib.check(L.mls_per_build(per.flags[i % ring].data_ptr(), B, N, per.prio.data_ptr(),
                                                                per.alpha, per.tree[i % ring].data_ptr(), st)), 10 * ring)
    first, usable = per._usable_rounds(4)
    u = torch.rand(M, dtype=torch.float64, device=dev)
    rho, ep, ag = (torch.empty(M, dtype=torch.int32, device=dev) for _ in range(3))
    sample_ms = event_ms(lambda i=0: _lib.check(L.mls_per_sample(per.tree.data_ptr(), ring, B, N, first, usable, u.data_ptr(), M,
                                                                 rho.data_ptr(), ep.data_ptr(), ag.data_ptr(), None, st)), 200)
    td = torch.randn(M, dtype=torch.float32, device=dev)
    update_ms = event_ms(lambda i=0: _lib.check(L.mls_per_update(per.tree.data_ptr(), ring, B, N, rho.data_ptr(), ep.data_ptr(),
                                                                 ag.data_ptr(), td.data_ptr(), M, per.alpha, per.eps,
                                                                 per.prio.data_ptr(), per.prio[1:].data_ptr(), st)), 200)
    tree_mb = per.tree[0].numel() * 8 / 1e6
    out = {
        "ring_rounds": ring, "pairs": pairs,
        "update_ms_median": {k: round(v, 4) for k, v in med.items()},
        "update_ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()},
        "prioritized_over_uniform": round(med["prioritized"] / med["uniform"] - 1.0, 4),
        "kernel_us": {"build_per_round": round(build_ms * 1e3, 2), "sample_M4096": round(sample_ms * 1e3, 2),
                      "update_M4096": round(update_ms * 1e3, 2)},
        "build_share_of_round": round(build_ms / ROUND_MS, 5),
        "build_note": (f"rotating over {ring} slots of {tree_mb:.1f} MB trees "
                       f"({'fits' if ring * tree_mb < 126 else 'exceeds'} the 126 MB L2); share against the {ROUND_MS} ms rollout round"),
    }
    print(json.dumps(out), flush=True)
    del col, env, uni, per, pol, net
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=30)
    ap.add_argument("--rings", type=int, nargs="+", default=[8, 64])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("per_overhead.py needs a GPU")
    dev = torch.device("cuda")
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    print(json.dumps({"card": torch.cuda.get_device_name(), "power_limit": power, "N": N, "B": B, "M": M}), flush=True)
    pool = bench.load_pool(N, G)
    tuples = bench.load_tuples(N, G, 65536)
    for ring in args.rings:
        run(ring, args.pairs, pool, tuples, dev)


if __name__ == "__main__":
    main()
