"""fp32 vs bf16 training precision of the DQN update, per network family (GPU).

    python scripts/train_precision.py [--models l_dgn,dgn_r,hl_dgn] [--samples 4096] [--profile]

For each model: the bench's training configuration (N = 50, 8192 episodes, replay ring of 8 rounds filled by the collector,
bf16 rollout), then one ``DQNPolicy.update`` of ``--samples`` transitions timed with CUDA events, fp32 and bf16 training
precision alternating in the same process after every shape is warmed up; the median of 9 per precision.  Then, on one
sampled batch, max |dq| of bf16 against fp32 and the relative L2 gradient error of every parameter (worst three listed).
``--profile`` instead prints a torch.profiler kernel table of one update per precision (a separate run: tracing slows the host).
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
from melissa_b200.data_parallel import FlatParameters, FusedAdam
from melissa_b200.networks import NETWORKS
from melissa_b200.networks.autograd import q_values
from melissa_b200.policy import Batch, BatchedCollector, DQNPolicy
from melissa_b200.replay import DeviceReplay

N, B, G = 50, 8192, 1024


def setup(model, dev, tuples, pool):
    torch.manual_seed(9)
    kw = dict(aggregator="max") if model == "hl_dgn" else {}
    net = NETWORKS[model](5, 128, 2, 4, N, dueling_param=({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]}),
                          device=str(dev), **kw).to(dev)
    net.set_precision("bf16")
    optim = FusedAdam(FlatParameters(net), lr=1e-3)
    pol = DQNPolicy(net, optim, 0.99, 4, 500, eps=0.05)
    env = BatchedGraphEnv(B, N, pool, device=dev, want_info=True)
    replay = DeviceReplay(B, N, 8, device=dev)
    col = BatchedCollector(agents_num=N, policy=pol, env=env, buffer=replay, exploration_noise=True,
                           tuples=ResetTuplesDevice(*tuples, N, dev, pool_size=G))
    for _ in range(8):
        col.iterate(0.05)
    return net, pol, replay


def timed_update(pol, replay, m):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    pol.update(m, replay)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def accuracy(net, replay, m):
    rho, ep, ag = replay.sample_indices(m, 4)
    rows = Batch(replay.gather(rho, ep, ag, 4, 0.99)).obs
    target = torch.linspace(-1, 1, rows.shape[0], device=rows.device)
    res = {}
    for prec in ("fp32", "bf16"):
        net.set_train_precision(prec)
        net.zero_grad(set_to_none=True)
        q = q_values(net, rows)
        ((q[:, 0] - target).pow(2).mean() + q[:, 1].mean()).backward()
        res[prec] = (q.detach(), {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None})
    (q32, g32), (q16, g16) = res["fp32"], res["bf16"]
    # TransformerConv's key bias has an exact gradient of zero (softmax shift invariance): its error is reported against the
    # key weights' gradient instead
    rel = {k: float((g16[k] - g).norm() / g.norm()) for k, g in g32.items() if float(g.norm()) > 0 and not k.endswith("lin_key.bias")}
    key_bias = {k: float((g16[k] - g).norm() / g32[k[:-4] + "weight"].norm()) for k, g in g32.items() if k.endswith("lin_key.bias")}
    dq = float((q16 - q32).abs().max())
    return dq, float(q32.abs().max()), rel, key_bias


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", default="l_dgn,dgn_r,hl_dgn")
    ap.add_argument("--samples", type=int, default=4096)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    dev = torch.device("cuda")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    print(q.stdout.strip() or q.stderr.strip())
    pool = bench.load_pool(N, G)
    tuples = bench.load_tuples(N, G, 65536)
    m = args.samples
    print(f"N = {N}, {B} episodes, replay ring 8 rounds, {m} samples per update; median of 9 updates per precision, alternating")
    for model in args.models.split(","):
        net, pol, replay = setup(model, dev, tuples, pool)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            for prec in ("fp32", "bf16"):
                net.set_train_precision(prec)
                for _ in range(3):
                    pol.update(m, replay)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    pol.update(m, replay)
                    torch.cuda.synchronize()
                print(f"== {model} {prec}: one update")
                print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20, max_name_column_width=70))
            continue
        times = {"fp32": [], "bf16": []}
        for prec in ("fp32", "bf16"):                        # warm up every shape of both paths
            net.set_train_precision(prec)
            for _ in range(3):
                timed_update(pol, replay, m)
        for _ in range(9):
            for prec in ("fp32", "bf16"):
                net.set_train_precision(prec)
                times[prec].append(timed_update(pol, replay, m))
        med = {p: sorted(t)[len(t) // 2] for p, t in times.items()}
        dq, qmax, rel, key_bias = accuracy(net, replay, m)
        worst = sorted(rel.items(), key=lambda kv: -kv[1])[:3]
        print(f"{model:7s} update fp32 {med['fp32']:.3f} ms  bf16 {med['bf16']:.3f} ms  ({med['fp32'] / med['bf16']:.2f}x)  "
              f"max|dq| {dq:.2e} (max|q| {qmax:.3f})  grad rel err max {worst[0][1]:.2e}  worst: "
              + ", ".join(f"{k} {v:.2e}" for k, v in worst)
              + "".join(f"  {k} err / |key weight grad| {v:.2e}" for k, v in key_bias.items()))
        del net, pol, replay
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
