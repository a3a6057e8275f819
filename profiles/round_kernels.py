"""Per-kernel GPU time of the headline rollout rounds under torch.profiler (CUDA activity), run in a process of its own:

    python profiles/round_kernels.py OUT.txt [bench.py arguments]

Runs bench.py's main with the given arguments inside the profiler and writes one line per kernel name: launches,
total and mean time.  Tracing slows the host, so take step times from bench.py itself, not from this run."""
import os
import runpy
import sys

import torch
from torch.profiler import ProfilerActivity, profile

out, args = sys.argv[1], sys.argv[2:]
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, root)
sys.argv = [os.path.join(root, "bench.py"), *args]
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    try:
        runpy.run_path(sys.argv[0], run_name="__main__")
    except SystemExit:
        pass
    torch.cuda.synchronize()
rows = [e for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA and e.count > 0]
rows.sort(key=lambda e: -e.device_time_total)
total = sum(e.device_time_total for e in rows)
with open(out, "w") as f:
    f.write(f"# bench.py {' '.join(args)} ; {torch.cuda.get_device_name()} ; all launches of the run (warm-up and timed rounds)\n")
    f.write(f"{'share':>6} {'launches':>8} {'total_ms':>10} {'mean_us':>9}  kernel\n")
    for e in rows:
        f.write(f"{100 * e.device_time_total / total:5.1f}% {e.count:8d} {e.device_time_total / 1e3:10.3f} "
                f"{e.device_time_total / e.count:9.1f}  {e.key[:140]}\n")
