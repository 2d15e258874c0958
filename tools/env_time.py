"""Per-launch timing of env_step_kernel on BASELINE.json configs[1] (65,536 games, tic + encode, in-kernel actions, in-place
reset): median / p05 / p95 over per-launch CUDA events, the algorithmic GB/s and the fraction of the measured HBM copy peak.
  [ASZ_LIB=tools/libasz_b200_<variant>.so] python tools/env_time.py [launches]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from alphasnake_zero_b200.engine import Engine  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 600
G = 65536
if "LOCAL_RANK" in os.environ:
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
nccl_mode = sys.argv[3] if len(sys.argv) > 3 else ""


def nccl_init():
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    dist.barrier()


if nccl_mode == "nccl":           # communicator first, engine second
    nccl_init()
eng = Engine(side=11, snakes=4, health_dec=1, games=G, seed=1)
eng.reset()
if nccl_mode == "nccl_after":     # engine first
    _ = eng.planes
    nccl_init()
kw = dict(spawn_mode=2, tic=True, encode=True, auto_reset=True, random_actions=True)
for _ in range(50):
    eng.step(**kw)
torch.cuda.synchronize()
t0 = eng.totals()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
ev[0].record()
for i in range(n):
    eng.step(**kw)
    ev[i + 1].record()
torch.cuda.synchronize()
t1 = eng.totals()
d = np.array([ev[i].elapsed_time(ev[i + 1]) * 1000 for i in range(n)])
tot_us = ev[0].elapsed_time(ev[n]) * 1000
planes_n, tics = t1["planes"] - t0["planes"], t1["tics"] - t0["tics"]
bytes_per_launch = (planes_n * 5292 + tics * 256) / n
peak = 6458.1
try:
    peak = float(json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass
gbs = bytes_per_launch / (tot_us / n) / 1e3
print("%s pitched: %d launches, %.1f us/launch (events per launch: median %.1f, p05 %.1f, p95 %.1f, max %.1f) | %.0f MB algorithmic per launch, "
      "%.0f GB/s = %.3f of %.0f GB/s | %.3e env steps/s" % (os.environ.get("ASZ_LIB", "libasz_b200.so"), n, tot_us / n,
       np.median(d), np.percentile(d, 5), np.percentile(d, 95), d.max(), bytes_per_launch / 1e6, gbs, gbs / peak, peak, tics / (tot_us * 1e-6)))
