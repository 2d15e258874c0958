"""Self-play throughput of one BASELINE.json configuration on this process's GPU (one process per GPU under torchrun;
games shard by game id with no collective on the hot path, SURVEY.md 8(e)).

  python tools/bench_selfplay.py --config 3|4|5 [--world 8] [--turns 2] [--dtype bf16|fp8]
  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/bench_selfplay.py --config 4

--world: number of GPUs the configuration is sharded over; the per-GPU share of the games is what runs here
(configs[3]: 32,768 games x 200 sims over 8 GPUs = 4,096 per GPU; configs[4]: 8,192 games of 19x19 x 8 snakes x 400 sims
over 8 GPUs = 1,024 per GPU).  Under torchrun the aggregate over the ranks that really ran is printed as well.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

CONFIGS = {3: dict(side=11, snakes=4, games=4096, breadth=100, world=1, label="configs[2]"),
           4: dict(side=11, snakes=4, games=32768, breadth=200, world=8, label="configs[3]"),
           5: dict(side=19, snakes=8, games=8192, breadth=400, world=8, label="configs[4]")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--world", type=int, default=0, help="GPUs the configuration is sharded over (default: the config's own)")
    ap.add_argument("--turns", type=int, default=2)
    ap.add_argument("--stub", action="store_true", help="stub value function (search kernels only)")
    ap.add_argument("--prewarm-tics", type=int, default=32, help="uniform-random tics (with reset) before the search starts")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp8"],
                    help="value network: bf16 (reference) or the opt-in fp8 tower (built and calibrated before the timed turns)")
    args = ap.parse_args()
    import torch
    rank = int(os.environ.get("RANK", "0")); nproc = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    c = CONFIGS[args.config]
    world = args.world or c["world"]
    games = c["games"] // world
    if nproc > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
        dist.barrier()
    from alphasnake_zero_b200.utils import alpha_nnet
    bf16_net = alpha_nnet.AlphaNNet
    if args.dtype != "bf16":
        # bench.selfplay_leg builds its AlphaNNet by name from this module: hand it one of the requested dtype for this call
        class Net(bf16_net):
            def __init__(self, *a, **k):
                super().__init__(*a, dtype=args.dtype, **k)
        alpha_nnet.AlphaNNet = Net
    try:
        r = bench.selfplay_leg(rank, games, c["breadth"], 8, args.turns, 1, use_net=not args.stub, side=c["side"], snakes=c["snakes"],
                               label="%s, 1/%d of the games per GPU" % (c["label"], world), prewarm_tics=args.prewarm_tics)
    finally:
        alpha_nnet.AlphaNNet = bf16_net
    if args.dtype != "bf16" and not args.stub:
        r["workload"] = r["workload"].replace("bf16 tcgen05 value net", "%s tcgen05 value net" % args.dtype)
        r.pop("net_roofline", None)                       # its peak is the bf16 one
    r["dtype"] = "stub" if args.stub else args.dtype
    r["ranks_run"] = nproc
    if nproc > 1:
        rates = ("sims_per_sec", "node_visits_per_sec", "nn_evals_per_sec", "subgame_tics_per_sec")
        t = torch.tensor([r["seconds"]] + [r[k] * r["seconds"] for k in rates], dtype=torch.float64, device="cuda")
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        r["seconds"] = float(mx[0])
        for i, k in enumerate(rates):
            r[k] = float(sm[1 + i]) / float(mx[0])          # whole job: work of all ranks / slowest rank's time
        r["aggregate_over_gpus"] = nproc
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(r))


if __name__ == "__main__":
    main()
