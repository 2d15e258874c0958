"""Pit throughput: the device arena (asz_pit_run behind pit_mp_game_runner.MPGameRunner.run) against the Python loop of the same
runner (native=False), with two random-init native AlphaNNets, at the shapes of pit.py (1,000 games, 1 vs 1 on 11x11), test_pit.py
(300 games, 1 vs 3 and 3 vs 1) and one large shape (16,384 games, 2 vs 2).  Both paths play the same seeded match; the script
checks that they return the same winners.  Prints one JSON line.
  python tools/bench_pit.py [--no-loop-above G] [--shapes name,name]"""
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet  # noqa: E402
from alphasnake_zero_b200.utils.pit_agent import Agent  # noqa: E402
from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner  # noqa: E402

SHAPES = {  # name: (side, snakes, games, Alice's snakes)
    "pit_py_1v1": (11, 2, 1000, 1),
    "test_pit_1v3": (11, 4, 300, 1),
    "test_pit_3v1": (11, 4, 300, 3),
    "large_2v2": (11, 4, 16384, 2),
}


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def play(side, S, G, acnt, nets, native, seed=5):
    gr = MPGameRunner(side, side, S, 1, G, seed=seed)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    winners = gr.run(Agent(nets[0]), Agent(nets[1]), acnt, native=native)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return gr, winners, wall


def main():
    skip_loop_above = 1 << 30
    if "--no-loop-above" in sys.argv:
        skip_loop_above = int(sys.argv[sys.argv.index("--no-loop-above") + 1])
    names = list(SHAPES)
    if "--shapes" in sys.argv:
        names = sys.argv[sys.argv.index("--shapes") + 1].split(",")
    if not torch.cuda.is_available():
        raise SystemExit("bench_pit.py measures the device pit: it needs a CUDA device")
    nets = [AlphaNNet(input_shape=(21, 21, 3), seed=s) for s in (1, 2)]
    for native in (True, False):                    # warm-up: module loads, first allocations, first forwards of both paths
        play(11, 2, 64, 1, nets, native)
    out = {"gpu": gpu_info(), "nets": "random init, seeds 1 and 2", "health_dec": 1}
    for name in names:
        side, S, G, acnt = SHAPES[name]
        gr, w_arena, t_arena = play(side, S, G, acnt, nets, True)
        st = gr.engine.pit_stats()
        r = {"games": G, "snakes": S, "alice_snakes": acnt, "turns": st["turns"], "network_evals": st["net_rows"],
             "arena": {"wall_s": t_arena, "games_per_s": G / t_arena, "evals_per_s": st["net_rows"] / t_arena,
                       "ms_per_turn": t_arena * 1e3 / max(st["turns"], 1), "forward_ms": st["forward_ms"],
                       "forward_share": st["forward_ms"] * 1e-3 / t_arena}}
        del gr
        if G <= skip_loop_above:
            _, w_loop, t_loop = play(side, S, G, acnt, nets, False)
            r["loop"] = {"wall_s": t_loop, "games_per_s": G / t_loop, "evals_per_s": st["net_rows"] / t_loop,
                         "ms_per_turn": t_loop * 1e3 / max(st["turns"], 1)}
            r["same_winners"] = w_loop == w_arena
            r["speedup"] = t_loop / t_arena
        else:
            r["loop"] = "not measured"
        out[name] = r
    print(json.dumps(out))


if __name__ == "__main__":
    main()
