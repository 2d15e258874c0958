"""Search pit throughput: pit_mp_game_runner.MPGameRunner.run with the search Agent (training=False, depth 8) on both sides, two
random-init native AlphaNNets, at pit.py's shape (1,000 games, 1 vs 1 on 11x11).  For each breadth, the device arena (native=None)
and the runner's Python loop (native=False) play the same seeded match; the script checks that they return the same winners.
Reports wall time per match, turns, network evaluations per second (both sides' searchers), the share of the arena's wall time
spent in the searches (copy + root-turn search, host clock: every search ends in a host synchronisation), and loop / arena.
Prints one JSON line.
  python tools/bench_search_pit.py [--breadths 32,128] [--games 1000] [--no-loop]"""
import json
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from bench_pit import gpu_info  # noqa: E402
from alphasnake_zero_b200.utils.agent import Agent  # noqa: E402
from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet  # noqa: E402
from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner  # noqa: E402

SIDE, SNAKES, ALICE, DEPTH, BASE = 11, 2, 1, 8, 100


def play(G, breadth, nets, native, seed=5):
    gr = MPGameRunner(SIDE, SIDE, SNAKES, 1, G, seed=seed)
    agents = [Agent(n, softmax_base=BASE, training=False, max_MCTS_depth=DEPTH, max_MCTS_breadth=breadth) for n in nets]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    winners = gr.run(agents[0], agents[1], ALICE, native=native)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    evals = sum(q.search_stats()["evals"] for _, q in gr._searchers)
    return gr, winners, wall, evals


def main():
    breadths = [32, 128]
    if "--breadths" in sys.argv:
        breadths = [int(b) for b in sys.argv[sys.argv.index("--breadths") + 1].split(",")]
    G = int(sys.argv[sys.argv.index("--games") + 1]) if "--games" in sys.argv else 1000
    if not torch.cuda.is_available():
        raise SystemExit("bench_search_pit.py measures the device pit: it needs a CUDA device")
    nets = [AlphaNNet(input_shape=(2 * SIDE - 1, 2 * SIDE - 1, 3), seed=s) for s in (1, 2)]
    for b in breadths:                                # warm-up: module loads, first allocations, both paths at every breadth
        for native in (None, False):
            play(16, b, nets, native)
    out = {"gpu": gpu_info(), "nets": "random init, seeds 1 and 2", "games": G, "snakes": SNAKES, "alice_snakes": ALICE,
           "side": SIDE, "health_dec": 1, "depth": DEPTH, "softmax_base": BASE}
    for b in breadths:
        gr, w_arena, t_arena, evals = play(G, b, nets, None)
        st = gr.engine.pit_stats()
        r = {"turns": st["turns"], "network_evals": evals, "searched_rows": st["search_rows"],
             "arena": {"wall_s": t_arena, "ms_per_turn": t_arena * 1e3 / max(st["turns"], 1), "evals_per_s": evals / t_arena,
                       "search_s": st["search_ms"] * 1e-3, "search_share": st["search_ms"] * 1e-3 / t_arena}}
        del gr
        if "--no-loop" not in sys.argv:
            _, w_loop, t_loop, evals_loop = play(G, b, nets, False)
            r["loop"] = {"wall_s": t_loop, "ms_per_turn": t_loop * 1e3 / max(st["turns"], 1), "evals_per_s": evals_loop / t_loop}
            r["same_winners"] = w_loop == w_arena
            r["same_evals"] = evals_loop == evals
            r["loop_over_arena"] = t_loop / t_arena
        else:
            r["loop"] = "not measured"
        out["breadth_%d" % b] = r
    print(json.dumps(out))


if __name__ == "__main__":
    main()
