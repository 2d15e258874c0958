"""A CI-sized pass over every kernel of the engine, meant to be run under compute-sanitizer (one tool per gpurun call):
  compute-sanitizer --tool memcheck python tools/sanitize_run.py
  compute-sanitizer --tool racecheck python tools/sanitize_run.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from alphasnake_zero_b200 import _lib  # noqa: E402
from alphasnake_zero_b200.engine import Engine  # noqa: E402
from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet  # noqa: E402
from alphasnake_zero_b200.net import NativeNet  # noqa: E402


def main():
    for side, S in ((11, 4), (7, 4), (19, 8)):
        eng = Engine(side=side, snakes=S, health_dec=1, games=96, seed=1, max_depth=4, max_breadth=8, softmax_base=2.0, training=True,
                     table_log2=14)
        eng.reset()
        for _ in range(6):
            eng.step(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=True, auto_reset=True, random_actions=True, keys=True)
        net = AlphaNNet(input_shape=(2 * side - 1, 2 * side - 1, 3), seed=0, backend="native")
        net._native = NativeNet(net.weights, "cuda", chunk_images=64)
        q, mv = eng.search(net=net._native)
        act = torch.where(mv < 3, mv, torch.ones_like(mv))
        eng.step(actions=act, spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=False, auto_reset=True)
        q, mv = eng.search(value_fn=None)
        torch.cuda.synchronize()
        st = eng.search_stats()
        assert st["evals"] > 0 and np.isfinite(q.cpu().numpy()).all()
        eng.close()
        # one pit per board size: the network against a stand-in player (asz_pit_*), stepwise with a replayed trace, then in one call
        pit = Engine(side=side, snakes=S, health_dec=3, games=48, seed=2)
        pit.reset()
        pit.pit_begin(net._native, 0, S // 2)
        moves = torch.empty(48, 8, dtype=torch.uint8, device="cuda")
        cells = torch.full((48,), -1, dtype=torch.int32, device="cuda")
        for _ in range(3):
            pit.pit_turn(spawn_cells=cells, spawn_mode=_lib.SPAWN_REPLAY, moves=moves)
        try:
            pit.pit_finish()
        except _lib.AszError:
            pass                                  # games still running after three turns: the results so far are written
        pit.reset()
        w, d, turns = pit.pit_run(net._native, 1, S // 2)
        torch.cuda.synchronize()
        assert (d >= 1).all() and turns == d.max()
        print("side %d ok: %d evals, pit of %d turns" % (side, st["evals"], turns))
        pit.close()


if __name__ == "__main__":
    main()
