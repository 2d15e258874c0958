"""One generation of AlphaSnake-Zero training on the B200 engine: the body of AlphaSnakeZeroTrainer.train
(alpha_snake_zero_trainer.py:52-91) with the drop-in classes, followed by a pit of the new net against the old one
(pit.py:28-35).  Small defaults so that it finishes in about a minute on one GPU:

  python examples/selfplay_generation.py [--games 256] [--breadth 32] [--depth 8] [--pit-games 100]
"""
import argparse
import os
import sys
from random import sample
from time import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from alphasnake_zero_b200.utils.agent import Agent  # noqa: E402
from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet  # noqa: E402
from alphasnake_zero_b200.utils.mp_game_runner import MPGameRunner  # noqa: E402
from alphasnake_zero_b200.utils import pit_agent, pit_mp_game_runner  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=256)
    ap.add_argument("--breadth", type=int, default=32)
    ap.add_argument("--depth", type=int, default=8)
    ap.add_argument("--pit-games", type=int, default=100)
    ap.add_argument("--name", default="Example")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp8"],
                    help="value network of the native backend: bf16 (reference) or the opt-in fp8 tower")
    a = ap.parse_args()
    iteration, health_dec, lr = 0, 9, 1e-4                                 # train.py:6-13, trainer :42-47
    nnet = AlphaNNet(input_shape=(21, 21, 3), dtype=a.dtype).copy_and_compile()
    t0 = time()
    Alice = Agent(nnet, 2 + iteration, True, a.depth, a.breadth)           # :52
    gr = MPGameRunner(11, 11, 4, health_dec, a.games, verbose=False)       # :53
    gr.run(Alice)                                                          # :54
    print("self-play: %d games, %d training records, %.1f s" % (a.games, len(Alice.records), time() - t0))
    print("log: wall %.3f body %.3f head %.3f starve %.3f food %.3f length %.2f" %
          (gr.wall_collision, gr.body_collision, gr.head_collision, gr.starvation, gr.food_eaten, gr.game_length))
    batch_size = 2048                                                      # :63-75
    batches = min(5, len(Alice.records) // batch_size)
    samples = batch_size * batches
    if samples == 0 or samples > len(Alice.records):
        batch_size = samples = len(Alice.records)
    idx = sample(range(len(Alice.records)), samples)
    X = [Alice.records[i] for i in idx]
    V = [Alice.values[i] for i in idx]
    Alice.clear()
    X += list(np.flip(X, axis=2))                                          # mirror_states / mirror_values, :93-100
    V += list(np.flip(V, axis=1))
    new = nnet.copy_and_compile(learning_rate=lr)                          # :79
    t0 = time()
    new.train(X, V, batch_size=batch_size)                                 # :81
    print("training on %d samples: %.1f s" % (len(X), time() - t0))
    new = new.copy_and_compile()
    new.save(a.name + str(iteration + 1))                                  # :91
    t0 = time()
    winners = pit_mp_game_runner.MPGameRunner(11, 11, 2, health_dec, a.pit_games).run(pit_agent.Agent(new), pit_agent.Agent(nnet), 1)
    wins = sum(w == 0 for w in winners); losses = sum(w == 1 for w in winners)
    print("pit, new vs old, %d games of 2 snakes: %d wins, %d losses, %d draws, %.1f s" %
          (a.pit_games, wins, losses, a.pit_games - wins - losses, time() - t0))


if __name__ == "__main__":
    main()
