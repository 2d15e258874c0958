"""What the fp8 tower costs in play: trains generations in bf16 (the body of examples/selfplay_generation.py, from a seeded
random-init network), then, with the last generation's weights,
  * pits a search Agent on the fp8 network against one on the bf16 network: pit.py's shape (1v1, depth 8, breadth 32,
    training=False), both seatings from the same seeded starts; fp8's score (win 1, draw 1/2) with its 95 % interval;
  * compares the two networks over seeded engine planes (uniform-random games): value error of fp8 against bf16 on the moves
    the obstacle mask leaves open, and how often the masked argmax (the move pit_agent.Agent plays) agrees;
  * times the fp8 network's quantization + calibration (NativeNet creation and update), against creating a bf16 network.

  python tools/fp8_strength.py [--generations 3] [--games 256] [--pit-games 1000] [--planes 65536] [--out DIR]
                               [--weights DIR/weights.npz] [--parts cost,values,pit]
--out also saves the trained weights (weights.npz); --weights starts from such a file instead of training.
"""
import argparse
import copy
import json
import math
import os
import sys
from random import sample, seed as py_seed
from time import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from alphasnake_zero_b200 import _lib  # noqa: E402
from alphasnake_zero_b200.engine import Engine  # noqa: E402
from alphasnake_zero_b200.net import NativeNet  # noqa: E402
from alphasnake_zero_b200.utils import pit_mp_game_runner  # noqa: E402
from alphasnake_zero_b200.utils.agent import Agent  # noqa: E402
from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet, flatten_weights, load_weights  # noqa: E402
from alphasnake_zero_b200.utils.mp_game_runner import MPGameRunner  # noqa: E402

HEALTH_DEC, LR = 9, 1e-4        # train.py / alpha_snake_zero_trainer.py, as in examples/selfplay_generation.py


def train_generations(n_gen, games, depth, breadth):
    nnet = AlphaNNet(input_shape=(21, 21, 3), seed=0).copy_and_compile()
    log = []
    for it in range(n_gen):
        t0 = time()
        alice = Agent(nnet, 2 + it, True, depth, breadth)
        MPGameRunner(11, 11, 4, HEALTH_DEC, games, seed=it, verbose=False).run(alice)
        bs = 2048
        batches = min(5, len(alice.records) // bs)
        samples = bs * batches
        if samples == 0:
            bs = samples = len(alice.records)
        idx = sample(range(len(alice.records)), samples)
        X = [alice.records[i] for i in idx]
        V = [alice.values[i] for i in idx]
        alice.clear()
        X += list(np.flip(X, axis=2))
        V += list(np.flip(V, axis=1))
        new = nnet.copy_and_compile(learning_rate=LR)
        new.train(X, V, batch_size=bs)
        nnet = new.copy_and_compile()
        log.append({"generation": it + 1, "records_trained": len(X), "seconds": time() - t0})
        print(json.dumps(log[-1]), flush=True)
    return nnet.weights, log


def pit(w, n_games, depth, breadth, base):
    f8 = AlphaNNet(weights=copy.deepcopy(w), dtype="fp8")
    bf = AlphaNNet(weights=copy.deepcopy(w))
    agent = lambda n: Agent(n, base, False, depth, breadth)
    scores, out = [], {}
    for seat, (alice, bob) in (("fp8_first", (f8, bf)), ("bf16_first", (bf, f8))):
        t0 = time()
        winners = pit_mp_game_runner.MPGameRunner(11, 11, 2, HEALTH_DEC, n_games, seed=1234).run(agent(alice), agent(bob), 1)
        fp8_id = 0 if seat == "fp8_first" else 1
        s = [1.0 if w_ == fp8_id else 0.5 if w_ is None else 0.0 for w_ in winners]
        scores += s
        out[seat] = {"fp8_wins": s.count(1.0), "bf16_wins": s.count(0.0), "draws": s.count(0.5), "seconds": time() - t0}
        print(seat, json.dumps(out[seat]), flush=True)
    m = float(np.mean(scores))
    half = 1.96 * float(np.std(scores, ddof=1)) / math.sqrt(len(scores))
    out["fp8_score"] = m
    out["fp8_score_95ci"] = [m - half, m + half]
    out["games"] = len(scores)
    return out


def engine_planes(n, seed=4242, games=4096, snakes=4):
    """n planes the engine encodes from seeded uniform-random games (every 4th tic, finished games reset), (game, snake) order"""
    eng = Engine(side=11, snakes=snakes, games=games, seed=seed)
    eng.reset()
    out, have, t = [], 0, 0
    while have < n:
        t += 1
        eng.step(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=True, auto_reset=True, random_actions=True)
        if t % 4 == 0:
            p = eng.rows()[1].contiguous()
            out.append(p)
            have += p.shape[0]
    eng.close()
    return torch.cat(out)[:n]


def masked(v, X):
    """AlphaNNet.v's obstacle mask (alpha_nnet.py:67-72) on device"""
    cy, cx = X.shape[1] // 2, X.shape[2] // 2
    m = torch.stack([X[:, cy, cx - 1, 1] >= 0.04, X[:, cy - 1, cx, 1] >= 0.04, X[:, cy, cx + 1, 1] >= 0.04], 1)
    return torch.where(m, torch.full_like(v, -1.0), v), m


def value_agreement(w, n):
    X = engine_planes(n)
    f8 = NativeNet(w, "cuda", dtype="fp8")
    bf = NativeNet(w, "cuda")
    a, m = masked(f8.forward(X), X)
    b, _ = masked(bf.forward(X), X)
    open_ = ~m
    d = (a - b).abs()[open_].double()
    return {"planes": n, "open_moves": int(open_.sum()), "value_err_max": float(d.max()), "value_err_mean": float(d.mean()),
            "value_err_p99": float(torch.quantile(d[:1 << 24].float(), 0.99)),
            "argmax_agreement": float((a.argmax(1) == b.argmax(1)).double().mean()), "act_scale": f8.act_scale}


def calibration_cost(w):
    def timed(fn):
        torch.cuda.synchronize(); t0 = time(); r = fn(); torch.cuda.synchronize(); return r, time() - t0
    timed(lambda: NativeNet(w, "cuda"))                                   # warm: module load, engine kernels
    _, t_bf = timed(lambda: NativeNet(w, "cuda"))
    f8, t_f8 = timed(lambda: NativeNet(w, "cuda", dtype="fp8"))
    _, t_up = timed(lambda: f8.update(w))
    return {"create_bf16_s": t_bf, "create_fp8_s": t_f8, "update_fp8_s": t_up, "calibration_planes": int(f8.calibration.shape[0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--generations", type=int, default=3)
    ap.add_argument("--games", type=int, default=256)
    ap.add_argument("--depth", type=int, default=8)
    ap.add_argument("--breadth", type=int, default=32)
    ap.add_argument("--base", type=float, default=100.0, help="softmax_base of the pit agents (agent.py's default)")
    ap.add_argument("--pit-games", type=int, default=1000)
    ap.add_argument("--planes", type=int, default=65536)
    ap.add_argument("--out", default="")
    ap.add_argument("--weights", default="")
    ap.add_argument("--parts", default="cost,values,pit")
    a = ap.parse_args()
    parts = set(a.parts.split(","))
    py_seed(7)
    np.random.seed(7)
    torch.manual_seed(7)
    res = {"gpu": torch.cuda.get_device_name(0)}
    if a.weights:
        w = load_weights(a.weights)
        res["weights"] = a.weights
    else:
        w, res["generations"] = train_generations(a.generations, a.games, a.depth, a.breadth)
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            np.savez(os.path.join(a.out, "weights.npz"), *flatten_weights(w), side=w["side"])
    if "cost" in parts:
        res["calibration_cost"] = calibration_cost(w)
        print(json.dumps(res["calibration_cost"]), flush=True)
    if "values" in parts:
        res["values"] = value_agreement(w, a.planes)
        print(json.dumps(res["values"]), flush=True)
    if "pit" in parts:
        res["pit"] = pit(w, a.pit_games, a.depth, a.breadth, a.base)
        res["pit"].update(depth=a.depth, breadth=a.breadth, softmax_base=a.base, snakes="1v1")
        print(json.dumps(res["pit"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        json.dump(res, open(os.path.join(a.out, "fp8_strength_%s.json" % "_".join(sorted(parts))), "w"), indent=1)


if __name__ == "__main__":
    main()
