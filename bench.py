#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 self-play engine.

Workload at N=1 (BASELINE.json configs[1]): 65,536 lockstep 11x11 4-snake games, uniform-random joint actions,
native food spawn, in-place reset of finished games, every live snake's fp32 NHWC plane encoded every tic.
A "step" is one lockstep tic of all games = one launch of the fused tic+encode kernel.  N>1: one process per GPU
(torchrun), every rank steps its own 65,536 games (weak scaling, no collective on the data path).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions of every field.
--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so that two builds run
with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SIDE, SNAKES, HEALTH_DEC, CHANCE, GAMES = 11, 4, 1, 0.15, 65536
PLANE_BYTES = 21 * 21 * 3 * 4          # 5,292 B (SURVEY.md 8(d))
STATE_BYTES = 128                      # nominal compact record, read + write => 2x (SURVEY.md 8(d))
METRIC, UNIT = "env_steps_per_sec", "env steps/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe): NVML polled every 2 ms from a
    thread (nvidia-smi -lms as fallback when the NVML binding is missing)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.proc, self.stop_flag, self.t = index, [], None, False, None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: resolve through the PCI bus id of the CUDA device
            import torch
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.handle = h
                        break
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def sample_now(self):
        """one sample taken by the caller's thread (the launches of the timed region are queued and still executing)"""
        if self.nvml is None:
            return
        n = self.nvml
        try:
            sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
            get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            mask = get_reasons(self.handle)
            pre = "nvmlClocksEventReason" if hasattr(n, "nvmlClocksEventReasonHwSlowdown") else "nvmlClocksThrottleReason"
            bits = [getattr(n, pre + k) for k in ("HwSlowdown", "HwThermalSlowdown", "SwThermalSlowdown", "SwPowerCap")]
            self.rows.append([str(sm), str(mx), "0"] + ["Active" if mask & b else "Not Active" for b in bits])
        except Exception:
            pass

    def _poll(self):
        n = self.nvml
        bits = [(n.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (n.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (n.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (n.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")] \
            if hasattr(n, "nvmlClocksEventReasonHwSlowdown") else \
               [(n.nvmlClocksThrottleReasonHwSlowdown, "hw_slowdown"), (n.nvmlClocksThrottleReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_thermal_slowdown"), (n.nvmlClocksThrottleReasonSwPowerCap, "sw_power_cap")]
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mask = get_reasons(self.handle)
                self.rows.append([str(sm), str(mx), "0"] + ["Active" if mask & b else "Not Active" for b, _ in bits])
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            if self.t is not None:
                self.t.join(timeout=1)
        elif not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        else:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for n, v in zip(self.NAMES, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml, 2 ms poll" if self.nvml is not None else "nvidia-smi -lms 100"}


def cpu_baseline(target_s=12.0):
    """The CPU oracle (C restatement of the reference, kind "port") on the same workload, all host threads, on a
    bounded sample sized for ~target_s seconds."""
    from oracle import oracle as orc
    orc.build()
    cores = os.cpu_count() or 1
    t0 = time.time()
    orc.env_run(2048, SIDE, SIDE, SNAKES, HEALTH_DEC, CHANCE, 0, 20, encode=True, n_threads=cores)
    rate = 2048 * 20 / max(time.time() - t0, 1e-6)
    tics = 100
    g = int(max(2048, min(GAMES, rate * target_s / tics)))
    t0 = time.time()
    st = orc.env_run(g, SIDE, SIDE, SNAKES, HEALTH_DEC, CHANCE, 0, tics, encode=True, n_threads=cores)
    dt = time.time() - t0
    return {"value": st["steps"] / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d games x %d tics (tic + encode of every live snake, %.2f planes/step), C oracle, %d threads, %.1f s"
                      % (g, tics, st["planes"] / st["steps"], cores, dt)}


REF_CODE = os.path.join(ROOT, "baseline", "_ref", "code")


def _import_reference():
    """the UNMODIFIED reference (baseline/_ref/code, vendored by baseline/vendor_reference.py from /root/reference) with the one
    NumPy >= 2.3 shim of SURVEY.md 8(c): Game.make_state returns an ndarray subclass that still has .tostring (agent.py:175)"""
    import numpy as np
    if not os.path.isdir(os.path.join(REF_CODE, "utils")):
        return None
    if REF_CODE not in sys.path:
        sys.path.insert(0, REF_CODE)
    import utils.agent as ra
    import utils.game as rg
    import utils.mp_game_runner as rr
    if not getattr(rg.Game, "_asz_shim", False):
        class _Sub(np.ndarray):
            def tostring(self):
                return self.tobytes()
        orig = rg.Game.make_state
        rg.Game.make_state = lambda self, you, last_move: orig(self, you, last_move).view(_Sub)
        rg.Game._asz_shim = True
    return rg, ra, rr


def python_reference_env(target_s=6.0):
    """BASELINE.md 3.1: the reference's own Game (pure Python) with uniform-random moves, tic + get_states() every tic, one core."""
    import random
    mods = _import_reference()
    if mods is None:
        return {"unavailable": "baseline/_ref/code is missing (run baseline/vendor_reference.py where /root/reference exists)"}
    rg = mods[0]
    random.seed(0)
    g = rg.Game(0, SIDE, SIDE, SNAKES, HEALTH_DEC)
    steps = planes = 0
    t0 = time.time()
    while time.time() - t0 < target_s:
        for _ in range(50):
            if g.tic([random.randrange(3) for _ in g.snakes]) != 0:
                g = rg.Game(0, SIDE, SIDE, SNAKES, HEALTH_DEC)
            else:
                planes += len(g.get_states())
            steps += 1
    dt = time.time() - t0
    return {"value": steps / dt, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": "unmodified reference utils/game.py: Game.tic + Game.get_states() with uniform-random moves, %d tics, %.2f planes/step, "
                      "single core (the reference is single threaded), %.1f s" % (steps, planes / max(steps, 1), dt)}


def python_reference_selfplay(games=4, breadth=50, depth=8):
    """BASELINE.md 3.2 / configs[0], bounded: the unmodified reference Agent.make_moves (MCTSAgent + MCTSMPGameRunner inside) for one
    root turn, with a torch-CPU fp32 network of identical architecture behind the AlphaNNet.v contract (TensorFlow is not
    installable here)."""
    import contextlib
    import io
    import random
    import numpy as np
    import torch
    mods = _import_reference()
    if mods is None:
        return {"unavailable": "baseline/_ref/code is missing"}
    rg, ra, rr = mods
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    net = AlphaNNet(input_shape=(2 * SIDE - 1, 2 * SIDE - 1, 3), seed=0, backend="torch", dtype="fp32", device="cpu")
    evals = [0]

    class Shim:
        def v(self, X):
            evals[0] += len(X)
            return net.v(np.array(X))
    random.seed(0); np.random.seed(0)
    gs = {i: rg.Game(i, SIDE, SIDE, SNAKES, HEALTH_DEC) for i in range(games)}
    alice = ra.Agent(Shim(), 2, True, depth, breadth)
    ids = [i for g in gs.values() for i in g.get_ids()]
    t0 = time.time()
    with contextlib.redirect_stdout(io.StringIO()):
        alice.make_moves(gs, ids)
    dt = time.time() - t0
    sims = games * (breadth // 8) * 8
    return {"sims_per_sec": sims / dt, "nn_evals_per_sec": evals[0] / dt, "cores": os.cpu_count() or 1, "torch_threads": torch.get_num_threads(),
            "kind": "reference (unmodified utils/agent.py + utils/game.py) + torch-CPU fp32 network behind AlphaNNet.v",
            "sample": "configs[0] bounded: %d games x breadth %d (%d sims/move), depth %d, one root turn, %.1f s" % (games, breadth, (breadth // 8) * 8, depth, dt)}


def selfplay_api_leg(rank, games, breadth, depth, turns):
    """The same self-play loop through the reference-facing Python API (MPGameRunner.run + Agent.make_moves): host lists of
    ids and moves; the training records (agent.py:93-97) stay in HBM (asz_records_append), only the moves cross PCIe."""
    import torch
    from alphasnake_zero_b200.utils.agent import Agent
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    from alphasnake_zero_b200.utils.mp_game_runner import MPGameRunner
    net = AlphaNNet(input_shape=(2 * SIDE - 1, 2 * SIDE - 1, 3), seed=0, backend="native")
    alice = Agent(net, 2, True, depth, breadth)
    gr = MPGameRunner(SIDE, SIDE, SNAKES, HEALTH_DEC, games, seed=5 + rank, verbose=False)
    gr._make_engine(alice)
    for _ in range(32):                              # games of every age, as in selfplay_leg
        gr.engine.step(spawn_mode=2, tic=True, encode=False, auto_reset=True, random_actions=True)
    gr.run(alice, max_turns=1)                       # warm-up root turn
    torch.cuda.synchronize()
    s0 = gr.engine.search_stats()
    n0 = len(alice.records)
    t0 = time.time()
    gr.run(alice, max_turns=turns)
    torch.cuda.synchronize()
    dt = time.time() - t0
    s1 = gr.engine.search_stats()
    n_rec = len(alice.records) - n0
    t1 = time.time()
    X, V, bs = alice.sample_training_batch()           # alpha_snake_zero_trainer.py:62-77, 93-100: sample + mirror, one gather kernel
    torch.cuda.synchronize()
    return {"sims_per_sec": (s1["subgames"] - s0["subgames"]) / dt, "nn_evals_per_sec": (s1["evals"] - s0["evals"]) / dt,
            "root_turns": turns, "seconds": dt, "records": n_rec, "records_resident": "HBM (asz_records_append: one encode launch per turn)",
            "d2h_bytes_per_turn": games * 8 + games * (SNAKES + 1 + 8), "h2d_bytes_per_turn": games * 8,
            "training_batch": {"rows": int(X.shape[0]), "batch_size": bs, "seconds": time.time() - t1, "where": "device (asz_records_gather, mirrored)"},
            "api": "MPGameRunner(%d games).run(Agent(net, 2, True, %d, %d), max_turns=%d) after 32 uniform-random tics with in-place "
                   "reset; host lists of ids and moves; records and root Q stay on the device" % (games, depth, breadth, turns)}


NET_FLOPS = {11: 1043724288, 19: 3240040448}   # per evaluation, 2 * MAC, convolutions + dense (SURVEY.md 8(d))


def selfplay_leg(rank, games, breadth, depth, turns, warm, use_net=True, side=SIDE, snakes=SNAKES, label="configs[2]", prewarm_tics=32):
    """configs[2] of BASELINE.json (also [3] and [4] per GPU through tools/bench_selfplay.py): self-play root turns with
    the search kernels and the hand-written value network.  A simulation = one sub-game rollout (agent.py:37-56)."""
    import torch
    from alphasnake_zero_b200.engine import Engine
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    from alphasnake_zero_b200 import _lib
    eng = Engine(side=side, snakes=snakes, health_dec=HEALTH_DEC, food_chance=CHANCE, games=games, seed=77 + rank,
                 max_depth=depth, max_breadth=breadth, softmax_base=2.0, training=True)
    eng.reset()
    # games of every age: uniform-random play with in-place reset first, so that the timed root turns see the live-snake
    # mix of running self-play (fresh games only: all snakes alive => the shallowest searches, agent.py:45)
    for _ in range(prewarm_tics):
        eng.step(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=False, auto_reset=True, random_actions=True)
    live = float(eng.alive_mask().float().sum().item()) / games
    net = AlphaNNet(input_shape=(2 * side - 1, 2 * side - 1, 3), seed=0, backend="native") if use_net else None
    nat = net._get_native() if use_net else None

    def root_turn():
        q, mv = eng.search(net=nat)
        act = torch.where(mv < 3, mv, torch.ones_like(mv))
        eng.step(actions=act, spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=False, auto_reset=True)
    for _ in range(warm):
        root_turn()
    torch.cuda.synchronize()
    s0 = eng.search_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(turns):
        root_turn()
    e1.record()
    torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3
    s1 = eng.search_stats()
    d = {k: s1[k] - s0[k] for k in ("evals", "node_visits", "subgames", "subgame_tics")}
    out = {"workload": "%s: %dx%d board, %d snakes, %d games x breadth %d (%d sims/move), depth %d, base 2, %s, Q cache on" %
                       (label, side, side, snakes, games, breadth, (breadth // min(8, breadth)) * min(8, breadth), depth,
                        "bf16 tcgen05 value net (random init)" if use_net else "stub value function (search kernels only)"),
           "root_turns": turns, "seconds": dt, "sims_per_sec": d["subgames"] / dt, "node_visits_per_sec": d["node_visits"] / dt,
           "nn_evals_per_sec": d["evals"] / dt, "subgame_tics_per_sec": d["subgame_tics"] / dt,
           "hit_rate": 1.0 - d["evals"] / max(d["node_visits"], 1), "evals_per_sim": d["evals"] / max(d["subgames"], 1),
           "table_overflow": s1["overflow"], "tag_collisions": s1["collisions"],
           "start_state": "%d uniform-random tics with in-place reset before the search starts: %.2f live snakes per game" % (prewarm_tics, live)}
    if use_net:
        flops = NET_FLOPS[side]
        out["net_tflops"] = d["evals"] * flops / dt / 1e12
        try:
            pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"]
            out["net_roofline"] = {"bound": "tensor", "achieved": out["net_tflops"], "peak": pk, "unit": "TFLOP/s",
                                   "frac": out["net_tflops"] / pk}
        except Exception:
            pass
    eng.close()
    return out


def cpu_selfplay_baseline(games=4, breadth=100, depth=8):
    """The GPU self-play leg's own shape (configs[2]: breadth 100 = 96 sims/move, depth 8, base 2, games of every age) on the host
    cores, bounded to a few games: the C port of the reference's search with a torch-CPU fp32 network of identical
    architecture as AlphaNNet.v (TensorFlow is not installable here).  One root turn."""
    import numpy as np
    import torch
    from oracle import oracle as orc
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    net = AlphaNNet(input_shape=(2 * SIDE - 1, 2 * SIDE - 1, 3), seed=0, backend="torch", dtype="fp32", device="cpu")
    gs = []
    for gi in range(games):
        g = orc.OracleGame(SIDE, SIDE, SNAKES, HEALTH_DEC); g.init_native(0, gi, 0); g.set_ids(gi, 0); gs.append(g)
    orc.env_run(games, SIDE, SIDE, SNAKES, HEALTH_DEC, CHANCE, 0, 32, encode=False, n_threads=1, games=gs)   # games of every age, like the GPU leg
    agent = orc.OracleAgent(base=2.0, training=True, max_depth=depth, max_breadth=breadth, value_fn=lambda X: net.v(np.array(X)))
    t0 = time.time()
    agent.make_moves(gs, games, root_turn=0, seed=0)
    dt = time.time() - t0
    return {"sims_per_sec": agent.stat("subgames") / dt, "node_visits_per_sec": agent.stat("node_visits") / dt,
            "nn_evals_per_sec": agent.stat("evals") / dt, "cores": os.cpu_count() or 1, "torch_threads": torch.get_num_threads(),
            "kind": "port (C search) + torch-CPU fp32 network", "sample": "configs[2] bounded: %d of 4096 games x breadth %d (%d sims/move), "
            "depth %d, after 32 uniform-random tics, one root turn, %.1f s" % (games, breadth, (breadth // 8) * 8, depth, dt)}


def run_reference(args, rank, world):
    """The reference arm: the reference's CPU implementation of the same path (its C port, oracle/asz_oracle.c -- the
    reference itself is Python + TensorFlow and does not exist on the GPU box, DESIGN.md 7) on all host threads.
    One step = the 65,536 env steps of the GPU arm's step, run as 8,192 persistent games x 8 tics (a bounded sample of
    the games, the same number of tics + plane encodes)."""
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    cores = os.cpu_count() or 1
    g, tics = 8192, GAMES // 8192
    games = []
    for gi in range(g):
        og = orc.OracleGame(SIDE, SIDE, SNAKES, HEALTH_DEC)
        og.init_native(0, gi, 0)
        games.append(og)
    arr = orc.env_handles(games)
    for _ in range(args.warmup):
        orc.env_run(g, SIDE, SIDE, SNAKES, HEALTH_DEC, CHANCE, 0, tics, encode=True, n_threads=cores, games=arr)
    t0 = time.time()
    steps = planes = 0
    for _ in range(args.steps):
        st = orc.env_run(g, SIDE, SIDE, SNAKES, HEALTH_DEC, CHANCE, 0, tics, encode=True, n_threads=cores, games=arr)
        steps += st["steps"]; planes += st["planes"]
    dt = time.time() - t0
    v = steps / dt
    sample = "%d games x %d tics per step (= the %d env steps of one GPU step), all %d host threads, C port of the reference " \
             "(oracle/asz_oracle.c)" % (g, tics, GAMES, cores)
    emit(({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u16/f32", "data": "synthetic",
        "config": {"workload": "configs[1]: 11x11, 4 snakes, lockstep games, uniform-random actions, tic + fp32 plane encode",
                   "games_per_step": g, "tics_per_step": tics, "planes_per_step": planes / max(steps, 1)},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "python_reference": python_reference_env(4.0)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


DUMP_PLANES = 4096     # planes in the dump: a fixed sample of the step's rows (one per live snake, ~1 GB of planes in all)


def dump_outputs(eng, out_dir):
    """What one eng.step of the timed loop hands its caller, as .npy files: the row count, every row id (game * 8 + snake),
    the per-game ended flags and rewards (integers, stored as float64: exact), and a fixed, seeded sample of the fp32 planes
    with the ids of the sampled rows.  Rows are put in row-id order first: the kernel hands rows out in whatever order its
    warps finish, so the raw order differs from run to run while the set of rows does not."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = int(eng.row_count.item())
    ids = eng.row_ids[:n]
    order = torch.argsort(ids)
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_PLANES), replace=False))
    sel = order[torch.from_numpy(pick).to(order.device)]
    out = {"row_count": np.array([n], np.float64),
           "row_ids": ids[order].cpu().numpy().astype(np.float64),
           "ended": eng.ended.cpu().numpy().astype(np.float64),
           "rewards": eng.rewards.cpu().numpy().astype(np.float64),
           "planes_sample_row_ids": ids[sel].cpu().numpy().astype(np.float64),
           "planes_sample": eng.planes[:n][sel].cpu().numpy()}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from alphasnake_zero_b200 import _lib
    from alphasnake_zero_b200.engine import Engine
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    K, W = args.steps, max(args.warmup, 3)
    eng = Engine(side=SIDE, snakes=SNAKES, health_dec=HEALTH_DEC, food_chance=CHANCE, games=GAMES, seed=1000 + rank)
    eng.reset()
    _ = eng.planes
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    kw = dict(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=True, auto_reset=True, random_actions=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- leg 1: device-resident throughput ("value") and the kernel roofline -----------------------------------
    for _ in range(W):
        eng.step(**kw)
    barrier()
    t_before = eng.totals()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(K):
        eng.step(**kw)
    ev1.record()
    if rank == 0:
        sampler.sample_now()      # the K launches are queued and executing: a sample from this thread is inside the region
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    t_after = eng.totals()
    if args.dump_outputs and rank == 0:     # before the untimed pass below steps the games on
        dump_outputs(eng, args.dump_outputs)
    # per-launch percentiles from a second, untimed pass with an event after every launch (the events themselves cost ~1 us per
    # launch, which is why they are not in the timed region): a launch-time distribution with two modes would show here
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    step_ev[0].record()
    for i in range(K):
        eng.step(**kw)
        step_ev[i + 1].record()
    torch.cuda.synchronize()
    per_launch = np.array([step_ev[i].elapsed_time(step_ev[i + 1]) * 1e3 for i in range(K)])      # us
    launch_us = {"p05": float(np.percentile(per_launch, 5)), "p50": float(np.median(per_launch)), "p95": float(np.percentile(per_launch, 95)),
                 "max": float(per_launch.max()), "what": "CUDA events around every launch of a second pass of K launches right after the "
                                                          "timed region (kernel + the event)"}
    steps_local = t_after["tics"] - t_before["tics"]
    planes_local = t_after["planes"] - t_before["planes"]

    # ---- leg 2: end to end through the C ABI with HOST buffers -----------------------------------------------------
    rng = np.random.default_rng(rank)
    n_pool = 8
    act_pool = [torch.from_numpy(rng.integers(0, 3, size=(GAMES, 8), dtype=np.uint8)).pin_memory() for _ in range(n_pool)]
    h_ended = torch.zeros(GAMES, dtype=torch.uint8).pin_memory()
    h_rewards = torch.zeros(GAMES, 8, dtype=torch.int8).pin_memory()
    rows = C.c_int32(0)
    L = _lib.lib()
    flags = _lib.STEP_TIC | _lib.STEP_ENCODE | _lib.STEP_AUTO_RESET

    def e2e_step(i):
        _lib.check(L.asz_env_step_host(eng.h, flags, _lib.SPAWN_NATIVE, C.c_void_p(act_pool[i % n_pool].data_ptr()), None,
                                       C.c_void_p(h_ended.data_ptr()), C.c_void_p(h_rewards.data_ptr()), C.byref(rows),
                                       None, None, eng.stream))

    def timed_e2e(run_steps):
        for i in range(W):
            e2e_step(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_b = eng.totals()
        barrier()
        e0.record()
        run_steps()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), eng.totals()["tics"] - t_b["tics"]

    # (a) one synchronous call per step: copy in, launch, results out, wait -- nothing of step k+1 starts before step k is back
    def sync_steps():
        for i in range(K):
            e2e_step(i)
    e2e_sync_ms, e2e_sync_steps_local = timed_e2e(sync_steps)

    # (b) the same steps as submit / wait with two steps in flight (the uniform-random moves of configs[1] do not depend on the
    # previous step's result): every step still brings its own actions from pinned host memory and lands its own ended / rewards /
    # row count in host memory inside the timed region, but the copy of step k+1 runs under the kernel of step k.
    h_ended2 = [h_ended, torch.zeros(GAMES, dtype=torch.uint8).pin_memory()]
    h_rewards2 = [h_rewards, torch.zeros(GAMES, 8, dtype=torch.int8).pin_memory()]
    kw_host = dict(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=True, auto_reset=True)
    e2e_rows = [0]

    def piped_steps():
        t_prev = eng.submit_host(act_pool[0], h_ended2[0], h_rewards2[0], **kw_host)
        for i in range(1, K):
            t_next = eng.submit_host(act_pool[i % n_pool], h_ended2[i & 1], h_rewards2[i & 1], **kw_host)
            e2e_rows[0] += eng.wait_host(t_prev)
            t_prev = t_next
        e2e_rows[0] += eng.wait_host(t_prev)
    e2e_ms, e2e_steps_local = timed_e2e(piped_steps)

    # what the headline e2e number does NOT do: ship the planes to the host.  The consumer of the planes is the value network on
    # the same GPU; a caller that wants them in host memory pays PCIe for ~1 GB per step (reported once, rank 0, 3 steps).
    planes_to_host = None
    if rank == 0 and not args.no_selfplay:
        try:
            h_planes = torch.empty(GAMES * SNAKES, 2 * SIDE - 1, 2 * SIDE - 1, 3).pin_memory()
            h_ids = torch.empty(GAMES * SNAKES, dtype=torch.int32).pin_memory()

            def e2e_planes_step(i):
                _lib.check(L.asz_env_step_host(eng.h, flags, _lib.SPAWN_NATIVE, C.c_void_p(act_pool[i % n_pool].data_ptr()), None,
                                               C.c_void_p(h_ended.data_ptr()), C.c_void_p(h_rewards.data_ptr()), C.byref(rows),
                                               C.c_void_p(h_planes.data_ptr()), C.c_void_p(h_ids.data_ptr()), eng.stream))
            e2e_planes_step(0)
            torch.cuda.synchronize()
            tb = eng.totals()
            t0 = time.time()
            for i in range(3):
                e2e_planes_step(i)
            torch.cuda.synchronize()
            dt = time.time() - t0
            planes_to_host = {"value": (eng.totals()["tics"] - tb["tics"]) / dt, "unit": UNIT, "d2h_bytes_per_step": int(rows.value) * PLANE_BYTES,
                              "note": "asz_env_step_host with h_planes: every plane copied to pinned host memory (PCIe bound); not the "
                                      "product path, shown so that nobody reads the e2e figure as including it"}
            del h_planes, h_ids
        except Exception as ex:
            planes_to_host = {"error": repr(ex)}

    # ---- leg 3: self-play (search + value network) on every rank ------------------------------------------------------
    sp = {}
    if not args.no_selfplay:
        for key, use_net in (("mcts", True), ("mcts_search_only", False)):
            try:
                barrier()
                r = selfplay_leg(rank, args.sp_games, 100, 8, args.sp_turns, 1, use_net=use_net)
                if world > 1:   # whole-job aggregate: sum of the work of all ranks / slowest rank's time
                    rates = ("sims_per_sec", "node_visits_per_sec", "nn_evals_per_sec", "subgame_tics_per_sec")
                    t = torch.tensor([r["seconds"]] + [r[k] * r["seconds"] for k in rates], dtype=torch.float64, device=dev)
                    mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
                    sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
                    r["seconds"] = float(mx[0])
                    for i, k in enumerate(rates):
                        r[k] = float(sm[1 + i]) / float(mx[0])
                    if "net_tflops" in r:
                        r["net_tflops_all_gpus"] = r["nn_evals_per_sec"] * 1043724288 / 1e12
                    r["aggregate_over_gpus"] = world
                sp[key] = r
            except Exception as ex:   # the headline line must still be printed
                sp[key] = {"error": repr(ex)}
        if world == 1:
            try:
                sp["mcts_e2e"] = selfplay_api_leg(rank, args.sp_games, 100, 8, args.sp_turns)
            except Exception as ex:
                sp["mcts_e2e"] = {"error": repr(ex)}

    # ---- per-generation weight broadcast (the only collective of the design, outside the hot loop; SURVEY.md 8(e)) ------
    # Real weights through alphasnake_zero_b200.parallel: every rank starts from DIFFERENT random weights, rank 0's are pushed
    # into every rank's live native network (asz_net_update_weights), a checksum proves all ranks hold the same bits and the
    # network outputs agree; then the hand-off of a sampled training batch and of the log counters, all on device tensors.
    bcast = None
    if world > 1:
        from alphasnake_zero_b200 import parallel
        from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet, flatten_weights
        try:
            net = AlphaNNet(input_shape=(2 * SIDE - 1, 2 * SIDE - 1, 3), seed=100 + rank, backend="native")
            net._get_native()
            differ_before = not parallel.weights_equal_all_ranks(net.weights)
            for _ in range(2):
                parallel.broadcast_weights(net, src=0)
            barrier()
            t0 = time.time()
            parallel.broadcast_weights(net, src=0)
            barrier()
            whole_ms = (time.time() - t0) * 1e3
            equal = parallel.weights_equal_all_ranks(net.weights)
            # the device copies really changed: identical outputs on every rank for the same planes
            gen = torch.Generator(device="cpu"); gen.manual_seed(7)
            probe = torch.rand(64, 2 * SIDE - 1, 2 * SIDE - 1, 3, generator=gen).to(dev)
            v = net.v_device(probe).double().sum().reshape(1)
            vmin, vmax = v.clone(), v.clone()
            dist.all_reduce(vmin, op=dist.ReduceOp.MIN); dist.all_reduce(vmax, op=dist.ReduceOp.MAX)
            n_par = sum(a.size for a in flatten_weights(net.weights))
            flat = torch.zeros(n_par, dtype=torch.float32, device=dev)
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(10):
                dist.broadcast(flat, src=0)
            b1.record()
            barrier()
            t = torch.tensor([b0.elapsed_time(b1) / 10.0, whole_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            # sampled training batch: 5 x 2048 records drawn over the union of the ranks' stores, only those rows move
            local_planes = torch.rand(20000, 2 * SIDE - 1, 2 * SIDE - 1, 3, device=dev)
            local_values = torch.rand(20000, 3, device=dev)
            barrier()
            t0 = time.time()
            X, V, bs = parallel.gather_sampled_batch(20000, lambda idx: (local_planes[idx.to(dev)], local_values[idx.to(dev)]),
                                                     (2 * SIDE - 1, 2 * SIDE - 1, 3), dst=0)
            barrier()
            batch_ms = (time.time() - t0) * 1e3
            counters = parallel.reduce_counters([1.0, 2.0, 3.0, 4.0, 5.0, 6.0], 1, dst=0)
            bcast = {"bytes": int(n_par * 4), "ms": float(t[0]), "end_to_end_ms": float(t[1]),
                     "weights_equal_all_ranks": bool(equal and differ_before), "outputs_equal_all_ranks": bool(float(vmin) == float(vmax)),
                     "sampled_batch": {"rows": None if X is None else int(X.shape[0]), "batch_size": bs, "ms": batch_ms,
                                       "what": "parallel.gather_sampled_batch: 5 x 2048 of 20,000 records per rank, tensor gather over NCCL"},
                     "counters_reduced": counters == [1.0, 2.0, 3.0, 4.0, 5.0, 6.0] if counters is not None else None,
                     "what": "parallel.broadcast_weights(AlphaNNet) over NCCL: rank 0's weights and BN buffers into every rank's live native "
                             "network (asz_net_update_weights), once per generation, outside every timed region above; `ms` is the "
                             "collective alone (device events), `end_to_end_ms` includes flattening, the host copy and the operand rebuild"}
        except Exception as ex:
            bcast = {"error": repr(ex)}

    # ---- reduce over ranks: max time, sum of work ----------------------------------------------------------------
    vals = torch.tensor([ms, e2e_ms, float(steps_local), float(planes_local), float(e2e_steps_local), e2e_sync_ms, float(e2e_sync_steps_local)],
                        dtype=torch.float64, device=dev)
    rank_ms = None
    if world > 1:
        allv = [torch.zeros_like(vals) for _ in range(world)]
        dist.all_gather(allv, vals)
        rank_ms = {"device_resident": [round(float(v[0]) / K, 5) for v in allv], "e2e": [round(float(v[1]) / K, 5) for v in allv],
                   "e2e_synchronous": [round(float(v[5]) / K, 5) for v in allv]}
        mx = vals.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = vals.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, e2e_ms, e2e_sync_ms = float(mx[0]), float(mx[1]), float(mx[5])
        steps_all, planes_all, e2e_steps_all, e2e_sync_steps_all = float(sm[2]), float(sm[3]), float(sm[4]), float(sm[6])
    else:
        steps_all, planes_all, e2e_steps_all = float(steps_local), float(planes_local), float(e2e_steps_local)
        e2e_sync_steps_all = float(e2e_sync_steps_local)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = steps_all / (ms * 1e-3)
    peak, peak_src = peaks()
    # roofline of the dominant (only) kernel: algorithmic bytes per launch on THIS rank / average launch duration
    bytes_per_launch = (planes_local * PLANE_BYTES + steps_local * 2 * STATE_BYTES) / K
    launch_s = (ev0.elapsed_time(ev1) * 1e-3) / K
    achieved = bytes_per_launch / launch_s / 1e9
    traffic = None
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tf):
        try:
            traffic = json.load(open(tf)).get("env_step_kernel_bytes_per_launch")
        except Exception:
            traffic = None
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16/f32", "data": "synthetic",
        "config": {"workload": "configs[1]: %d lockstep 11x11 4-snake games per GPU, uniform-random joint actions (in-kernel Philox), "
                               "native food spawn, in-place reset, tic + fp32 NHWC plane encode of every live snake" % GAMES,
                   "games_per_gpu": GAMES, "planes_per_step": planes_all / max(steps_all, 1),
                   "l2": "each launch writes %.0f MB of planes (> 126 MB L2); the 21 MB of game records may stay L2 resident"
                         % (bytes_per_launch / 1e6),
                   "plane_layout": "fp32 NHWC rows, 5,312 B apart (asz_plane_pitch: 5,292 B plane + 20 B pad, 32-byte aligned rows)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "env_step_kernel (pitched rows, warp_encode_game_v3b)", "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": bytes_per_launch,
                     "note": "algorithmic bytes count 5,292 B per plane; the kernel writes 5,312 B (rows padded to 32-byte sectors)"},
        "e2e": {"value": e2e_steps_all / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": GAMES * 8,
                "d2h_bytes_per_step": GAMES + GAMES * 8 + 4,
                "note": "asz_env_submit_host / asz_env_wait_host, two steps in flight: every step copies its pinned host actions in and "
                        "lands its per-game ended/rewards + row count in host memory inside the timed region; the copy of step k+1 runs "
                        "under the kernel of step k; planes stay in HBM for the network",
                "synchronous": {"value": e2e_sync_steps_all / (e2e_sync_ms * 1e-3), "unit": UNIT,
                                "note": "asz_env_step_host: one blocking call per step (copy in, launch, results out, wait)"}},
        "gpu_launches": K, "clocks": clocks, "launch_us": launch_us,
    }
    if planes_to_host is not None:
        out["e2e_planes_to_host"] = planes_to_host
    out.update(sp)
    if rank_ms is not None:   # ms per step of every rank: the aggregate above is paced by the slowest one (DESIGN.md 4.1)
        out["rank_ms_per_step"] = rank_ms
    if bcast is not None:
        out["weight_broadcast"] = bcast
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline()
        try:      # the reference's own Python next to its C port (BASELINE.md 3.1)
            out["cpu_baseline"]["python_reference"] = python_reference_env()
        except Exception as ex:
            out["cpu_baseline"]["python_reference"] = {"error": repr(ex)}
        if not args.no_selfplay:
            try:
                out["mcts_cpu_baseline"] = cpu_selfplay_baseline()
            except Exception as ex:
                out["mcts_cpu_baseline"] = {"error": repr(ex)}
            try:  # BASELINE.md 3.2
                out["mcts_cpu_baseline"]["python_reference"] = python_reference_selfplay()
            except Exception as ex:
                out["mcts_cpu_baseline"]["python_reference"] = {"error": repr(ex)}
    emit(out)
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None


def emit(obj):
    """the ONE JSON line goes to the process's original stdout; everything libraries print (NCCL's version banner,
    warnings) was redirected to stderr in main()."""
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)          # fd 1 now points at stderr for every library in this process
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle leg (profiling runs)")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the self-play (MCTS + value net) leg")
    ap.add_argument("--sp-games", type=int, default=4096, help="root games of the self-play leg (configs[2]: 4096)")
    ap.add_argument("--sp-turns", type=int, default=2, help="timed root turns of the self-play leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
