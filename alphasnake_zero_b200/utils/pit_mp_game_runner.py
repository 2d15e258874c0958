"""pit MPGameRunner -- mirror of code/utils/pit_mp_game_runner.py:3-63 (two agents, argmax policy, early exit).
When both agents are pit_agent.Agent over a native AlphaNNet, the whole match runs on the device (asz_pit_*: the planes never
leave HBM, one host wait per turn); any other agent is driven by the loop below, over the same fused tic+encode kernel."""
import numpy as np
import torch

from ..engine import Engine
from .. import _lib
from .._lib import AszError
from . import alpha_nnet, pit_agent


class MPGameRunner:

    def __init__(self, height=11, width=11, snake_cnt=4, health_dec=1, game_cnt=1, seed=0, device=None):
        self.height, self.width, self.snake_cnt, self.health_dec, self.game_cnt = height, width, snake_cnt, health_dec, game_cnt
        self.engine = Engine(side=height, snakes=snake_cnt, health_dec=health_dec, games=game_cnt, seed=seed, device=device)
        self.engine.reset()

    # Alice and Bob are agents using different nets
    def run(self, Alice, Bob, Alice_snake_cnt=None, spawn_trace=None, move_log=None, native=None):
        """pit_mp_game_runner.py:14-63.  Extensions for trace replay (tests): spawn_trace[turn] = int32 [game_cnt] food cell
        spawned in that turn's tic (-1 none) instead of the engine's RNG; move_log (a list) receives per turn a uint8
        [game_cnt, 8] array of the moves played (255 = no move).
        native=None: the device arena when both agents are pit_agent.Agent over a native AlphaNNet of this board side on this
        device, the loop otherwise; native=False: the loop; native=True: the arena, or AszError when it cannot be used.
        Both give the same winners, moves and final game states.  A game that is already finished when the match begins is a
        draw on the arena (the reference's loop fails on it)."""
        if Alice_snake_cnt is None:
            Alice_snake_cnt = self.snake_cnt // 2
        if native is not False:
            nets = self._arena_nets(Alice, Bob)
            if nets is not None:
                return self._run_arena(nets, Alice_snake_cnt, spawn_trace, move_log)
            if native:
                raise AszError("the device pit needs pit_agent.Agent over a native AlphaNNet for side %d on %s on both sides"
                               % (self.height, self.engine.device))
        return self._run_loop(Alice, Bob, Alice_snake_cnt, spawn_trace, move_log)

    def _arena_nets(self, Alice, Bob):
        """(Alice's NativeNet, Bob's NativeNet) when both agents are exactly pit_agent.Agent over an AlphaNNet whose `v` is
        the native forward + float32 obstacle mask, for this runner's board side and device; else None"""
        nets = []
        for agent in (Alice, Bob):
            if type(agent) is not pit_agent.Agent or type(agent.nnet) is not alpha_nnet.AlphaNNet:
                return None
            nnet = agent.nnet
            if nnet.backend not in ("auto", "native") or nnet.weights is None or int(nnet.weights["side"]) != self.height:
                return None
            dev = nnet.device.index if nnet.device.index is not None else torch.cuda.current_device()
            if nnet.device.type != "cuda" or dev != self.engine.device.index:
                return None
            nets.append(nnet._get_native())
        return nets

    def _run_arena(self, nets, Alice_snake_cnt, spawn_trace, move_log):
        eng = self.engine
        if spawn_trace is None and move_log is None:
            winners, _, _ = eng.pit_run(nets[0], nets[1], Alice_snake_cnt)
        else:
            running = eng.pit_begin(nets[0], nets[1], Alice_snake_cnt)
            trace = None
            if spawn_trace is not None:
                trace = torch.from_numpy(np.ascontiguousarray(np.asarray(spawn_trace, np.int32))).to(eng.device)
            logs, turn = [], 0
            while running:
                if trace is not None and turn >= trace.shape[0]:
                    eng.pit_finish()          # raises: games are still running, the results so far are attached
                moves = torch.empty(self.game_cnt, 8, dtype=torch.uint8, device=eng.device) if move_log is not None else None
                if trace is not None:
                    running = eng.pit_turn(spawn_cells=trace[turn], spawn_mode=_lib.SPAWN_REPLAY, moves=moves)
                else:
                    running = eng.pit_turn(spawn_mode=_lib.SPAWN_NATIVE, moves=moves)
                if moves is not None:
                    logs.append(moves)
                turn += 1
            winners, _, _ = eng.pit_finish()
            if move_log is not None:
                move_log.extend(m.cpu().numpy() for m in logs)
        return [None if w < 0 else int(w) for w in winners]

    def _run_loop(self, Alice, Bob, Alice_snake_cnt, spawn_trace, move_log):
        eng = self.engine
        winners = [None] * self.game_cnt
        running = np.ones(self.game_cnt, bool)
        eng.step(tic=False, encode=True)
        turn = -1
        while running.any():
            turn += 1
            planes, rows = eng.encode_rows(refresh=False)
            rows = rows.astype(np.int64)
            g, s = rows // 8, rows % 8
            keep = running[g]
            a_idx = np.nonzero(keep & (s < Alice_snake_cnt))[0]     # pit_mp_game_runner.py:30-33
            b_idx = np.nonzero(keep & (s >= Alice_snake_cnt))[0]
            moves_a = Alice.make_moves(planes[torch.from_numpy(a_idx).to(planes.device)], [(int(g[i]), int(s[i])) for i in a_idx])
            moves_b = Bob.make_moves(planes[torch.from_numpy(b_idx).to(planes.device)], [(int(g[i]), int(s[i])) for i in b_idx])
            actions = np.ones((self.game_cnt, 8), np.uint8)
            actions[g[a_idx], s[a_idx]] = np.asarray(moves_a, np.uint8)
            actions[g[b_idx], s[b_idx]] = np.asarray(moves_b, np.uint8)
            if move_log is not None:
                played = np.full((self.game_cnt, 8), 255, np.uint8)
                played[g[a_idx], s[a_idx]] = np.asarray(moves_a, np.uint8)
                played[g[b_idx], s[b_idx]] = np.asarray(moves_b, np.uint8)
                move_log.append(played)
            if spawn_trace is not None:
                cells = torch.from_numpy(np.maximum(np.asarray(spawn_trace[turn], np.int32), -1)).to(eng.device)
                eng.step(actions=torch.from_numpy(actions).to(eng.device), spawn_cells=cells, spawn_mode=_lib.SPAWN_REPLAY,
                         tic=True, encode=True)
            else:
                eng.step(actions=torch.from_numpy(actions).to(eng.device), spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=True)
            ended = eng.ended.cpu().numpy().astype(bool)
            rw = eng.rewards.cpu().numpy()
            alive = eng.alive_mask().cpu().numpy()
            for gi in np.nonzero(running)[0]:
                if ended[gi]:                                        # pit_mp_game_runner.py:44-48
                    w = np.nonzero(rw[gi, :self.snake_cnt] == 1)[0]
                    if len(w):
                        winners[gi] = int(w[0])
                    running[gi] = False
                else:                                                # :49-60 the team with snakes left wins
                    live = np.nonzero(alive[gi])[0]
                    A = (live < Alice_snake_cnt).any()
                    B = (live >= Alice_snake_cnt).any()
                    if not A or not B:
                        winners[gi] = int(live[0])
                        running[gi] = False
        return winners
