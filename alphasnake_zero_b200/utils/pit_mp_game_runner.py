"""pit MPGameRunner -- mirror of code/utils/pit_mp_game_runner.py:3-63 (two agents, early exit).
Either side may be pit_agent.Agent (argmax of the network) or the search Agent of utils/agent.py with training=False (argmax of
the root Q of a full root-turn search with that side's own network and Q table).  When every side is one of these over a native
AlphaNNet (or, for a search side, over agent.StubNet), the whole match runs on the device (asz_pit_*: the planes never leave HBM,
one host wait per turn plus the search's own); any other agent is driven by the loop below, over the same fused tic+encode kernel
and the same search kernels."""
import numpy as np
import torch

from ..engine import Engine
from .. import _lib
from .._lib import AszError
from . import agent as search_agent
from . import alpha_nnet, pit_agent


class MPGameRunner:

    def __init__(self, height=11, width=11, snake_cnt=4, health_dec=1, game_cnt=1, seed=0, device=None):
        self.height, self.width, self.snake_cnt, self.health_dec, self.game_cnt = height, width, snake_cnt, health_dec, game_cnt
        self.seed = seed
        self.engine = Engine(side=height, snakes=snake_cnt, health_dec=health_dec, games=game_cnt, seed=seed, device=device)
        self.engine.reset()
        self._searchers = [None, None]     # per side: ((depth, breadth, softmax_base), searcher Engine), kept across matches

    # Alice and Bob are agents using different nets
    def run(self, Alice, Bob, Alice_snake_cnt=None, spawn_trace=None, move_log=None, native=None):
        """pit_mp_game_runner.py:14-63.  Extensions for trace replay (tests): spawn_trace[turn] = int32 [game_cnt] food cell
        spawned in that turn's tic (-1 none) instead of the engine's RNG; move_log (a list) receives per turn a uint8
        [game_cnt, 8] array of the moves played (255 = no move).
        Alice and Bob are pit_agent.Agent or utils.agent.Agent (the search agent; training=True raises ValueError, a pit keeps no
        records).  A search side plays Agent.make_moves(training=False) over the running games on a searcher engine of its own:
        its network values every snake inside its search, its own Q table is cleared when a match begins and ages across the
        match's turns, and its snakes play the argmaxs of their root Q.  The runner creates one searcher per search side and
        keeps it for later matches (a new one when the side's depth, breadth or softmax_base changes); its seed is
        seed * 2 + 1 + side (mod 2^64) for this runner's `seed`, side 0 = Alice, 1 = Bob.
        native=None: the device arena when every side is pit_agent.Agent over a native AlphaNNet, or the search Agent over a native
        AlphaNNet or agent.StubNet, of this board side on this device; the loop otherwise (a torch network, any other agent);
        native=False: the loop; native=True: the arena, or AszError when it cannot be used.  Both give the same winners, moves and
        final game states.  A game that is already finished when the match begins is a draw on the arena (the reference's loop
        fails on it)."""
        if Alice_snake_cnt is None:
            Alice_snake_cnt = self.snake_cnt // 2
        for agent in (Alice, Bob):
            if isinstance(agent, search_agent.Agent) and agent.training:
                raise ValueError("a pit plays search agents with training=False (a pit keeps no records)")
        if native is not False:
            players = self._arena_players(Alice, Bob)
            if players is not None:
                return self._run_arena(players, (Alice, Bob), Alice_snake_cnt, spawn_trace, move_log)
            if native:
                raise AszError("the device pit needs, on both sides, pit_agent.Agent over a native AlphaNNet or the search Agent over "
                               "a native AlphaNNet or StubNet, for side %d on %s" % (self.height, self.engine.device))
        return self._run_loop(Alice, Bob, Alice_snake_cnt, spawn_trace, move_log)

    def _native_net(self, nnet):
        """the NativeNet of an AlphaNNet whose `v` is the native forward + float32 obstacle mask, for this runner's board side and
        device; else None"""
        if type(nnet) is not alpha_nnet.AlphaNNet:
            return None
        if nnet.backend not in ("auto", "native") or nnet.weights is None or int(nnet.weights["side"]) != self.height:
            return None
        dev = nnet.device.index if nnet.device.index is not None else torch.cuda.current_device()
        if nnet.device.type != "cuda" or dev != self.engine.device.index:
            return None
        return nnet._get_native()

    def _arena_players(self, Alice, Bob):
        """per side the arena's player (a NativeNet, or 1: the engine's stub value function) when both agents can play on the
        arena; else None"""
        players = []
        for agent in (Alice, Bob):
            if type(agent) is pit_agent.Agent:
                player = self._native_net(agent.nnet)
            elif type(agent) is search_agent.Agent:
                value_fn, net = agent.search_values()
                player = None if value_fn is not None else 1 if net is None else self._native_net(agent.nnet)
            else:
                player = None
            if player is None:
                return None
            players.append(player)
        return players

    def _searcher(self, side, agent):
        """the searcher engine of a search side, created with the agent's search settings and training=False"""
        cfg = (int(agent.max_MCTS_depth), int(agent.max_MCTS_breadth), float(agent.softmax_base))
        if self._searchers[side] is None or self._searchers[side][0] != cfg:
            seed = (self.seed * 2 + 1 + side) % (1 << 64)
            eng = Engine(side=self.height, snakes=self.snake_cnt, health_dec=self.health_dec, games=self.game_cnt, seed=seed,
                         max_depth=cfg[0], max_breadth=cfg[1], softmax_base=cfg[2], training=False, device=self.engine.device)
            self._searchers[side] = (cfg, eng)
        return self._searchers[side][1]

    def _searchers_of(self, agents):
        return [self._searcher(side, a) if isinstance(a, search_agent.Agent) else None for side, a in enumerate(agents)]

    def _run_arena(self, players, agents, Alice_snake_cnt, spawn_trace, move_log):
        eng = self.engine
        for side, q in enumerate(self._searchers_of(agents)):
            eng.pit_set_search(side, q)
        if spawn_trace is None and move_log is None:
            winners, _, _ = eng.pit_run(players[0], players[1], Alice_snake_cnt)
        else:
            running = eng.pit_begin(players[0], players[1], Alice_snake_cnt)
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

    def _search_moves(self, agent, searcher, running, g, s):
        """a search side's moves for the rows (g, s): its root-turn search over the running games, copied into its searcher"""
        searcher.copy_root_games_from(self.engine, skip=torch.from_numpy(~running))
        value_fn, net = agent.search_values()
        _, mv = searcher.search(value_fn=value_fn, net=net)
        moves = mv.cpu().numpy()[g, s]
        if (moves > 2).any():
            raise AszError("search returned no move for a live snake")
        return moves

    def _run_loop(self, Alice, Bob, Alice_snake_cnt, spawn_trace, move_log):
        eng = self.engine
        searchers = self._searchers_of((Alice, Bob))
        for q in searchers:
            if q is not None:
                q.search_clear()                                     # as the arena's begin: a match starts from an empty table
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
            moves = []
            for agent, q, idx in ((Alice, searchers[0], a_idx), (Bob, searchers[1], b_idx)):
                if q is None:
                    moves.append(agent.make_moves(planes[torch.from_numpy(idx).to(planes.device)], [(int(g[i]), int(s[i])) for i in idx]))
                else:                                                # a side with no snake to move does not search
                    moves.append(self._search_moves(agent, q, running, g[idx], s[idx]) if len(idx) else [])
            moves_a, moves_b = moves
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
