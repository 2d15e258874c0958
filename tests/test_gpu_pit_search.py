"""GPU: pits in which a side plays the search Agent (agent.py:25-111, training=False) with its own network and Q table.
 (1) the arena with stand-in sides against a composition of two CPU-oracle search agents: every move, winners, decided turns,
     final game states, each side's Q table and search counters (decided games are never searched);
 (2) the arena and the runner's Python loop with random-init native networks, move for move;
 (3) argument errors, training agents, and Q table overflow with the results so far attached."""
import numpy as np
import pytest

from tests.helpers import KeyStubNet, assert_dump_equal

pytestmark = pytest.mark.gpu

WORDS = (1, 0)                     # stand-in key word of Alice / Bob, as in tests/test_gpu_pit.py
SEEDS = (101, 202)                 # searcher seeds of Alice / Bob


def _engine(**kw):
    from alphasnake_zero_b200.engine import Engine
    return Engine(**kw)


def _argmaxs(V):                   # pit_agent.py:15-28
    return [(0 if v[0] > v[2] else 2) if v[0] > v[1] else (1 if v[1] > v[2] else 2) for v in V]


def _oracle_pit(games, S, acnt, seed, kinds, D, B, base):
    """pit_mp_game_runner.py:14-63 over oracle games with native spawn, each side an oracle search agent (its own table, seed,
    stand-in word) or the stand-in's argmax.  Decided games keep being stepped with move 1, as the arena does.
    Returns (moves per turn [G, 8] with 255 = no move, winners, decided turn, oracle agents, sub-games searched per side)."""
    from oracle import oracle as orc
    G = len(games)
    agents = []
    for side, kind in enumerate(kinds):
        if kind == "search":
            a = orc.OracleAgent(base=base, training=False, max_depth=D, max_breadth=B,
                                value_fn=None if WORDS[side] == 1 else KeyStubNet(WORDS[side]).v)
            a.set_rhat_mode(True)   # the kernels' order: every r-hat of a step from the values before the step's backups
            agents.append(a)
        else:
            agents.append(None)
    root_turn = [0, 0]
    searched = [0, 0]
    running = np.ones(G, bool)                 # fresh or auto-reset games: none is finished when the match begins
    ended = np.zeros(G, bool)
    winners, decided = np.full(G, -1), np.full(G, -1)
    log, turn = [], 0
    while running.any():
        live = {gi: games[gi].live_ids() for gi in range(G) if not ended[gi]}
        act = {gi: {sid: 1 for sid in ids} for gi, ids in live.items()}
        played = np.full((G, 8), 255, np.uint8)
        for side in (0, 1):
            rows = [(gi, sid) for gi in np.nonzero(running)[0] for sid in live[gi] if (sid < acnt) == (side == 0)]
            if not rows:
                continue
            if agents[side] is None:
                planes = np.array([games[gi].make_state(live[gi].index(sid)) for gi, sid in rows])
                mv = _argmaxs(KeyStubNet(WORDS[side]).v(planes))
            else:
                run_ids = list(np.nonzero(running)[0])
                omv, _ = agents[side].make_moves([games[gi] for gi in run_ids], G, root_turn=root_turn[side], seed=SEEDS[side])
                root_turn[side] += 1
                searched[side] += len(run_ids) * min(8, B) * (B // min(8, B))   # P sub-games per game in each epoch
                at = {}
                k = 0
                for gi in run_ids:
                    for sid in live[gi]:
                        at[(gi, sid)] = int(omv[k]); k += 1
                mv = [at[r] for r in rows]
            for (gi, sid), m in zip(rows, mv):
                act[gi][sid] = m
                played[gi, sid] = m
        log.append(played)
        turn += 1
        for gi, ids in live.items():
            g = games[gi]
            if g.tic(np.array([act[gi][sid] for sid in ids], np.int32), spawn_mode=2, chance=0.15, seed=seed):
                ended[gi] = True
            if not running[gi]:
                continue
            if ended[gi]:
                w = np.nonzero(g.dump()["snake"][:, 5] == 1)[0]
                winners[gi] = int(w[0]) if len(w) else -1
            else:
                lv = g.live_ids()
                if not (all(s < acnt for s in lv) or all(s >= acnt for s in lv)):
                    continue
                winners[gi] = lv[0] if lv else -1
            decided[gi] = turn
            running[gi] = False
    return log, winners, decided, agents, searched


def _seeded_games(side, S, G, seed, dec, warm_tics):
    """the engine's root games and the oracle's, from the same seed; warm_tics of uniform-random play with in-place reset give
    a mid-game start (games of every age)"""
    import os
    from oracle import oracle as orc
    eng = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=seed)
    eng.reset()
    games = []
    for gi in range(G):
        g = orc.OracleGame(side, side, S, dec); g.init_native(seed, gi, 0); g.set_ids(gi, 0); games.append(g)
    if warm_tics:
        for _ in range(warm_tics):
            eng.step(spawn_mode=2, tic=True, encode=False, auto_reset=True, random_actions=True)
        orc.env_run(G, side, side, S, dec, 0.15, seed, warm_tics, encode=False, n_threads=os.cpu_count() or 1, games=games)
    for gi in range(G):
        assert_dump_equal(eng.get_state(gi), games[gi].dump(), "game %d at the start" % gi)
    return eng, games


@pytest.mark.parametrize("side,S,acnt,G,D,B,dec,warm,kinds", [
    (11, 2, 1, 24, 4, 8, 3, 0, ("search", "search")),
    (11, 4, 2, 16, 4, 16, 3, 0, ("search", "search")),
    (7, 4, 3, 16, 3, 8, 5, 0, ("search", "search")),
    (19, 8, 4, 4, 4, 8, 3, 20, ("search", "search")),
    (11, 2, 1, 24, 4, 8, 3, 0, ("search", "argmax")),
    (11, 4, 2, 16, 4, 8, 3, 0, ("argmax", "search"))])
def test_search_pit_against_oracle(side, S, acnt, G, D, B, dec, warm, kinds):
    """stand-in search sides (key words 1 / 0, their own seeds and tables) on the arena, stepwise with a move log, against the
    oracle's composition: moves, winners, decided turns, final states; tables (keys, N, ages exact, W to reassociation) and
    search counters.  Decided games are not searched: the sub-games counted are those of the running games only."""
    import torch
    base, seed = 2.0, 31
    eng, games = _seeded_games(side, S, G, seed, dec, warm)
    searchers = [None, None]
    for s in (0, 1):
        if kinds[s] == "search":
            searchers[s] = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=SEEDS[s], max_depth=D, max_breadth=B,
                                   softmax_base=base, training=False)
            searchers[s].reset()
            searchers[s].search(value_fn=None)          # a used table: the match must start from a cleared one
        eng.pit_set_search(s, searchers[s])
    running = eng.pit_begin(WORDS[0], WORDS[1], acnt)
    log = []
    while running:
        moves = torch.empty(G, 8, dtype=torch.uint8, device="cuda")
        running = eng.pit_turn(spawn_mode=2, moves=moves)
        log.append(moves.cpu().numpy())
    winners, decided, turns = eng.pit_finish()
    want_log, want_w, want_d, agents, searched = _oracle_pit(games, S, acnt, seed, kinds, D, B, base)
    for t, (a, b) in enumerate(zip(log, want_log)):
        assert np.array_equal(a, b), "moves differ in turn %d" % t
    assert turns == len(log) == len(want_log)
    assert np.array_equal(decided, want_d) and np.array_equal(winners, want_w)
    for gi in range(G):
        assert_dump_equal(eng.get_state(gi), games[gi].dump(), "game %d at the end" % gi)
    st = eng.pit_stats()
    assert st["search_rows"] == sum(int((m[:, :acnt] != 255).sum()) * (kinds[0] == "search") +
                                    int((m[:, acnt:] != 255).sum()) * (kinds[1] == "search") for m in log)
    if G > 4:
        assert decided.min() < turns, "no game was decided early"
    for s in (0, 1):
        if searchers[s] is None:
            continue
        tab, otab = searchers[s].table(), agents[s].table()
        oo = np.lexsort((otab["keys"][:, 1], otab["keys"][:, 0]))
        assert len(tab["keys"]) > 0
        assert np.array_equal(tab["keys"], otab["keys"][oo]), "side %d: key sets differ" % s
        assert np.array_equal(tab["N"], otab["N"][oo]) and np.array_equal(tab["age"], otab["age"][oo])
        np.testing.assert_allclose(tab["W"], otab["W"][oo], rtol=0, atol=1e-4)
        ss = searchers[s].search_stats()
        assert ss["subgames"] == searched[s] == agents[s].stat("subgames")
        assert ss["evals"] == agents[s].stat("evals") and ss["node_visits"] == agents[s].stat("node_visits")
        assert ss["overflow"] == 0 and ss["collisions"] == 0
        team = slice(0, acnt) if s == 0 else slice(acnt, S)
        assert searchers[s].search_info()["root_turn"] == sum(int((m[:, team] != 255).any()) for m in log)


def _nets(side, backend="native"):
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    kw = dict(backend="torch", dtype="fp32") if backend == "torch" else {}
    return [AlphaNNet(input_shape=(2 * side - 1, 2 * side - 1, 3), seed=s, **kw) for s in (1, 2)]


def _agent(kind, nnet):
    from alphasnake_zero_b200.utils.agent import Agent
    from alphasnake_zero_b200.utils.pit_agent import Agent as PitAgent
    if kind == "argmax":
        return PitAgent(nnet)
    return Agent(nnet, softmax_base=2.0, training=False, max_MCTS_depth=4, max_MCTS_breadth=8)


@pytest.mark.parametrize("kinds", [("search", "search"), ("search", "argmax"), ("argmax", "search")])
def test_arena_equals_loop_with_search_agents(kinds):
    """two random-init native AlphaNNets: the arena (native=None) and the loop (native=False) run the same search and network
    kernels, so they play the same match: winners, every move, the final state of every game"""
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner
    side, S, G, acnt = 11, 2, 64, 1
    nets = _nets(side)
    out = []
    for native in (None, False):
        gr = MPGameRunner(side, side, S, 3, G, seed=9)
        log = []
        w = gr.run(_agent(kinds[0], nets[0]), _agent(kinds[1], nets[1]), acnt, move_log=log, native=native)
        out.append((gr, w, log))
    (ga, wa, la), (gl, wl, ll) = out
    st = ga.engine.pit_stats()
    assert st["turns"] == len(la) > 0 and st["search_rows"] > 0            # native=None chose the arena
    assert gl.engine.pit_stats()["turns"] == 0                              # native=False: the loop
    assert wa == wl
    assert len(la) == len(ll)
    for t, (a, b) in enumerate(zip(la, ll)):
        assert np.array_equal(a, b), "moves differ in turn %d" % t
    for gi in range(G):
        assert_dump_equal(ga.engine.get_state(gi), gl.engine.get_state(gi), "game %d" % gi)
    assert any(w is not None for w in wa)
    # the runner keeps its searchers: a second match from the same start begins with cleared tables and is the same match
    searchers = [q for q in ga._searchers if q is not None]
    ga.engine.reset()
    assert ga.run(_agent(kinds[0], nets[0]), _agent(kinds[1], nets[1]), acnt) == wa
    assert [q for q in ga._searchers if q is not None] == searchers


def test_torch_network_search_side_runs_on_the_loop():
    """a search side over backend="torch" is played by the loop (Engine.search with value_fn=nnet.v_device): the match completes
    with legal moves"""
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner
    (t, _), (n, _) = _nets(11, "torch"), _nets(11)
    gr = MPGameRunner(11, 11, 2, 10, 8, seed=3)
    log = []
    w = gr.run(_agent("search", t), _agent("argmax", n), 1, move_log=log)
    assert len(w) == 8 and len(log) > 0
    assert gr.engine.pit_stats()["turns"] == 0
    for m in log:
        assert ((m == 255) | (m < 3)).all()
    assert any((m[:, 0] < 3).any() for m in log)


def test_training_search_agent_is_refused():
    from alphasnake_zero_b200.utils.agent import Agent, StubNet
    from alphasnake_zero_b200.utils.pit_agent import Agent as PitAgent
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner
    (n,) = _nets(11)[:1]
    gr = MPGameRunner(11, 11, 2, 1, 4, seed=1)
    for native in (None, False):
        with pytest.raises(ValueError):
            gr.run(Agent(StubNet(), training=True, max_MCTS_depth=2, max_MCTS_breadth=8), PitAgent(n), 1, native=native)


def test_searcher_argument_errors():
    import torch
    from alphasnake_zero_b200._lib import AszError
    G = 8
    eng = _engine(side=11, snakes=4, health_dec=1, games=G, seed=1)
    eng.reset()

    def searcher(**kw):
        cfg = dict(side=11, snakes=4, health_dec=1, games=G, seed=2, max_depth=2, max_breadth=8, training=False)
        cfg.update(kw)
        return _engine(**cfg)
    bad = [searcher(games=G + 1), searcher(side=7), searcher(snakes=2), searcher(max_breadth=0, max_depth=0),
           searcher(training=True), searcher(health_dec=2), eng]
    for q in bad:
        for side in (0, 1):
            eng.pit_set_search(side, q)
            with pytest.raises(AszError, match="error -1.*searcher"):
                eng.pit_begin(1, 0, 2)
            with pytest.raises(AszError, match="error -1"):
                eng.pit_run(1, 0, 2)
            eng.pit_set_search(side, None)
    q = searcher()
    eng.pit_set_search(0, q); eng.pit_set_search(1, q)
    with pytest.raises(AszError, match="error -1.*both sides"):
        eng.pit_begin(1, 0, 2)
    eng.pit_set_search(1, None)
    with pytest.raises(AszError, match="error -1"):
        eng.pit_set_search(2, q)
    assert eng.pit_begin(1, 0, 2) == G                       # one matching searcher is accepted
    eng.pit_turn()
    eng.pit_set_search(0, None)
    # asz_copy_root_games refuses engines of another shape or device, and a self-copy
    for other in (searcher(games=G + 1), searcher(side=7), searcher(snakes=2)):
        with pytest.raises(AszError, match="error -1"):
            other.copy_root_games_from(eng)
    with pytest.raises(AszError, match="error -1"):
        eng.copy_root_games_from(eng)
    # a copy is the source's games, with the skipped ones finished
    skip = torch.zeros(G, dtype=torch.bool); skip[3] = True
    q.copy_root_games_from(eng, skip=skip)
    for gi in range(G):
        got, want = q.get_state(gi), eng.get_state(gi)
        assert_dump_equal(got, want, "game %d" % gi)
        assert got["counters"][7] == (1 if gi == 3 else want["counters"][7])
    torch.cuda.synchronize()


def test_table_overflow_is_a_capacity_error_with_results():
    """a searcher whose Q table (2^10 slots) fills within a few turns (entries live for max_depth root turns): asz_pit_run stops in
    the turn that overflowed with ASZ_ERR_CAPACITY and the results so far written, which the Engine attaches to the error"""
    from alphasnake_zero_b200._lib import AszError
    G = 64
    eng = _engine(side=11, snakes=4, health_dec=1, games=G, seed=1)
    eng.reset()
    q = _engine(side=11, snakes=4, health_dec=1, games=G, seed=2, max_depth=4, max_breadth=16, training=False, table_log2=10)
    eng.pit_set_search(0, q)
    with pytest.raises(AszError, match="error -4.*overflow") as ei:
        eng.pit_run(1, 0, 2)
    w, d, turns = ei.value.partial
    assert turns >= 1 and turns == eng.pit_stats()["turns"] and len(w) == G
    assert ((d == -1) | ((d >= 1) & (d <= turns))).all() and (w[d == -1] == -1).all() and (d == -1).any()
    assert q.search_stats()["overflow"] > 0
    with pytest.raises(AszError, match="error -3"):
        eng.pit_turn()                                           # the match is closed
