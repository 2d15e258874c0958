"""GPU: the device pit (asz_pit_*, utils/pit_mp_game_runner.MPGameRunner.run on the arena) plays the reference's matches:
the recorded pit fixtures move for move, seeded native-spawn matches against the CPU oracle, and the Python loop with real
networks down to the final state of every game."""
import numpy as np
import pytest

from tests.helpers import KeyStubNet, assert_dump_equal, load

pytestmark = pytest.mark.gpu

PITS = ["1v1", "2v2", "1v3", "3v1_7x7"]


def _engine(**kw):
    from alphasnake_zero_b200.engine import Engine
    return Engine(**kw)


def _nets(side, seeds=(1, 2)):
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    return [AlphaNNet(input_shape=(2 * side - 1, 2 * side - 1, 3), seed=s) for s in seeds]


@pytest.mark.parametrize("name", PITS)
def test_arena_replays_reference_pit_fixtures(name):
    """the stepwise arena with stand-in players (Alice key word 1, Bob key word 0) and the recorded food cells: every move of every
    turn, the number of turns and the winner list of the unmodified reference"""
    import torch
    from alphasnake_zero_b200 import _lib
    from tests.test_gpu_env import init_dump
    z = load("pit_%s.npz" % name)
    side, S, dec, G = int(z["H"]), int(z["S"]), int(z["health_dec"]), int(z["G"])
    acnt = S // 2 if int(z["alice_cnt"]) < 0 else int(z["alice_cnt"])
    eng = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=1)
    for gi in range(G):
        nf = int(z["init_nfood"][gi])
        eng.set_state(gi, init_dump(side, S, z["init_start"][gi], z["init_last"][gi], z["init_food"][gi][:nf]))
    trace = torch.from_numpy(np.ascontiguousarray(z["spawn"].astype(np.int32))).cuda()
    running = eng.pit_begin(1, 0, acnt)
    assert running == G
    t = 0
    while running:
        moves = torch.empty(G, 8, dtype=torch.uint8, device="cuda")
        running = eng.pit_turn(spawn_cells=trace[t], spawn_mode=_lib.SPAWN_REPLAY, moves=moves)
        assert np.array_equal(moves.cpu().numpy(), z["moves"][t]), "moves differ in turn %d" % t
        t += 1
    winners, decided, turns = eng.pit_finish()
    assert turns == t == z["moves"].shape[0]
    assert winners.tolist() == z["winners"].tolist()
    assert decided.max() == turns and decided.min() >= 1
    st = eng.pit_stats()
    assert st["turns"] == turns and st["net_rows"] == 0 and st["stub_rows"] == int((z["moves"] != 255).sum())


def _oracle_pit(side, S, acnt, G, seed, dec=1):
    """tests/test_oracle_pit.py's loop with native food spawn: (winners, decided turn) per game"""
    from oracle import oracle as orc
    from tests.test_oracle_pit import argmaxs
    nets = (KeyStubNet(1), KeyStubNet(0))
    games = {}
    for gi in range(G):
        g = orc.OracleGame(side, side, S, dec)
        g.init_native(seed, gi, 0)
        games[gi] = g
    winners, decided = np.full(G, -1), np.full(G, -1)
    turn = 0
    while games:
        rows, planes = [], []
        for gi, g in games.items():
            for k, sid in enumerate(g.live_ids()):
                rows.append((gi, sid))
                planes.append(g.make_state(k))
        planes = np.array(planes)
        team = np.array([sid >= acnt for _, sid in rows])
        mv = np.zeros(len(rows), np.int32)
        for b in (0, 1):
            if (team == b).any():
                mv[team == b] = argmaxs(nets[b].v(planes[team == b]))
        per = {}
        for (gi, sid), m in zip(rows, mv):
            per.setdefault(gi, []).append(m)
        turn += 1
        for gi in list(games):
            g = games[gi]
            ended = g.tic(np.array(per.get(gi, []), np.int32), spawn_mode=2, chance=0.15, seed=seed)
            if ended:
                w = np.nonzero(g.dump()["snake"][:, 5] == 1)[0]
                winners[gi] = int(w[0]) if len(w) else -1
            else:
                live = g.live_ids()
                if all(s < acnt for s in live) or all(s >= acnt for s in live):
                    winners[gi] = live[0] if live else -1
                else:
                    continue
            decided[gi] = turn
            del games[gi]
    return winners, decided, turn


@pytest.mark.parametrize("side,S,acnt", [(11, 2, 1), (11, 4, 2), (7, 4, 3), (19, 8, 4)])
def test_native_spawn_match_against_oracle(side, S, acnt):
    """asz_pit_run (one call, engine RNG food) with stand-in players against the oracle's games: winner and decided turn of every
    one of 512 games"""
    G, seed = 512, 31
    eng = _engine(side=side, snakes=S, health_dec=1, games=G, seed=seed)
    eng.reset()
    winners, decided, turns = eng.pit_run(1, 0, acnt)
    want_w, want_d, want_turns = _oracle_pit(side, S, acnt, G, seed)
    assert np.array_equal(decided, want_d), np.nonzero(decided != want_d)[0][:10]
    assert np.array_equal(winners, want_w), np.nonzero(winners != want_w)[0][:10]
    assert turns == want_turns
    assert len(set(winners.tolist())) > 1


def _two_runs(side, S, G, acnt, nets, seed=7, dec=1):
    """the same match on the arena (stepwise with a move log) and on the Python loop: winners, move logs, final states"""
    from alphasnake_zero_b200.utils.pit_agent import Agent as PitAgent
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner as PitRunner
    out = []
    for native in (True, False):
        gr = PitRunner(side, side, S, dec, G, seed=seed)
        log = []
        w = gr.run(PitAgent(nets[0]), PitAgent(nets[1]), acnt, move_log=log, native=native)
        out.append((gr, w, log))
    (ga, wa, la), (gl, wl, ll) = out
    assert wa == wl
    assert len(la) == len(ll)
    for t, (a, b) in enumerate(zip(la, ll)):
        assert np.array_equal(a, b), "moves differ in turn %d" % t
    for gi in range(G):
        da, dl = ga.engine.get_state(gi), gl.engine.get_state(gi)
        for k in ("snake", "owner", "dist", "food", "counters"):
            assert np.array_equal(da[k], dl[k]), (gi, k)
    assert ga.engine.pit_stats()["net_rows"] == sum(int((m != 255).sum()) for m in la)
    return wa, ga


@pytest.mark.parametrize("side,S,G,acnt,shared", [(11, 2, 256, 1, False), (11, 4, 128, 2, False), (19, 4, 32, 2, False),
                                                  (11, 4, 128, 2, True)])
def test_arena_equals_python_loop_with_networks(side, S, G, acnt, shared):
    """two random-init native AlphaNNets (or one on both sides): the arena and the loop play the same match, move for move"""
    from alphasnake_zero_b200.utils.pit_agent import Agent as PitAgent
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner as PitRunner
    a, b = _nets(side)
    nets = (a, a) if shared else (a, b)
    winners, ga = _two_runs(side, S, G, acnt, nets)
    assert any(w is not None for w in winners)
    # the one-call path (asz_pit_run) gives the same match as the stepwise calls
    gr = PitRunner(side, side, S, 1, G, seed=7)
    assert gr.run(PitAgent(nets[0]), PitAgent(nets[1]), acnt) == winners
    assert gr.engine.pit_stats()["turns"] > 0                    # native=None chose the arena
    for gi in range(0, G, 5):
        assert_dump_equal(gr.engine.get_state(gi), ga.engine.get_state(gi), "game %d" % gi)


@pytest.mark.parametrize("acnt", [0, 4])
def test_empty_team_is_decided_after_the_first_tic(acnt):
    a, b = _nets(11)
    winners, _ = _two_runs(11, 4, 32, acnt, (a, b))
    eng = _engine(side=11, snakes=4, health_dec=1, games=64, seed=3)
    eng.reset()
    w, decided, turns = eng.pit_run(1, 0, acnt)
    assert turns == 1 and (decided == 1).all()


def test_single_game():
    a, b = _nets(11)
    _two_runs(11, 2, 1, 1, (a, b), seed=12)


def test_argument_and_state_errors():
    import torch
    from alphasnake_zero_b200._lib import AszError
    eng = _engine(side=11, snakes=4, health_dec=1, games=8, seed=1)
    eng.reset()
    with pytest.raises(AszError, match="error -3"):
        eng.pit_turn()                                           # no begin
    with pytest.raises(AszError, match="error -3"):
        eng.pit_finish()
    assert eng.pit_begin(1, 0, 2) == 8
    (n7,) = _nets(7, seeds=(1,))
    with pytest.raises(AszError, match="error -1.*side 7"):
        eng.pit_begin(n7._get_native(), 0, 2)                    # a network of another board side
    with pytest.raises(AszError, match="error -3"):
        eng.pit_turn()                                           # a failed begin abandons the match in progress
    with pytest.raises(AszError, match="error -1"):
        eng.pit_begin(1, 0, 5)                                   # alice_snakes outside 0..S
    with pytest.raises(AszError, match="error -1"):
        eng.pit_begin(2, 0, 2)                                   # stub word
    eng.pit_begin(1, 0, 2)
    with pytest.raises(AszError, match="error -1"):
        eng.pit_turn(spawn_mode=1)                               # replay without cells
    eng.pit_turn()
    with pytest.raises(AszError, match="error -3.*still running") as ei:
        eng.pit_finish()
    w, d, turns = ei.value.partial
    assert turns == 1 and ((d == -1) | (d == 1)).all() and (w[d == -1] == -1).all()
    with pytest.raises(AszError, match="error -3"):
        eng.pit_turn()                                           # finished: no match open
    torch.cuda.synchronize()


def test_max_turns_and_trace_end_write_partial_results():
    from alphasnake_zero_b200._lib import AszError
    from alphasnake_zero_b200.utils.pit_agent import Agent as PitAgent
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner as PitRunner
    full = _engine(side=11, snakes=4, health_dec=3, games=256, seed=4)
    full.reset()
    w_full, d_full, turns_full = full.pit_run(1, 0, 2)
    k = int(np.median(d_full))
    assert 1 < k < turns_full
    eng = _engine(side=11, snakes=4, health_dec=3, games=256, seed=4)
    eng.reset()
    with pytest.raises(AszError, match="error -3") as ei:
        eng.pit_run(1, 0, 2, max_turns=k)
    w, d, turns = ei.value.partial
    assert turns == k
    done = d_full <= k
    assert np.array_equal(d[done], d_full[done]) and np.array_equal(w[done], w_full[done])
    assert (d[~done] == -1).all() and (w[~done] == -1).all()
    # the trace of a replayed match runs out while games are running
    a, b = _nets(11)
    gr = PitRunner(11, 11, 2, 1, 16, seed=2)
    with pytest.raises(AszError, match="error -3") as ei:
        gr.run(PitAgent(a), PitAgent(b), 1, spawn_trace=np.full((3, 16), -1, np.int32), native=True)
    w, d, turns = ei.value.partial
    assert turns == 3 and (d == -1).any()


def test_game_finished_before_the_match_is_a_draw_at_turn_0():
    from alphasnake_zero_b200 import _lib
    eng = _engine(side=7, snakes=4, health_dec=9, games=64, seed=5)
    eng.reset()
    eng.alive_mask()                                             # binds the record views
    for _ in range(60):                                          # uniform-random play without reset until some games are over
        eng.step(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=False, random_actions=True)
        finished = ((eng._meta_view[:, 7] & 1) == 1).cpu().numpy()
        if finished.sum() >= 8:
            break
    assert 0 < finished.sum() < 64
    w, d, turns = eng.pit_run(1, 0, 2)
    assert (d[finished] == 0).all() and (w[finished] == -1).all()
    assert (d[~finished] >= 1).all() and turns == d.max()


def test_runner_chooses_the_arena_only_for_native_pit_agents():
    from alphasnake_zero_b200._lib import AszError
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    from alphasnake_zero_b200.utils.pit_agent import Agent as PitAgent
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner as PitRunner
    t = [AlphaNNet(input_shape=(21, 21, 3), seed=s, backend="torch", dtype="fp32") for s in (1, 2)]
    gr = PitRunner(11, 11, 2, 1, 8, seed=4)
    assert len(gr.run(PitAgent(t[0]), PitAgent(t[1]), 1)) == 8
    assert gr.engine.pit_stats()["turns"] == 0                   # the torch backend goes through the loop
    with pytest.raises(AszError):
        PitRunner(11, 11, 2, 1, 8, seed=4).run(PitAgent(KeyStubNet(1)), PitAgent(KeyStubNet(0)), 1, native=True)
    a, _ = _nets(11)
    (n7,) = _nets(7, seeds=(1,))
    with pytest.raises(AszError):
        PitRunner(11, 11, 2, 1, 8, seed=4).run(PitAgent(a), PitAgent(n7), 1, native=True)


def test_failed_run_leaves_no_match_and_no_partial_results():
    """an asz_pit_run that cannot start abandons the match in progress: a later finish is the plain state error, with no results"""
    from alphasnake_zero_b200._lib import AszError
    eng = _engine(side=11, snakes=2, health_dec=1, games=8, seed=1)
    eng.reset()
    eng.pit_begin(1, 0, 1)
    eng.pit_turn()
    with pytest.raises(AszError, match="error -1") as ei:
        eng.pit_run(1, 0, 3)                                     # alice_snakes outside 0..S
    assert not hasattr(ei.value, "partial")
    with pytest.raises(AszError, match="error -3") as ei:
        eng.pit_finish()
    assert not hasattr(ei.value, "partial")
    with pytest.raises(AszError, match="error -1"):
        eng.pit_run(1, 0, 1, max_turns=-1)
    with pytest.raises(AszError, match="error -3"):
        eng.pit_turn()
