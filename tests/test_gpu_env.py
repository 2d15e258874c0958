"""GPU parity: the CUDA lockstep tic + fused plane encode (through the C ABI) against
 (1) the fixtures produced by the unmodified reference, (2) the CPU oracle on seeded full-size runs."""
import os

import numpy as np
import pytest

from tests.helpers import assert_dump_equal, digest, golden_dump, load

pytestmark = pytest.mark.gpu

ENVS = ["11x11x4", "11x11x4_dec9", "7x7x4", "19x19x8", "11x11x2", "7x7x8"]


def _engine(**kw):
    from alphasnake_zero_b200.engine import Engine
    return Engine(**kw)


def init_dump(side, S, start, last, food):
    Cn = side * side
    snake = np.zeros((S, 6), np.int32); owner = np.full(Cn, -1, np.int32); dist = np.zeros(Cn, np.int32)
    fd = np.zeros(Cn, np.int32)
    for i in range(S):
        c = int(start[i][0]) * side + int(start[i][1])
        snake[i] = [1, 100, 3, int(last[i]), c, 0]
        owner[c] = i; dist[c] = 3
    for (y, x) in food:
        fd[int(y) * side + int(x)] = 1
    return dict(snake=snake, owner=owner, dist=dist, food=fd, counters=np.zeros(8, np.int32))


@pytest.mark.parametrize("name", ENVS)
def test_env_replay_against_reference(name):
    import torch
    z = load("env_%s.npz" % name)
    side, S, dec = int(z["H"]), int(z["S"]), int(z["health_dec"])
    gp = z["game_ptr"]
    G = len(gp) - 1
    eng = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=1)
    for gi in range(G):
        nf = int(z["init_nfood"][gi])
        eng.set_state(gi, init_dump(side, S, z["init_start"][gi], z["init_last"][gi], z["init_food"][gi][:nf]))
    live_ids = [list(range(S)) for _ in range(G)]
    full = {(int(t), int(k)): i for i, (t, k) in enumerate(z["full_idx"])}
    max_len = int((gp[1:] - gp[:-1]).max())
    n_planes = 0
    for step in range(max_len):
        actions = np.ones((G, 8), np.uint8)
        spawn = np.full(G, -1, np.int32)
        running = []
        for gi in range(G):
            t = int(gp[gi]) + step
            if t >= int(gp[gi + 1]):
                continue
            running.append(gi)
            n = int(z["nlive"][t])
            assert n == len(live_ids[gi])
            for k, sid in enumerate(live_ids[gi]):
                actions[gi, sid] = z["moves"][t][k]
            spawn[gi] = int(z["spawn"][t])
        eng.step(actions=torch.from_numpy(actions).cuda(), spawn_cells=torch.from_numpy(spawn).cuda(), spawn_mode=1,
                 tic=True, encode=True)
        ids, planes = eng.rows()
        planes = planes.cpu().numpy()
        ended = eng.ended.cpu().numpy()
        row_of = {int(i): r for r, i in enumerate(ids)}
        for gi in running:
            t = int(gp[gi]) + step
            want = golden_dump(z, t)
            assert_dump_equal(eng.get_state(gi), want, "%s game %d tic %d" % (name, gi, t))
            assert int(ended[gi]) == int(z["ended"][t])
            live_ids[gi] = [s for s in range(S) if want["snake"][s][0] == 1]
            d0, d1 = int(z["dig_ptr"][t]), int(z["dig_ptr"][t + 1])
            if z["ended"][t]:
                assert all((gi * 8 + s) not in row_of for s in range(S))   # ended games produce no rows
                continue
            assert d1 - d0 == len(live_ids[gi])
            for k, sid in enumerate(live_ids[gi]):
                p = planes[row_of[gi * 8 + sid]]
                assert digest(p) == z["digests"][d0 + k], (name, gi, t, k)
                if (t, k) in full:
                    assert np.array_equal(p.view(np.uint32), z["full_planes"][full[(t, k)]].view(np.uint32))
                n_planes += 1
        # finished games must not change any more and must not emit rows
        assert len(ids) == sum(len(live_ids[g]) for g in running if not z["ended"][int(gp[g]) + step])
    assert n_planes > 0
    eng.close()


def test_edge_cases_against_reference():
    import torch
    z = load("edge_cases.npz")
    n = len(z["names"])
    for dec in sorted(set(z["health_dec"].tolist())):
        idx = [i for i in range(n) if int(z["health_dec"][i]) == dec]
        eng = _engine(side=11, snakes=4, health_dec=dec, games=len(idx), seed=0)
        for j, i in enumerate(idx):
            eng.set_state(j, {k: z["before_" + k][i] for k in ("snake", "owner", "dist", "food", "counters")})
        # planes of the hand-built states
        eng.step(tic=False, encode=True)
        ids, planes = eng.rows()
        planes = planes.cpu().numpy()
        row_of = {int(v): r for r, v in enumerate(ids)}
        for j, i in enumerate(idx):
            pb = z["planes_before"][int(z["pb_ptr"][i]):int(z["pb_ptr"][i + 1])]
            live = [s for s in range(4) if z["before_snake"][i][s][0] == 1]
            assert len(pb) == len(live)
            for k, sid in enumerate(live):
                assert np.array_equal(planes[row_of[j * 8 + sid]].view(np.uint32), pb[k].view(np.uint32)), z["names"][i]
        actions = np.ones((len(idx), 8), np.uint8)
        for j, i in enumerate(idx):
            live = [s for s in range(4) if z["before_snake"][i][s][0] == 1]
            for k, sid in enumerate(live):
                actions[j, sid] = z["moves"][i][k]
        eng.step(actions=torch.from_numpy(actions).cuda(), spawn_mode=0, tic=True, encode=True)
        ids, planes = eng.rows()
        planes = planes.cpu().numpy()
        row_of = {int(v): r for r, v in enumerate(ids)}
        ended = eng.ended.cpu().numpy()
        for j, i in enumerate(idx):
            name = str(z["names"][i])
            after = {k: z["after_" + k][i] for k in ("snake", "owner", "dist", "food", "counters")}
            assert_dump_equal(eng.get_state(j), after, name)
            assert int(ended[j]) == int(z["ended"][i]), name
            if z["ended"][i]:
                continue
            pa = z["planes_after"][int(z["pa_ptr"][i]):int(z["pa_ptr"][i + 1])]
            live = [s for s in range(4) if after["snake"][s][0] == 1]
            for k, sid in enumerate(live):
                assert np.array_equal(planes[row_of[j * 8 + sid]].view(np.uint32), pa[k].view(np.uint32)), name
        eng.close()


def test_edge_sequences_against_reference():
    """multi-tic scenarios recorded from the reference: a head-on winner ends a tic alive with health <= 0 (game.py:156-165 is an
    elif chain; the packed record keeps health signed), then starves / eats / hits the wall / wins again; health_dec 9, 3, 1.
    States, counters, `ended` and every plane (food channel (101 - health) * 0.01 > 1) bit for bit after every tic."""
    import torch
    z = load("edge_sequences.npz")
    keys = ("snake", "owner", "dist", "food", "counters")
    n = len(z["names"])
    assert int(z["min_health"].min()) < 0
    for dec in sorted(set(z["health_dec"].tolist())):
        idx = [i for i in range(n) if int(z["health_dec"][i]) == dec]
        eng = _engine(side=11, snakes=4, health_dec=dec, games=len(idx), seed=0, food_chance=0.0)
        live = {}
        for j, i in enumerate(idx):
            eng.set_state(j, {k: z["before_" + k][i] for k in keys})
            live[j] = [s for s in range(4) if z["before_snake"][i][s][0] == 1]
        max_t = max(int(z["tic_ptr"][i + 1] - z["tic_ptr"][i]) for i in idx)
        for step in range(max_t):
            actions = np.ones((len(idx), 8), np.uint8)
            running = []
            for j, i in enumerate(idx):
                t = int(z["tic_ptr"][i]) + step
                if t >= int(z["tic_ptr"][i + 1]):
                    continue
                running.append((j, i, t))
                for k, sid in enumerate(live[j]):
                    actions[j, sid] = z["moves"][t][k]
            # spawn mode NATIVE with food_chance 0: the reference's guard (game.py:130) means nothing is ever spawned
            eng.step(actions=torch.from_numpy(actions).cuda(), spawn_mode=2, tic=True, encode=True)
            ids, planes = eng.rows()
            planes = planes.cpu().numpy()
            row_of = {int(v): r for r, v in enumerate(ids)}
            ended = eng.ended.cpu().numpy()
            for j, i, t in running:
                name = "%s tic %d" % (z["names"][i], step)
                after = {k: z["after_" + k][t] for k in keys}
                got = eng.get_state(j)
                assert_dump_equal(got, after, name)
                assert int(ended[j]) == int(z["ended"][t]), name
                live[j] = [s for s in range(4) if after["snake"][s][0] == 1]
                pl = z["planes"][int(z["pl_ptr"][t]):int(z["pl_ptr"][t + 1])]
                assert len(pl) == (0 if z["ended"][t] else len(live[j])), name
                for k, sid in enumerate(live[j][:len(pl)]):
                    assert np.array_equal(planes[row_of[j * 8 + sid]].view(np.uint32), pl[k].view(np.uint32)), name
        eng.close()


@pytest.mark.parametrize("dec,G,tics", [(9, 768, 320), (3, 512, 320)])
def test_long_survival_run_against_oracle(dec, G, tics):
    """The trainer's health_dec 9 and 3 (alpha_snake_zero_trainer.py:42-47) with play that survives long enough to starve:
    every snake picks uniformly among the moves its own plane shows as free (ch1 of the three cells around the centre),
    the same actions go to the engine (asz_env_step) and to the oracle, food spawns natively on both sides, ended games
    restart in place.  EVERY game is compared every 40 tics and at the end; the run must contain starvations and snakes that
    ended a tic alive with health <= 0 (game.py:156-165)."""
    import torch
    from oracle import oracle as orc
    seed, side, S = 4242 + dec, 11, 4
    eng = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=seed)
    eng.reset()
    games = []
    for gi in range(G):
        g = orc.OracleGame(side, side, S, dec); g.init_native(seed, gi, 0); games.append(g)
    episode = [0] * G
    gen = torch.Generator(device="cpu"); gen.manual_seed(seed)
    rng = np.random.default_rng(seed)
    c = side - 1
    nonpositive, since_injection = 0, 99
    for t in range(tics):
        eng.step(tic=False, encode=True)
        n = int(eng.row_count.item())
        ids = eng.row_ids[:n].long()
        pl = eng.planes[:n]
        blocked = torch.stack([pl[:, c, c - 1, 1], pl[:, c - 1, c, 1], pl[:, c, c + 1, 1]], 1) >= 0.04
        score = torch.rand(n, 3, generator=gen).cuda() + (~blocked).float() * 2.0       # a free move always beats a blocked one
        mv = score.argmax(1).to(torch.uint8)
        actions = torch.ones(G * 8, dtype=torch.uint8, device="cuda")
        actions[ids] = mv
        eng.step(actions=actions.view(G, 8), spawn_mode=2, tic=True, encode=False, auto_reset=True)
        ah = actions.view(G, 8).cpu().numpy()
        for gi, g in enumerate(games):
            lv = g.live_ids()
            if g.tic(ah[gi, lv].astype(np.int32), spawn_mode=2, chance=0.15, seed=seed):
                episode[gi] += 1
                g.init_native(seed, gi, episode[gi])
            elif since_injection < 3:
                sn = g.dump()["snake"]
                nonpositive += int(((sn[:, 0] == 1) & (sn[:, 1] <= 0)).sum())
        since_injection += 1
        if t % 40 == 39 or t == tics - 1:
            for gi, g in enumerate(games):
                want = g.dump()
                got = eng.get_state(gi)
                assert_dump_equal(got, want, "dec %d game %d tic %d" % (dec, gi, t))
                assert got["counters"][6] == episode[gi]
                if t != tics - 1:
                    # natural play almost never brings a LONGER snake with health <= health_dec into a head-on collision, so
                    # every 40 tics all live snakes get a low health on both sides; the next tics then contain head-on winners
                    # that stay alive with health <= 0 and starve (or eat) one tic later
                    live = want["snake"][:, 0] == 1
                    want["snake"][live, 1] = rng.integers(1, 2 * dec + 1, size=int(live.sum()))
                    g.load_dump(want)
                    eng.set_state(gi, want, episode=episode[gi])
            since_injection = 0
    tot = eng.totals()
    assert tot["starve"] > 0 and tot["head"] > 0 and tot["episodes"] == sum(episode) > 0
    assert nonpositive > 0, "no snake ended a tic alive with health <= 0"
    eng.close()


def test_food_chance_zero_never_spawns():
    """game.py:130 `if self.food_spawn_chance > 0.0`: chance 0 with the native spawn mode never spawns, not even on an empty board"""
    import torch
    eng = _engine(side=11, snakes=2, health_dec=1, games=4, seed=3, food_chance=0.0)
    d = init_dump(11, 2, [(1, 1), (9, 9)], [1, 3], [])
    for gi in range(4):
        eng.set_state(gi, d)
    act = torch.ones(4, 8, dtype=torch.uint8, device="cuda")
    for _ in range(6):
        eng.step(actions=act, spawn_mode=2, tic=True, encode=False)
        assert all(eng.get_state(gi)["food"].sum() == 0 for gi in range(4))
    eng.close()
    eng = _engine(side=11, snakes=2, health_dec=1, games=4, seed=3, food_chance=1e-12)
    for gi in range(4):
        eng.set_state(gi, d)
    eng.step(actions=act, spawn_mode=2, tic=True, encode=False)
    assert all(eng.get_state(gi)["food"].sum() == 1 for gi in range(4))    # a board without food always gets one
    eng.close()


@pytest.mark.parametrize("side,S,dec,G,tics", [(11, 4, 1, 4096, 120), (7, 4, 9, 1024, 80), (19, 8, 1, 512, 150),
                                               (11, 2, 3, 1000, 60), (7, 8, 1, 333, 60),
                                               (11, 4, 1, 65536, 24),       # BASELINE.json configs[1] at full size
                                               # odd game counts above the single-game tail of a launch (3 games per resident warp):
                                               # scheduling tickets of two games, single games at the end of the launch and an odd
                                               # last game, on every board size
                                               (11, 4, 1, 20001, 30), (19, 8, 1, 4001, 20), (7, 4, 9, 12001, 24)])
def test_native_run_against_oracle(side, S, dec, G, tics):
    """Seeded native runs (engine RNG for layouts, actions and food; auto reset): every game's final state, the
    totals and an order-free checksum over every plane written must equal the oracle's, bit for bit."""
    import torch
    from oracle import oracle as orc
    seed = 1234 + side
    eng = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=seed)
    eng.reset()
    if G % 2 and G > 4000:     # the odd game counts: pair tickets first, then single games, the last of them alone in its ticket
        from tests.test_gpu_env_planes import launch_layout
        pairs, _ = launch_layout(side, G, torch.cuda.get_device_properties(eng.device).multi_processor_count)
        assert pairs > 0 and 2 * pairs < G and (G - 2 * pairs) % 2 == 1, (G, pairs)
    csum = torch.zeros((), dtype=torch.int64, device="cuda")
    planes = 0
    # initial planes are not part of the oracle's env_run accounting (it encodes after every tic)
    for _ in range(tics):
        eng.step(spawn_mode=2, tic=True, encode=True, auto_reset=True, random_actions=True, keys=True)
        n = int(eng.row_count.item())
        planes += n
        csum += eng.keys[:n, 0].sum()
    games = []
    for gi in range(G):
        g = orc.OracleGame(side, side, S, dec); g.init_native(seed, gi, 0); games.append(g)
    st = orc.env_run(G, side, side, S, dec, 0.15, seed, tics, encode=True, n_threads=os.cpu_count() or 1, games=games)
    tot = eng.totals()
    assert tot["tics"] == st["steps"] == G * tics
    assert tot["episodes"] == st["episodes"] and st["episodes"] > 0
    assert [tot[k] for k in ("wall", "body", "head", "starve", "food_eaten", "game_length")] == st["counters"]
    assert planes == st["planes"]
    assert (int(csum.item()) & 0xFFFFFFFFFFFFFFFF) == st["plane_checksum"]
    for gi in range(0, G, 1 if G <= 4096 else G // 1024):
        want = games[gi].dump()
        got = eng.get_state(gi)
        assert_dump_equal(got, want, "game %d" % gi)
        assert got["counters"][6] == want["counters"][6]   # episode
    eng.close()


def test_env_submit_wait_host_pipeline_equals_synchronous_steps():
    """asz_env_submit_host / asz_env_wait_host with two steps in flight: per-step host results, row counts and the final game
    states equal those of the same steps through the synchronous asz_env_step_host; a third submit without a wait is an error."""
    import ctypes as C
    import torch
    from alphasnake_zero_b200 import _lib
    from alphasnake_zero_b200.engine import AszError
    G, T = 512, 60
    rng = np.random.default_rng(5)
    acts = [torch.from_numpy(rng.integers(0, 3, size=(G, 8), dtype=np.uint8)).pin_memory() for _ in range(T)]
    ea, eb = _engine(side=11, snakes=4, games=G, seed=11), _engine(side=11, snakes=4, games=G, seed=11)
    ea.reset(); eb.reset()
    L = _lib.lib()
    flags = _lib.STEP_TIC | _lib.STEP_ENCODE | _lib.STEP_AUTO_RESET
    # synchronous reference run
    end_s = torch.zeros(G, dtype=torch.uint8).pin_memory(); rew_s = torch.zeros(G, 8, dtype=torch.int8).pin_memory()
    rows = C.c_int32(0)
    want = []
    for t in range(T):
        _lib.check(L.asz_env_step_host(ea.h, flags, 2, C.c_void_p(acts[t].data_ptr()), None, C.c_void_p(end_s.data_ptr()),
                                       C.c_void_p(rew_s.data_ptr()), C.byref(rows), None, None, ea.stream))
        want.append((end_s.numpy().copy(), rew_s.numpy().copy(), rows.value))
    # pipelined run: submit t+1 before waiting for t
    end_p = [torch.zeros(G, dtype=torch.uint8).pin_memory() for _ in range(2)]
    rew_p = [torch.zeros(G, 8, dtype=torch.int8).pin_memory() for _ in range(2)]
    kw = dict(spawn_mode=2, tic=True, encode=True, auto_reset=True)
    tickets = [eb.submit_host(acts[0], end_p[0], rew_p[0], **kw)]
    seen_end = 0
    for t in range(T):
        if t + 1 < T:
            tickets.append(eb.submit_host(acts[t + 1], end_p[(t + 1) & 1], rew_p[(t + 1) & 1], **kw))
            if t == 0:
                with pytest.raises(AszError):                       # two steps in flight already
                    eb.submit_host(acts[2], end_p[0], rew_p[0], **kw)
        n = eb.wait_host(tickets[t])
        w_end, w_rew, w_rows = want[t]
        assert n == w_rows, t
        assert np.array_equal(end_p[t & 1].numpy(), w_end) and np.array_equal(rew_p[t & 1].numpy(), w_rew), t
        seen_end += int(w_end.sum())
    assert seen_end > 0
    with pytest.raises(AszError):
        eb.wait_host(tickets[-1])                                   # already waited for
    torch.cuda.synchronize()
    for gi in range(0, G, 17):
        assert_dump_equal(eb.get_state(gi), ea.get_state(gi), "game %d" % gi)
    ta, tb = ea.totals(), eb.totals()
    assert all(ta[k] == tb[k] for k in ("tics", "planes", "episodes", "wall", "body", "head", "starve", "food_eaten"))
    ea.close(); eb.close()


def test_env_step_host_roundtrip():
    """asz_env_step_host: host buffers in, host results out (the e2e path of bench.py)."""
    import ctypes as C
    import torch
    from alphasnake_zero_b200 import _lib
    eng = _engine(side=11, snakes=4, games=256, seed=3)
    eng.reset()
    G = 256
    actions = torch.ones(G, 8, dtype=torch.uint8).pin_memory()
    ended = torch.zeros(G, dtype=torch.uint8).pin_memory()
    rewards = torch.zeros(G, 8, dtype=torch.int8).pin_memory()
    planes = torch.zeros(G * 4, 21, 21, 3).pin_memory()
    ids = torch.zeros(G * 4, dtype=torch.int32).pin_memory()
    rows = C.c_int32(0)
    L = _lib.lib()
    flags = _lib.STEP_TIC | _lib.STEP_ENCODE
    for t in range(5):
        _lib.check(L.asz_env_step_host(eng.h, flags, 2, C.c_void_p(actions.data_ptr()), None,
                                       C.c_void_p(ended.data_ptr()), C.c_void_p(rewards.data_ptr()), C.byref(rows),
                                       C.c_void_p(planes.data_ptr()), C.c_void_p(ids.data_ptr()), eng.stream))
    n = rows.value
    assert 0 < n <= G * 4
    # results written into pinned memory by the kernel (zero-copy), into pageable memory by copies, and the device-resident
    # results of an identical engine stepped through asz_env_step must agree
    ea, eb, ec = (_engine(side=11, snakes=4, games=256, seed=3) for _ in range(3))
    for x in (ea, eb, ec):
        x.reset()
    end_pin = torch.zeros(G, dtype=torch.uint8).pin_memory(); rew_pin = torch.zeros(G, 8, dtype=torch.int8).pin_memory()
    end_pg = np.zeros(G, np.uint8); rew_pg = np.zeros((G, 8), np.int8)
    act_d = torch.ones(G, 8, dtype=torch.uint8, device="cuda")
    r2 = C.c_int32(0)
    seen_end = 0
    for t in range(40):
        _lib.check(L.asz_env_step_host(ea.h, _lib.STEP_TIC, 2, C.c_void_p(actions.data_ptr()), None, C.c_void_p(end_pin.data_ptr()),
                                       C.c_void_p(rew_pin.data_ptr()), C.byref(r2), None, None, ea.stream))
        _lib.check(L.asz_env_step_host(eb.h, _lib.STEP_TIC, 2, C.c_void_p(actions.data_ptr()), None, end_pg.ctypes.data_as(C.c_void_p),
                                       rew_pg.ctypes.data_as(C.c_void_p), C.byref(r2), None, None, eb.stream))
        ec.step(actions=act_d, spawn_mode=2, tic=True, encode=False)
        torch.cuda.synchronize()
        assert np.array_equal(end_pin.numpy(), end_pg) and np.array_equal(rew_pin.numpy(), rew_pg), t
        assert np.array_equal(end_pg, ec.ended.cpu().numpy()) and np.array_equal(rew_pg, ec.rewards.cpu().numpy()), t
        seen_end += int(end_pg.sum())
    assert seen_end > 0
    for x in (ea, eb, ec):
        x.close()
    # all snakes went straight for 5 tics from a start cell next to the wall: planes must match get_state-derived oracle
    from oracle import oracle as orc
    order = np.argsort(ids[:n].numpy())
    for r in order[:64]:
        gid, sid = int(ids[r]) // 8, int(ids[r]) % 8
        g = orc.OracleGame(11, 11, 4, 1)
        d = eng.get_state(gid)
        g.load_dump(d)
        k = g.live_ids().index(sid)
        assert np.array_equal(g.make_state(k).view(np.uint32), planes[r].numpy().view(np.uint32))
    eng.close()


def test_no_cpu_fallback_symbols():
    from alphasnake_zero_b200 import _lib
    L = _lib.lib()
    for name, _, _ in _lib.SYMBOLS:
        assert hasattr(L, name)
