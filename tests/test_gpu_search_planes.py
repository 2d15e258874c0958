"""The planes the value network is fed during self-play, bit for bit against the CPU oracle's make_state:
 (1) every row of the search's evaluation batch (`search_step_kernel` -> `warp_encode<G, false>`), step by step, at all three
     board sizes, with the stub value function and with the native network; rows the step did not write must stay untouched,
     and the plane bytes must carry the key the table was probed with;
 (2) every training record of the device store (`asz_records_append`) and the sampled, mirrored batch (`records_gather_kernel`).
The oracle replays the trace the device recorded and hands its miss planes of each step to a value-function callback, which
compares them with the device's rows of the same step."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.helpers import SENTINEL, assert_dump_equal, load, plane_features

def eval_row_floats(eng):
    """Floats between consecutive rows of the evaluation batch (asz_search_eval_planes): dense planes."""
    return int(eng.L.asz_plane_floats(eng.h))


# ---- the comparator (runs without a GPU: test_plane_checker_on_cpu) ---------------------------------------------------------

def _keys(planes):
    from oracle import oracle as orc
    return [orc.plane_key(p) for p in planes]


def compare_step(label, got, want, got_keys=None, want_keys=None, limit=4):
    """got: the device's evaluation rows of one search step [n, N, N, 3] float32, want: the oracle's miss planes of the same
    step.  Rows are paired by plane key (the probe deduplicates, so keys are unique within a step) and compared as uint32
    words.  Returns a list of failure messages, empty when both steps hold the same set of planes bit for bit."""
    got_keys = _keys(got) if got_keys is None else got_keys
    want_keys = _keys(want) if want_keys is None else want_keys
    fails = []
    if len(got) != len(want):
        fails.append("%s: %d device rows, %d oracle rows" % (label, len(got), len(want)))
    gi = {k: i for i, k in enumerate(got_keys)}
    wi = {k: j for j, k in enumerate(want_keys)}
    if len(gi) != len(got_keys):
        fails.append("%s: %d device rows repeat a key of the same step" % (label, len(got_keys) - len(gi)))
    pairs = [(i, wi[k]) for k, i in gi.items() if k in wi]
    lost = [i for k, i in gi.items() if k not in wi]
    extra = [j for k, j in wi.items() if k not in gi]
    if lost or extra:
        fails.append("%s: key sets differ: %d device rows have a key the oracle's step lacks, %d oracle rows a key the "
                     "device's step lacks" % (label, len(lost), len(extra)))
        if extra:     # say where: pair each (of the first few) with the unmatched oracle row it differs from least
            w = want[extra].view(np.uint32).reshape(len(extra), -1)
            for i in lost[:limit]:
                pairs.append((i, extra[int(np.argmin((w != got[i].view(np.uint32).reshape(-1)).sum(axis=1)))]))
    if pairs:
        a = np.array([p[0] for p in pairs]); b = np.array([p[1] for p in pairs])
        g, w = got[a].view(np.uint32), want[b].view(np.uint32)
        diff = np.flatnonzero((g != w).reshape(len(pairs), -1).any(axis=1))
        for r in diff[:limit]:
            y, x, c = (int(v) for v in np.argwhere(g[r] != w[r])[0])
            fails.append("%s, row %d: first difference at pixel (%d, %d) channel %d: got %r (0x%08x), want %r (0x%08x)" % (
                label, int(a[r]), y, x, c, float(got[a[r]][y, x, c]), int(g[r][y, x, c]), float(want[b[r]][y, x, c]),
                int(w[r][y, x, c])))
        if len(diff) > limit:
            fails.append("%s: %d rows differ in all" % (label, len(diff)))
    return fails


# ---- the device side: one root turn through the C ABI, the per-step loop of Engine.search -----------------------------------

class _Step:
    def __init__(self, epoch, step, planes, values, raw):
        self.epoch, self.step, self.planes, self.values, self.raw = epoch, step, planes, values, raw
        self.n = len(planes)
        self.keys = _keys(planes)


def _device_turn(eng, info, nat, tree):
    """asz_search_begin / epoch_begin / step_probe -> values -> step_sample (recording the trace) / finish.  Before every probe
    the whole evaluation buffer (with its slack) is filled with SENTINEL; after it, rows [0, n) hold no SENTINEL word and
    everything past them is untouched.  Returns the steps with host copies of their rows and values."""
    import torch
    from alphasnake_zero_b200._lib import check
    L, h, st = eng.L, eng.h, eng.stream
    R, N, stride = info["max_rows"], eng.N, eval_row_floats(eng)
    flat = eng._wrap(L.asz_search_eval_planes(h), (R * stride + 4,), torch.float32)     # + the 16 bytes of slack
    words = flat.view(torch.int32)
    values = eng._wrap(L.asz_search_eval_values(h), (R, 3), torch.float32)
    n = C.c_int32(0)
    steps = []
    check(L.asz_search_begin(h, st))
    for ep in range(info["epochs"]):
        check(L.asz_search_epoch_begin(h, st))
        for step in range(1, info["max_steps"] + 2):
            words.fill_(SENTINEL)
            check(L.asz_search_step_probe(h, C.byref(n), st))
            k = n.value
            assert 0 <= k <= R
            assert not bool((words[:k * stride] == SENTINEL).any()), "epoch %d step %d: a word of rows [0, %d) was not written" % (ep, step, k)
            assert bool((words[k * stride:] == SENTINEL).all()), "epoch %d step %d: a word past row %d was written" % (ep, step, k)
            if step > info["max_steps"]:
                assert k == 0, "the closing probe of epoch %d wrote %d planes that are never evaluated" % (ep, k)
                continue
            planes = torch.as_strided(flat, (k, N, N, 3), (stride, 3 * N, 3, 1))
            raw = None
            if nat is None:
                check(L.asz_search_stub_values(h, st))
            elif k > 0:      # search_run's network path: asz_net_forward, then asz_obstacle_mask
                nat.forward(planes, out=values[:k])
                raw = values[:k].cpu().numpy()
                check(L.asz_obstacle_mask(h, C.c_void_p(flat.data_ptr()), k, C.c_void_p(values.data_ptr()), st))
            check(L.asz_search_step_sample(h, None, C.c_void_p(tree.data_ptr()), 2, st))
            steps.append(_Step(ep, step, planes.cpu().numpy(), values[:k].cpu().numpy(), raw))
    check(L.asz_search_finish(h, None, None, None, st))
    torch.cuda.synchronize()
    return steps


class _OracleValues:
    """value_fn of the oracle agent.  The oracle calls it once per step with misses, so call k gets the oracle's miss planes
    of the k-th device step with misses; they are compared with that step's device rows.  Stub: the oracle's own stub value
    (what value_fn=None gives), and the device's value of each key must equal it.  Network: the device's value of that key.
    Failures are collected here (the callback runs inside ctypes) and asserted by the caller."""

    def __init__(self, steps, side, turn, native):
        self.steps = [s for s in steps if s.n > 0]
        self.side, self.turn, self.native = side, turn, native
        self.calls, self.fails = 0, []

    def __call__(self, pl):
        try:
            return self._values(np.array(pl, np.float32))
        except Exception as ex:        # an exception would not cross the ctypes boundary
            self.fails.append("turn %d, oracle step %d: %r" % (self.turn, self.calls, ex))
            return np.zeros((len(pl), 3), np.float32)

    def _values(self, want):
        from oracle import oracle as orc
        k = self.calls
        self.calls += 1
        keys = _keys(want)
        stub = np.array([orc.obstacle_mask(p, self.side, self.side, orc.stub_value(key)) for p, key in zip(want, keys)], np.float32)
        if k >= len(self.steps):
            self.fails.append("turn %d: the oracle has a step with misses beyond the device's %d" % (self.turn, len(self.steps)))
            return stub
        s = self.steps[k]
        label = "turn %d step %d (epoch %d, depth step %d)" % (self.turn, k, s.epoch, s.step)
        self.fails += compare_step(label, s.planes, want, s.keys, keys)
        dev = {key: s.values[i] for i, key in enumerate(s.keys)}
        if not self.native:
            bad = [j for j, key in enumerate(keys) if key in dev and not np.array_equal(dev[key].view(np.uint32), stub[j].view(np.uint32))]
            if bad:
                self.fails.append("%s: %d stub values differ, first %s (device) vs %s (oracle)" % (label, len(bad), dev[keys[bad[0]]], stub[bad[0]]))
            return stub
        return np.array([dev.get(key, np.zeros(3, np.float32)) for key in keys], np.float32)


# ---- one case: seeded or fixture start, a few root turns, everything compared ---------------------------------------------------

def edge_layout(side, S):
    """(start cells, last moves, food) of a start with snake k's head on board edge k % 4, facing away from that edge.  A head
    that got where it is by moving always has a board cell behind it, so this is how the board window reaches the plane edge
    behind the viewer (the plane's first rows and its first floats)."""
    c = side // 2
    start, last = [], []
    for k in range(S):
        p = c - 3 * (k // 4)
        start.append([(side - 1, p), (0, p), (p, 0), (p, side - 1)][k % 4])
        last.append([0, 2, 1, 3][k % 4])
    return np.array(start, np.int32), np.array(last, np.int32), np.array([(1, 1), (side - 2, side - 2)], np.int32)


def _run_case(side, S, G, D, breadth, base=2.0, training=True, turns=2, warm=0, fixture=None, net=False, records=False,
              edge_game=False, table_log2=18, seed=77):
    import torch
    from oracle import oracle as orc
    from tests.test_gpu_env import _engine
    dec = 1
    if fixture is not None:
        z = load("mcts_%s.npz" % fixture)
        side, S, G, dec = int(z["H"]), int(z["S"]), int(z["G"]), int(z["health_dec"])
        D, breadth, base, training = int(z["D"]), int(z["breadth"]), float(z["base"]), bool(z["training"])
    n_fixed = G if fixture is not None else 0
    if edge_game:
        G += 1
    eng = _engine(side=side, snakes=S, health_dec=dec, games=G, seed=seed, max_depth=D, max_breadth=breadth, softmax_base=base,
                  training=training, table_log2=table_log2)
    eng.reset()
    info = eng.search_info()
    stride = eval_row_floats(eng)
    games = []
    for gi in range(G):
        g = orc.OracleGame(side, side, S, dec)
        if gi < n_fixed:
            d = {k: z["t0_before_%s" % k][gi] for k in ("snake", "owner", "dist", "food", "counters")}
            eng.set_state(gi, d)
            g.load_dump(d)
        else:
            g.init_native(seed, gi, 0)
        g.set_ids(gi, 0)
        games.append(g)
    if warm:
        for _ in range(warm):
            eng.step(spawn_mode=2, tic=True, encode=False, auto_reset=True, random_actions=True)
        orc.env_run(G, side, side, S, 1, 0.15, seed, warm, encode=False, n_threads=os.cpu_count() or 1, games=games)
        for gi in range(0, G, 7):
            assert_dump_equal(eng.get_state(gi), games[gi].dump(), "game %d after the warm-up" % gi)
    if edge_game:      # one more game, started over from edge_layout on both sides
        from tests.test_gpu_env import init_dump
        start, last, food = edge_layout(side, S)
        eng.set_state(G - 1, init_dump(side, S, start, last, food))
        games[-1].init_explicit(start, last, food)
        games[-1].set_ids(G - 1, 0)
    nat = None
    if net:
        from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
        an = AlphaNNet(input_shape=(2 * side - 1, 2 * side - 1, 3), seed=4, backend="native")
        an.weights["dense2_w"] = (an.weights["dense2_w"] * 5).astype(np.float32)   # spread the values, |v| well below 1
        nat = an._get_native()
    if records:
        eng.records_enable(64)          # 64 rows: the store has to grow several times
    replay = _OracleValues([], side, 0, net)
    agent = orc.OracleAgent(base=base, training=training, max_depth=D, max_breadth=breadth, value_fn=replay)
    q_atol = 2e-5 if net else 5e-6
    spawn = 0 if fixture is not None else 2      # fixture starts: no food spawn between root turns on either side
    done = [False] * G
    stats = dict(rows=0, steps=0, phases=set(), epochs=set(), max_step=0, edges=set(), heads=False, food=False,
                 food_above_1=False, first_n=[], records=0)
    rec_ids, rec_turns = [], []
    for t in range(turns):
        live = [g for gi, g in enumerate(games) if not done[gi]]
        if not live:
            break
        evals0 = eng.search_stats()["evals"]
        tree = torch.full((info["epochs"], info["max_steps"], G * info["P"], S), 255, dtype=torch.uint8, device="cuda")
        steps = _device_turn(eng, info, nat, tree)
        stats["first_n"].append(steps[0].n)
        if records:
            eng.records_append()          # Agent.make_moves's order: after the search, before the root tic
        q, mv = _root_q_moves(eng)
        # the stored bytes carry the key the table was probed with: one evaluation per new key, each key in the table
        keys = [k for s in steps for k in s.keys]
        assert len(set(keys)) == len(keys), "turn %d: an evaluation-batch key repeats within the root turn" % t
        assert len(keys) == eng.search_stats()["evals"] - evals0
        tab = eng.table()
        in_table = {(int(a), int(b)) for a, b in tab["keys"]}
        missing = [k for k in keys if k not in in_table]
        assert not missing, "turn %d: %d evaluation rows carry a key that is not in the table" % (t, len(missing))
        for s in steps:
            if s.raw is not None:    # asz_obstacle_mask on these planes: AlphaNNet.v's mask of the raw outputs
                want = np.array([orc.obstacle_mask(p, side, side, r) for p, r in zip(s.planes, s.raw)], np.float32)
                assert np.array_equal(s.values.view(np.uint32), want.view(np.uint32)), "turn %d: obstacle mask" % t
            if s.n:
                f = plane_features(s.planes)
                stats["rows"] += s.n; stats["steps"] += 1
                stats["phases"] |= set(((np.arange(s.n, dtype=np.int64) * stride) & 3).tolist())
                stats["epochs"].add(s.epoch); stats["max_step"] = max(stats["max_step"], s.step)
                stats["edges"] |= f["edges"]
                for k in ("heads", "food", "food_above_1"):
                    stats[k] = stats[k] or f[k]
        # the oracle replays the recorded trace; its value function compares the planes of every step
        replay.__init__(steps, side, t, net)
        ids = [(gi, s) for gi in range(G) if not done[gi] for s in games[gi].live_ids()]
        root_moves = np.array([mv[gi, s] for gi, s in ids], np.uint8)
        assert np.all(root_moves < 3)
        omv, oq = agent.make_moves(live, G, root_turn=t, tree_moves=np.ascontiguousarray(tree.cpu().numpy()),
                                   root_moves=root_moves.copy(), replay=True)
        assert not replay.fails, "\n".join(replay.fails[:12])
        assert replay.calls == len(replay.steps), "turn %d: %d device steps with misses, the oracle evaluated %d" % (
            t, len(replay.steps), replay.calls)
        np.testing.assert_allclose(np.array([q[gi, s] for gi, s in ids]), oq, rtol=0, atol=q_atol)
        if training:
            assert np.array_equal(omv, root_moves)
        otab = agent.table()
        oo = np.lexsort((otab["keys"][:, 1], otab["keys"][:, 0]))
        assert np.array_equal(tab["keys"], otab["keys"][oo]), "key sets differ at turn %d" % t
        assert np.array_equal(tab["N"], otab["N"][oo]) and np.array_equal(tab["age"], otab["age"][oo])
        np.testing.assert_allclose(tab["W"], otab["W"][oo], rtol=0, atol=2e-4 if net else 1e-4)
        st = eng.search_stats()
        assert st["evals"] == agent.stat("evals") and st["node_visits"] == agent.stat("node_visits")
        assert st["collisions"] == 0 and st["overflow"] == 0 and agent.stat("alias_errors") == 0
        if records:
            rec_ids += [gi * 8 + s for gi, s in ids]
            rec_turns += [t] * len(ids)
            _check_records_turn(eng, agent, side, t, rec_ids, rec_turns, q_atol)
        # root tic on both sides with the device's root moves
        actions = np.ones((G, 8), np.uint8)
        for (gi, s), m in zip(ids, root_moves):
            actions[gi, s] = m
        eng.step(actions=torch.from_numpy(actions).cuda(), spawn_mode=spawn, tic=True, encode=False)
        r0 = 0
        for gi in range(G):
            if done[gi]:
                continue
            n = games[gi].n_live
            if games[gi].tic(root_moves[r0:r0 + n].astype(np.int32), spawn_mode=spawn, chance=0.15, seed=seed):
                done[gi] = True
            r0 += n
        for gi in list(range(0, G, 5)) + [G - 1]:
            assert_dump_equal(eng.get_state(gi), games[gi].dump(), "root game %d after turn %d" % (gi, t))
    if records:
        stats["records"] = _check_gather(eng, agent, side, rec_ids, rec_turns)
    stats["max_rows"] = info["max_rows"]
    eng.close()
    return stats


def _root_q_moves(eng):
    import torch
    q = eng._wrap(eng.L.asz_search_root_q(eng.h), (eng.G, 8, 3), torch.float32).cpu().numpy()
    mv = eng._wrap(eng.L.asz_search_root_moves(eng.h), (eng.G, 8), torch.uint8).cpu().numpy()
    return q, mv


# ---- training records --------------------------------------------------------------------------------------------------------

def _store(eng):
    """(planes, values, ids, turns) of the record store on the host, planes read at the engine's row pitch"""
    pl, va, ids, tu = eng.records_views()
    return pl.cpu().numpy(), va.cpu().numpy(), ids.cpu().numpy(), tu.cpu().numpy()


def _check_records_turn(eng, agent, side, t, rec_ids, rec_turns, q_atol):
    """the store's rows of root turn t, in ids order, against the records the oracle agent appended in that turn"""
    pl, va, ids, tu = _store(eng)
    assert len(pl) == len(rec_ids) == eng.records_count()
    sel = np.flatnonzero(tu == t)
    sel = sel[np.argsort(ids[sel], kind="stable")]
    want_ids = np.array([i for i, u in zip(rec_ids, rec_turns) if u == t])
    assert np.array_equal(ids[sel], want_ids), "turn %d: record ids" % t
    oplanes, oq = agent.records(side, side)
    assert len(oplanes) == len(rec_ids)
    op, oqt = oplanes[-len(sel):], oq[-len(sel):]
    fails = compare_step("records of turn %d" % t, pl[sel], op, [(i,) for i in range(len(sel))], [(i,) for i in range(len(sel))])
    assert not fails, "\n".join(fails)
    np.testing.assert_allclose(va[sel], oqt, rtol=0, atol=q_atol)


def _gather(eng, idx, mirror):
    """asz_records_gather into outputs filled with zeros first, so that a row the kernel does not write reads 0, not NaN"""
    import torch
    from alphasnake_zero_b200._lib import check
    d_idx = torch.as_tensor(np.asarray(idx, np.int64)).cuda()
    n = len(idx)
    m = 2 * n if mirror else n
    X = torch.zeros(m, eng.N, eng.N, 3, dtype=torch.float32, device="cuda")
    V = torch.zeros(m, 3, dtype=torch.float32, device="cuda")
    check(eng.L.asz_records_gather(eng.h, C.c_void_p(d_idx.data_ptr()), n, int(mirror), C.c_void_p(X.data_ptr()),
                                   C.c_void_p(V.data_ptr()), eng.stream))
    return X.cpu().numpy(), V.cpu().numpy()


def _check_gather(eng, agent, side, rec_ids, rec_turns):
    """the trainer's sampled batch with mirrored copies (alpha_snake_zero_trainer.py:70-77, 93-100) against numpy.flip of the
    oracle's records; indices -1 and count give all-NaN planes and values, mirrored copies included"""
    pl, va, ids, tu = _store(eng)
    count = eng.records_count()
    order = np.lexsort((ids, tu))                     # store rows in the oracle's order: per turn, ids order
    assert np.array_equal(ids[order], rec_ids) and np.array_equal(tu[order], rec_turns)
    oplanes, oq = agent.records(side, side)
    orc_of = np.empty(count, np.int64); orc_of[order] = np.arange(count)
    rng = np.random.default_rng(side)
    good = rng.choice(count, size=min(count, 300), replace=False)
    idx = np.concatenate([good, [-1, count]])
    n, m = len(idx), len(good)
    X, V = _gather(eng, idx, True)
    want = oplanes[orc_of[good]]
    u = lambda a: np.ascontiguousarray(a).view(np.uint32)
    assert np.array_equal(u(X[:m]), u(want))
    assert np.array_equal(u(X[n:n + m]), u(np.flip(want, axis=2)))               # mirror_states: the width axis
    c = eng.N // 2                                                               # N is odd: the centre column stays put
    assert np.array_equal(u(X[n:n + m, :, c]), u(X[:m, :, c])) and not np.array_equal(u(X[n:n + m]), u(X[:m]))
    assert np.array_equal(u(V[:m]), u(va[good])) and np.array_equal(u(V[n:n + m]), u(np.flip(va[good], axis=1)))
    np.testing.assert_allclose(V[:m], oq[orc_of[good]], rtol=0, atol=2e-5)
    for lo in (m, n + m):                                                        # -1 and count, and their mirrored copies
        assert np.isnan(X[lo:lo + 2]).all(), "an out-of-range index must give an all-NaN plane"
        assert np.isnan(V[lo:lo + 2]).all(), "an out-of-range index must give all-NaN values"
    X1, V1 = _gather(eng, idx, False)
    assert np.array_equal(u(X1[:m]), u(want)) and np.isnan(X1[m:]).all() and np.isnan(V1[m:]).all()
    return count


# ---- the cases ------------------------------------------------------------------------------------------------------------------

def _report(name, s):
    print("%s: %d evaluation rows in %d steps, phases %s, epochs %s, steps up to %d, edges %s, heads %s, food %s, food > 1 %s, "
          "step-1 rows %s of %d, %d records" % (name, s["rows"], s["steps"], sorted(s["phases"]), sorted(s["epochs"]),
                                                s["max_step"], sorted(s["edges"]), s["heads"], s["food"], s["food_above_1"],
                                                s["first_n"], s["max_rows"], s["records"]))


def _assert_exercised(name, s, food_above_1=False):
    """the comparison was not vacuous: rows of every 16-byte phase, board windows on all four plane edges, other snakes' heads and
    food, rows of two epochs and of depth steps >= 3"""
    assert s["phases"] == {0, 1, 2, 3}, (name, s["phases"])
    assert s["edges"] == {"top", "bottom", "left", "right"}, (name, s["edges"])
    assert s["heads"] and s["food"], name
    assert len(s["epochs"]) >= 2 and s["max_step"] >= 3, (name, s["epochs"], s["max_step"])
    if food_above_1:
        assert s["food_above_1"], "%s: no row with food above 1.0 (viewer health <= 0)" % name


SEEDED = {   # side, S, G, D, breadth, base, training, warm-up tics, turns, records
    "7x7x4": (7, 4, 32, 4, 16, 100.0, False, 6, 3, False),
    "11x11x2": (11, 2, 40, 6, 16, 10.0, True, 0, 3, False),
    "11x11x4": (11, 4, 64, 8, 32, 2.0, True, 10, 2, True),
    "19x19x8": (19, 8, 8, 8, 16, 3.0, True, 20, 3, True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SEEDED))
def test_eval_planes_and_records_from_seeded_starts(name):
    side, S, G, D, B, base, training, warm, turns, records = SEEDED[name]
    s = _run_case(side, S, G, D, B, base=base, training=training, turns=turns, warm=warm, records=records, edge_game=True)
    _report(name, s)
    _assert_exercised(name, s)
    if records:
        assert s["records"] > 64


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["11x11x4_neghealth_dec9", "11x11x4_neghealth_dec3", "19x19x8_mid"])
def test_eval_planes_from_fixture_starts(fixture):
    """hand-built / mid-game starts: sub-games with a head-on winner alive at health <= 0 (its food reads above 1.0), and 19x19x8
    with 3-4 live snakes; root tics between turns without food spawn"""
    s = _run_case(0, 0, 0, 0, 0, turns=2, fixture=fixture, edge_game=True)
    _report(fixture, s)
    _assert_exercised(fixture, s, food_above_1="neghealth" in fixture)


@pytest.mark.gpu
@pytest.mark.parametrize("side,S,G", [(7, 4, 24), (11, 4, 16)])
def test_eval_planes_and_records_with_the_native_network(side, S, G):
    """the value network reads the rows it is handed: search_run's asz_net_forward + asz_obstacle_mask, and the oracle is given
    the device's value of each key"""
    name = "%dx%dx%d native" % (side, side, S)
    s = _run_case(side, S, G, 8, 16, turns=3, warm=6, net=True, records=(side == 7), edge_game=True)
    _report(name, s)
    _assert_exercised(name, s)


@pytest.mark.gpu
@pytest.mark.parametrize("side,S", [(7, 4), (11, 4), (19, 8)])
def test_eval_planes_fill_the_whole_buffer(side, S):
    """breadth 1 on a fresh table: step 1 evaluates every snake of every game, so the batch is full and its last row ends at the
    end of the allocation"""
    s = _run_case(side, S, 64, 2, 1, turns=1, seed=80)     # seed 80: no two of the 64 x S root planes are equal at any size
    _report("%dx%dx%d full" % (side, side, S), s)
    assert s["first_n"] == [s["max_rows"]] == [64 * S]
    assert s["phases"] == {0, 1, 2, 3}


# ---- the checker itself, without a GPU -------------------------------------------------------------------------------------

def test_plane_checker_on_cpu():
    """compare_step on the oracle's miss planes (captured through its value function) against themselves, permuted within each
    step: no failure; a changed wall float, a changed board pixel, a last float left at the sentinel and a row moved to the
    next step are each reported"""
    from oracle import oracle as orc
    side, S, G, seed = 7, 4, 8, 3
    games = []
    for gi in range(G):
        g = orc.OracleGame(side, side, S, 1); g.init_native(seed, gi, 0); g.set_ids(gi, 0); games.append(g)
    orc.env_run(G, side, side, S, 1, 0.15, seed, 4, encode=False, games=games)
    captured = []

    def capture(pl):
        p = np.array(pl, np.float32)
        captured.append(p)
        return np.array([orc.obstacle_mask(x, side, side, orc.stub_value(orc.plane_key(x))) for x in p], np.float32)
    agent = orc.OracleAgent(base=2.0, training=True, max_depth=6, max_breadth=16, value_fn=capture)
    agent.make_moves([g for g in games if g.n_live > 0], G, root_turn=0, seed=seed)
    assert len(captured) >= 3 and sum(len(p) for p in captured) > 100
    rng = np.random.default_rng(0)
    perm = [p[rng.permutation(len(p))] for p in captured]
    for k, (got, want) in enumerate(zip(perm, captured)):
        assert compare_step("step %d" % k, got, want) == []
    k = max(range(len(captured)), key=lambda i: len(captured[i]))     # a step with several rows
    want = captured[k]
    r = len(want) // 2

    def mutated(f):
        got = want.copy()
        f(got)
        return compare_step("step %d" % k, got, want)

    # 1. one wall float: the first background pixel of row r gets 1.0 in channel 0
    wall = np.argwhere((want[r, ..., 0] == 0) & (want[r, ..., 1] == 1) & (want[r, ..., 2] == 0))[0]
    f = mutated(lambda g: g[r, wall[0], wall[1]].__setitem__(0, 1.0))
    assert any("pixel (%d, %d) channel 0" % tuple(wall) in x for x in f), f
    # 2. one board pixel (the first non-wall pixel of row r): a new key, and the difference is still found
    y, x = np.argwhere(~((want[r, ..., 0] == 0) & (want[r, ..., 1] == 1) & (want[r, ..., 2] == 0)))[0]
    f = mutated(lambda g: g[r, y, x].__setitem__(1, g[r, y, x, 1] + np.float32(0.02)))
    assert any("key sets differ" in m for m in f) and any("pixel (%d, %d) channel 1" % (y, x) in m for m in f), f
    # 3. the last float of a row left at the sentinel
    f = mutated(lambda g: g[r].reshape(-1).view(np.uint32).__setitem__(-1, SENTINEL))
    n = want.shape[1] - 1
    assert any("pixel (%d, %d) channel 2" % (n, n) in x and "0x%08x" % SENTINEL in x for x in f), f
    # 4. a row moved to the next step
    nxt = captured[k + 1] if k + 1 < len(captured) else captured[k - 1]
    f1 = compare_step("step a", np.delete(want, r, axis=0), want)
    f2 = compare_step("step b", np.concatenate([nxt, want[r:r + 1]]), nxt)
    assert any("device rows" in x for x in f1) and any("key sets differ" in x for x in f1)
    assert any("device rows" in x for x in f2) and any("key sets differ" in x for x in f2)
    # the features the GPU cases require are there in the oracle's own rows
    feats = plane_features(np.concatenate(captured))
    assert feats["heads"] and feats["food"]
