"""Every plane the fused tic + encode (`env_step_kernel` -> `warp_encode_game_v3b`) writes, bit for bit against the CPU oracle's
make_state, at the game counts the benchmark runs: the network's input batch, the engine's internal buffer of the host-buffer
path, a caller's short buffer and the record store (`row_base > 0`).  Per compared launch every row is paired with the oracle's
row of the same (game, snake) id, every pad word must have been written and nothing past the last row may be; the row ids must
keep a game's rows together in ascending snake id.  Engine and oracle games are stepped in lockstep: in-kernel random actions
(the oracle restates the same Philox streams) or actions supplied by the caller on both sides."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.helpers import SENTINEL, plane_features, plane_keys

ROW_FREE = -1            # row_ids are filled with this before a compared launch: an id nobody wrote
KIND = ("a single ticket", "game A of a pair ticket", "game B of a pair ticket")


# ---- the launch's scheduling tickets (restated from EnvLaunch<SIDE>::launch, asz_env.cu) -----------------------------------------

def launch_layout(side, G, n_sm):
    """(pair tickets, games handed out one by one at most): EnvLaunch's grid of min(ceil(G / WARPS), n_sm * MINB) CTAs of WARPS
    warps; the last kTailRounds = 3 games of every warp are single tickets, every game before them is in a ticket of two"""
    warps, minb = (4, 2) if side >= 19 else (8, 3)
    blocks = min((G + warps - 1) // warps, n_sm * minb)
    tail = 3 * blocks * warps
    return max(0, G - tail) // 2, tail


def ticket_kinds(G, pairs):
    """per game: 0 single ticket, 1 game A (2t) of pair ticket t, 2 game B (2t + 1)"""
    k = np.zeros(G, np.int8)
    k[0:2 * pairs:2] = 1
    k[1:2 * pairs:2] = 2
    return k


# ---- the comparator (plain NumPy: test_plane_comparator_reports_planted_faults runs it without a GPU) ---------------------------

def new_coverage():
    return dict(rows=0, launches=0, kinds=set(), rots=set(), w0=set(), edges=set(), heads=False, food=False,
                food_above_1=False, reset_rows=0, rows_per_game=set())


def _cover(cov, wid, wpl, kinds, viewer, reset, g0):
    f = plane_features(wpl)
    cov["rows"] += len(wid)
    cov["edges"] |= f["edges"]
    for k in ("heads", "food", "food_above_1"):
        cov[k] = cov[k] or f[k]
    games = wid // 8
    cov["kinds"] |= set(np.unique(kinds[games]).tolist())
    cov["rows_per_game"] |= set(np.unique(np.bincount(games - g0)).tolist()) - {0}
    if reset is not None:
        cov["reset_rows"] += int(reset[games].sum())
    if viewer is not None:     # packed snake records (asz_game.cuh pack_snake): head cell, last move = the plane's rotation
        N = wpl.shape[1]
        side, U = (N + 1) // 2, (N - 1) // 2
        v = viewer[games, wid % 8]
        head, rot = (v & 0xFFFF).astype(np.int64), ((v >> 40) & 3).astype(np.int64)
        hy, hx = head // side, head % side
        i0 = np.select([rot == 0, rot == 1, rot == 2], [U - hy, hx, hy], U - hx)     # first plane row of the board window
        cov["rots"] |= set(np.unique(rot).tolist())
        cov["w0"] |= set(np.unique((i0 * 3 * N) & 7).tolist())


def compare_step(label, n, row_ids, rows, tail, want, G, pitch, plane, kinds=None, grown=None, cap=None, filled=True, keys=None,
                 cov=None, viewer=None, reset=None, limit=4):
    """One compared launch.  n: the row count it reported; row_ids: its ids in kernel order; rows: uint32 [>= min(n, cap), pitch],
    the rows as written, pad words included; tail: the uint32 words from row min(n, cap) to the end of the allocation (its slack
    included); want(g0, g1) -> the oracle's (ids, planes) of games [g0, g1) in (game, snake id) order.  kinds: ticket kind per
    game (ticket_kinds); grown: how much totals()["planes"] grew; cap: rows the buffer holds (None: all n fit); filled: the
    buffer was filled with SENTINEL before the launch (else pad words and the tail are not checked); keys: uint64 [n, 2] plane
    keys in kernel order.  Returns a list of failure messages, empty when the launch wrote what the oracle says."""
    fails = []
    kinds = np.zeros(G, np.int8) if kinds is None else kinds
    m = n if cap is None else min(n, cap)
    ids = np.asarray(row_ids[:m]).astype(np.int64)

    def where(r):
        i = int(ids[r])
        g = i // 8
        return "row %d (game %d snake %d, %s)" % (r, g, i % 8, KIND[kinds[g]] if 0 <= g < G else "no such game")
    order = np.argsort(ids, kind="stable")
    sids = ids[order]
    dup = np.flatnonzero(sids[1:] == sids[:-1])
    if len(dup):
        r = order[dup[0] + 1]
        fails.append("%s: %d row ids repeat; first: %s, also at row %d" % (label, len(dup), where(r), order[dup[0]]))
    gm = ids // 8
    if m > 1:
        runs = gm[np.flatnonzero(np.r_[True, gm[1:] != gm[:-1]])]
        rs = np.sort(runs)
        split = rs[1:][rs[1:] == rs[:-1]]
        if len(split):
            at = np.flatnonzero(gm == split[0])
            fails.append("%s: the rows of %d games are not contiguous; first: game %d (%s) at rows %s" % (
                label, len(np.unique(split)), split[0], KIND[kinds[split[0]]] if 0 <= split[0] < G else "no such game", at[:8].tolist()))
        bad = np.flatnonzero((gm[1:] == gm[:-1]) & (ids[1:] <= ids[:-1]))
        if len(bad):
            fails.append("%s: %d rows break ascending snake id within their game; first: %s after snake %d" % (
                label, len(bad), where(bad[0] + 1), ids[bad[0]] % 8))
    if filled and pitch > plane and m:
        pad = np.flatnonzero((rows[:m, plane:] == SENTINEL).any(axis=1))
        if len(pad):
            w = plane + int(np.flatnonzero(rows[pad[0], plane:] == SENTINEL)[0])
            fails.append("%s: %d rows leave a pad word unwritten; first: %s, word %d of %d" % (label, len(pad), where(pad[0]), w, pitch))
    if filled:
        tb = np.flatnonzero(np.asarray(tail) != SENTINEL)
        if len(tb):
            w = m * pitch + int(tb[0])
            fails.append("%s: %d words past row %d were written; first: word %d (row %d, word %d of the row)" % (
                label, len(tb), m, w, w // pitch, w % pitch))
    n_want, n_missing, n_diff, missing = 0, 0, 0, []
    matched = np.zeros(len(sids), bool)
    chunk = max(64, (1 << 25) // (8 * plane))           # games per oracle chunk: ~128 MB of oracle planes
    for g0 in range(0, G, chunk):
        wid, wpl = want(g0, min(G, g0 + chunk))
        wid = np.asarray(wid).astype(np.int64)
        n_want += len(wid)
        if not len(wid):
            continue
        j = np.searchsorted(sids, wid)
        jc = np.minimum(j, max(len(sids) - 1, 0))
        ok = (j < len(sids)) & (sids[jc] == wid) if len(sids) else np.zeros(len(wid), bool)
        if cap is None or n <= cap:
            n_missing += int((~ok).sum())
            missing += wid[~ok][:limit].tolist()
        matched[jc[ok]] = True
        r = order[jc[ok]]
        wk = wpl[ok]
        w = wk.reshape(len(r), plane).view(np.uint32)
        g = rows[r, :plane]
        d = np.flatnonzero((g != w).any(axis=1))
        for q in d[:max(0, limit - n_diff)]:
            c = int(np.flatnonzero(g[q] != w[q])[0])
            N = wpl.shape[2]
            (y, x), ch = divmod(c // 3, N), c % 3
            fails.append("%s, %s: first difference at pixel (%d, %d) channel %d: got %r (0x%08x), want %r (0x%08x)" % (
                label, where(r[q]), y, x, ch, float(g[q:q + 1, c].view(np.float32)[0]), int(g[q, c]),
                float(wk[q].reshape(-1)[c]), int(w[q, c])))
        n_diff += len(d)
        if keys is not None:
            kw = plane_keys(wk)
            kd = np.flatnonzero((np.asarray(keys)[r] != kw).any(axis=1))
            if len(kd):
                fails.append("%s: %d plane keys differ; first: %s, got %s want %s" % (label, len(kd), where(r[kd[0]]),
                                                                                      np.asarray(keys)[r[kd[0]]], kw[kd[0]]))
        if cov is not None:
            _cover(cov, wid[ok], wk, kinds, viewer, reset, g0)
    if n_diff > limit:
        fails.append("%s: %d rows differ in all" % (label, n_diff))
    if n_missing:
        fails.append("%s: %d oracle rows have no row; first ids %s" % (label, n_missing, missing))
    extra = order[~matched]
    if len(extra):
        fails.append("%s: %d rows carry an id the oracle has no row for; first: %s" % (label, len(extra), where(extra[0])))
    if n != n_want:
        fails.insert(0, "%s: row_count is %d, the oracle has %d rows" % (label, n, n_want))
    if grown is not None and grown != n:
        fails.insert(0, "%s: totals()['planes'] grew by %d, row_count is %d" % (label, grown, n))
    if cov is not None:
        cov["launches"] += 1
    return fails


def oracle_rows(games, n_threads):
    """want(g0, g1) of compare_step: the oracle's batch encoder over a slice of games (None = a finished game, no rows)"""
    from oracle import oracle as orc

    def want(g0, g1):
        ids, planes = orc.env_encode(games[g0:g1], n_threads)
        return ids.astype(np.int64) + 8 * g0, planes
    return want


# ---- the device side -------------------------------------------------------------------------------------------------------------

def _engine(**kw):
    from alphasnake_zero_b200.engine import Engine
    return Engine(**kw)


class Case:
    """One engine and its oracle games in lockstep, with the coverage of every compared launch."""

    def __init__(self, name, side, S, dec, G, seed):
        import torch
        from oracle import oracle as orc
        self.name, self.side, self.S, self.dec, self.G, self.seed = name, side, S, dec, G, seed
        self.eng = _engine(side=side, snakes=S, health_dec=dec, food_chance=0.15, games=G, seed=seed)
        self.eng.reset()
        self.games = []
        for gi in range(G):
            g = orc.OracleGame(side, side, S, dec)
            g.init_native(seed, gi, 0)
            self.games.append(g)
        self.handles = orc.env_handles(self.games)
        self.done = np.zeros(G, bool)        # finished without a restart: the game emits no rows on either side
        self.threads = os.cpu_count() or 1
        n_sm = torch.cuda.get_device_properties(self.eng.device).multi_processor_count
        self.pairs, self.tail = launch_layout(side, G, n_sm)
        self.kinds = ticket_kinds(G, self.pairs)
        self.cov = new_coverage()
        self.rng = np.random.default_rng(seed)
        _ = self.eng.planes

    def close(self):
        self.eng.close()

    # -- stepping both sides
    def oracle_random(self, tics):
        from oracle import oracle as orc
        orc.env_run(self.G, self.side, self.side, self.S, self.dec, 0.15, self.seed, tics, encode=False, n_threads=self.threads,
                    games=self.handles)

    def warm(self, tics):
        for _ in range(tics):
            self.eng.step(spawn_mode=2, tic=True, encode=False, auto_reset=True, random_actions=True)
        self.oracle_random(tics)

    def actions(self):
        return self.rng.integers(0, 3, size=(self.G, 8), dtype=np.uint8)

    def oracle_actions(self, acts, auto_reset=True):
        """OracleGame.tic with the caller's actions; a game that ends restarts as episode + 1 (auto_reset) or is done.
        Returns (ended uint8 [G], rewards int8 [G, 8]) as the engine reports them."""
        ended = np.zeros(self.G, np.uint8)
        rewards = np.zeros((self.G, 8), np.int8)
        for gi, g in enumerate(self.games):
            if self.done[gi]:
                continue
            lv = g.live_ids()
            e = g.tic(acts[gi, lv].astype(np.int32), spawn_mode=2, chance=0.15, seed=self.seed)
            d = g.dump()
            rewards[gi, :self.S] = d["snake"][:, 5]
            if e:
                ended[gi] = 1
                if auto_reset:
                    g.init_native(self.seed, gi, int(d["counters"][6]) + 1)
                else:
                    self.done[gi] = True
        return ended, rewards

    # -- one compared launch
    def compare(self, label, launch, oracle_step, fill=True, keys=False, planes=None, cap=None, row_ids=None, count=None,
                reset_rows=True):
        """launch(): the engine's launch; oracle_step(): the same step on the oracle side.  planes: the flat float32 buffer the
        launch writes (default: the engine's batch, eng._planes_flat), cap: its rows when it is shorter than the batch."""
        import torch
        eng = self.eng
        flat = eng._planes_flat if planes is None else planes
        ids_buf = eng.row_ids if row_ids is None else row_ids
        if fill:
            flat.view(torch.int32).fill_(SENTINEL)
            ids_buf.fill_(ROW_FREE)
        before = eng.totals()["planes"]
        launch()
        oracle_step()
        torch.cuda.synchronize()
        n = int(eng.row_count.item()) if count is None else count()
        grown = eng.totals()["planes"] - before
        m = n if cap is None else min(n, cap)
        words = flat.view(torch.int32)
        pitch = eng.pitch
        rows = words[:m * pitch].cpu().numpy().view(np.uint32).reshape(m, pitch)
        tail = words[m * pitch:].cpu().numpy().view(np.uint32)
        ids = ids_buf[:m].cpu().numpy()
        if fill and cap is not None:
            assert bool((ids_buf[m:] == ROW_FREE).all()), "%s: a row id past row %d was written" % (label, m)
        ptrs = (C.c_void_p * 3)()
        from alphasnake_zero_b200._lib import check
        check(eng.L.asz_internal_state(eng.h, ptrs))
        viewer = eng._wrap64(ptrs[1], (self.G, 8)).cpu().numpy().view(np.uint64)
        reset = eng.ended.cpu().numpy().astype(bool) if reset_rows else None
        k = eng.keys[:n].cpu().numpy().view(np.uint64) if keys else None
        games = [None if d else g for g, d in zip(self.games, self.done)]
        fails = compare_step("%s, %s" % (self.name, label), n, ids, rows, tail, oracle_rows(games, self.threads), self.G,
                             pitch, eng.plane, kinds=self.kinds, grown=grown, cap=cap, filled=fill, keys=k, cov=self.cov,
                             viewer=viewer, reset=reset)
        assert not fails, "\n".join(fails[:12])
        return n

    def random_step(self, label, fill=True, keys=False, auto_reset=True):
        return self.compare(label, lambda: self.eng.step(spawn_mode=2, tic=True, encode=True, auto_reset=auto_reset,
                                                         random_actions=True, keys=keys),
                            lambda: self.oracle_random(1), fill=fill, keys=keys)

    def edge_step(self):
        """one encode-only launch after a few games (of both ticket kinds) restart on both sides from a layout with snake k's head
        on board edge k % 4, facing away from it: only a head that did not move there has the plane's first rows (W0 = 0, no wall
        before the window) in its board window"""
        from tests.test_gpu_env import init_dump
        c, step = self.side // 2, 2 if self.side == 7 else 3
        start = np.array([[(self.side - 1, p), (0, p), (p, 0), (p, self.side - 1)][k % 4]
                          for k, p in ((k, c - step * (k // 4)) for k in range(self.S))], np.int32)
        last = np.array([[0, 2, 1, 3][k % 4] for k in range(self.S)], np.int32)
        food = np.array([(1, 1), (self.side - 2, self.side - 2)], np.int32)
        for gi in sorted({0, 1, 2, 3, self.G // 2, self.G - 2, self.G - 1}):
            if gi < 0 or gi >= self.G:
                continue
            self.eng.set_state(gi, init_dump(self.side, self.S, start, last, food), episode=0)
            self.games[gi].init_explicit(start, last, food)
            self.games[gi].set_ids(gi, 0)
            self.done[gi] = False
        return self.compare("encode only, edge layouts", lambda: self.eng.step(tic=False, encode=True), lambda: None,
                            reset_rows=False)

    def action_step(self, label, auto_reset=True):
        import torch
        acts = self.actions()
        out = {}
        n = self.compare(label, lambda: self.eng.step(actions=torch.from_numpy(acts).cuda(), spawn_mode=2, tic=True, encode=True,
                                                      auto_reset=auto_reset),
                         lambda: out.update(r=self.oracle_actions(acts, auto_reset)))
        ended, rewards = out["r"]
        assert np.array_equal(self.eng.ended.cpu().numpy(), ended), "%s, %s: ended" % (self.name, label)
        self.check_rewards(label, self.eng.rewards.cpu().numpy(), rewards)
        return n

    def check_rewards(self, label, got, want):
        """rewards of every game against the oracle's, dumped after the tic and before a restart"""
        bad = np.flatnonzero((got != want).any(axis=1))
        assert not len(bad), "%s, %s: rewards of %d games differ; first: game %d %s vs %s" % (
            self.name, label, len(bad), bad[0], got[bad[0]], want[bad[0]])

    def report(self):
        c = self.cov
        print("%s: %d rows in %d launches, %d pair tickets, tickets %s, rotations %s, W0 & 7 %s, edges %s, heads %s, food %s, "
              "food > 1 %s, %d rows of games reset in the step, rows per game %s" % (
                  self.name, c["rows"], c["launches"], self.pairs, sorted(KIND[k] for k in c["kinds"]), sorted(c["rots"]),
                  sorted(c["w0"]), sorted(c["edges"]), c["heads"], c["food"], c["food_above_1"], c["reset_rows"],
                  sorted(c["rows_per_game"])))

    def assert_exercised(self, pairs=True, reset=True, food_above_1=False):
        """the comparison was not vacuous"""
        c, name = self.cov, self.name
        if pairs:
            assert self.pairs > 0 and c["kinds"] == {0, 1, 2}, (name, self.pairs, c["kinds"])
        assert c["rots"] == {0, 1, 2, 3}, (name, c["rots"])
        N = 2 * self.side - 1
        assert c["w0"] == {(i0 * 3 * N) & 7 for i0 in range(self.side)}, (name, c["w0"])      # all 8 at 11x11 and 19x19
        assert c["edges"] == {"top", "bottom", "left", "right"}, (name, c["edges"])
        assert c["heads"] and c["food"], name
        if reset:
            assert c["reset_rows"] > 0, "%s: no rows of a game reset in place in the step" % name
        if self.S == 8:       # a game with one snake left has ended, so a game emits 2 to 8 rows
            assert set(range(2, 9)) <= c["rows_per_game"], (name, c["rows_per_game"])
        if food_above_1:
            assert c["food_above_1"], "%s: no row with food above 1.0" % name


# ---- the cases -------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_benchmark_engine_planes():
    """bench.py's engine (11x11x4, health_dec 1, 65,536 games, random actions, native spawn, auto reset, keys off): 4 launches
    from reset, 40 uncompared tics, 4 launches on games of every age (2 over the previous launch's rows), 1 with keys; then one
    encode-only launch (edge layouts in a few games) and 2 launches without auto reset, in which finished games emit no rows"""
    c = Case("benchmark 11x11x4", 11, 4, 1, 65536, 1000)
    for t in range(4):
        c.random_step("step %d from reset" % t)
    c.warm(40)
    for t in range(4):
        c.random_step("step %d after 40 tics%s" % (t, " (no sentinel fill)" if t >= 2 else ""), fill=t < 2)
    c.random_step("step with keys", keys=True)
    c.edge_step()
    for t in range(2):
        c.action_step("caller actions without auto reset %d" % t, auto_reset=False)
    assert c.done.sum() > 0
    c.report()
    c.assert_exercised()
    c.close()


@pytest.mark.gpu
def test_caller_action_planes():
    """actions from the caller (the ACTS instantiation): eng.step, asz_env_submit_host / asz_env_wait_host (the engine's internal
    buffer) and asz_env_step_host into pinned and pageable host planes (the dense strided copy)"""
    import torch
    from alphasnake_zero_b200 import _lib
    c = Case("caller actions 11x11x4", 11, 4, 1, 65536, 2024)
    c.warm(12)
    for t in range(3):
        c.action_step("eng.step %d" % t)
    c.edge_step()
    eng, L, G = c.eng, c.eng.L, c.G
    flags = _lib.STEP_TIC | _lib.STEP_ENCODE | _lib.STEP_AUTO_RESET
    R = G * c.S
    internal = eng._wrap(L.asz_internal_planes(eng.h), (R * eng.pitch + 8,), torch.float32)
    internal_ids = eng._wrap(L.asz_internal_row_ids(eng.h), (R,), torch.int32)
    acts = torch.from_numpy(c.actions()).pin_memory()
    end_p, rew_p = torch.zeros(G, dtype=torch.uint8).pin_memory(), torch.zeros(G, 8, dtype=torch.int8).pin_memory()
    res, rows = {}, {}

    def submit():
        tk = eng.submit_host(acts, end_p, rew_p, spawn_mode=2, tic=True, encode=True, auto_reset=True)
        rows["n"] = eng.wait_host(tk)
    c.compare("submit_host + wait_host", submit, lambda: res.update(r=c.oracle_actions(acts.numpy())), planes=internal,
              row_ids=internal_ids, count=lambda: rows["n"], reset_rows=False)
    assert np.array_equal(end_p.numpy(), res["r"][0])
    c.check_rewards("submit_host", rew_p.numpy(), res["r"][1])
    # asz_env_step_host: rows dense on the host (PLANE floats apart), the host buffers filled with the sentinel first
    for pinned in (True, False):
        label = "asz_env_step_host, %s h_planes" % ("pinned" if pinned else "pageable")
        a = c.actions()
        h_acts = torch.from_numpy(a).pin_memory()
        words = np.full(R * eng.plane + 64, SENTINEL, np.uint32)
        h_ids = np.full(R, ROW_FREE, np.int32)
        if pinned:
            pl_t = torch.from_numpy(words.view(np.int32)).pin_memory()
            words = pl_t.numpy().view(np.uint32)
        n = C.c_int32(0)
        before = eng.totals()["planes"]
        _lib.check(L.asz_env_step_host(eng.h, flags, 2, C.c_void_p(h_acts.data_ptr()), None, C.c_void_p(end_p.data_ptr()),
                                       C.c_void_p(rew_p.data_ptr()), C.byref(n), words.ctypes.data_as(C.c_void_p),
                                       h_ids.ctypes.data_as(C.c_void_p), eng.stream))
        ended, rewards = c.oracle_actions(a)
        grown = eng.totals()["planes"] - before
        n = n.value
        games = [None if d else g for g, d in zip(c.games, c.done)]
        fails = compare_step("%s, %s" % (c.name, label), n, h_ids, words[:n * eng.plane].reshape(n, eng.plane),
                             words[n * eng.plane:], oracle_rows(games, c.threads), G, eng.plane, eng.plane, kinds=c.kinds,
                             grown=grown, cov=c.cov)
        assert not fails, "\n".join(fails[:12])
        assert np.array_equal(end_p.numpy(), ended), label
        c.check_rewards(label, rew_p.numpy(), rewards)
    c.report()
    c.assert_exercised()
    c.close()


@pytest.mark.gpu
def test_19x19x8_planes():
    """19x19x8 at 8,192 games (the 4-warp, 2-CTA launch): 3 launches from reset, 3 after 30 tics, 1 with keys, 1 with caller
    actions"""
    c = Case("19x19x8", 19, 8, 1, 8192, 1919)
    for t in range(3):
        c.random_step("step %d from reset" % t)
    c.warm(30)
    for t in range(3):
        c.random_step("step %d after 30 tics" % t)
    c.random_step("step with keys", keys=True)
    c.action_step("caller actions")
    c.edge_step()
    c.report()
    c.assert_exercised()
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("S,G", [(4, 65536), (8, 16384)])
def test_7x7_planes(S, G):
    """7x7 (three cells per lane: the CPL = 2 branch of load_lin): 3 launches from reset, 3 after 30 tics.  A 7x7 window starts
    on one of 7 plane rows, so W0 & 7 takes 7 of its 8 values here"""
    c = Case("7x7x%d" % S, 7, S, 1, G, 707 + S)
    for t in range(3):
        c.random_step("step %d from reset" % t)
    c.warm(30)
    for t in range(3):
        c.random_step("step %d after 30 tics" % t)
    c.edge_step()
    c.report()
    c.assert_exercised()
    c.close()


@pytest.mark.gpu
def test_ticket_boundary_planes():
    """game counts around the first pair ticket (T = 3 * blocks * WARPS single games at most: T and T + 1 have no pair, T + 2 and
    T + 3 one), and 1 and 5 games; 2 launches each"""
    import torch
    n_sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    _, T = launch_layout(11, 1 << 20, n_sm)
    for G, want_pairs in [(T, 0), (T + 1, 0), (T + 2, 1), (T + 3, 1), (1, 0), (5, 0)]:
        c = Case("11x11x2 at %d games" % G, 11, 2, 1, G, 300 + G % 97)
        assert c.pairs == want_pairs, (G, c.pairs)
        for t in range(2):
            c.random_step("step %d" % t)
        c.report()
        if G > 1000:
            assert c.cov["kinds"] == ({0, 1, 2} if want_pairs else {0})
        c.close()


@pytest.mark.gpu
def test_low_health_planes():
    """health_dec 9 with low health injected on both sides (as test_long_survival_run_against_oracle does): the next 3 launches
    carry head-on winners alive at health <= 0, whose food reads above 1.0"""
    c = Case("11x11x4 health_dec 9", 11, 4, 9, 16384, 99)
    c.warm(5)
    for gi, g in enumerate(c.games):
        d = g.dump()
        live = d["snake"][:, 0] == 1
        d["snake"][live, 1] = c.rng.integers(1, 2 * c.dec + 1, size=int(live.sum()))
        g.load_dump(d)
        c.eng.set_state(gi, d, episode=int(d["counters"][6]))
    for t in range(3):
        c.random_step("step %d after the injection" % t)
    c.edge_step()
    c.report()
    c.assert_exercised(food_above_1=True)
    c.close()


@pytest.mark.gpu
def test_short_batch_planes():
    """a caller buffer of 100,003 rows inside a larger sentinel allocation: the rows that fit equal the oracle's rows of their
    ids, nothing past row 100,003 is written, row_count is the full count"""
    import torch
    c = Case("short batch 11x11x4", 11, 4, 1, 65536, 5)
    cap, eng = 100003, c.eng
    flat = torch.empty((cap + 4000) * eng.pitch + 8, dtype=torch.float32, device=eng.device)
    view = torch.as_strided(flat, (cap, eng.N, eng.N, 3), (eng.pitch, 3 * eng.N, 3, 1))
    n = c.compare("caller buffer of %d rows" % cap, lambda: eng.step(spawn_mode=2, tic=True, encode=True, auto_reset=True,
                                                                    random_actions=True, planes=view),
                  lambda: c.oracle_random(1), planes=flat, cap=cap)
    assert n > cap
    c.report()
    c.close()


@pytest.mark.gpu
def test_record_store_planes():
    """asz_records_append (row_base = records held) into a store of 1,000 rows that grows: every stored row of both appends
    against the oracle, by id and append"""
    import torch
    c = Case("records 11x11x4", 11, 4, 1, 16384, 31)
    eng = c.eng
    eng.records_enable(1000)
    zeros = torch.zeros(c.G * 8 * 3, dtype=torch.float32, device=eng.device)
    for k in range(2):
        c.warm(3 + 7 * k)
        count0 = eng.records_count()
        want = oracle_rows(list(c.games), c.threads)
        count = eng.records_append(root_q=zeros)
        _, _, ids, turns = eng.records_views()
        assert count > count0 and bool((turns[count0:count] == k).all())
        flat = eng._wrap(eng.L.asz_records_planes(eng.h), (count * eng.pitch,), torch.int32)      # rows `pitch` floats apart
        words = flat[count0 * eng.pitch:].cpu().numpy().view(np.uint32).reshape(-1, eng.pitch)
        fails = compare_step("%s, append %d (row_base %d)" % (c.name, k, count0), count - count0, ids[count0:count].cpu().numpy(),
                             words, np.zeros(0, np.uint32), want, c.G, eng.pitch, eng.plane, kinds=c.kinds, filled=False, cov=c.cov)
        assert not fails, "\n".join(fails[:12])
    assert eng.records_count() > 1000
    c.report()
    c.close()


# ---- without a GPU ---------------------------------------------------------------------------------------------------------------

def _oracle_games(side, S, G, tics, seed=3, dec=1):
    from oracle import oracle as orc
    games = []
    for gi in range(G):
        g = orc.OracleGame(side, side, S, dec)
        g.init_native(seed, gi, 0)
        games.append(g)
    orc.env_run(G, side, side, S, dec, 0.15, seed, tics, encode=False, games=games)
    return games


def test_batch_encoder_equals_make_state():
    """oracle.env_encode against OracleGame.make_state / live_ids: 8-snake games, games with no live snake, finished games"""
    from oracle import oracle as orc
    for side, S, G, tics in [(11, 4, 200, 7), (19, 8, 60, 12), (7, 8, 80, 3)]:
        games = _oracle_games(side, S, G, tics)
        for gi in range(0, G, 9):                 # every 9th game: all snakes dead
            d = games[gi].dump()
            d["snake"][:, 0] = 0
            games[gi].load_dump(d)
            assert games[gi].n_live == 0
        batch = [None if gi % 13 == 5 else g for gi, g in enumerate(games)]
        ids, planes = orc.env_encode(batch, n_threads=4)
        want_ids, want = [], []
        for gi, g in enumerate(batch):
            if g is None:
                continue
            for k, s in enumerate(g.live_ids()):
                want_ids.append(gi * 8 + s)
                want.append(g.make_state(k))
        assert len(want) > G and (S < 8 or any(g.n_live == 8 for g in games))
        assert np.array_equal(ids, np.array(want_ids, np.int32))
        assert np.array_equal(planes.view(np.uint32), np.array(want).view(np.uint32))
    assert orc.env_encode([], 2)[1].shape[0] == 0


def test_plane_comparator_reports_planted_faults():
    """compare_step on oracle rows laid out as the kernel lays them out (tickets of two games with B's rows first, pitched rows,
    pad words 0, sentinel past the last row): nothing to report; each planted fault is reported and located"""
    from oracle import oracle as orc
    side, S, G, pairs = 11, 4, 96, 20
    games = _oracle_games(side, S, G, 6)
    want_ids, want_pl = orc.env_encode(games, 2)
    want_ids = want_ids.astype(np.int64)
    plane = want_pl[0].size
    pitch = (plane + 7) // 8 * 8
    kinds = ticket_kinds(G, pairs)
    # kernel order: tickets in a scrambled order, a pair's game B before its game A, a game's rows in ascending snake id
    tickets = [[2 * t + 1, 2 * t] for t in range(pairs)] + [[g] for g in range(2 * pairs, G)]
    rng = np.random.default_rng(1)
    seq = [g for t in rng.permutation(len(tickets)) for g in tickets[t]]
    rows_of = [np.flatnonzero(want_ids // 8 == g) for g in seq]
    perm = np.concatenate(rows_of)
    n = len(perm)
    words = np.full((n + 3) * pitch + 8, SENTINEL, np.uint32)
    rows = words[:n * pitch].reshape(n, pitch)
    rows[:, :plane] = want_pl[perm].reshape(n, -1).view(np.uint32)
    rows[:, plane:] = 0
    ids = want_ids[perm].astype(np.int32)
    want = lambda g0, g1: (want_ids[(want_ids >= 8 * g0) & (want_ids < 8 * g1)], want_pl[(want_ids >= 8 * g0) & (want_ids < 8 * g1)])

    def run(rows=rows, ids=ids, tail=words[n * pitch:], n=n, grown=n, keys=None):
        return compare_step("step", n, ids, rows, tail, want, G, pitch, plane, kinds=kinds, grown=grown, keys=keys)
    cov = new_coverage()
    assert compare_step("step", n, ids, rows, words[n * pitch:], want, G, pitch, plane, kinds=kinds, grown=n,
                        keys=plane_keys(want_pl[perm]), cov=cov) == []
    assert cov["kinds"] == {0, 1, 2} and cov["rows"] == n and cov["heads"] and cov["food"]
    N = 2 * side - 1
    # 1. one wall word: the first wall pixel of a row of game A of a pair gets 1.0 in channel 0
    r = int(np.flatnonzero(kinds[ids // 8] == 1)[1])
    P = want_pl[perm[r]]
    y, x = np.argwhere((P[..., 0] == 0) & (P[..., 1] == 1) & (P[..., 2] == 0))[0]
    bad = rows.copy(); bad[r, (y * N + x) * 3] = np.float32(1.0).view(np.uint32)
    f = run(rows=bad)
    loc = "row %d (game %d snake %d, game A of a pair ticket): first difference at pixel (%d, %d) channel 0" % (
        r, ids[r] // 8, ids[r] % 8, y, x)
    assert any(loc in m for m in f), f
    # 2. one board pixel of a single ticket's row, channel 1
    r = int(np.flatnonzero(kinds[ids // 8] == 0)[0])
    P = want_pl[perm[r]]
    y, x = np.argwhere(~((P[..., 0] == 0) & (P[..., 1] == 1) & (P[..., 2] == 0)))[0]
    bad = rows.copy(); bad[r, (y * N + x) * 3 + 1] ^= 1
    f = run(rows=bad)
    assert any("row %d (game %d snake %d, a single ticket): first difference at pixel (%d, %d) channel 1" % (
        r, ids[r] // 8, ids[r] % 8, y, x) in m for m in f), f
    # 3. a pad word left at the sentinel
    bad = rows.copy(); bad[7, pitch - 1] = SENTINEL
    f = run(rows=bad)
    assert any("pad word unwritten; first: row 7" in m and "word %d of %d" % (pitch - 1, pitch) in m for m in f), f
    # 4. a word written past row n: the first word of the slack after the last row
    tail = words[n * pitch:].copy(); tail[pitch + 2] = 0
    f = run(tail=tail)
    assert any("1 words past row %d were written; first: word %d (row %d, word 2" % (n, (n + 1) * pitch + 2, n + 1) in m for m in f), f
    # 5. a repeated id (row 12 carries row 40's id: 12's own id is missing, row 40's plane differs from row 12's)
    bad_ids = ids.copy(); bad_ids[12] = ids[40]
    f = run(ids=bad_ids)
    assert any("row ids repeat" in m for m in f) and any("oracle rows have no row" in m for m in f), f
    # 6. a game's rows split: one row of a 3-or-more-row game moved (with its id) to the end
    g = next(gg for gg in seq if (want_ids // 8 == gg).sum() >= 3)
    first = int(np.flatnonzero(ids // 8 == g)[0])
    mv = np.r_[np.arange(first), np.arange(first + 1, n), first]
    f = run(rows=rows[mv], ids=ids[mv])
    assert any("not contiguous; first: game %d" % g in m for m in f), f
    # 7. a game's rows out of snake order (rows and ids swapped together: every plane still matches its id)
    sw = np.arange(n); sw[first], sw[first + 1] = first + 1, first
    f = run(rows=rows[sw], ids=ids[sw])
    assert any("break ascending snake id" in m for m in f) and not any("difference" in m for m in f), f
    # 8. a row count off by one, and totals that grew by another number than the row count
    f = run(n=n - 1, grown=n - 1, tail=words[(n - 1) * pitch:])
    assert any("row_count is %d, the oracle has %d rows" % (n - 1, n) in m for m in f), f
    f = run(grown=n + 1)
    assert any("grew by %d, row_count is %d" % (n + 1, n) in m for m in f), f
    # 9. a wrong plane key
    k = plane_keys(want_pl[perm]); k[3, 1] ^= np.uint64(1)
    f = run(keys=k)
    assert any("1 plane keys differ; first: row 3" in m for m in f), f
