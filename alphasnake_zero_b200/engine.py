"""Python handle on one device-resident engine (include/asz_b200.h).  PyTorch is used only for device memory and
streams; all game, encode and search work happens in libasz_b200.so."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (SPAWN_NATIVE, SPAWN_NONE, SPAWN_REPLAY, STEP_AUTO_RESET, STEP_ENCODE, STEP_KEYS, STEP_RANDOM_ACT,
                   STEP_TIC, AszError, check)

__all__ = ["Engine", "AszError", "STEP_TIC", "STEP_ENCODE", "STEP_AUTO_RESET", "STEP_RANDOM_ACT", "STEP_KEYS",
           "SPAWN_NONE", "SPAWN_REPLAY", "SPAWN_NATIVE"]


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _np(a):
    return a.ctypes.data_as(C.c_void_p)


class Engine:
    def __init__(self, side=11, snakes=4, health_dec=1, food_chance=0.15, games=1, seed=0, max_depth=0, max_breadth=0,
                 softmax_base=100.0, training=False, table_log2=0, numpy1_mask=False, device=None):
        if not torch.cuda.is_available():
            raise AszError("no CUDA device: alphasnake_zero_b200 has no CPU fallback")
        if isinstance(device, torch.device):
            device = device.index
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self.L = _lib.lib()
        self.side, self.S, self.G = side, snakes, games
        self.N = 2 * side - 1
        self.plane = self.N * self.N * 3
        cfg = _lib.Config(side, snakes, health_dec, food_chance, games, seed, max_depth, max_breadth, softmax_base,
                          int(training), table_log2, int(numpy1_mask))
        self.cfg = cfg
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(self.L.asz_engine_create(C.byref(h), C.byref(cfg)))
        self.h = h
        dev = self.device
        self.pitch = int(self.L.asz_plane_pitch(self.h))      # floats between rows of the engine's plane buffers (32-byte rows)
        self.max_rows = games * snakes
        self._planes = None
        self.row_ids = torch.zeros(self.max_rows, dtype=torch.int32, device=dev)
        self.row_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.ended = torch.zeros(games, dtype=torch.uint8, device=dev)
        self.rewards = torch.zeros(games, 8, dtype=torch.int8, device=dev)
        self.keys = None
        self._pit_open = False
        self._pit_searchers = [None, None]     # attached searcher engines, kept alive while attached

    def close(self):
        if getattr(self, "h", None):
            self.L.asz_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def planes(self):
        """[G*S, N, N, 3] float32 batch buffer (allocated on first use).  Rows are `pitch` floats apart (the plane size rounded
        up to 8 floats: every plane starts on a 32-byte sector, the one layout the encode kernel writes), so this is a strided
        view; `.contiguous()` / indexing give dense copies."""
        if self._planes is None:
            # empty, not zeros: a 1.4 GB fill would leave the L2 full of dirty lines right before the first launch (DESIGN.md 4.1)
            self._planes_flat = torch.empty(self.max_rows * self.pitch + 8, dtype=torch.float32, device=self.device)
            self._planes = torch.as_strided(self._planes_flat, (self.max_rows, self.N, self.N, 3), (self.pitch, 3 * self.N, 3, 1))
        return self._planes

    def _plane_pitch_of(self, t):
        """self.pitch for a [rows, N, N, 3] view with the engine's row pitch (see `planes`); the encode writes whole rows of
        `pitch` floats, so a tensor with any other layout is refused"""
        if tuple(t.shape[1:]) != (self.N, self.N, 3) or t.dtype != torch.float32:
            raise AszError("planes must be float32 [rows, %d, %d, 3]" % (self.N, self.N))
        if tuple(t.stride()) != (self.pitch, 3 * self.N, 3, 1):
            raise AszError("planes must have the engine's row pitch: rows %d floats apart (asz_plane_pitch)" % self.pitch)
        return self.pitch

    def reset(self):
        check(self.L.asz_reset(self.h, self.stream))

    # ---- state interchange -------------------------------------------------------------------------------------
    def get_state(self, game):
        Cn = self.side * self.side
        snake = np.zeros((self.S, 6), np.int32); owner = np.zeros(Cn, np.int32); dist = np.zeros(Cn, np.int32)
        food = np.zeros(Cn, np.int32); counters = np.zeros(8, np.int32)
        check(self.L.asz_get_state(self.h, game, _np(snake), _np(owner), _np(dist), _np(food), _np(counters)))
        return dict(snake=snake, owner=owner, dist=dist, food=food, counters=counters)

    def set_state(self, game, d, episode=0):
        """d: canonical dump (asz_get_state); `episode` is the episode counter of the game's RNG streams (0 for a fresh game)."""
        a = {k: np.ascontiguousarray(d[k], dtype=np.int32) for k in ("snake", "owner", "dist", "food")}
        cnt = np.zeros(8, np.int32)
        c = np.asarray(d["counters"]).astype(np.int32)
        cnt[:6] = c[:6]
        cnt[6] = episode
        cnt[7] = 0
        check(self.L.asz_set_state(self.h, game, _np(a["snake"]), _np(a["owner"]), _np(a["dist"]), _np(a["food"]), _np(cnt)))

    # ---- lockstep step -----------------------------------------------------------------------------------------
    def step(self, actions=None, spawn_cells=None, spawn_mode=SPAWN_NATIVE, tic=True, encode=True, auto_reset=False,
             random_actions=False, keys=False, planes=None):
        """One fused launch.  actions: uint8 cuda tensor [G, 8]; spawn_cells: int32 cuda tensor [G].
        Returns nothing; results are in self.row_count / row_ids / planes / ended / rewards (device tensors)."""
        flags = (STEP_TIC if tic else 0) | (STEP_ENCODE if encode else 0) | (STEP_AUTO_RESET if auto_reset else 0) | \
                (STEP_RANDOM_ACT if random_actions else 0) | (STEP_KEYS if keys else 0)
        a = _lib.StepArgs()
        a.flags = flags
        a.spawn_mode = spawn_mode
        a.d_actions = actions.data_ptr() if actions is not None else None
        a.d_spawn_cells = spawn_cells.data_ptr() if spawn_cells is not None else None
        if encode:
            pl = self.planes if planes is None else planes
            a.d_planes = pl.data_ptr()
            a.max_rows = pl.shape[0]
            a.plane_pitch = self._plane_pitch_of(pl)
        a.d_row_ids = self.row_ids.data_ptr()
        if keys:
            if self.keys is None:
                self.keys = torch.zeros(self.max_rows, 2, dtype=torch.int64, device=self.device)
            a.d_keys = self.keys.data_ptr()
        a.d_row_count = self.row_count.data_ptr()
        a.d_ended = self.ended.data_ptr()
        a.d_rewards = self.rewards.data_ptr()
        check(self.L.asz_env_step(self.h, C.byref(a), self.stream))

    def submit_host(self, h_actions, h_ended, h_rewards, spawn_mode=SPAWN_NATIVE, tic=True, encode=True, auto_reset=False,
                    random_actions=False, h_spawn_cells=None):
        """asz_env_submit_host: one step with HOST buffers (pinned torch tensors or None), enqueued without waiting.  Returns the
        ticket for wait_host; two steps may be in flight (the inputs of the second are copied under the kernel of the first)."""
        flags = (STEP_TIC if tic else 0) | (STEP_ENCODE if encode else 0) | (STEP_AUTO_RESET if auto_reset else 0) | \
                (STEP_RANDOM_ACT if random_actions else 0)
        ticket = C.c_int32(-1)
        check(self.L.asz_env_submit_host(self.h, flags, spawn_mode, _ptr(h_actions), _ptr(h_spawn_cells), _ptr(h_ended),
                                         _ptr(h_rewards), self.stream, C.byref(ticket)))
        return ticket.value

    def wait_host(self, ticket):
        """asz_env_wait_host: blocks until the step's host results are complete; returns the number of plane rows it wrote."""
        rows = C.c_int32(0)
        check(self.L.asz_env_wait_host(self.h, ticket, C.byref(rows)))
        return rows.value

    def totals(self):
        t = np.zeros(16, np.uint64)
        check(self.L.asz_get_totals(self.h, _np(t)))
        return dict(zip(("wall", "body", "head", "starve", "food_eaten", "game_length", "episodes", "tics", "planes"), t.tolist()))

    # ---- convenience used by tests and the drop-in classes -------------------------------------------------------
    def rows(self):
        """(row_ids numpy [n], planes torch view [n, N, N, 3]) of the last encode, sorted by (game, snake)."""
        n = int(self.row_count.item())
        ids = self.row_ids[:n]
        order = torch.argsort(ids)
        return ids[order].cpu().numpy(), self.planes[:n][order]

    # ---- search (Agent.make_moves) -------------------------------------------------------------------------------
    def search_info(self):
        info = np.zeros(8, np.int32)
        check(self.L.asz_search_info(self.h, _np(info)))
        return dict(zip(("P", "epochs", "max_steps", "n_sub", "max_rows", "table_log2", "root_turn", "epoch"), info.tolist()))

    def _wrap(self, ptr, shape, dtype):
        """torch view of an engine-owned device buffer (no copy)."""
        n = int(np.prod(shape))
        itemsize = torch.empty((), dtype=dtype).element_size()
        iface = {"shape": (n,), "typestr": {1: "|u1", 4: "<f4"}[itemsize] if dtype != torch.int32 else "<i4",
                 "data": (int(ptr), False), "version": 3}
        holder = type("_Buf", (), {"__cuda_array_interface__": iface})()
        return torch.as_tensor(holder, device=self.device).view(dtype).view(*shape)

    def search(self, value_fn=None, trace=None, trace_mode=0, root_trace=None, net=None, sync_steps=False):
        """One root turn of the search for the engine's current root games.
        net: a NativeNet -- the whole root turn runs in one native call (asz_search_run_net), the product path.
        value_fn(planes[n, N, N, 3] float32 cuda) -> [n, 3] float32 cuda raw network outputs (the obstacle mask of
        AlphaNNet.v is applied here): a Python-driven loop for reference networks (tests).
        Neither = the deterministic stub value function (no host sync in the loops; sync_steps=True drives the same stub
        through the per-step calls, reading the miss count back every step like the network path does).
        trace: uint8 cuda tensor [epochs, max_steps, G*P, S]; trace_mode 0 none / 1 replay / 2 record.
        Returns (root_q [G, 8, 3] float32, root_moves [G, 8] uint8, 255 = no row) as views of engine buffers."""
        st = self.stream
        tp = C.c_void_p(trace.data_ptr()) if trace is not None else None
        rp = C.c_void_p(root_trace.data_ptr()) if root_trace is not None else None
        if net is not None:
            check(self.L.asz_search_run_net(self.h, net.h, tp, trace_mode, rp, st))
        elif value_fn is None and not sync_steps:
            check(self.L.asz_search_run_stub(self.h, tp, trace_mode, rp, st))
        else:
            info = self.search_info()
            planes = self._wrap(self.L.asz_search_eval_planes(self.h), (info["max_rows"], self.N, self.N, 3), torch.float32)
            values = self._wrap(self.L.asz_search_eval_values(self.h), (info["max_rows"], 3), torch.float32)
            n = C.c_int32(0)
            check(self.L.asz_search_begin(self.h, st))
            for _ in range(info["epochs"]):
                check(self.L.asz_search_epoch_begin(self.h, st))
                for step in range(1, info["max_steps"] + 2):
                    check(self.L.asz_search_step_probe(self.h, C.byref(n), st))
                    if step <= info["max_steps"]:
                        if value_fn is None:
                            check(self.L.asz_search_stub_values(self.h, st))
                        elif n.value > 0:
                            v = value_fn(planes[:n.value])
                            values[:n.value].copy_(v)
                            check(self.L.asz_obstacle_mask(self.h, C.c_void_p(planes.data_ptr()), n.value,
                                                           C.c_void_p(values.data_ptr()), st))
                        check(self.L.asz_search_step_sample(self.h, None, tp, trace_mode, st))
            check(self.L.asz_search_finish(self.h, rp, None, None, st))
        q = self._wrap(self.L.asz_search_root_q(self.h), (self.G, 8, 3), torch.float32)
        mv = self._wrap(self.L.asz_search_root_moves(self.h), (self.G, 8), torch.uint8)
        return q, mv

    def search_clear(self):
        check(self.L.asz_search_clear(self.h, self.stream))

    def search_stats(self):
        s = np.zeros(16, np.uint64)
        check(self.L.asz_search_stats(self.h, _np(s)))
        names = ("evals", "node_visits", "hits", "subgames", "subgame_tics", "collisions", "inserts", "recreated",
                 "occupied", "overflow", "compactions", "mid_turn_compactions")
        return dict(zip(names, s.tolist()))

    def table(self, cap=None):
        cnt = C.c_int32(0)
        check(self.L.asz_search_table_dump(self.h, 0, None, None, None, None, C.byref(cnt)))
        n = cnt.value if cap is None else min(cap, cnt.value)
        keys = np.zeros((max(n, 1), 2), np.uint64); W = np.zeros((max(n, 1), 3), np.float32); N = np.zeros((max(n, 1), 3), np.float32)
        age = np.zeros(max(n, 1), np.int32)
        if n > 0:
            check(self.L.asz_search_table_dump(self.h, n, _np(keys), _np(W), _np(N), _np(age), C.byref(cnt)))
        keys, W, N, age = keys[:n], W[:n], N[:n], age[:n]
        order = np.lexsort((keys[:, 1], keys[:, 0]))
        return dict(keys=keys[order], W=W[order], N=N[order], Q=(W / N)[order] if n else W, age=age[order])

    # ---- training records kept on the device (Agent.records / Agent.values, agent.py:21-23, 93-97) ---------------------
    def records_enable(self, capacity_rows):
        check(self.L.asz_records_enable(self.h, int(capacity_rows)))
        self.records_capacity = int(capacity_rows)

    def records_append(self, root_q=None):
        """root states + root Q rows of every live snake into the device store; returns the number of records held."""
        n = C.c_int64(0)
        check(self.L.asz_records_append(self.h, _ptr(root_q), C.byref(n), self.stream))
        return n.value

    def records_count(self):
        n = C.c_int64(0)
        check(self.L.asz_records_count(self.h, C.byref(n)))
        return n.value

    def records_clear(self):
        check(self.L.asz_records_clear(self.h))

    def records_gather(self, idx, mirror=True):
        """alpha_snake_zero_trainer.py:70-77, 93-100: (X [m, N, N, 3], V [m, 3]) device tensors, m = 2n with the mirrored copies
        after the n originals when mirror.  idx: int64 indices (any array-like or a cuda tensor)."""
        idx = torch.as_tensor(idx, dtype=torch.int64).to(self.device).contiguous()
        n = idx.numel()
        m = 2 * n if mirror else n
        X = torch.empty(m, self.N, self.N, 3, dtype=torch.float32, device=self.device)
        V = torch.empty(m, 3, dtype=torch.float32, device=self.device)
        check(self.L.asz_records_gather(self.h, _ptr(idx), n, int(bool(mirror)), _ptr(X), _ptr(V), self.stream))
        return X, V

    def records_views(self):
        """(planes [n, N, N, 3], values [n, 3], ids [n] int32 = game*8 + snake, turns [n] int32) views of the store"""
        n = max(self.records_count(), 1)       # the store may have grown: wrap what is filled, not a remembered capacity
        flat = self._wrap(self.L.asz_records_planes(self.h), (n * self.pitch,), torch.float32)      # rows are `pitch` floats apart
        pl = torch.as_strided(flat, (n, self.N, self.N, 3), (self.pitch, 3 * self.N, 3, 1))
        va = self._wrap(self.L.asz_records_values(self.h), (n, 3), torch.float32)
        ids = self._wrap(self.L.asz_records_ids(self.h), (n,), torch.int32)
        tu = self._wrap(self.L.asz_records_turns(self.h), (n,), torch.int32)
        n = self.records_count()
        return pl[:n], va[:n], ids[:n], tu[:n]

    # ---- pit: pit_mp_game_runner.MPGameRunner.run with pit_agent.Agent on both sides, on the device ----------------
    # A player is a NativeNet, or 0 / 1: the stand-in player valued from that word of the plane key (tests).
    @staticmethod
    def _pit_player(p):
        if isinstance(p, int):
            return _lib.PitPlayer(None, p)
        return _lib.PitPlayer(p.h.value, 0)

    def pit_begin(self, alice, bob, alice_snakes):
        """asz_pit_begin: a match of `alice` (snake ids < alice_snakes) against `bob` on the current root games.  Returns the
        number of games running."""
        a, b = self._pit_player(alice), self._pit_player(bob)
        running = C.c_int32(0)
        self._pit_open = False
        check(self.L.asz_pit_begin(self.h, C.byref(a), C.byref(b), int(alice_snakes), C.byref(running), self.stream))
        self._pit_open = True
        return running.value

    def pit_turn(self, spawn_cells=None, spawn_mode=SPAWN_NATIVE, moves=None):
        """asz_pit_turn: one turn; spawn_cells int32 cuda [G] for SPAWN_REPLAY, moves uint8 cuda [G, 8] receives the moves played
        (255 = none).  Returns the number of games still running."""
        running = C.c_int32(0)
        check(self.L.asz_pit_turn(self.h, spawn_mode, _ptr(spawn_cells), _ptr(moves), C.byref(running), self.stream))
        return running.value

    def _pit_results(self, rc_of, written_on_state):
        """written_on_state: ASZ_ERR_STATE from this call means 'games still running, results so far written' (and so does
        ASZ_ERR_CAPACITY, a searcher's Q table overflow, from asz_pit_run)"""
        winners = torch.empty(self.G, dtype=torch.int32, device=self.device)
        decided = torch.empty(self.G, dtype=torch.int32, device=self.device)
        turns = C.c_int32(0)
        rc = rc_of(_ptr(winners), _ptr(decided), C.byref(turns))
        if rc != 0 and not (rc in (_lib.ASZ_ERR_STATE, _lib.ASZ_ERR_CAPACITY) and written_on_state):
            check(rc)                     # nothing was written
        res = (winners.cpu().numpy(), decided.cpu().numpy(), turns.value)
        if rc != 0:
            err = AszError("asz error %d: %s" % (rc, self.L.asz_last_error().decode()))
            err.partial = res             # (winners, decided_turn, turns) of the games decided so far
            raise err
        return res

    def pit_finish(self):
        """asz_pit_finish -> (winners int32 [G] with -1 = draw, decided_turn int32 [G], turns).  Games still running raise
        AszError with the results so far in `.partial` (winner -1 and decided_turn -1 for the running games)."""
        open_match, self._pit_open = self._pit_open, False      # asz_pit_finish closes the match
        return self._pit_results(lambda w, d, t: self.L.asz_pit_finish(self.h, w, d, t, self.stream), open_match)

    def pit_run(self, alice, bob, alice_snakes, max_turns=0):
        """asz_pit_run: the whole match with native food spawn, one call; results as pit_finish."""
        a, b = self._pit_player(alice), self._pit_player(bob)
        self._pit_open = False            # asz_pit_run abandons a match in progress and closes its own
        # its ASZ_ERR_STATE comes only from the closing asz_pit_finish: results so far written (begin and turn fail otherwise)
        return self._pit_results(lambda w, d, t: self.L.asz_pit_run(self.h, C.byref(a), C.byref(b), int(alice_snakes),
                                                                    int(max_turns), w, d, t, self.stream), True)

    def pit_stats(self):
        s = np.zeros(4, np.float64)
        check(self.L.asz_pit_stats(self.h, _np(s)))
        r = np.zeros(2, np.float64)
        check(self.L.asz_pit_search_stats(self.h, _np(r)))
        return dict(turns=int(s[0]), net_rows=int(s[1]), stub_rows=int(s[2]), forward_ms=float(s[3]), search_rows=int(r[0]),
                    search_ms=float(r[1]))

    def pit_set_search(self, side, searcher):
        """asz_pit_set_search: `searcher` (an Engine with search configured and training=False, or None to detach) plays side 0
        (Alice) or 1 (Bob) of the next pit_begin / pit_run as the search Agent, valued by that side's player (its network, or
        the stand-in reading key word 0 / 1)."""
        check(self.L.asz_pit_set_search(self.h, int(side), searcher.h if searcher is not None else None))
        self._pit_searchers[int(side)] = searcher

    def copy_root_games_from(self, src, skip=None):
        """asz_copy_root_games: this engine's root games become copies of `src`'s (same board side, snake count, game count and
        device); skip: bool / uint8 cuda tensor [G], games where it is set arrive finished, so a search here leaves them alone."""
        if skip is not None:
            skip = skip.to(device=self.device, dtype=torch.uint8).contiguous()
        check(self.L.asz_copy_root_games(self.h, src.h, _ptr(skip), self.stream))

    # ---- helpers for the drop-in classes ---------------------------------------------------------------------------
    def alive_mask(self):
        """bool [G, S] (device): snake alive and game not finished."""
        if not hasattr(self, "_snk_view"):
            ptrs = (C.c_void_p * 3)()
            check(self.L.asz_internal_state(self.h, ptrs))
            self._snk_view = self._wrap64(ptrs[1], (self.G, 8))
            self._meta_view = self._wrap(ptrs[2], (self.G, 8), torch.int32)
        alive = ((self._snk_view >> 42) & 1).bool()[:, :self.S]
        live_game = (self._meta_view[:, 7] & 1) == 0
        return alive & live_game[:, None]

    def _wrap64(self, ptr, shape):
        n = int(np.prod(shape))
        iface = {"shape": (n,), "typestr": "<i8", "data": (int(ptr), False), "version": 3}
        holder = type("_Buf", (), {"__cuda_array_interface__": iface})()
        return torch.as_tensor(holder, device=self.device).view(*shape)

    def encode_rows(self, refresh=True):
        """(planes [n, N, N, 3] device view, row ids numpy [n]) of the current root states."""
        if refresh:
            self.step(tic=False, encode=True)
        n = int(self.row_count.item())
        return self.planes[:n], self.row_ids[:n].cpu().numpy()

    def states_of(self, game):
        planes, rows = self.encode_rows()
        sel = [i for i, r in enumerate(rows) if r // 8 == game]
        sel.sort(key=lambda i: rows[i])
        ph = planes.cpu().numpy()
        return [ph[i] for i in sel]
