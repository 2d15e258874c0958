"""ctypes binding of the CPU oracle (oracle/asz_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  Never imported by the
product package (alphasnake_zero_b200).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libasz_oracle.so")


def build(force=False):
    src = [os.path.join(_HERE, f) for f in ("asz_oracle.c", "asz_oracle.h", "Makefile")]
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "CC=gcc"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


class EnvStats(C.Structure):
    _fields_ = [("steps", C.c_uint64), ("planes", C.c_uint64), ("episodes", C.c_uint64),
                ("plane_checksum", C.c_uint64), ("counters", C.c_uint64 * 6)]


class Trace(C.Structure):
    _fields_ = [("mode", C.c_int), ("seed", C.c_uint64), ("root_turn", C.c_uint32), ("max_steps", C.c_int),
                ("total_games", C.c_int), ("tree_moves", C.c_void_p), ("root_moves", C.c_void_p)]


VALUE_FN = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        vp, i32, u32, u64 = C.c_void_p, C.c_int, C.c_uint32, C.c_uint64
        L.og_new.restype = vp; L.og_new.argtypes = [i32] * 4
        L.og_free.argtypes = [vp]
        L.og_clone.restype = vp; L.og_clone.argtypes = [vp]
        L.og_init_explicit.argtypes = [vp, vp, vp, vp, i32]
        L.og_init_native.argtypes = [vp, u64, u32, u32]
        L.og_tic.restype = i32; L.og_tic.argtypes = [vp, vp, i32, i32, u32, u64]
        L.og_n_live.restype = i32; L.og_n_live.argtypes = [vp]
        L.og_live_ids.argtypes = [vp, vp]
        L.og_make_state.argtypes = [vp, i32, vp]
        L.og_dump.argtypes = [vp] * 6
        L.og_set_ids.argtypes = [vp, u32, u32]
        L.og_load_dump.argtypes = [vp] * 6
        L.og_philox.argtypes = [u32, u32, u32, u32, u64, vp]
        L.og_plane_key.argtypes = [vp, i32, vp]
        L.og_stub_value.argtypes = [vp, vp]
        L.og_obstacle_mask.argtypes = [vp, i32, i32, vp]
        L.oenv_run.argtypes = [vp, i32, i32, i32, i32, i32, u32, u64, i32, i32, i32, C.POINTER(EnvStats)]
        L.oenv_encode.restype = i32; L.oenv_encode.argtypes = [vp, i32, i32, vp, vp]
        L.oa_new.restype = vp; L.oa_new.argtypes = [C.c_double, i32, i32, i32, vp, vp]
        L.oa_free.argtypes = [vp]; L.oa_clear.argtypes = [vp]
        L.oa_set_rhat_mode.argtypes = [vp, i32]
        L.oa_make_moves.restype = i32; L.oa_make_moves.argtypes = [vp, vp, i32, C.POINTER(Trace), vp, vp]
        L.oa_table_size.restype = i32; L.oa_table_size.argtypes = [vp]
        L.oa_table_dump.restype = i32; L.oa_table_dump.argtypes = [vp, i32, vp, vp, vp, vp, vp]
        L.oa_stat.restype = u64; L.oa_stat.argtypes = [vp, i32]
        L.oa_n_records.restype = i32; L.oa_n_records.argtypes = [vp]
        L.oa_get_record.argtypes = [vp, i32, vp, vp]
        L.og_softermax.argtypes = [vp, C.c_double, vp]
        L.og_argmax3.restype = i32; L.og_argmax3.argtypes = [vp]
        L.og_choice3.restype = i32; L.og_choice3.argtypes = [vp, C.c_double]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def chance_threshold(chance):
    """u32 threshold of the engine's spawn coin: spawn iff philox_u32 <= threshold (game.py:131 `random() <= chance`)."""
    if chance <= 0.0:
        return 0                                   # game.py:130: a chance of 0 disables spawning altogether
    return int(min(max(int(chance * 4294967296.0), 1), 4294967295))


class OracleGame:
    """Game of code/utils/game.py, restated (oracle/asz_oracle.c)."""

    def __init__(self, H=11, W=11, S=4, health_dec=1, _handle=None):
        self.H, self.W, self.S, self.health_dec = H, W, S, health_dec
        self.h = _handle if _handle is not None else lib().og_new(H, W, S, health_dec)
        if not self.h:
            raise ValueError("unsupported game shape")

    def __del__(self):
        if getattr(self, "h", None):
            lib().og_free(self.h)
            self.h = None

    def clone(self):
        return OracleGame(self.H, self.W, self.S, self.health_dec, _handle=lib().og_clone(self.h))

    def init_explicit(self, start_yx, last_moves, food_yx):
        s = np.ascontiguousarray(start_yx, dtype=np.int32).reshape(-1)
        m = np.ascontiguousarray(last_moves, dtype=np.int32)
        f = np.ascontiguousarray(food_yx, dtype=np.int32).reshape(-1)
        lib().og_init_explicit(self.h, _p(s), _p(m), _p(f), len(f) // 2)

    def init_native(self, seed, game_id, episode=0):
        lib().og_init_native(self.h, seed, game_id, episode)

    def load_dump(self, d):
        a = {k: np.ascontiguousarray(d[k], dtype=np.int32) for k in ("snake", "owner", "dist", "food", "counters")}
        lib().og_load_dump(self.h, _p(a["snake"]), _p(a["owner"]), _p(a["dist"]), _p(a["food"]), _p(a["counters"]))

    def set_ids(self, game_id, episode=0):
        lib().og_set_ids(self.h, game_id, episode)

    def tic(self, moves, spawn_mode=0, spawn_cell=-1, chance=0.15, seed=0):
        m = np.ascontiguousarray(moves, dtype=np.int32)
        return lib().og_tic(self.h, _p(m), spawn_mode, spawn_cell, chance_threshold(chance), seed)

    @property
    def n_live(self):
        return lib().og_n_live(self.h)

    def live_ids(self):
        out = np.zeros(8, dtype=np.int32)
        lib().og_live_ids(self.h, _p(out))
        return out[: self.n_live].tolist()

    def make_state(self, k):
        out = np.empty((2 * self.H - 1, 2 * self.W - 1, 3), dtype=np.float32)
        lib().og_make_state(self.h, k, _p(out))
        return out

    def get_states(self):
        return [self.make_state(k) for k in range(self.n_live)]

    def dump(self):
        Cn = self.H * self.W
        snake = np.zeros((self.S, 6), dtype=np.int32)
        owner = np.zeros(Cn, dtype=np.int32); dist = np.zeros(Cn, dtype=np.int32); food = np.zeros(Cn, dtype=np.int32)
        counters = np.zeros(8, dtype=np.int32)
        lib().og_dump(self.h, _p(snake), _p(owner), _p(dist), _p(food), _p(counters))
        return dict(snake=snake, owner=owner, dist=dist, food=food, counters=counters)


def philox(c0, c1, c2, c3, seed):
    out = np.zeros(4, dtype=np.uint32)
    lib().og_philox(c0, c1, c2, c3, seed, _p(out))
    return out


def plane_key(plane):
    p = np.ascontiguousarray(plane, dtype=np.float32)
    key = np.zeros(2, dtype=np.uint64)
    lib().og_plane_key(_p(p), p.size // 3, _p(key))
    return int(key[0]), int(key[1])


def stub_value(key):
    k = np.array(key, dtype=np.uint64)
    v = np.zeros(3, dtype=np.float32)
    lib().og_stub_value(_p(k), _p(v))
    return v


def obstacle_mask(plane, H, W, v):
    p = np.ascontiguousarray(plane, dtype=np.float32)
    v = np.ascontiguousarray(v, dtype=np.float32).copy()
    lib().og_obstacle_mask(_p(p), H, W, _p(v))
    return v


def env_run(G, H=11, W=11, S=4, health_dec=1, chance=0.15, seed=0, tics=100, encode=True, n_threads=1, games=None):
    st = EnvStats()
    arr = None
    if games is not None:   # a list of OracleGame, or the ctypes array env_handles() made of one (reused between calls)
        arr = games if isinstance(games, C.Array) else (C.c_void_p * G)(*[g.h for g in games])
    lib().oenv_run(arr, G, H, W, S, health_dec, chance_threshold(chance), seed, tics, int(bool(encode)), n_threads,
                   C.byref(st))
    return dict(steps=st.steps, planes=st.planes, episodes=st.episodes, plane_checksum=st.plane_checksum,
                counters=list(st.counters))


def env_encode(games, n_threads=1):
    """make_state of every live snake of every game, in (game, snake id) order: (ids int32 [n] = game * 8 + snake id,
    planes float32 [n, 2H-1, 2W-1, 3]).  games: OracleGame or None (a finished game: no rows); all of one shape."""
    arr = (C.c_void_p * len(games))(*[g.h if g is not None else None for g in games])
    shape = next(((2 * g.H - 1, 2 * g.W - 1, 3) for g in games if g is not None), (1, 1, 3))
    n = lib().oenv_encode(arr, len(games), 1, None, None) if len(games) else 0
    planes = np.empty((n,) + shape, dtype=np.float32)
    ids = np.empty(n, dtype=np.int32)
    if n:
        lib().oenv_encode(arr, len(games), n_threads, _p(planes), _p(ids))
    return ids, planes


def env_handles(games):
    """ctypes array of the games' handles, to be passed as env_run(games=...) repeatedly without rebuilding it"""
    return (C.c_void_p * len(games))(*[g.h for g in games])


def softermax(z, base):
    z = np.ascontiguousarray(z, dtype=np.float32)
    out = np.zeros(3, dtype=np.float32)
    lib().og_softermax(_p(z), float(base), _p(out))
    return out


def argmax3(z):
    z = np.ascontiguousarray(z, dtype=np.float32)
    return lib().og_argmax3(_p(z))


def choice3(p, u):
    p = np.ascontiguousarray(p, dtype=np.float32)
    return lib().og_choice3(_p(p), float(u))


class OracleAgent:
    """Agent + MCTSAgent + MCTSMPGameRunner of agent.py / mp_game_runner.py, restated."""

    def __init__(self, base=100, training=False, max_depth=8, max_breadth=128, value_fn=None):
        self._cb = None
        cb = None
        if value_fn is not None:
            def _tramp(ctx, planes, n, H, W, vout):
                pl = np.ctypeslib.as_array(planes, shape=(n, 2 * H - 1, 2 * W - 1, 3))
                v = np.ascontiguousarray(value_fn(pl), dtype=np.float32)
                C.memmove(vout, v.ctypes.data, 12 * n)
            self._cb = VALUE_FN(_tramp)
            cb = C.cast(self._cb, C.c_void_p)
        self.h = lib().oa_new(float(base), int(training), max_depth, max_breadth, cb, None)
        self.base, self.training, self.D, self.breadth = base, training, max_depth, max_breadth
        self.parallel = min(8, max_breadth)
        self.epochs = max_breadth // self.parallel

    def __del__(self):
        if getattr(self, "h", None):
            lib().oa_free(self.h)
            self.h = None

    def clear(self):
        lib().oa_clear(self.h)

    def set_rhat_mode(self, before_backups):
        """False (default) = the reference's order: r-hat of a row is computed inside the backup loop from a live alias of the
        table entry (agent.py:180,214); True = every r-hat of a step from the values before the step's backups."""
        lib().oa_set_rhat_mode(self.h, int(bool(before_backups)))

    def make_moves(self, games, total_games, root_turn=0, seed=0, tree_moves=None, root_moves=None, replay=False):
        """games: list of live OracleGame (their game_id must be set).  tree_moves: uint8 array
        [epochs, D, total_games*parallel, S] (read in replay mode, written otherwise)."""
        S = games[0].S
        n_rows_max = len(games) * S
        tr = Trace()
        tr.mode = 1 if replay else 0
        tr.seed = seed; tr.root_turn = root_turn; tr.max_steps = max(self.D, 1); tr.total_games = total_games
        tr.tree_moves = tree_moves.ctypes.data if tree_moves is not None else None
        if root_moves is None:
            root_moves = np.full(n_rows_max, 255, dtype=np.uint8)
        tr.root_moves = root_moves.ctypes.data
        arr = (C.c_void_p * len(games))(*[g.h for g in games])
        moves = np.zeros(n_rows_max, dtype=np.int32)
        q = np.zeros((n_rows_max, 3), dtype=np.float32)
        n = lib().oa_make_moves(self.h, arr, len(games), C.byref(tr), _p(moves), _p(q))
        return moves[:n].copy(), q[:n].copy()

    def table(self):
        n = lib().oa_table_size(self.h)
        keys = np.zeros((n, 2), dtype=np.uint64)
        Q = np.zeros((n, 3), dtype=np.float32); Wt = np.zeros((n, 3), dtype=np.float32); N = np.zeros((n, 3), dtype=np.float32)
        age = np.zeros(n, dtype=np.int32)
        lib().oa_table_dump(self.h, n, _p(keys), _p(Q), _p(Wt), _p(N), _p(age))
        return dict(keys=keys, Q=Q, W=Wt, N=N, age=age)

    def stat(self, which):
        names = dict(evals=0, node_visits=1, hits=2, subgames=3, subgame_tics=4, alias_errors=7)
        return lib().oa_stat(self.h, names[which])

    def records(self, H, W):
        n = lib().oa_n_records(self.h)
        planes = np.zeros((n, 2 * H - 1, 2 * W - 1, 3), dtype=np.float32)
        q = np.zeros((n, 3), dtype=np.float32)
        for i in range(n):
            lib().oa_get_record(self.h, i, _p(planes[i]), _p(q[i]))
        return planes, q
