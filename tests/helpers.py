"""Shared helpers for the parity tests."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def digest(plane):
    return np.frombuffer(hashlib.blake2b(np.ascontiguousarray(plane).tobytes(), digest_size=8).digest(), np.uint64)[0]


def assert_dump_equal(got, want, ctx=""):
    """canonical dumps: last_move is only meaningful for live snakes; episode/game_id are engine bookkeeping."""
    gs, ws = np.asarray(got["snake"]).astype(np.int64), np.asarray(want["snake"]).astype(np.int64)
    alive = ws[:, 0] == 1
    assert np.array_equal(gs[:, 0], ws[:, 0]), "alive %s\n%s\n%s" % (ctx, gs, ws)
    assert np.array_equal(gs[alive][:, 1:5], ws[alive][:, 1:5]), "snake table %s\n%s\n%s" % (ctx, gs, ws)
    assert np.array_equal(gs[:, 5], ws[:, 5]), "rewards %s\n%s\n%s" % (ctx, gs, ws)
    for k in ("owner", "dist", "food"):
        assert np.array_equal(np.asarray(got[k]).astype(np.int64), np.asarray(want[k]).astype(np.int64)), "%s %s" % (k, ctx)
    assert np.array_equal(np.asarray(got["counters"])[:6], np.asarray(want["counters"])[:6]), "counters %s %s %s" % (
        ctx, got["counters"], want["counters"])


def golden_dump(z, t):
    return dict(snake=z["snake"][t], owner=z["owner"][t], dist=z["dist"][t], food=z["food"][t], counters=z["counters"][t])


SENTINEL = 0x7FBADBAD        # a NaN with a payload no encoder writes: fills plane buffers to mark the words nobody wrote


def plane_features(planes):
    """What a set of rows exercises: board window on each plane edge, other snakes' heads, food, food above 1.0."""
    P = np.asarray(planes)
    board = ~((P[..., 0] == 0) & (P[..., 1] == 1) & (P[..., 2] == 0))
    c = P.shape[1] // 2
    off = np.ones(P.shape[1:3], bool); off[c, c] = False
    return dict(edges={e for e, v in (("top", board[:, 0, :]), ("bottom", board[:, -1, :]), ("left", board[:, :, 0]),
                                      ("right", board[:, :, -1])) if v.any()},
                heads=bool((P[:, off, 0] != 0).any()), food=bool((P[:, off, 2] != 0).any()),
                food_above_1=bool((P[:, off, 2] > 1.0).any()))


# ---- deterministic stand-in value functions (AlphaNNet.v contract, alpha_nnet.py:61-76) -------------------------------
# Defined on the plane bytes; tests/golden/make_golden.py gives these to the reference's agents, the GPU tests give them
# to the mirror's agents, so both sides see identical values for identical planes.
def _fmix64(k):
    k = k ^ (k >> np.uint64(33))
    k = k * np.uint64(0xff51afd7ed558ccd)
    k = k ^ (k >> np.uint64(33))
    k = k * np.uint64(0xc4ceb9fe1a85ec53)
    k = k ^ (k >> np.uint64(33))
    return k


def plane_keys(X):
    """X: (n, h, w, 3) float32 -> (n, 2) uint64, the engine's 128-bit plane key (asz_common.cuh key_accumulate)."""
    X = np.ascontiguousarray(X, dtype=np.float32)
    n = X.shape[0]
    u = X.view(np.uint32).reshape(n, -1, 3).astype(np.uint64)
    a, b, c = u[..., 0], u[..., 1], u[..., 2]
    p = np.arange(u.shape[1], dtype=np.uint64)[None, :]
    wall = (a == 0) & (b == np.uint64(0x3F800000)) & (c == 0)
    x = (a << np.uint64(32)) | b
    y = (c << np.uint64(32)) | p
    with np.errstate(over="ignore"):
        h0 = _fmix64(_fmix64(y ^ np.uint64(0x9E3779B97F4A7C15)) ^ x)
        h1 = _fmix64(_fmix64(x ^ np.uint64(0xC2B2AE3D27D4EB4F)) + y)
        h0 = np.where(wall, np.uint64(0), h0).sum(axis=1, dtype=np.uint64)
        h1 = np.where(wall, np.uint64(0), h1).sum(axis=1, dtype=np.uint64)
    h0 = np.where(h0 == 0, np.uint64(1), h0)
    return np.stack([h0, h1], axis=1)


class KeyStubNet:
    """.v(X): value of action a = 16 bits of word `word` of the plane key, then the obstacle mask (NumPy >= 2 semantics).
    word 1 is the engine's built-in stub value function; word 0 is a second, different player for the pit tests."""

    def __init__(self, word=1):
        self.word = word
        self.calls = []

    def v(self, X):
        if hasattr(X, "detach"):
            X = X.detach().cpu().numpy()
        X = np.array(X, dtype=np.float32)
        if len(X) == 0:
            return np.zeros((0, 3), np.float32)
        keys = plane_keys(X)
        V = np.zeros((len(X), 3), np.float32)
        for i in range(3):
            xs = ((keys[:, self.word] >> np.uint64(16 * i)) & np.uint64(0xFFFF)).astype(np.float32)
            V[:, i] = (xs - np.float32(32767.5)) * np.float32(1.0 / 32768.0)
        cy, cx = X.shape[1] // 2, X.shape[2] // 2
        thr = np.float32(0.04)
        V[X[:, cy, cx - 1, 1] >= thr, 0] = -1.0
        V[X[:, cy - 1, cx, 1] >= thr, 1] = -1.0
        V[X[:, cy, cx + 1, 1] >= thr, 2] = -1.0
        self.calls.append(len(X))
        return V
