"""Empty, ragged and overflowing inputs through the C ABI: nothing to encode, nothing to evaluate, every game finished,
a plane batch smaller than the number of live snakes, a Q table that is too small."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _engine(**kw):
    from alphasnake_zero_b200.engine import Engine
    return Engine(**kw)


def test_network_on_empty_and_ragged_batches():
    import torch
    from alphasnake_zero_b200.net import NativeNet
    from oracle import net_oracle as no
    w = no.init_weights(11, seed=2, randomize_bn=True)
    net = NativeNet(w, "cuda", chunk_images=64)
    out = net.forward(torch.zeros(0, 21, 21, 3, device="cuda"))
    assert tuple(out.shape) == (0, 3)
    x = torch.rand(131, 21, 21, 3, device="cuda")
    full = net.forward(x).cpu().numpy()
    for n in (1, 63, 64, 65, 130):                     # below / at / above the pass size, odd remainders
        part = net.forward(x[:n]).cpu().numpy()
        assert np.array_equal(part.view(np.uint32), full[:n].view(np.uint32)), n


def test_all_games_finished_produce_no_rows_and_no_moves():
    import torch
    from alphasnake_zero_b200 import _lib
    eng = _engine(side=7, snakes=4, health_dec=9, games=64, seed=5, max_depth=4, max_breadth=8, softmax_base=2.0, training=True,
                  table_log2=14)
    eng.reset()
    for _ in range(400):                               # uniform-random play without reset: every game ends
        eng.step(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=False, auto_reset=False, random_actions=True)
    assert not bool(eng.alive_mask().any().item())
    before = eng.get_state(3)
    eng.step(spawn_mode=_lib.SPAWN_NATIVE, tic=True, encode=True, auto_reset=False, random_actions=True)
    assert int(eng.row_count.item()) == 0 and int(eng.ended.sum().item()) == 0       # finished games do not tic, end or encode again
    after = eng.get_state(3)
    for k in ("snake", "owner", "dist", "food", "counters"):
        assert np.array_equal(before[k], after[k]), k
    q, mv = eng.search(value_fn=None)                  # a search over finished games: no rows, no moves, no evaluations
    assert bool((mv == 255).all().item())
    assert eng.search_stats()["evals"] == 0
    eng.close()


def test_pitched_plane_batch_smaller_than_the_live_rows():
    """max_rows below the number of live snakes: the rows that fit are complete planes, the counter still says how many
    rows there were, nothing is written past the buffer"""
    import torch
    eng = _engine(side=11, snakes=4, games=256, seed=9)
    eng.reset()
    eng.step(tic=False, encode=True)
    n = int(eng.row_count.item())
    assert n == 1024
    ids_full = eng.row_ids[:n].cpu().numpy().copy()
    full = eng.planes[:n].cpu().numpy()
    ref = {int(i): full[r] for r, i in enumerate(ids_full)}
    flat = torch.full(((100 + 8) * eng.pitch,), 7.0, device="cuda")
    small = torch.as_strided(flat, (100, 21, 21, 3), (eng.pitch, 3 * 21, 3, 1))
    eng.step(tic=False, encode=True, planes=small)
    assert int(eng.row_count.item()) == 1024            # rows that existed, not rows that fit
    assert bool((flat[100 * eng.pitch:] == 7.0).all().item())      # nothing past the 100 rows
    ids = eng.row_ids[:100].cpu().numpy()
    got = small.cpu().numpy()
    for r in range(100):
        assert np.array_equal(got[r].view(np.uint32), ref[int(ids[r])].view(np.uint32))
    eng.close()


def test_table_overflow_fails_the_turn_but_not_the_engine():
    """a table far too small: the turn fails with ASZ_ERR_CAPACITY (a dropped row would play an arbitrary move), the counters say
    why, the outputs that were written are well formed, and the engine keeps working after Agent.clear"""
    from alphasnake_zero_b200.engine import AszError
    eng = _engine(side=11, snakes=4, games=64, seed=2, max_depth=8, max_breadth=32, softmax_base=2.0, training=True, table_log2=10)
    eng.reset()
    with pytest.raises(AszError, match="overflow"):
        eng.search(value_fn=None)
    st = eng.search_stats()
    assert st["overflow"] > 0 and st["evals"] > 0
    q = eng._wrap(eng.L.asz_search_root_q(eng.h), (64, 8, 3), torch_float32())
    assert np.isfinite(q.cpu().numpy()).all()
    eng.search_clear()
    assert eng.search_stats()["overflow"] == 0
    eng.close()


def torch_float32():
    import torch
    return torch.float32


def test_argument_errors_are_reported():
    import torch
    from alphasnake_zero_b200 import _lib
    from alphasnake_zero_b200.engine import AszError
    eng = _engine(side=11, snakes=4, games=8, seed=1)
    eng.reset()
    a = _lib.StepArgs()
    a.flags = _lib.STEP_TIC                             # a tic without actions and without STEP_RANDOM_ACT
    a.spawn_mode = _lib.SPAWN_NATIVE
    assert _lib.lib().asz_env_step(eng.h, C.byref(a), eng.stream) != 0
    assert b"d_actions" in _lib.lib().asz_last_error()
    # the encode writes rows asz_plane_pitch() floats apart: dense rows (0 or the plane size) are refused, not reinterpreted
    for pitch in (0, int(_lib.lib().asz_plane_floats(eng.h))):
        a = _lib.StepArgs()
        a.flags = _lib.STEP_ENCODE
        a.d_planes = eng.planes.data_ptr()
        a.d_row_ids = eng.row_ids.data_ptr()
        a.d_row_count = eng.row_count.data_ptr()
        a.max_rows = eng.max_rows
        a.plane_pitch = pitch
        assert _lib.lib().asz_env_step(eng.h, C.byref(a), eng.stream) != 0
        assert b"asz_plane_pitch" in _lib.lib().asz_last_error()
    with pytest.raises(AszError):
        eng.step(tic=False, encode=True, planes=torch.zeros(8, 21, 21, 3, device="cuda"))
    with pytest.raises(AszError):
        eng.search(value_fn=None)                       # the engine was created without a search configuration
    eng.close()


def test_host_pipeline_edge_cases():
    """asz_env_submit_host / asz_env_wait_host at the edges: one game, an odd number of games, pageable result buffers, missing
    inputs, and an engine closed while a step is still in flight."""
    import torch
    from alphasnake_zero_b200.engine import AszError
    for G in (1, 3):
        a, b = _engine(side=7, snakes=2, games=G, seed=4), _engine(side=7, snakes=2, games=G, seed=4)
        a.reset(); b.reset()
        acts = torch.ones(G, 8, dtype=torch.uint8).pin_memory()
        end_pin = torch.zeros(G, dtype=torch.uint8).pin_memory(); rew_pin = torch.zeros(G, 8, dtype=torch.int8).pin_memory()
        end_pg = torch.zeros(G, dtype=torch.uint8); rew_pg = torch.zeros(G, 8, dtype=torch.int8)        # pageable
        for _ in range(12):
            ra = a.wait_host(a.submit_host(acts, end_pin, rew_pin, spawn_mode=2, auto_reset=True))
            rb = b.wait_host(b.submit_host(acts, end_pg, rew_pg, spawn_mode=2, auto_reset=True))
            assert ra == rb
            assert torch.equal(end_pin, end_pg) and torch.equal(rew_pin, rew_pg)
        with pytest.raises(AszError):
            a.submit_host(None, end_pin, rew_pin, spawn_mode=2)                  # a tic with caller-supplied moves needs them
        with pytest.raises(AszError):
            a.submit_host(acts, end_pin, rew_pin, spawn_mode=1)                  # replayed spawns need the cells
        a.submit_host(acts, end_pin, rew_pin, spawn_mode=2)                      # ... and never waited for
        a.close(); b.close()
    torch.cuda.synchronize()
