"""GPU numerics of the value network: the hand-written tcgen05 kernels against the float64 CPU restatement
(oracle/net_oracle.py; TF itself is not runnable here, see its header) and against the plain PyTorch forward.
Tolerance: 2e-2 absolute on the tanh outputs for the bf16 path, 1e-5 for the fp32 PyTorch path (BASELINE.json)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def game_planes(side, S, n, seed=1):
    from oracle import oracle as orc
    rng = np.random.default_rng(seed)
    X = []
    gid = 0
    while len(X) < n:
        g = orc.OracleGame(side, side, S, 1); g.init_native(seed, gid); gid += 1
        for t in range(30):
            X += g.get_states()
            if g.tic(rng.integers(0, 3, g.n_live).astype(np.int32), spawn_mode=2, seed=seed):
                break
    return np.array(X[:n], np.float32)


@pytest.mark.parametrize("side,S,n,chunk", [(11, 4, 37, 1024), (11, 4, 300, 128), (7, 4, 20, 64), (19, 8, 9, 16)])
def test_native_net_matches_oracle(side, S, n, chunk):
    import torch
    from alphasnake_zero_b200.net import NativeNet
    from oracle import net_oracle as no
    w = no.init_weights(side, seed=5, randomize_bn=True)
    w["dense2_w"] = (w["dense2_w"] * 1.5).astype(np.float32)   # use a good part of the tanh range
    X = game_planes(side, S, n)
    m = min(n, 48)
    want = no.forward(w, X[:m])                     # float64 restatement of the reference network
    want_q = no.forward(w, X[:m], bf16=True)        # same, with the CUDA path's bf16 storage points emulated
    net = NativeNet(w, "cuda", chunk_images=chunk)
    got = net.forward(torch.from_numpy(X).cuda()).cpu().numpy()
    assert np.isfinite(got).all()
    assert np.abs(want).max() > 0.05                # the comparison is not vacuous
    err_q = np.abs(got[:m] - want_q).max()
    assert err_q < 2e-2, err_q                      # (the structural check is test_native_net_layer_by_layer)
    err = np.abs(got[:m] - want).max()
    assert err < 2e-2, err                          # bf16 tolerance of BASELINE.json's north star
    # batch invariance: the same plane gives the same bits wherever it sits in the batch
    perm = np.random.default_rng(0).permutation(n)
    got2 = net.forward(torch.from_numpy(X[perm]).cuda()).cpu().numpy()
    assert np.array_equal(got2.view(np.uint32), got[perm].view(np.uint32))


def test_native_net_vs_torch_bf16_and_alphannet_v():
    import torch
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    from oracle import net_oracle as no
    w = no.init_weights(11, seed=9, randomize_bn=True)
    X = game_planes(11, 4, 64, seed=3)
    a = AlphaNNet(weights=w, backend="native")
    b = AlphaNNet(weights=w, backend="torch", dtype="fp32")
    va, vb = a.v(X), b.v(X)
    assert va.shape == vb.shape == (64, 3) and va.dtype == np.float32
    assert np.array_equal(va == -1.0, vb == -1.0)          # obstacle mask identical
    assert np.abs(va - vb).max() < 2e-2
    assert a._get_native() is not None


@pytest.mark.parametrize("side,S", [(11, 4), (7, 4), (19, 8)])
def test_native_net_layer_by_layer(side, S):
    """every convolution of the tower against the bf16-emulating restatement: errors stay at the 1-2 bf16 ulp level
    (rounding ties decided differently by fp32 and float64 accumulation), a wrong tap / fold / residual would not"""
    import torch
    from alphasnake_zero_b200.net import NativeNet
    from oracle import net_oracle as no
    w = no.init_weights(side, seed=5, randomize_bn=True)
    X = game_planes(side, S, 6)
    want = no.forward_layers(w, X)
    net = NativeNet(w, "cuda", chunk_images=8)
    xs = torch.from_numpy(X).cuda()
    for layer in range(9):
        got = net.debug_layer(xs, layer).cpu().numpy().astype(np.float64)
        ref = want[layer]
        scale = np.abs(ref).max()
        err = np.abs(got - ref).max()
        print("layer %d: max |ref| %.3f, max err %.5f" % (layer, scale, err))
        assert err <= 0.0079 * scale + 1e-3, (layer, err, scale)     # 2 bf16 ulp of the largest activation


@pytest.mark.parametrize("side,S,n,chunk", [(11, 4, 700, 256), (7, 4, 90, 32), (19, 8, 40, 16)])
def test_chunked_forward_bit_identical(side, S, n, chunk):
    """a forward split into several passes of chunk_images gives the same bits as one pass over the whole batch (chunk sizes
    chosen so that several passes and a ragged last pair tile occur)"""
    import torch
    from alphasnake_zero_b200.net import NativeNet
    from oracle import net_oracle as no
    w = no.init_weights(side, seed=11, randomize_bn=True)
    X = torch.from_numpy(game_planes(side, S, n, seed=7)).cuda()
    chunked = NativeNet(w, "cuda", chunk_images=chunk).forward(X).cpu().numpy()
    whole = NativeNet(w, "cuda", chunk_images=n).forward(X).cpu().numpy()
    assert np.isfinite(whole).all() and np.abs(whole).max() > 0.01
    assert np.array_equal(chunked.view(np.uint32), whole.view(np.uint32))


def test_weight_update_equals_a_fresh_network():
    """asz_net_update_weights (the per-generation weight push): after AlphaNNet.set_weights the SAME native network object gives
    bit-identical outputs to a network created from the new weights, and differs from the old ones"""
    import torch
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet, init_weights
    X = torch.from_numpy(game_planes(11, 4, 300, seed=9)).cuda()
    a = AlphaNNet(input_shape=(21, 21, 3), seed=1)
    old = a.v_device(X).clone()
    nat = a._get_native()
    w2 = init_weights((21, 21, 3), seed=2)
    a.set_weights(w2)
    assert a._get_native() is nat                       # same object, new operands
    new = a.v_device(X).clone()
    fresh = AlphaNNet(input_shape=(21, 21, 3), seed=2).v_device(X)
    assert torch.equal(new, fresh) and not torch.equal(new, old)


def test_parallel_collectives_on_nccl():
    """parallel.py over the nccl backend (world size 1 on this box; the 8-GPU bench leg runs the same calls): device tensors
    for every collective, weights pushed into the live native network"""
    import socket
    import torch
    import torch.distributed as dist
    from alphasnake_zero_b200 import parallel
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=0, world_size=1)
    try:
        net = AlphaNNet(input_shape=(21, 21, 3), seed=5)
        net._get_native()
        parallel.broadcast_weights(net, src=0)
        assert parallel.weights_equal_all_ranks(net.weights)
        assert parallel.reduce_counters([4.0, 2.0, 0, 0, 6.0, 20.0], 2, dst=0) == [2.0, 1.0, 0.0, 0.0, 3.0, 10.0]
        planes = torch.rand(50, 21, 21, 3, device="cuda"); values = torch.rand(50, 3, device="cuda")
        X, V, bs = parallel.gather_sampled_batch(50, lambda idx: (planes[idx.cuda()], values[idx.cuda()]), (21, 21, 3), batch_size=16,
                                                 max_batches=2, dst=0)
        assert X.shape == (32, 21, 21, 3) and V.shape == (32, 3) and bs == 16 and X.is_cuda
    finally:
        dist.destroy_process_group()
