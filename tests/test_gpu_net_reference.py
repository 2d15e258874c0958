"""Value network, element by element: every convolution of the tower and the dense head of the tcgen05 kernels
(csrc/asz_net.cu) against a float64 reference of the same operation, at the batch sizes production runs.

Each layer is isolated: the reference of layer L is computed from the kernel's own exported output of layer L-1 (exact
bf16 values) and, for the second convolution of a residual block, the kernel's own block input as the residual.  So
errors do not compound, and every element is held to a bound derived from the arithmetic the kernel does (bf16
operands, fp32 accumulation, fp32 epilogue, bf16 store), not to a tolerance fitted to what it happens to produce.

With z = sum a*w in float64, S = sum |a|*|w| (the same convolution over absolute values), the folded BatchNorm scale s
and bias b (the fp32 operands of NativeNet) and the residual r:
    f = s*z + b (+ r),  ref = max(f, 0),
    |got - ref| <= ulp_bf16(max(|got|, |ref|)) + |s|*GAMMA*S + 2^-22*(|s*z| + |b| + |r|)
where GAMMA = 2^-16 covers fp32 accumulation over the 144 MMA steps of a layer ((144 + 16) * 2^-24 ~ 2^-16.7).
The head convolution (layer 8) and the fp32 dense head propagate these bounds through their own fp32 sums (head_terms,
dense_reference).

The GPU shapes reach what only production batches use: 20+ super-tiles per CTA pair (both TMEM accumulator pairs, both
parities of their barriers, the A halves refilled, resident weights reused, every starting stage of the 17-stage weight
ring at 19x19), ragged last tiles, and at 19x19 the chunk_images=16384 of AlphaNNet, whose activation operands lie past
4 GB.  The CPU test rehearses the checker against oracle/net_oracle.py and shows that it is not vacuous."""
import numpy as np
import pytest

GAMMA = 2.0 ** -16      # fp32 accumulation over <= 160 steps (tensor-core K steps, the 128-term head sum)
FP32 = 2.0 ** -22       # fp32 epilogue: two roundings of (s*z + b) + r, with a factor 2 to spare
U32 = 2.0 ** -24        # unit roundoff of fp32 (the dense head's probabilistic bound)
LAMBDA = 8.0            # its confidence: Hoeffding, 2 exp(-LAMBDA^2 / 2) = 3e-14 per output
SLICE = 512             # images per slice of the float64 reference (bounds its memory)

CASES = [   # side, snakes, images, chunk_images
    (7, 4, 4093, 4096),       # 21-22 super-tiles per pair, ragged last tile; resident weights
    (11, 4, 4001, 4096),      # 51-52 super-tiles per pair, ragged last tile; resident weights
    (19, 8, 1021, 16384),     # 38-39 super-tiles per pair: every start stage of the 17-stage ring; operands past 4 GB
]


# ---- float64 reference and bounds (device agnostic: the CPU test runs them on the oracle) ---------------------------------

def bf16_rne(t):
    """float tensor -> float64 holding its round-to-nearest-even bf16 value (what torch's bf16 cast and NativeNet do)"""
    import torch
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def ulp_bf16(x):
    """one bf16 ulp at |x| (0 at 0): 2^(floor(log2 |x|) - 7)"""
    import torch
    x = x.abs()
    _, e = torch.frexp(x)
    return torch.where(x > 0, torch.ldexp(torch.ones_like(x), e - 8), torch.zeros_like(x))


def conv_operands(w, layer, device, exact=False):
    """(W [128, cin, 3, 3] float64, s [128], b [128]) of convolution `layer` (0..8) as the kernel consumes them: bf16
    weights, the fp32 BatchNorm fold of NativeNet.  exact=True: unrounded weights and a float64 fold (the oracle's
    arithmetic)."""
    import torch
    from alphasnake_zero_b200 import net
    names = ["conv0"] + ["res%d_conv%d" % (b, j) for b in range(4) for j in range(2)]
    bns = ["bn0"] + ["res%d_bn%d" % (b, j) for b in range(4) for j in range(2)]
    k = torch.from_numpy(np.asarray(w[names[layer]], np.float32)).permute(3, 2, 0, 1).contiguous()   # HWIO -> OIHW
    W = k.to(torch.float64) if exact else bf16_rne(k)
    if exact:
        p = {q: w[bns[layer]][q].astype(np.float64) for q in ("gamma", "beta", "mean", "var")}
        s = p["gamma"] / np.sqrt(p["var"] + net.BN_EPS)
        b = p["beta"] - p["mean"] * s
    else:
        s, b = net._fold(w[bns[layer]])
    f64 = lambda a: torch.as_tensor(np.asarray(a, np.float64), device=device)
    return W.to(device), f64(s), f64(b)


def conv_terms(a, ops, r=None):
    """a [n, cin, N, N] float64 (the layer's input), r [n, 128, N, N] or None -> (f, e): f = s*conv(a) + b (+ r) in float64
    and e = the bound on |fp32 f - f| (accumulation + epilogue)"""
    import torch.nn.functional as F
    W, s, b = ops
    z = F.conv2d(a, W, padding=1)
    S = F.conv2d(a.abs(), W.abs(), padding=1)
    s4, b4 = s.view(1, -1, 1, 1), b.view(1, -1, 1, 1)
    sz = s4 * z
    f = sz + b4
    mag = sz.abs() + b4.abs()
    if r is not None:
        f = f + r
        mag = mag + r.abs()
    return f, s4.abs() * GAMMA * S + FP32 * mag


def layer_excess(got, f, e):
    """per-element |got - ref| and its bound for a stored bf16 layer output"""
    import torch
    ref = f.clamp_min(0)
    err = (got - ref).abs()
    return err, ulp_bf16(torch.maximum(got.abs(), ref)) + e


def head_terms(f, e, head_w, head_scale, head_bias):
    """layer 8: hq_c = bf16(relu(f_c)) stays inside the kernel, then head = relu(hs * sum_c hw_c * hq_c + hb) in fp32.
    f, e [n, 128, N, N] -> (ref [n, 1, N, N], bound)"""
    hq = f.clamp_min(0)
    d = e + ulp_bf16(hq + e)                                             # |bf16(relu(fp32 f)) - relu(f)|
    hw = head_w.view(1, -1, 1, 1).abs()
    acc = (hq * head_w.view(1, -1, 1, 1)).sum(1, keepdim=True)
    pre = head_scale * acc + head_bias
    bound = abs(head_scale) * ((hw * d).sum(1, keepdim=True) + GAMMA * (hw * (hq + d)).sum(1, keepdim=True)) \
        + FP32 * ((head_scale * acc).abs() + abs(head_bias))
    return pre.clamp_min(0), bound


def head_operands(w, device, exact=False):
    import torch
    from alphasnake_zero_b200 import net
    hw = torch.as_tensor(np.asarray(w["head_conv"], np.float32).reshape(-1).astype(np.float64), device=device)
    if exact:
        p = {q: w["head_bn"][q].astype(np.float64) for q in ("gamma", "beta", "mean", "var")}
        hs = p["gamma"] / np.sqrt(p["var"] + net.BN_EPS)
        hb = p["beta"] - p["mean"] * hs
    else:
        hs, hb = net._fold(w["head_bn"])
    return hw, float(hs[0]), float(hb[0])


def dense_reference(head, w):
    """head [n, N, N] float64 (the kernel's layer-8 activations) -> (ref [n, 3], bound [n, 3]) of Dense(128) + ReLU +
    Dense(3) + tanh.

    dense_head_kernel sums dense1 as four fp32 fma chains over quarters of the padded raster (raster order, zero terms at
    the padding), adds them to the bias in order q = 0..3, then runs dense2 as one fp32 fma chain from the bias.  Step k of
    a chain rounds by delta_k with |delta_k| <= u |s_k| (s_k its partial sum, u = 2^-24), and to first order an output
    moves by c_k delta_k, where c_k = |w2[unit, out]| for a step of a hidden unit (ReLU is 1-Lipschitz) and 1 for a step of
    dense2.  The worst case, u * sum_k c_k |s_k|, comes to ~2e-3 at 19x19: it assumes all ~185,000 roundings of an output
    line up, and it could not tell a tanh.approx.f32 (~5e-4) from tanhf.  The bound used is the probabilistic one of
    Higham & Mary (SIAM J. Sci. Comput. 41(5), 2019): with independent, mean-zero roundings, Hoeffding's inequality gives
    |sum_k c_k delta_k| <= LAMBDA * u * sqrt(sum_k c_k^2 s_k^2) except with probability 2 exp(-LAMBDA^2 / 2) = 3e-14 per
    output.  tanhf adds at most 2 ulp."""
    import torch
    dev = head.device
    n, N = head.shape[0], head.shape[1]
    side = (N + 1) // 2
    pitch = 2 * side
    stride = pitch * pitch
    f64 = lambda a: torch.as_tensor(np.asarray(a, np.float32).astype(np.float64), device=dev)
    w1, b1, w2, b2 = f64(w["dense1_w"]), f64(w["dense1_b"]), f64(w["dense2_w"]), f64(w["dense2_b"])
    hr = torch.zeros(n, pitch, pitch, dtype=torch.float64, device=dev)
    hr[:, :N, :N] = head
    hr = hr.reshape(n, stride)
    w1r = torch.zeros(pitch, pitch, 128, dtype=torch.float64, device=dev)
    w1r[:N, :N] = w1.view(N, N, 128)
    w1r = w1r.reshape(stride, 128)
    qlen = (stride + 3) // 4
    v = b1.expand(n, 128)
    var = torch.zeros(n, 128, dtype=torch.float64, device=dev)         # sum of s_k^2 over the roundings of a hidden unit
    for q in range(4):
        seg = slice(q * qlen, min(stride, (q + 1) * qlen))
        cs = (hr[:, seg, None] * w1r[None, seg, :]).cumsum(1)            # [n, len, 128] partial sums of the chain
        v = v + cs[:, -1]
        var = var + cs.square().sum(1) + v.square()                      # the chain, then its addition to v
    hid = v.clamp_min(0)
    cs2 = b2 + (hid[:, :, None] * w2[None]).cumsum(1)                   # [n, 128, 3]
    o = cs2[:, -1]
    var_o = (var[:, :, None] * w2.square()[None]).sum(1) + cs2.square().sum(1)
    t = torch.tanh(o)
    return t, LAMBDA * U32 * var_o.sqrt() + 2 * U32 * t.abs()


# ---- inputs -------------------------------------------------------------------------------------------------------------

def fuzz_planes(side, n, seed):
    """n planes that are no game position: full-mantissa uniform values in [-1.5, 1.5], exact round-to-nearest-even ties
    of bf16 (halfway between two bf16 neighbours, e.g. 1 + 2^-8 and -(1 + 3 * 2^-8)), an all-zero and an all -1 plane"""
    rng = np.random.default_rng(seed)
    N = 2 * side - 1
    nu = (n - 2) // 2
    nt = n - 2 - nu
    uni = rng.uniform(-1.5, 1.5, (nu, N, N, 3)).astype(np.float32)
    m = rng.integers(0, 128, (nt, N, N, 3))
    ex = rng.integers(-3, 1, (nt, N, N, 3))
    sg = rng.choice([-1.0, 1.0], (nt, N, N, 3))
    ties = (sg * ((128 + m) * 2.0 ** (ex - 7) + 2.0 ** (ex - 8))).astype(np.float32)
    ties[0, 0, 0, :2] = [1 + 2 ** -8, -(1 + 3 * 2 ** -8)]
    return np.concatenate([np.zeros((1, N, N, 3), np.float32), uni, ties, -np.ones((1, N, N, 3), np.float32)])


def mixed_planes(side, S, n, seed=1):
    """game planes (test_gpu_net.game_planes) with a quarter of fuzz planes spread among them; the last plane is all -1,
    so the ragged last tile holds large values at the border"""
    from tests.test_gpu_net import game_planes
    nf = max(4, n // 4)
    X = np.concatenate([game_planes(side, S, n - nf, seed=seed), fuzz_planes(side, nf, seed)])
    X = X[np.random.default_rng(seed).permutation(n)]
    last = int(np.flatnonzero((X == -1).all(axis=(1, 2, 3)))[0])
    X[[last, n - 1]] = X[[n - 1, last]]
    return np.ascontiguousarray(X)


def wide_weights(side):
    """init_weights(seed=5, randomize_bn=True) with dense2 scaled so that the outputs use a good part of the tanh range"""
    from oracle import net_oracle as no
    w = no.init_weights(side, seed=5, randomize_bn=True)
    w["dense2_w"] = (w["dense2_w"] * 1.5).astype(np.float32)
    return w


# ---- the checker ----------------------------------------------------------------------------------------------------------

def _nchw(t):
    """[n, N, N, C] -> float64 [n, C, N, N]"""
    return t.permute(0, 3, 1, 2).double()


def check_tower(layers, X, w, device, exact=False):
    """layers(L) -> the exported output of layer L [n, N, N, 128] (L = 8: [n, N, N, 1]); X the input planes.
    -> (per layer a dict: violations, worst err/bound, nonzero mask per position [n, N, N], nonzero fraction;
        the layer-8 head activations [n, N, N] float64)"""
    import torch
    planes = torch.as_tensor(X, device=device)
    n = planes.shape[0]
    hw, hs, hb = head_operands(w, device, exact)
    out, report, keep = [], [], {}
    for L in range(9):
        got_all = layers(L)
        keep[L] = got_all
        keep.pop(L - 3, None)                                   # only L-1 and L-2 are inputs of later layers
        ops = conv_operands(w, L, device, exact)
        viol, worst, nz = 0, 0.0, []
        for i in range(0, n, SLICE):
            sl = slice(i, i + SLICE)
            a = (planes[sl].to(torch.float64) if exact else bf16_rne(planes[sl])).permute(0, 3, 1, 2) if L == 0 else _nchw(keep[L - 1][sl])
            r = _nchw(keep[L - 2][sl]) if L >= 2 and L % 2 == 0 else None
            f, e = conv_terms(a, ops, r)
            got = _nchw(got_all[sl])
            if L < 8:
                err, bound = layer_excess(got, f, e)
            else:
                ref, bound = head_terms(f, e, hw, hs, hb)
                err = (got - ref).abs()
            bad = err > bound
            viol += int(bad.sum())
            ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0))
            worst = max(worst, float(ratio.max()))
            nz.append((got != 0).any(1))
        report.append(dict(layer=L, violations=viol, worst=worst, nonzero=torch.cat(nz),
                           frac=float((got_all != 0).double().mean())))
    return report, keep[8][..., 0].to(torch.float64)


def check_dense(head, values, w):
    """head [n, N, N] float64 (layer 8 of the kernel), values [n, 3] (forward of the kernel) -> (violations, worst ratio, max bound)"""
    import torch
    viol, worst, bmax = 0, 0.0, 0.0
    for i in range(0, head.shape[0], SLICE):
        ref, bound = dense_reference(head[i:i + SLICE], w)
        err = (values[i:i + SLICE].to(torch.float64) - ref).abs()
        viol += int((err > bound).sum())
        worst = max(worst, float((err / bound).max()))
        bmax = max(bmax, float(bound.max()))
    return viol, worst, bmax


# ---- CPU rehearsal against the oracle ------------------------------------------------------------------------------------

def _oracle_case():
    from oracle import net_oracle as no
    from tests.test_gpu_net import game_planes
    w = wide_weights(7)
    X = game_planes(7, 4, 2, seed=1)
    return no, w, X


def _as_layers(outs):
    import torch
    return lambda L: torch.as_tensor(np.asarray(outs[L], np.float64)).to(torch.float32)


def _violations(report):
    return [r["violations"] for r in report]


def test_checker_against_the_oracle_on_cpu():
    """the helpers restate the oracle's float64 arithmetic; the oracle's own bf16 emulation passes the checker, and a 2-ulp
    error, two swapped taps of one weight or inputs truncated instead of rounded to bf16 are all reported"""
    import torch
    no, w, X = _oracle_case()
    # 1. before rounding: the helpers restate net_oracle to 1e-12 (relative to each layer's largest activation)
    exact = no.forward_layers(w, X, bf16=False)
    planes = torch.as_tensor(X).to(torch.float64).permute(0, 3, 1, 2)
    hw, hs, hb = head_operands(w, "cpu", exact=True)
    for L in range(9):
        a = planes if L == 0 else torch.as_tensor(exact[L - 1]).permute(0, 3, 1, 2)
        r = torch.as_tensor(exact[L - 2]).permute(0, 3, 1, 2) if L >= 2 and L % 2 == 0 else None
        f, _ = conv_terms(a, conv_operands(w, L, "cpu", exact=True), r)
        ref = head_terms(f, torch.zeros_like(f), hw, hs, hb)[0] if L == 8 else f.clamp_min(0)
        want = torch.as_tensor(exact[L]).permute(0, 3, 1, 2)
        assert float((ref - want).abs().max()) <= 1e-12 * float(want.abs().max()), L
    head = torch.as_tensor(exact[8][..., 0])
    dense, _ = dense_reference(head, w)
    want = no.forward(w, X)
    assert np.abs(dense.numpy() - want).max() <= 1e-12 * np.abs(want).max()
    assert np.abs(want).max() > 0.05

    # 2. the oracle's bf16 emulation (bf16 planes, weights and layer outputs; float64 sums) as "kernel output": no violation
    outs = no.forward_layers(w, X, bf16=True)
    report, head_q = check_tower(_as_layers(outs), X, w, "cpu")
    print("oracle as kernel, worst err/bound per layer:", ["%.3f" % r["worst"] for r in report])
    assert _violations(report) == [0] * 9
    for r in report:
        assert r["frac"] > 0.05, r["layer"]
    v, worst, bmax = check_dense(head_q, torch.as_tensor(no.forward(w, X, bf16=True)), w)
    print("dense: worst err/bound %.3g, largest bound %.3g" % (worst, bmax))
    assert v == 0 and bmax < 1e-4

    # 3a. one element off by 2 bf16 ulp (the largest output of the first layer and of a middle one)
    for L in (0, 3):
        bad = [o.copy() for o in outs]
        idx = np.unravel_index(np.argmax(bad[L]), bad[L].shape)
        bad[L][idx] += 2 * float(ulp_bf16(torch.tensor(bad[L][idx], dtype=torch.float64)))
        report, _ = check_tower(_as_layers(bad), X, w, "cpu")
        assert report[L]["violations"] >= 1, L
        assert all(r["violations"] == 0 for r in report[:L])
    # 3b. two taps of one weight swapped (one input / output channel pair of one convolution)
    ws = {k: (v if not isinstance(v, np.ndarray) else v.copy()) for k, v in w.items()}
    k = ws["res1_conv1"]
    k[0, 1, 5, 9], k[1, 0, 5, 9] = k[1, 0, 5, 9], k[0, 1, 5, 9]
    report, _ = check_tower(_as_layers(no.forward_layers(ws, X, bf16=True)), X, w, "cpu")
    assert report[4]["violations"] >= 1 and all(r["violations"] == 0 for r in report[:4])
    # 3c. planes truncated to bf16 (toward zero) instead of rounded to nearest even
    Xt = (X.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32)
    report, _ = check_tower(_as_layers(no.forward_layers(w, Xt, bf16=True)), X, w, "cpu")
    assert report[0]["violations"] >= 1
    # 3d. the dense head with tanh off by a relative 2^-11 (the size of tanh.approx.f32's error)
    vals = torch.as_tensor(no.forward(w, X, bf16=True))
    v, _, _ = check_dense(head_q, vals * (1 + 2.0 ** -11), w)
    assert v >= 1


# ---- on the B200 -----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def case():
    """side -> the network of CASES with its inputs, per-layer report, head activations and forward values (built once)"""
    import torch
    built = {}

    def get(side):
        if side not in built:
            side_, S, n, chunk = next(c for c in CASES if c[0] == side)
            w = wide_weights(side)
            X = torch.from_numpy(mixed_planes(side, S, n)).cuda()
            net = NativeNet(w, "cuda", chunk_images=chunk)
            report, head = check_tower(lambda L: net.debug_layer(X, L), X, w, X.device)
            built[side] = dict(w=w, X=X, n=n, chunk=chunk, net=net, report=report, head=head, values=net.forward(X).clone())
        return built[side]
    yield get
    built.clear()
    torch.cuda.empty_cache()


def NativeNet(*a, **k):
    from alphasnake_zero_b200.net import NativeNet as cls
    return cls(*a, **k)


@pytest.mark.gpu
@pytest.mark.parametrize("side", [c[0] for c in CASES])
def test_every_layer_within_its_bound_at_production_shapes(case, side):
    """all 9 convolutions, every element, at 20-52 super-tiles per CTA pair; and the comparison is not vacuous: every layer
    has many nonzero outputs, at the border too, and in every super-tile that a pair runs after its second"""
    import torch
    c = case(side)
    N, pitch = 2 * side - 1, 2 * side
    n_tiles = (c["n"] * pitch * pitch + 511) // 512
    pairs = min(n_tiles, torch.cuda.get_device_properties(0).multi_processor_count // 2)
    assert n_tiles >= 20 * pairs                                   # well past the first two super-tiles of every pair
    img, y, x = torch.meshgrid(*(torch.arange(k, device=c["X"].device) for k in (c["n"], N, N)), indexing="ij")
    tile = (img * pitch * pitch + y * pitch + x) // 512
    print("side %d, %d images, %d super-tiles over %d pairs: worst err/bound per layer %s" % (
        side, c["n"], n_tiles, pairs, " ".join("%.3f" % r["worst"] for r in c["report"])))
    for r in c["report"]:
        nz = r["nonzero"]
        assert r["violations"] == 0, (r["layer"], r["violations"], r["worst"])
        assert r["frac"] > 0.25, r
        assert nz[:, 0].any() and nz[:, -1].any() and nz[:, :, 0].any() and nz[:, :, -1].any(), r["layer"]
        per_tile = torch.bincount(tile[nz], minlength=n_tiles)
        assert bool((per_tile[2 * pairs:] > 0).all()), r["layer"]


@pytest.mark.gpu
@pytest.mark.parametrize("side", [c[0] for c in CASES])
def test_dense_head_within_its_bound(case, side):
    """forward() against Dense(128) + ReLU + Dense(3) + tanh in float64 of the kernel's own layer-8 activations"""
    import torch
    c = case(side)
    v, worst, bmax = check_dense(c["head"], c["values"], c["w"])
    print("side %d: dense head worst err/bound %.3f, largest bound %.3g" % (side, worst, bmax))
    assert v == 0, (v, worst)
    assert bmax < 1e-4 and float(c["values"].abs().max()) > 0.5 and bool(torch.isfinite(c["values"]).all())


@pytest.mark.gpu
@pytest.mark.parametrize("side,n,dense2", [(11, 1023, 1.5), (19, 15, 1.5), (7, 1, 1.5), (11, 1023, 0.25), (11, 1023, 0.05)])
def test_dense_head_ragged_groups_and_unsaturated_tanh(side, n, dense2):
    """8 images per CTA of dense_head_kernel: counts of 8k+7 and a single image leave the last group ragged.  dense2 scaled
    down keeps the outputs in tanh's steep range (|t| ~ 0.3 and ~ 0.07), where an approximate tanh would show"""
    import torch
    from oracle import net_oracle as no
    S = 8 if side == 19 else 4
    w = no.init_weights(side, seed=5, randomize_bn=True)
    w["dense2_w"] = (w["dense2_w"] * dense2).astype(np.float32)
    X = torch.from_numpy(mixed_planes(side, S, max(n, 16), seed=3)[-n:]).cuda()
    net = NativeNet(w, "cuda", chunk_images=n)
    head = net.debug_layer(X, 8)[..., 0].double()
    v, worst, bmax = check_dense(head, net.forward(X), w)
    print("side %d, %d images, dense2 x %g: dense head worst err/bound %.3f, largest bound %.3g" % (side, n, dense2, worst, bmax))
    assert v == 0, (v, worst)


def _bits(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("pitch", [1328, 1361])
def test_pitched_input_with_nan_padding(case, pitch):
    """planes read in place from rows `pitch` floats apart (1,328 = the engine's 32-byte row pitch at 11x11, and an odd
    pitch), with NaN in the floats between rows: the same bits as the contiguous forward"""
    import torch
    c = case(11)
    n, N = c["n"], 21
    flat = torch.full((n * pitch,), float("nan"), device=c["X"].device)
    view = flat.as_strided((n, N, N, 3), (pitch, 3 * N, 3, 1))
    view.copy_(c["X"])
    got = c["net"].forward(view)
    assert bool(torch.isfinite(got).all())
    assert np.array_equal(_bits(got), _bits(c["values"]))


@pytest.mark.gpu
def test_balanced_passes_equal_one_pass(case):
    """4,001 images through chunk_images=1000: 5 passes of 801 / 797 images give the bits of the one-pass forward (which
    test_dense_head_within_its_bound checks against the reference)"""
    c = case(11)
    got = NativeNet(c["w"], "cuda", chunk_images=1000).forward(c["X"])
    assert np.array_equal(_bits(got), _bits(c["values"]))


@pytest.mark.gpu
def test_reused_network_equals_fresh_ones(case):
    """one object through forward(4001), forward(37), debug_layer(6 images) and forward(1): each result has the bits of a
    fresh object's, so nothing left in the activation buffers past the last tile of a smaller call leaks into it"""
    import torch
    c = case(11)
    X, w = c["X"], c["w"]
    a = NativeNet(w, "cuda", chunk_images=c["chunk"])
    fresh = lambda: NativeNet(w, "cuda", chunk_images=c["chunk"])
    assert np.array_equal(_bits(a.forward(X)), _bits(c["values"]))
    small = X[-37:]
    assert np.array_equal(_bits(a.forward(small)), _bits(fresh().forward(small)))
    for L in (0, 7, 8):
        assert np.array_equal(_bits(a.debug_layer(X[:6], L)), _bits(fresh().debug_layer(X[:6], L))), L
    one = a.forward(X[-1:])
    assert np.array_equal(_bits(one), _bits(c["values"][-1:]))
    assert np.array_equal(_bits(one), _bits(fresh().forward(X[-1:])))
    del a
    torch.cuda.empty_cache()
