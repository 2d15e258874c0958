"""The fp8 (e4m3) value network (NativeNet(dtype="fp8"), AlphaNNet(dtype="fp8")), element by element, at the shapes of
test_gpu_net_reference.py.

An fp8 network stores every layer's output as e4m3 codes c = e4m3(y / act_scale[L]) (round to nearest even, saturating
at +-448) and runs convolutions 1..8 on them with e4m3 weights q (net.quantize_fp8).  Each layer is isolated as in the
bf16 test: the float64 reference of layer L starts from the kernel's own exported layer L-1 (debug_layer: c * act_scale,
exact) and, for the second convolution of a block, its own block input:
    f = s' * sum (a / act_scale[L-1]) * q + b (+ r),   y = max(f, 0) / act_scale[L]
with s' the fp32 folded scale of quantize_fp8 (it includes the weight and input scales).  The products of two e4m3 values
are exact in fp32, so the bf16 test's accumulation and epilogue bound e applies unchanged (GAMMA = 2^-16 covers 72 K = 32
MMAs plus the 32 products inside one: (72 + 32) * 2^-24 < 2^-16).  Rounding is monotonic, so the stored code must lie
between the codes of (f - e) and (f + e):
    e4m3(max(f - e, 0) / act_scale) <= c <= e4m3(max(f + e, 0) / act_scale)
These two are the same code except when f lies within e of a rounding midpoint; the tests count how often that happens.
If kind::f8f6f4 accumulated with less than fp32 precision, codes next to midpoints would fall outside this interval, and
the printed worst distance (in units of e) would grow past 1.

The per-layer reference takes its operands from net.quantize_fp8, the code that makes the kernel's; a CPU test holds
those operands against a float64 quantizer written apart from it (independent_quantization).  The CPU tests also check the
e4m3 rounding of these helpers against torch.float8_e4m3fn, the purity of the quantization and calibration arithmetic, and
that the checker is not vacuous."""
import numpy as np
import pytest

from tests.test_gpu_net_reference import (CASES, SLICE, _bits, _nchw, bf16_rne, check_dense, conv_operands, conv_terms,
                                          head_operands, head_terms, mixed_planes, wide_weights)

E4M3_MAX = 448.0


# ---- e4m3 arithmetic and the fp8 reference (device agnostic) --------------------------------------------------------------

def e4m3_rne(x):
    """float64 tensor -> float64 holding its e4m3 (fn) value: nearest even, 3 mantissa bits, subnormals below 2^-6 in steps
    of 2^-9, saturating at +-448 (cvt.rn.satfinite.e4m3x2.f32)"""
    import torch
    _, e = torch.frexp(x.abs())                                       # |x| = m 2^e, m in [0.5, 1)
    quantum = torch.ldexp(torch.ones_like(x), torch.clamp(e - 1, min=-6) - 3)
    return (torch.round(x / quantum) * quantum).clamp(-E4M3_MAX, E4M3_MAX)    # torch.round: half to even


def fp8_operands(q8, layer, device):
    """(W [128, 128, 3, 3] float64 of the e4m3 weights, s' [128], b [128]) of convolution `layer` (1..8)"""
    import torch
    W = torch.from_numpy(q8[layer]["q"]).permute(3, 2, 0, 1).to(torch.float64).contiguous()
    f64 = lambda a: torch.as_tensor(np.asarray(a, np.float64), device=device)
    return W.to(device), f64(q8[layer]["scale"]), f64(q8[layer]["bias"])


def layer_terms(L, a_prev, r, w, q8, act, device, planes=None):
    """(f, e) of layer L from the dequantized layer L-1 (or the planes for L = 0) and residual r"""
    if L == 0:
        return conv_terms(bf16_rne(planes).permute(0, 3, 1, 2), conv_operands(w, 0, device), None)
    return conv_terms(a_prev / act[L - 1], fp8_operands(q8, L, device), r)


def code_interval(f, e, scale):
    """codes (as values) the kernel may store for f +- e"""
    return e4m3_rne((f - e).clamp_min(0) / scale), e4m3_rne((f + e).clamp_min(0) / scale)


def emulate(w, X, act, device="cpu"):
    """the fp8 tower in float64 (no fp32 rounding): dequantized outputs of layers 0..7 [n, N, N, 128] and the head [n, N, N, 1]"""
    import torch
    from alphasnake_zero_b200 import net
    q8 = net.quantize_fp8(w, act)
    hw, hs, hb = head_operands(w, device)
    planes = torch.as_tensor(X, device=device)
    outs = []
    for L in range(9):
        a = _nchw(outs[L - 1]) if L else None
        r = _nchw(outs[L - 2]) if L >= 2 and L % 2 == 0 else None
        f, _ = layer_terms(L, a, r, w, q8, act, device, planes)
        if L == 8:
            o = head_terms(f, torch.zeros_like(f), hw, hs, hb)[0]
        else:
            o = e4m3_rne(f.clamp_min(0) / act[L]) * act[L]
        outs.append(o.permute(0, 2, 3, 1).contiguous())
    return outs


def check_tower_fp8(layers, X, w, act, device):
    """layers(L) -> the kernel's exported output of layer L.  -> (per layer a dict: violations, near-midpoint elements,
    saturated elements, worst: for the codes that are not the nearest-even one, the largest distance of the value from the
    midpoint they straddle, in units of e (at most 1 unless there is a violation); the layer-8 head float64)"""
    import torch
    from alphasnake_zero_b200 import net
    q8 = net.quantize_fp8(w, act)
    planes = torch.as_tensor(X, device=device)
    n = planes.shape[0]
    hw, hs, hb = head_operands(w, device)
    report, keep = [], {}
    for L in range(9):
        got_all = layers(L)
        keep[L] = got_all
        keep.pop(L - 3, None)
        viol = near = flips = sat = 0
        worst = 0.0
        finite = bool(torch.isfinite(got_all).all())
        for i in range(0, n, SLICE):
            sl = slice(i, i + SLICE)
            a = _nchw(keep[L - 1][sl]) if L else None
            r = _nchw(keep[L - 2][sl]) if L >= 2 and L % 2 == 0 else None
            f, e = layer_terms(L, a, r, w, q8, act, device, planes[sl])
            got = _nchw(got_all[sl])
            if L < 8:
                c = got / act[L]
                lo, hi = code_interval(f, e, act[L])
                bad = (c < lo) | (c > hi)
                near += int((lo != hi).sum())
                sat += int((c == E4M3_MAX).sum())
                mid = e4m3_rne(f.clamp_min(0) / act[L])             # the nearest-even code of the float64 value
                dist = (f.clamp_min(0) / act[L] - (c + mid) / 2).abs() * act[L] / e.clamp_min(1e-300)
                worst = max(worst, float(torch.where(c != mid, dist, torch.zeros_like(dist)).max()))
                flips += int((c != mid).sum())
            else:
                ref, bound = head_terms(f, e, hw, hs, hb)
                err = (got - ref).abs()
                bad = err > bound
                worst = max(worst, float((err / bound.clamp_min(1e-300)).max()))
            viol += int(bad.sum())
        report.append(dict(layer=L, violations=viol, near=near, flips=flips, saturated=sat, worst=worst, finite=finite,
                           frac=float((got_all != 0).double().mean()), size=got_all.numel()))
    return report, keep[8][..., 0].to(torch.float64)


def independent_quantization(w, act):
    """float64 restatement of the fp8 operands, apart from net.quantize_fp8: per layer 1..8 the weight scale amax / 448
    over each output channel's kernel (1 for an all-zero channel), the weights divided by it and rounded with e4m3_rne, the
    BatchNorm fold gamma / sqrt(var + 1e-3), beta - mean * that, and scale' = fold * weight scale * act[layer - 1]
    -> {layer: (q HWIO, x = the unrounded k / w_scale, scale', bias)} in float64"""
    import torch
    out = {}
    for L in range(1, 9):
        name = "res%d_conv%d" % ((L - 1) // 2, (L - 1) % 2)
        bn = w["res%d_bn%d" % ((L - 1) // 2, (L - 1) % 2)]
        k = np.asarray(w[name], np.float64)
        amax = np.abs(k).reshape(-1, k.shape[3]).max(0)
        ws = np.where(amax > 0, amax / 448.0, 1.0)
        x = k / ws
        q = e4m3_rne(torch.from_numpy(x)).numpy()
        g, be, mu, var = (np.asarray(bn[t], np.float64) for t in ("gamma", "beta", "mean", "var"))
        fold = g / np.sqrt(var + 1e-3)
        out[L] = (q, x, fold * ws * act[L - 1], be - mu * fold)
    return out


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_quantizer_against_an_independent_restatement_on_cpu():
    """net.quantize_fp8, which makes the kernel's operands, against independent_quantization: the same e4m3 weight in every
    position except where k / w_scale lies within float32 rounding of a midpoint (net divides in float32; counted), scale'
    and bias to float32 rounding.  A fold without the weight scale, without act_scale or with act_scale[i] instead of
    act_scale[i-1] would not pass."""
    import torch
    from alphasnake_zero_b200 import net
    w = wide_weights(11)
    act = [2.0 ** -k for k in (7, 7, 6, 6, 6, 5, 5, 5, 5)]
    mine = net.quantize_fp8(w, act)
    ref = independent_quantization(w, act)
    ties = total = 0
    for L in range(1, 9):
        q, x, sc, b = ref[L]
        got = mine[L]["q"].astype(np.float64)
        diff = got != q
        # the float32 quotient may round across a midpoint: only there may the codes differ, and by one step
        mids = (e4m3_rne(torch.from_numpy(x * (1 - 2.0 ** -22))).numpy() != e4m3_rne(torch.from_numpy(x * (1 + 2.0 ** -22))).numpy())
        assert not (diff & ~mids).any(), L
        ties += int(diff.sum())
        total += q.size
        assert np.abs(q).reshape(-1, 128).max(0).min() == 448.0
        np.testing.assert_allclose(mine[L]["scale"], sc, rtol=2.0 ** -22, atol=0)
        np.testing.assert_allclose(mine[L]["bias"], b, rtol=2.0 ** -21, atol=2.0 ** -30)
    print("weights rounded across a midpoint by the float32 quotient: %d of %d" % (ties, total))
    assert ties <= 1e-4 * total
    # the checks above are not vacuous: each of these mistakes is visible in them
    for bad in (dict(act=[1.0] * 9), dict(act=act[1:] + [1.0])):
        other = net.quantize_fp8(w, bad["act"])
        assert any(not np.allclose(other[L]["scale"], ref[L][2], rtol=2.0 ** -22, atol=0) for L in range(1, 9))
    no_ws = ref[1][2] / (np.abs(np.asarray(w["res0_conv0"], np.float64)).reshape(-1, 128).max(0) / 448.0)
    assert not np.allclose(mine[1]["scale"], no_ws, rtol=2.0 ** -22, atol=0)


def test_e4m3_rounding_against_torch_on_cpu():
    """every finite e4m3 value, every midpoint between neighbours (and one float32 ulp either side of it), and values past
    the range: e4m3_rne and net.e4m3 agree with torch.float8_e4m3fn (which has no saturation: it gets the clamped value)"""
    import torch
    from alphasnake_zero_b200 import net
    codes = torch.arange(256, dtype=torch.int32).to(torch.uint8).view(torch.float8_e4m3fn).to(torch.float32)
    vals = np.unique(codes[torch.isfinite(codes)].numpy())
    assert vals.size == 253 and vals.max() == 448 and vals[vals > 0].min() == 2.0 ** -9
    mids = ((vals[1:].astype(np.float64) + vals[:-1]) / 2).astype(np.float32)
    assert np.array_equal(mids.astype(np.float64), (vals[1:].astype(np.float64) + vals[:-1]) / 2)   # exact in float32
    x = np.concatenate([vals, mids, np.nextafter(mids, np.float32(np.inf)), np.nextafter(mids, np.float32(-np.inf)),
                        np.float32([449, 463.9, 464, 465, 479, 480, 1e4, 3e38, -449, -464, -480, -1e4, -3e38])]).astype(np.float32)
    want = torch.from_numpy(np.clip(x, -E4M3_MAX, E4M3_MAX)).to(torch.float8_e4m3fn).to(torch.float64).numpy()
    got = e4m3_rne(torch.from_numpy(x).to(torch.float64)).numpy()
    assert np.array_equal(got, want)
    assert np.array_equal(net.e4m3(x)[0].astype(np.float64), want)
    assert np.abs(got[-13:]).max() == E4M3_MAX                      # saturation
    ties = np.isin(x, mids)
    assert ties.sum() >= 250                                         # half of them round down, half up (to the even code)


def test_quantization_and_calibration_are_pure_functions_on_cpu():
    """act_scales maps maxima to powers of two with the maximum in (56, 112] of the stored range, quantize_fp8 gives the same
    operands for the same inputs and leaves its inputs alone; the extreme weight of every output channel is +-448"""
    import copy
    from alphasnake_zero_b200 import net
    amax = [112.0, np.nextafter(np.float32(112), np.float32(200)), 56.0, 0.0, 3.1e-3, 7e5, 1.0, 2.0 ** -140, 111.9]
    s = net.act_scales(amax)
    assert s[:4] == [1.0, 2.0, 0.5, 1.0] and s[7] == 2.0 ** -125
    for a, k in zip(amax, s):
        m, _ = np.frexp(k)
        assert m == 0.5 and (a == 0 or a < 2.0 ** -120 or 56 < a / k <= 112), (a, k)
    assert net.act_scales(amax) == s
    w = wide_weights(7)
    w0 = copy.deepcopy(w)
    a = net.quantize_fp8(w, s)
    b = net.quantize_fp8(w, s)
    for L in range(1, 9):
        for k in ("codes", "scale", "bias", "w_scale"):
            assert np.array_equal(a[L][k], b[L][k]), (L, k)
        assert np.abs(a[L]["q"]).max(axis=(0, 1, 2)).min() == E4M3_MAX
        assert np.array_equal(a[L]["q"].view(np.uint32),
                              np.asarray(net.e4m3(a[L]["q"])[0]).view(np.uint32))     # already e4m3 values
    for k, v in w0.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, w[k]), k
        elif isinstance(v, dict):
            assert all(np.array_equal(v[q], w[k][q]) for q in v), k
    # act_scale[L-1] enters the folded scale of layer L, nothing else
    s2 = list(s)
    s2[2] *= 4
    c = net.quantize_fp8(w, s2)
    assert np.array_equal(c[3]["scale"], (a[3]["scale"].astype(np.float64) * 4).astype(np.float32))
    assert all(np.array_equal(c[L]["scale"], a[L]["scale"]) for L in range(1, 9) if L != 3)


def test_fp8_checker_rejects_a_perturbed_layer_on_cpu():
    """the float64 emulation passes the checker; one code moved up by an e4m3 step and two swapped weight taps are
    reported"""
    import torch
    from tests.test_gpu_net import game_planes
    from alphasnake_zero_b200 import net
    from oracle import net_oracle as no
    w = wide_weights(7)
    X = game_planes(7, 4, 2, seed=1)
    act = net.act_scales([np.abs(o).max() for o in no.forward_layers(w, X, bf16=True)])
    outs = emulate(w, X, act)
    lay = lambda o: (lambda L: o[L].to(torch.float32))
    report, _ = check_tower_fp8(lay(outs), X, w, act, "cpu")
    print("emulation as kernel:", [(r["violations"], r["near"], "%.2f" % r["worst"]) for r in report])
    assert [r["violations"] for r in report] == [0] * 9
    assert all(r["frac"] > 0.05 for r in report)
    for L in (0, 5):
        bad = [o.clone() for o in outs]
        flat = bad[L].view(-1)
        i = int(torch.nonzero((flat >= act[L]) & (flat < 400 * act[L]))[0, 0])
        flat[i] = float(e4m3_rne(torch.tensor(float(flat[i]) / act[L] * 1.13, dtype=torch.float64))) * act[L]   # a code up
        report, _ = check_tower_fp8(lay(bad), X, w, act, "cpu")
        assert report[L]["violations"] >= 1 and all(r["violations"] == 0 for r in report[:L]), L
    ws = {k: (v if not isinstance(v, np.ndarray) else v.copy()) for k, v in w.items()}
    k = ws["res1_conv1"]
    k[0, 1, 5, 9], k[1, 0, 5, 9] = k[1, 0, 5, 9], k[0, 1, 5, 9]
    report, _ = check_tower_fp8(lay(emulate(ws, X, act)), X, w, act, "cpu")
    assert report[4]["violations"] >= 1 and all(r["violations"] == 0 for r in report[:4])


def test_torch_backend_refuses_fp8_on_cpu():
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    with pytest.raises(ValueError):
        AlphaNNet(input_shape=(21, 21, 3), seed=1, backend="torch", dtype="fp8", device="cpu")


# ---- on the B200 -------------------------------------------------------------------------------------------------------------

def NativeNet(*a, **k):
    from alphasnake_zero_b200.net import NativeNet as cls
    return cls(*a, **k)


@pytest.fixture(scope="module")
def case():
    """side -> the fp8 network of CASES (default calibration) with its inputs, per-layer report, head and values"""
    import torch
    built = {}

    def get(side):
        if side not in built:
            side_, S, n, chunk = next(c for c in CASES if c[0] == side)
            if side == 19:
                chunk *= 2                  # e4m3 rows are half as wide: 32,768 images put the operands past 4 GB again
            w = wide_weights(side)
            X = torch.from_numpy(mixed_planes(side, S, n)).cuda()
            net = NativeNet(w, "cuda", chunk_images=chunk, dtype="fp8")
            report, head = check_tower_fp8(lambda L: net.debug_layer(X, L), X, w, net.act_scale, X.device)
            built[side] = dict(w=w, X=X, n=n, chunk=chunk, net=net, report=report, head=head, values=net.forward(X).clone())
        return built[side]
    yield get
    built.clear()
    torch.cuda.empty_cache()


def _print_report(tag, report):
    print(tag, "codes per layer: violations / within e of a midpoint / not the nearest-even code / saturated:",
          " ".join("%d/%.1e/%.1e/%d" % (r["violations"], r["near"] / r["size"], r["flips"] / r["size"], r["saturated"]) for r in report[:8]),
          "| worst |c - rne| in units of e: %s | head worst err/bound %.3f" % (
              " ".join("%.2f" % r["worst"] for r in report[:8]), report[8]["worst"]))


@pytest.mark.gpu
@pytest.mark.parametrize("side", [c[0] for c in CASES])
def test_every_fp8_layer_is_the_nearest_code(case, side):
    """every stored e4m3 code of the 9 convolutions is the nearest-even code of the float64 value, except where that value
    lies within the fp32 bound of a midpoint (counted); the head conv within its fp32 bound; nothing vacuous"""
    c = case(side)
    print("side %d, act_scale %s" % (side, c["net"].act_scale))
    _print_report("side %d:" % side, c["report"])
    for r in c["report"]:
        assert r["violations"] == 0, r
        assert r["finite"] and r["frac"] > 0.25, r
        assert r["near"] <= 5e-2 * r["size"] and r["flips"] <= r["near"], r


@pytest.mark.gpu
@pytest.mark.parametrize("side", [c[0] for c in CASES])
def test_fp8_dense_head_within_its_bound(case, side):
    import torch
    c = case(side)
    v, worst, bmax = check_dense(c["head"], c["values"], c["w"])
    print("side %d: fp8 dense head worst err/bound %.3f, largest bound %.3g" % (side, worst, bmax))
    assert v == 0 and bmax < 1e-4 and bool(torch.isfinite(c["values"]).all())


@pytest.mark.gpu
def test_fp8_end_to_end_against_the_emulation_and_float64(case):
    """A sanity check, not a derived bound: forward() of 64 planes against the float64 fp8 emulation and against float64
    (the bf16 network's error printed beside).  The per-layer test is the exact check: every code is the nearest-even code
    of its own layer's float64 value except the rare ones next to a midpoint.  But one code a step off moves the inputs of
    the next layer's codes, and with 3 mantissa bits some of those cross a midpoint too, so end to end the two towers drift
    apart by a cascade of such steps that no per-layer bound limits.  The test asks only that the drift stays well below
    fp8's own error against float64 (a tenth of its mean, half of its max)."""
    import torch
    from oracle import net_oracle as no
    c = case(11)
    X, w, act = c["X"][:64], c["w"], c["net"].act_scale
    outs = [o.cpu() for o in emulate(w, X, act, X.device)]
    from tests.test_gpu_net_reference import dense_reference
    emu, _ = dense_reference(outs[8][..., 0], w)
    got = c["values"][:64].cpu().double()
    exact = torch.from_numpy(no.forward(w, X.cpu().numpy()))
    bf = NativeNet(w, "cuda", chunk_images=64).forward(X).cpu().double()
    d_emu, d_64, d_bf = (got - emu).abs(), (got - exact).abs(), (bf - exact).abs()
    print("fp8 vs its emulation: max %.2e mean %.2e | fp8 vs float64: max %.3f mean %.4f | bf16 vs float64: max %.4f mean %.5f" % (
        d_emu.max(), d_emu.mean(), d_64.max(), d_64.mean(), d_bf.max(), d_bf.mean()))
    assert float(d_emu.mean()) < 0.1 * float(d_64.mean()) and float(d_emu.max()) < 0.5 * float(d_64.max())
    assert 0.005 < float(d_64.mean()) < 0.1 and float(d_64.max()) < 0.5


@pytest.mark.gpu
def test_fp8_saturation():
    """calibrated on half of a batch, then run on that batch times 16: activations run past 448 * act_scale, they are stored
    as 448, the checker (whose rounding saturates) still passes every element, and no NaN or inf appears"""
    import torch
    side, S, n = 11, 4, 1021
    w = wide_weights(side)
    X = torch.from_numpy(mixed_planes(side, S, n, seed=4)).cuda()
    net = NativeNet(w, "cuda", chunk_images=n, dtype="fp8", calibration=X[: n // 2].clone())
    X = X * 16
    report, head = check_tower_fp8(lambda L: net.debug_layer(X, L), X, w, net.act_scale, X.device)
    _print_report("saturation:", report)
    assert [r["violations"] for r in report] == [0] * 9
    assert all(r["finite"] for r in report)
    assert report[0]["saturated"] > 0 and sum(r["saturated"] for r in report[:8]) > 1000
    v = net.forward(X)
    assert bool(torch.isfinite(v).all())


@pytest.mark.gpu
def test_fp8_invariances(case):
    """bit-identical: a plane wherever it sits in the batch, pitched input with NaN padding, balanced passes against one
    pass, and two calibrations of the same weights"""
    import torch
    c = case(11)
    X, n, w = c["X"], c["n"], c["w"]
    perm = torch.from_numpy(np.random.default_rng(0).permutation(n)).cuda()
    assert np.array_equal(_bits(c["net"].forward(X[perm])), _bits(c["values"][perm]))
    for pitch in (1328, 1361):
        flat = torch.full((n * pitch,), float("nan"), device=X.device)
        view = flat.as_strided((n, 21, 21, 3), (pitch, 63, 3, 1))
        view.copy_(X)
        assert np.array_equal(_bits(c["net"].forward(view)), _bits(c["values"])), pitch
    again = NativeNet(w, "cuda", chunk_images=1000, dtype="fp8")
    assert again.act_scale == c["net"].act_scale
    assert np.array_equal(_bits(again.forward(X)), _bits(c["values"]))


@pytest.mark.gpu
def test_fp8_update_equals_a_fresh_network_and_abi_errors():
    """AlphaNNet(dtype="fp8").set_weights re-quantizes and re-calibrates the same native object: the bits of a fresh fp8
    network.  Updating with the other precision's weights, or with an act_scale that is not a power of two, is refused."""
    import ctypes as C
    import torch
    from alphasnake_zero_b200 import _lib
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet, init_weights
    from tests.test_gpu_net import game_planes
    X = torch.from_numpy(game_planes(11, 4, 300, seed=9)).cuda()
    a = AlphaNNet(input_shape=(21, 21, 3), seed=1, dtype="fp8")
    old = a.v_device(X).clone()
    nat = a._get_native()
    assert nat.dtype == "fp8"
    a.set_weights(init_weights((21, 21, 3), seed=2))
    assert a._get_native() is nat
    new = a.v_device(X).clone()
    fresh = AlphaNNet(input_shape=(21, 21, 3), seed=2, dtype="fp8")
    assert torch.equal(new, fresh.v_device(X)) and not torch.equal(new, old)
    assert fresh._get_native().act_scale == nat.act_scale
    bf = AlphaNNet(input_shape=(21, 21, 3), seed=2)._get_native()
    L = _lib.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert L.asz_net_update_weights(nat.h, C.byref(nat._nw.w), st) == _lib.ASZ_ERR_ARG
    assert L.asz_net_update_weights_fp8(bf.h, C.byref(nat._nw), st) == _lib.ASZ_ERR_ARG
    for bad in (3.0, 0.0, -1.0, float("inf"), float("nan"), 2.0 ** -130):
        nw = _lib.NetWeightsFP8(nat._nw.w, (C.c_float * 9)(*([1.0] * 8 + [bad])))
        assert L.asz_net_update_weights_fp8(nat.h, C.byref(nw), st) == _lib.ASZ_ERR_ARG, bad
        h = C.c_void_p()
        assert L.asz_net_create_fp8(C.byref(h), C.byref(nw), 16) == _lib.ASZ_ERR_ARG, bad
    assert torch.equal(a.v_device(X), new)                   # the refused calls changed nothing


@pytest.mark.gpu
def test_fp8_search_against_oracle_agent():
    """a root-turn search on the device with an fp8 network (asz_search_run_net) against the oracle agent whose value function
    calls the same network (AlphaNNet.v): same table keys and visit counts, Q within float reassociation"""
    import torch
    from alphasnake_zero_b200.engine import Engine
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    from oracle import oracle as orc
    net = AlphaNNet(input_shape=(21, 21, 3), seed=4, dtype="fp8")
    net.weights["dense2_w"] = (net.weights["dense2_w"] * 5).astype(np.float32)
    nat = net._get_native()
    G, S, D, B, seed = 6, 4, 8, 16, 31
    eng = Engine(side=11, snakes=S, games=G, seed=seed, max_depth=D, max_breadth=B, softmax_base=2.0, training=True, table_log2=18)
    eng.reset()
    info = eng.search_info()
    games = []
    for gi in range(G):
        g = orc.OracleGame(11, 11, S, 1); g.init_native(seed, gi, 0); g.set_ids(gi, 0); games.append(g)
    agent = orc.OracleAgent(base=2.0, training=True, max_depth=D, max_breadth=B, value_fn=net.v)
    for t in range(2):
        tree = torch.full((info["epochs"], info["max_steps"], G * info["P"], S), 255, dtype=torch.uint8, device="cuda")
        q, mv = eng.search(net=nat, trace=tree, trace_mode=2)
        mvh = mv.cpu().numpy()
        ids = [(gi, s) for gi in range(G) for s in games[gi].live_ids()]
        root = np.array([mvh[g, s] for g, s in ids], np.uint8)
        omv, oq = agent.make_moves(games, G, root_turn=t, tree_moves=np.ascontiguousarray(tree.cpu().numpy()), root_moves=root.copy(), replay=True)
        tab, otab = eng.table(), agent.table()
        oo = np.lexsort((otab["keys"][:, 1], otab["keys"][:, 0]))
        assert np.array_equal(tab["keys"], otab["keys"][oo]) and np.array_equal(tab["N"], otab["N"][oo])
        np.testing.assert_allclose(tab["W"], otab["W"][oo], rtol=0, atol=2e-4)
        got_q = np.array([q.cpu().numpy()[g, s] for g, s in ids])
        np.testing.assert_allclose(got_q, oq, rtol=0, atol=2e-5)
        assert np.abs(oq[oq > -1]).max() > 0.01
        actions = np.ones((G, 8), np.uint8)
        for (g, s), m in zip(ids, root):
            actions[g, s] = m
        eng.step(actions=torch.from_numpy(actions).cuda(), spawn_mode=2, tic=True, encode=False)
        r0 = 0
        for gi in range(G):
            n = games[gi].n_live
            games[gi].tic(root[r0:r0 + n].astype(np.int32), spawn_mode=2, chance=0.15, seed=seed)
            r0 += n
    eng.close()


@pytest.mark.gpu
def test_fp8_side_against_bf16_side_arena_equals_loop():
    """a search agent on an fp8 network against one on a bf16 network: the arena and the Python loop play the same match"""
    from alphasnake_zero_b200.utils.agent import Agent
    from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet
    from alphasnake_zero_b200.utils.pit_mp_game_runner import MPGameRunner
    from tests.helpers import assert_dump_equal
    nets = [AlphaNNet(input_shape=(21, 21, 3), seed=1, dtype="fp8"), AlphaNNet(input_shape=(21, 21, 3), seed=2)]
    agent = lambda nn: Agent(nn, softmax_base=2.0, training=False, max_MCTS_depth=4, max_MCTS_breadth=8)
    out = []
    for native in (None, False):
        gr = MPGameRunner(11, 11, 2, 3, 64, seed=9)
        log = []
        w = gr.run(agent(nets[0]), agent(nets[1]), 1, move_log=log, native=native)
        out.append((gr, w, log))
    (ga, wa, la), (gl, wl, ll) = out
    assert ga.engine.pit_stats()["turns"] == len(la) > 0 and gl.engine.pit_stats()["turns"] == 0
    assert wa == wl and len(la) == len(ll)
    for t, (a, b) in enumerate(zip(la, ll)):
        assert np.array_equal(a, b), "moves differ in turn %d" % t
    for gi in range(64):
        assert_dump_equal(ga.engine.get_state(gi), gl.engine.get_state(gi), "game %d" % gi)
