"""NativeNet -- host side of the hand-written value-network kernels (csrc/asz_net.cu): folds BatchNorm, lays the
weights out for the tcgen05 implicit GEMM and calls asz_net_forward.  PyTorch only owns the device memory.

dtype="fp8" (opt-in, outside the bf16 network's accuracy: DESIGN.md 4.3) quantizes here: residual convolutions 1..8 get
e4m3 weights with one scale per output channel (amax / 448), and every layer's output a power-of-two scale calibrated on
the bf16 network (act_scales).  Quantization and calibration are pure functions of the weights and the calibration planes,
so every rank that pushes the same weights ends up with the same operands."""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import check

BN_EPS = 1e-3


def _fold(bn):
    s = bn["gamma"].astype(np.float64) / np.sqrt(bn["var"].astype(np.float64) + BN_EPS)
    b = bn["beta"].astype(np.float64) - bn["mean"].astype(np.float64) * s
    return s.astype(np.float32), b.astype(np.float32)


def _conv3x3_layout(k, per=8):
    """HWIO (3,3,128,128) -> [tap][cin/per][cout][cin%per] (per = channels in 16 bytes: 8 bf16, 16 e4m3)"""
    kh, kw, cin, cout = k.shape
    t = k.reshape(kh * kw, cin // per, per, cout)        # [tap][kc][j][cout]
    return np.ascontiguousarray(np.transpose(t, (0, 1, 3, 2)))


def _conv0_layout(k):
    """HWIO (3,3,3,128) -> K = 27 (+5 zero) GEMM operand [1][4][cout][8], k = (dy*3+dx)*3 + c"""
    cout = k.shape[3]
    flat = np.zeros((32, cout), np.float32)
    flat[:27] = k.reshape(27, cout)
    return np.ascontiguousarray(np.transpose(flat.reshape(1, 4, 8, cout), (0, 1, 3, 2)))


CONV_NAMES = ["conv0"] + ["res%d_conv%d" % (b, j) for b in range(4) for j in range(2)]
BN_NAMES = ["bn0"] + ["res%d_bn%d" % (b, j) for b in range(4) for j in range(2)]
E4M3_MAX = 448.0
ACT_TARGET = E4M3_MAX / 4       # calibrated maxima land in (56, 112]: 4x headroom before a stored value saturates


def e4m3(a):
    """float32 array -> (values as float32, codes as uint8) of its e4m3 (fn) rounding: nearest even, clamped to +-448"""
    t = torch.from_numpy(np.clip(np.asarray(a, np.float32), -E4M3_MAX, E4M3_MAX)).to(torch.float8_e4m3fn)
    return t.to(torch.float32).numpy(), t.view(torch.uint8).numpy()


def quantize_fp8(weights, act_scale):
    """the operands of an fp8 network: per convolution i = 1..8 a dict of q (float32 HWIO, the e4m3 weights), codes (uint8,
    the same), w_scale [128] (amax over the output channel's kernel / 448, 1 for an all-zero channel), scale [128] =
    float32(bn_scale * w_scale * act_scale[i-1]) and bias [128] (the float32 BatchNorm fold).  The kernel computes
    acc * scale + bias from the e4m3 products acc = sum q * (stored input), where stored input = input / act_scale[i-1]."""
    out = {}
    for i in range(1, 9):
        k = np.asarray(weights[CONV_NAMES[i]], np.float32)
        amax = np.abs(k).max(axis=(0, 1, 2))
        ws = np.where(amax > 0, amax / np.float32(E4M3_MAX), np.float32(1)).astype(np.float32)
        q, codes = e4m3(k / ws)
        s, b = _fold(weights[BN_NAMES[i]])
        scale = (s.astype(np.float64) * ws.astype(np.float64) * float(act_scale[i - 1])).astype(np.float32)
        out[i] = dict(q=q, codes=codes, w_scale=ws, scale=scale, bias=b)
    return out


def act_scales(amax):
    """per-layer maxima of the bf16 network's outputs -> the fp8 network's act_scale: 2^ceil(log2(amax / 112)), 1 where
    amax is 0, kept in [2^-125, 2^126] (what asz_net_create_fp8 accepts)"""
    out = []
    for a in amax:
        a = float(a)
        if not a > 0:
            out.append(1.0)
            continue
        m, e = math.frexp(a / ACT_TARGET)               # = m * 2^e, m in [0.5, 1): exact for float32 maxima
        out.append(math.ldexp(1.0, min(126, max(-125, e - 1 if m == 0.5 else e))))
    return out


CALIBRATION_GAMES, CALIBRATION_SNAKES, CALIBRATION_TICS, CALIBRATION_SEED = 256, 4, 24, 8675309


def calibration_planes(side, device):
    """The default calibration set: every plane the engine encodes after tics 3, 6, ..., 24 of 256 seeded games of 4 snakes
    played with uniform random moves (native food spawn, finished games reset), in (game, snake) order: about 6,000 planes,
    the same on every device and in every run."""
    from .engine import Engine, SPAWN_NATIVE
    eng = Engine(side=side, snakes=CALIBRATION_SNAKES, games=CALIBRATION_GAMES, seed=CALIBRATION_SEED, device=device)
    try:
        with torch.cuda.device(eng.device):
            eng.reset()
            out = []
            for t in range(1, CALIBRATION_TICS + 1):
                eng.step(spawn_mode=SPAWN_NATIVE, tic=True, encode=True, auto_reset=True, random_actions=True)
                if t % 3 == 0:
                    out.append(eng.rows()[1].contiguous())
            return torch.cat(out)
    finally:
        eng.close()


def calibrate(weights, planes, device, chunk=1024):
    """act_scales of the maxima of every layer's output (asz_net_debug_layer) of the bf16 native network over `planes`"""
    n = planes.shape[0]
    net = NativeNet(weights, device, chunk_images=max(1, min(chunk, n)))
    amax = [0.0] * 9
    for i in range(0, n, chunk):
        for L in range(9):
            amax[L] = max(amax[L], float(net.debug_layer(planes[i:i + chunk], L).abs().max()))
    return act_scales(amax)


class NativeNet:

    def __init__(self, weights, device, chunk_images=16384, dtype="bf16", calibration=None):
        """dtype "bf16" (the reference network) or "fp8"; calibration: device planes [n, N, N, 3] for the fp8 activation
        scales (default: calibration_planes)"""
        if dtype not in ("bf16", "fp8"):
            raise ValueError("NativeNet dtype must be 'bf16' or 'fp8', not %r" % (dtype,))
        if not torch.cuda.is_available():
            raise _lib.AszError("no CUDA device: the native network has no CPU fallback")
        self.device = torch.device(device)
        self.L = _lib.lib()
        self.side = int(weights["side"])
        self.N = 2 * self.side - 1
        self.dtype = dtype
        self.calibration = calibration
        self.act_scale = None
        self._keep, self._nw = self._upload(weights)
        nw = self._nw
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            if dtype == "fp8":
                check(self.L.asz_net_create_fp8(C.byref(h), C.byref(nw), chunk_images))
            else:
                check(self.L.asz_net_create(C.byref(h), C.byref(nw), chunk_images))
        self.h = h

    def _upload(self, weights):
        """device copies of the weights in the layouts the kernels consume -> (tensors kept alive, asz_net_weights)"""
        dev = self.device
        keep = []

        def up(a, dtype):
            t = torch.from_numpy(np.ascontiguousarray(a)).to(dev).to(dtype).contiguous()
            keep.append(t)
            return t.data_ptr()
        nw = _lib.NetWeights()
        nw.side = self.side
        q8 = None
        if self.dtype == "fp8":
            if self.calibration is None:
                self.calibration = calibration_planes(self.side, dev)
            self.act_scale = calibrate(weights, self.calibration, dev)
            q8 = quantize_fp8(weights, self.act_scale)
        for i, (cn, bn) in enumerate(zip(CONV_NAMES, BN_NAMES)):
            if q8 is not None and i > 0:
                nw.w_conv[i] = up(_conv3x3_layout(q8[i]["codes"], 16), torch.uint8)
                nw.scale[i] = up(q8[i]["scale"], torch.float32)
                nw.bias[i] = up(q8[i]["bias"], torch.float32)
                continue
            k = weights[cn].astype(np.float32)
            lay = _conv0_layout(k) if i == 0 else _conv3x3_layout(k)
            nw.w_conv[i] = up(lay, torch.bfloat16)
            s, b = _fold(weights[bn])
            nw.scale[i] = up(s, torch.float32)
            nw.bias[i] = up(b, torch.float32)
        nw.head_w = up(weights["head_conv"].reshape(-1).astype(np.float32), torch.float32)
        hs, hb = _fold(weights["head_bn"])
        nw.head_scale, nw.head_bias = float(hs[0]), float(hb[0])
        nw.dense1_w = up(weights["dense1_w"].astype(np.float32), torch.float32)
        nw.dense1_b = up(weights["dense1_b"].astype(np.float32), torch.float32)
        nw.dense2_w = up(weights["dense2_w"].astype(np.float32), torch.float32)
        nw.dense2_b = up(weights["dense2_b"].astype(np.float32), torch.float32)
        if q8 is not None:
            nw = _lib.NetWeightsFP8(nw, (C.c_float * 9)(*self.act_scale))
        return keep, nw

    def update(self, weights):
        """new weights for the same network object (per-generation weight push): asz_net_update_weights; an fp8 network
        re-quantizes and re-calibrates (on the same calibration planes)"""
        assert int(weights["side"]) == self.side
        keep, nw = self._upload(weights)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        with torch.cuda.device(self.device):
            if self.dtype == "fp8":
                check(self.L.asz_net_update_weights_fp8(self.h, C.byref(nw), st))
            else:
                check(self.L.asz_net_update_weights(self.h, C.byref(nw), st))
            torch.cuda.current_stream(self.device).synchronize()      # the old arrays may be freed once nothing reads them
        self._keep, self._nw = keep, nw

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.L.asz_net_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def forward(self, planes, out=None):
        """planes [n, N, N, 3] float32 cuda (contiguous) -> [n, 3] float32 raw outputs."""
        assert planes.is_cuda and planes.dtype == torch.float32
        n = planes.shape[0]
        pitch = 0
        if n > 1 and not planes.is_contiguous() and tuple(planes.stride()[1:]) == (3 * self.N, 3, 1) and planes.stride(0) >= 3 * self.N * self.N:
            pitch = planes.stride(0)            # rows of an engine plane buffer (32-byte aligned rows): read in place
        else:
            planes = planes.contiguous()
        if out is None:
            out = torch.empty(n, 3, dtype=torch.float32, device=planes.device)
        if n > 0:
            st = C.c_void_p(torch.cuda.current_stream(planes.device).cuda_stream)
            if pitch:
                check(self.L.asz_net_forward_pitched(self.h, C.c_void_p(planes.data_ptr()), pitch, n, C.c_void_p(out.data_ptr()), st))
            else:
                check(self.L.asz_net_forward(self.h, C.c_void_p(planes.data_ptr()), n, C.c_void_p(out.data_ptr()), st))
        return out

    def debug_layer(self, planes, layer):
        """test hook: output of convolution `layer` as float32 [n, N, N, 128] (layer 8: [n, N, N, 1], the head conv).
        fp8: the stored e4m3 values times act_scale[layer] (exact)."""
        planes = planes.contiguous()
        n = planes.shape[0]
        out = torch.empty(n, self.N, self.N, 1 if layer == 8 else 128, dtype=torch.float32, device=planes.device)
        st = C.c_void_p(torch.cuda.current_stream(planes.device).cuda_stream)
        check(self.L.asz_net_debug_layer(self.h, C.c_void_p(planes.data_ptr()), n, layer, C.c_void_p(out.data_ptr()), st))
        return out
