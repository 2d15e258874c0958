"""NativeNet -- host side of the hand-written value-network kernels (csrc/asz_net.cu): folds BatchNorm, lays the
weights out for the tcgen05 implicit GEMM and calls asz_net_forward.  PyTorch only owns the device memory."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check

BN_EPS = 1e-3


def _fold(bn):
    s = bn["gamma"].astype(np.float64) / np.sqrt(bn["var"].astype(np.float64) + BN_EPS)
    b = bn["beta"].astype(np.float64) - bn["mean"].astype(np.float64) * s
    return s.astype(np.float32), b.astype(np.float32)


def _conv3x3_layout(k):
    """HWIO (3,3,128,128) -> [tap][cin/8][cout][cin%8]"""
    kh, kw, cin, cout = k.shape
    t = k.reshape(kh * kw, cin // 8, 8, cout)            # [tap][kc][j][cout]
    return np.ascontiguousarray(np.transpose(t, (0, 1, 3, 2)))


def _conv0_layout(k):
    """HWIO (3,3,3,128) -> K = 27 (+5 zero) GEMM operand [1][4][cout][8], k = (dy*3+dx)*3 + c"""
    cout = k.shape[3]
    flat = np.zeros((32, cout), np.float32)
    flat[:27] = k.reshape(27, cout)
    return np.ascontiguousarray(np.transpose(flat.reshape(1, 4, 8, cout), (0, 1, 3, 2)))


class NativeNet:

    def __init__(self, weights, device, chunk_images=16384):
        if not torch.cuda.is_available():
            raise _lib.AszError("no CUDA device: the native network has no CPU fallback")
        self.device = torch.device(device)
        self.L = _lib.lib()
        self.side = int(weights["side"])
        self.N = 2 * self.side - 1
        self._keep, self._nw = self._upload(weights)
        nw = self._nw
        h = C.c_void_p()
        with torch.cuda.device(self.device):
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
        names = ["conv0"] + ["res%d_conv%d" % (b, j) for b in range(4) for j in range(2)]
        bns = ["bn0"] + ["res%d_bn%d" % (b, j) for b in range(4) for j in range(2)]
        for i, (cn, bn) in enumerate(zip(names, bns)):
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
        return keep, nw

    def update(self, weights):
        """new weights for the same network object (per-generation weight push): asz_net_update_weights"""
        assert int(weights["side"]) == self.side
        keep, nw = self._upload(weights)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        with torch.cuda.device(self.device):
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
        """test hook: output of convolution `layer` as float32 [n, N, N, 128] (layer 8: [n, N, N, 1], the head conv)."""
        planes = planes.contiguous()
        n = planes.shape[0]
        out = torch.empty(n, self.N, self.N, 1 if layer == 8 else 128, dtype=torch.float32, device=planes.device)
        st = C.c_void_p(torch.cuda.current_stream(planes.device).cuda_stream)
        check(self.L.asz_net_debug_layer(self.h, C.c_void_p(planes.data_ptr()), n, layer, C.c_void_p(out.data_ptr()), st))
        return out
