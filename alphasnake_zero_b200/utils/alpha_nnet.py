"""AlphaNNet -- mirror of code/utils/alpha_nnet.py:8-109 (value network holder).

On the hot path only `v` matters (alpha_nnet.py:61-76): batched forward + obstacle mask.  The forward runs either
through the hand-written sm_100a kernels of libasz_b200.so (backend "native", the default: implicit-GEMM convolutions on
tcgen05 tensor cores, bf16 operands, fp32 accumulation; it raises when the library or a GPU is missing) or, only when asked
for by name, through plain PyTorch ops (backend "torch": the library baseline and fp32 reference of the numerics tests).  Weights are kept in the Keras layouts the reference's .h5 files use
(conv kernels HWIO, dense (in, out), BN gamma/beta/moving_mean/moving_variance).
dtype="fp8" selects the native fp8 (e4m3) tower instead (net.py; opt-in: its values are outside the bf16 network's 2e-2
accuracy, DESIGN.md 4.3); it has no PyTorch path.
"""
import numpy as np
import torch
import torch.nn.functional as F

K = 128
BN_EPS = 1e-3   # Keras BatchNormalization default epsilon


def _glorot(rng, shape, fan_in, fan_out):
    lim = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def init_weights(input_shape, seed=None):
    """Keras defaults of alpha_nnet.py:19-56: glorot-uniform kernels, zero biases, BN (1, 0, 0, 1)."""
    rng = np.random.default_rng(seed)
    n = int(input_shape[0])

    def bn(c):
        return dict(gamma=np.ones(c, np.float32), beta=np.zeros(c, np.float32), mean=np.zeros(c, np.float32),
                    var=np.ones(c, np.float32))
    w = {"side": (n + 1) // 2}
    w["conv0"] = _glorot(rng, (3, 3, 3, K), 27, 9 * K); w["bn0"] = bn(K)
    for b in range(4):
        for j in range(2):
            w["res%d_conv%d" % (b, j)] = _glorot(rng, (3, 3, K, K), 9 * K, 9 * K)
            w["res%d_bn%d" % (b, j)] = bn(K)
    w["head_conv"] = _glorot(rng, (1, 1, K, 1), K, 1); w["head_bn"] = bn(1)
    w["dense1_w"] = _glorot(rng, (n * n, K), n * n, K); w["dense1_b"] = np.zeros(K, np.float32)
    w["dense2_w"] = _glorot(rng, (K, 3), K, 3); w["dense2_b"] = np.zeros(3, np.float32)
    return w


def flatten_weights(w):
    """Keras get_weights() order: per layer kernel, (bias), gamma, beta, moving_mean, moving_variance."""
    out = []
    def bn(p):
        out.extend([p["gamma"], p["beta"], p["mean"], p["var"]])
    out.append(w["conv0"]); bn(w["bn0"])
    for b in range(4):
        for j in range(2):
            out.append(w["res%d_conv%d" % (b, j)]); bn(w["res%d_bn%d" % (b, j)])
    out.append(w["head_conv"]); bn(w["head_bn"])
    out.extend([w["dense1_w"], w["dense1_b"], w["dense2_w"], w["dense2_b"]])
    return out


class _VNet:
    """stand-in for the Keras Model attribute `v_net` (summary / get_weights / set_weights), test_weights.py:5-7."""

    def __init__(self, owner):
        self._o = owner

    def get_weights(self):
        return [np.array(a) for a in flatten_weights(self._o.weights)]

    def summary(self):
        tot = sum(a.size for a in self.get_weights())
        print("AlphaNNet value network: conv3x3(3->128) + 4 residual blocks + conv1x1 + dense(128) + dense(3); "
              "%d parameters and buffers" % tot)

    def predict(self, X):
        return self._o._forward_host(X)


class AlphaNNet:

    def __init__(self, model_name=None, input_shape=None, device=None, backend="auto", dtype="bf16", seed=None,
                 weights=None, calibration=None):
        """calibration: device planes [n, N, N, 3] on which dtype="fp8" calibrates its activation scales (default: the
        seeded set of net.calibration_planes)"""
        if dtype == "fp8" and backend == "torch":
            raise ValueError("dtype='fp8' runs on the native backend only: there is no PyTorch fp8 path")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.backend = backend
        self.dtype = dtype
        self.calibration = calibration
        self.weights = None
        self._torch = None
        self._native = None
        self.lr = 1e-4
        if weights is not None:
            self.weights = weights
        elif model_name:
            self.weights = load_weights(model_name)            # alpha_nnet.py:11-12
        elif input_shape:
            self.weights = init_weights(input_shape, seed)     # alpha_nnet.py:13-56
        self.v_net = _VNet(self)

    # ---- forward paths -----------------------------------------------------------------------------------------
    def _torch_params(self):
        if self._torch is None:
            w, dev = self.weights, self.device
            t = {}
            def conv(k):   # HWIO -> OIHW
                return torch.from_numpy(np.ascontiguousarray(np.transpose(k, (3, 2, 0, 1)))).to(dev)
            def bn(p):
                s = p["gamma"] / np.sqrt(p["var"] + BN_EPS)
                return torch.from_numpy(s.astype(np.float32)).to(dev), torch.from_numpy((p["beta"] - p["mean"] * s).astype(np.float32)).to(dev)
            t["conv0"] = conv(w["conv0"]); t["bn0"] = bn(w["bn0"])
            for b in range(4):
                for j in range(2):
                    t["res%d_conv%d" % (b, j)] = conv(w["res%d_conv%d" % (b, j)]); t["res%d_bn%d" % (b, j)] = bn(w["res%d_bn%d" % (b, j)])
            t["head_conv"] = conv(w["head_conv"]); t["head_bn"] = bn(w["head_bn"])
            for k in ("dense1_w", "dense1_b", "dense2_w", "dense2_b"):
                t[k] = torch.from_numpy(w[k]).to(dev)
            self._torch = t
        return self._torch

    def forward_torch(self, planes, dtype=torch.float32):
        """Plain PyTorch forward (library path): planes [n, N, N, 3] float32 cuda -> [n, 3] float32 raw outputs."""
        t = self._torch_params()
        x = planes.permute(0, 3, 1, 2).to(dtype).contiguous(memory_format=torch.channels_last)
        def cbr(x, ck, bk, res=None):
            y = F.conv2d(x, t[ck].to(dtype), padding=t[ck].shape[-1] // 2)
            s, b = t[bk]
            y = y * s.to(dtype).view(1, -1, 1, 1) + b.to(dtype).view(1, -1, 1, 1)
            if res is not None:
                y = y + res
            return F.relu(y)
        h = cbr(x, "conv0", "bn0")
        for b in range(4):
            sc = h
            h = cbr(h, "res%d_conv0" % b, "res%d_bn0" % b)
            h = cbr(h, "res%d_conv1" % b, "res%d_bn1" % b, sc)
        h = cbr(h, "head_conv", "head_bn")
        h = h.reshape(h.shape[0], -1).float()
        h = F.relu(h @ t["dense1_w"] + t["dense1_b"])
        return torch.tanh(h @ t["dense2_w"] + t["dense2_b"])

    def v_device(self, planes):
        """raw network outputs for device planes (no obstacle mask): the engine's value_fn.
        "native" (and "auto", its alias) is the product path: the hand-written kernels or an exception, never a silent
        library fallback.  "torch" is the explicit PyTorch/cuDNN path used as numerics reference and library baseline."""
        if self.backend == "torch":
            return self.forward_torch(planes, torch.bfloat16 if self.dtype == "bf16" else torch.float32)
        return self._get_native().forward(planes)

    def _get_native(self):
        if self._native is None:
            from ..net import NativeNet          # raises if libasz_b200.so is missing: no fallback
            self._native = NativeNet(self.weights, self.device, dtype="fp8" if self.dtype == "fp8" else "bf16",
                                     calibration=self.calibration)
        return self._native

    def set_weights(self, weights):
        """replace the weight dictionary and refresh every device copy `v` uses (the native network's operands through
        asz_net_update_weights, re-quantized and re-calibrated for fp8; the PyTorch parameters by rebuilding them): the
        per-generation weight push"""
        self.weights = weights
        self._torch = None
        if self._native is not None:
            self._native.update(weights)

    def _forward_host(self, X):
        X = np.ascontiguousarray(np.array(X, dtype=np.float32))
        out = []
        for i in range(0, len(X), 4096):
            out.append(self.v_device(torch.from_numpy(X[i:i + 4096]).to(self.device)).float().cpu().numpy())
        return np.concatenate(out) if out else np.zeros((0, 3), np.float32)

    # ---- reference surface -------------------------------------------------------------------------------------
    def v(self, X):
        """alpha_nnet.py:61-76: predict + obstacle mask; X list/array of NHWC planes (or a cuda tensor)."""
        if torch.is_tensor(X):
            Xh = X.detach().float().cpu().numpy()
        else:
            Xh = np.ascontiguousarray(np.array(X, dtype=np.float32))
        V = self._forward_host(Xh)
        cy, cx = Xh.shape[1] // 2, Xh.shape[2] // 2
        thr = np.float32(0.04)                      # NumPy >= 2 semantics (SURVEY.md D-11)
        V[Xh[:, cy, cx - 1, 1] >= thr, 0] = -1.0    # alpha_nnet.py:67-72
        V[Xh[:, cy - 1, cx, 1] >= thr, 1] = -1.0
        V[Xh[:, cy, cx + 1, 1] >= thr, 2] = -1.0
        return V

    def is_obstacle(self, value):
        return value >= 0.04

    def copy_and_compile(self, learning_rate=0.0001, TPU=None):
        """alpha_nnet.py:78-106: a copy with a fresh optimizer state (piecewise-constant LR x0.25 every 20 steps)."""
        import copy
        c = AlphaNNet(device=self.device, backend=self.backend, dtype=self.dtype, weights=copy.deepcopy(self.weights),
                      calibration=self.calibration)
        c.lr = learning_rate
        return c

    def train(self, X, Y, epochs=32, batch_size=2048):
        """alpha_nnet.py:58-59 (outside the self-play hot path; SURVEY.md 8(f) #1)."""
        from ..training import fit
        self.weights = fit(self, X, Y, epochs, batch_size, self.lr)
        self._torch = None
        self._native = None

    def save(self, name):
        """alpha_nnet.py:108-109: models/<name>.h5 in the layout of tf.keras 2.2.4's Model.save (written by the pure-NumPy HDF5 subset
        of utils/h5lite.py: no h5py needed), plus the same Keras-ordered weight list as models/<name>.npz (SURVEY.md 8(f) #3)."""
        import os
        from . import keras_h5
        os.makedirs("models", exist_ok=True)
        keras_h5.save(self.weights, "models/" + name + ".h5")
        np.savez("models/" + name + ".npz", side=self.weights["side"], *flatten_weights(self.weights))


def load_weights(path):
    """alpha_nnet.py:11-12: `model_name` is a path; a Keras .h5 model file (what the reference's train.py passes:
    "models/<name><generation>.h5"), an .npz written by save(), or a path without extension (.npz first, then .h5)."""
    import os
    if path.endswith(".h5") or (not path.endswith(".npz") and not os.path.exists(path + ".npz") and os.path.exists(path + ".h5")):
        from . import keras_h5
        return keras_h5.load(path if path.endswith(".h5") else path + ".h5")
    z = np.load(path if path.endswith(".npz") else path + ".npz")
    arrs = [z["arr_%d" % i] for i in range(len(z.files) - 1)]
    side = int(z["side"])
    w = {"side": side}
    it = iter(arrs)
    def bn():
        return dict(gamma=next(it), beta=next(it), mean=next(it), var=next(it))
    w["conv0"] = next(it); w["bn0"] = bn()
    for b in range(4):
        for j in range(2):
            w["res%d_conv%d" % (b, j)] = next(it); w["res%d_bn%d" % (b, j)] = bn()
    w["head_conv"] = next(it); w["head_bn"] = bn()
    w["dense1_w"] = next(it); w["dense1_b"] = next(it); w["dense2_w"] = next(it); w["dense2_b"] = next(it)
    return w
