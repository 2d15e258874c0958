"""Value-network throughput: hand-written tcgen05 path vs PyTorch (cuDNN) bf16/fp32.  python tools/bench_net.py [n]"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from alphasnake_zero_b200.utils.alpha_nnet import AlphaNNet, init_weights  # noqa: E402
from alphasnake_zero_b200.net import NativeNet  # noqa: E402

FLOPS = {7: None, 11: 1043724288, 19: 3240040448}


def main():
    argv = [a for a in sys.argv[1:] if not a.startswith("--")]
    n = int(argv[0]) if len(argv) > 0 else 16384
    side = int(argv[1]) if len(argv) > 1 else 11
    chunk = int(argv[2]) if len(argv) > 2 else 4096
    N = 2 * side - 1
    w = init_weights((N, N, 3), seed=0)
    x = torch.rand(n, N, N, 3, device="cuda") * 0.5
    out = {}
    tnet = AlphaNNet(weights=w, backend="torch")

    def timeit(fn, reps=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3
    for ch in sorted({chunk, 4 * chunk} if "--chunks" in sys.argv else {chunk}):
        nat = NativeNet(w, "cuda", chunk_images=ch)
        t = timeit(lambda: nat.forward(x))
        out["native_bf16_chunk%d" % ch] = {"evals_per_s": n / t, "tflops": n / t * FLOPS[side] / 1e12 if FLOPS[side] else None,
                                           "ms": t * 1e3}
        del nat
    if "--no-torch" in sys.argv:
        print(json.dumps({"n": n, "side": side, "chunk": chunk, **out}))
        return
    with torch.no_grad():
        for name, dt in (("torch_bf16", torch.bfloat16), ("torch_fp32", torch.float32)):
            bs = 4096
            t = timeit(lambda: [tnet.forward_torch(x[i:i + bs], dt) for i in range(0, n, bs)], reps=3)
            out[name] = {"evals_per_s": n / t, "tflops": n / t * FLOPS[side] / 1e12 if FLOPS[side] else None, "ms": t * 1e3}
    print(json.dumps({"n": n, "side": side, "chunk": chunk, **out}))


if __name__ == "__main__":
    main()
