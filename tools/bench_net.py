"""Value-network throughput: hand-written tcgen05 path vs PyTorch (cuDNN) bf16/fp32.
python tools/bench_net.py [n [side [chunk]]] [--dtype bf16|fp8|both] [--chunks] [--no-torch]   (or --dtype=...)
--dtype both times the bf16 and the fp8 native networks in alternating rounds and adds their ratio."""
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
    args = sys.argv[1:]
    dt = "bf16"
    for i, a in enumerate(args):                # --dtype=X or --dtype X
        if a.startswith("--dtype="):
            dt = a.split("=", 1)[1]
        elif a == "--dtype" and i + 1 < len(args):
            dt = args[i + 1]
            args[i + 1] = "--"
    if dt not in ("bf16", "fp8", "both"):
        sys.exit("--dtype must be bf16, fp8 or both")
    argv = [a for a in args if not a.startswith("--")]
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
    dtypes = ["bf16", "fp8"] if dt == "both" else [dt]
    for ch in sorted({chunk, 4 * chunk} if "--chunks" in sys.argv else {chunk}):
        nats = {d: NativeNet(w, "cuda", chunk_images=ch, dtype=d) for d in dtypes}
        times = {d: [] for d in dtypes}
        for _ in range(3):                      # alternating rounds: both dtypes see the same clocks and neighbours
            for d in dtypes:
                times[d].append(timeit(lambda: nats[d].forward(x)))
        for d in dtypes:
            t = min(times[d])
            out["native_%s_chunk%d" % (d, ch)] = {"evals_per_s": n / t, "tflops": n / t * FLOPS[side] / 1e12 if FLOPS[side] else None,
                                                 "ms": t * 1e3, "ms_rounds": [r * 1e3 for r in times[d]]}
        if len(dtypes) == 2:
            out["fp8_over_bf16_chunk%d" % ch] = min(times["bf16"]) / min(times["fp8"])
        del nats
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
