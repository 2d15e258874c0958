"""Where does env_step_kernel spend its cycles in the fast and in the slow regime (DESIGN.md 4.1)?
Builds a measurement copy of the library with -DASZ_ENV_PROFILE (phase timers, clock64 per warp) and prints the share of
warp-cycles per phase for: A device path, B encode only, C device path after B.
  python tools/env_profile.py build     (here, no GPU needed)
  ASZ_LIB=tools/libasz_b200_prof.so python tools/env_profile.py run"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROF_LIB = os.path.join(ROOT, "tools", "libasz_b200_prof.so")
sys.path.insert(0, ROOT)
if len(sys.argv) > 1 and sys.argv[1] == "build":
    from alphasnake_zero_b200 import build
    cmd = ["nvcc"] + build.NVCC_FLAGS + ["-DASZ_ENV_PROFILE", "-shared", "-o", PROF_LIB] + \
          [os.path.join(build.CSRC, f) for f in build.SOURCES] + ["-lcuda", "-ldl"]
    subprocess.check_call(cmd)
    print(PROF_LIB)
    sys.exit(0)
os.environ.setdefault("ASZ_LIB", PROF_LIB)
import ctypes as C
import numpy as np, torch
from alphasnake_zero_b200 import _lib
from alphasnake_zero_b200.engine import Engine
G = 65536
eng = Engine(side=11, snakes=4, health_dec=1, games=G, seed=1); eng.reset(); _ = eng.planes
kw = dict(spawn_mode=2, tic=True, encode=True, auto_reset=True, random_actions=True)
kw_enc = dict(tic=False, encode=True)
names = ("record wait", "tic", "write-back", "counter wait+prefetch", "cell view+row wait", "encode", "-", "-")
def phase(name, kw, n=300):
    h = np.zeros(8, np.uint64)
    _lib.check(_lib.lib().asz_internal_profile(eng.h, h.ctypes.data_as(C.c_void_p)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): eng.step(**kw)
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / n * 1000
    _lib.check(_lib.lib().asz_internal_profile(eng.h, h.ctypes.data_as(C.c_void_p)))
    tot = float(h[:6].sum())
    print("%-22s %.1f us/launch | kcycles per game: %s" % (name, us, ", ".join("%s %.2f" % (names[k], h[k] / n / G / 1e3) for k in range(6))))
for _ in range(20): eng.step(**kw)
phase("A tic+encode", kw); phase("A tic+encode", kw)
phase("B encode only", kw_enc)
phase("C tic+encode", kw); phase("C tic+encode", kw)
eng.planes.zero_()
phase("D after zero_", kw); phase("D after zero_", kw)
