#!/usr/bin/env python
"""Warp-time by kind of chunk, and the share of the face chunks spent in seismometer collection (face_collect).
usage: chunk_clocks.py <config> <deg> <n>   (R3D_TIMING=1 makes r3d_kernel_times print the clocks of the
libr3dgpu_clocks.so build, make -C radiative3d_b200/csrc clocks; the model comes from radiative3d_b200/workload_model.py)"""
import os, sys
os.environ["R3D_TIMING"] = "1"
_clk = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "radiative3d_b200", "libr3dgpu_clocks.so")
if os.path.exists(_clk):
    os.environ.setdefault("R3D_LIBRARY", _clk)
else:
    print("chunk_clocks.py: libr3dgpu_clocks.so not built (make -C radiative3d_b200/csrc clocks): per-chunk figures will be zero", file=sys.stderr)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from radiative3d_b200 import abi, engine, workload_model
cfg, deg, n = sys.argv[1], int(sys.argv[2]), int(float(sys.argv[3]))
m = workload_model.build_model(cfg, deg)
eng = engine.Engine(m)
eng.run_simulation(n, seed=1); eng.sync(); eng.reset(); eng.set_profiling(True)
eng.run_simulation(n, seed=2)
t = eng.sync()
kt = eng.kernel_times()
print(f"{cfg} deg {deg} n={n}: {t * 1e3:.2f} ms, {n / t:.3e} phonons/s; {kt}")
