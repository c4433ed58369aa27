#!/usr/bin/env python3
"""Front-end kernel time of one resident ble_wb40 capture-second, ONE batch at a time (no other lane on the GPU) and two in
flight: separates the kernel itself from what it suffers next to the other lane's kernels."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from snout_b200 import synth
from snout_b200.engine import RxEngine
x, _ = synth.wideband_capture_gpu(seconds=0.983, kind="ble", seed=4000, device=0)
eng = RxEngine("ble_wb40", max_samples=len(x), device=0, max_frames=1 << 17)
def serial(n):
    fe, tot = [], []
    for i in range(n):
        eng.process(x); eng.poll(copy=False)
        s = eng.stats(); fe.append(s["gpu_ms_frontend"]); tot.append(s["gpu_ms"])
    return np.median(fe[3:]), np.median(tot[3:])
def piped(n, depth=2):
    fe = []
    for _ in range(depth - 1):
        eng.process(x)
    t0 = time.perf_counter()
    for i in range(n):
        eng.process(x); eng.poll(copy=False); fe.append(eng.stats()["gpu_ms_frontend"])
    for _ in range(depth - 1):
        eng.poll(copy=False)
    torch.cuda.synchronize()
    return np.median(fe[3:]), (time.perf_counter() - t0) / n * 1e3
a = serial(25); b = piped(40)
c = piped(60, 3) if os.environ.get('AB_DEPTH3') else (float('nan'), float('nan'))
print(f"serial: frontend {a[0]:.4f} ms, batch {a[1]:.4f} ms | two in flight: frontend {b[0]:.4f} ms, wall/step {b[1]:.4f} ms | three in flight: frontend {c[0]:.4f} ms, wall/step {c[1]:.4f} ms")
