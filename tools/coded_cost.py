"""Cost of snrx_ble_coded: host wall time around RxEngine.ble_coded() (the call ends in a stream synchronise, so this is the
device time of its scan, decode and pointer rounds plus their launches and read-backs) on
  * the dense 0.98-s ble_wb40 capture of tools/aux_cost.py (legacy traffic on all 40 channels and 1M / 2M extended
    advertising, no Coded packet): mostly the scan of channels 37..39, and
  * a 0.98-s capture of Long Range events (synth.coded_adv_schedule),
with the step it follows (snrx_process + snrx_poll) timed the same way, and the device time of each kernel of the call from
torch.profiler (a separate pass of 5 calls, profiler on).  Prints one JSON line with the card's name and power limit.

    python tools/coded_cost.py [--reps 20] [--out results/coded_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from aux_cost import capture as dense_capture  # noqa: E402
from snout_b200 import chanplan, synth  # noqa: E402
from snout_b200.engine import RxEngine  # noqa: E402


def coded_capture(seconds: float = 0.98, seed: int = 9900):
    rng = np.random.default_rng(seed)
    n_ch = int(round(seconds * chanplan.NB_RATE))
    n_ch -= n_ch % chanplan.BLE_WINDOW
    streams, truth = synth.coded_adv_schedule(n_ch, rng, n_events=30, max_chain=2, event_gap=2000)
    x = synth.wideband_mix(streams)
    x = x + synth._awgn(len(x), np.random.default_rng(seed + 999), 4.0 * chanplan.WB_DECIM / 10 ** 2.5).astype(np.complex64)
    return x.astype(np.complex64), truth


def timed(x, reps):
    import torch
    xd = torch.from_numpy(x).cuda()
    with RxEngine("ble_wb40", max_samples=len(x)) as e:
        step, cost = [], []
        for k in range(reps + 3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            frames = e.process(xd).poll()
            t1 = time.perf_counter()
            lst = e.ble_coded()
            t2 = time.perf_counter()
            if k >= 3:
                step.append((t1 - t0) * 1e3)
                cost.append((t2 - t1) * 1e3)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                e.ble_coded()
            torch.cuda.synchronize()
        kernels = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            if t and ("coded" in ev.key or "aux" in ev.key or "scan" in ev.key):
                name = ev.key.split("(")[0].replace("void snrx::", "")
                kernels[name] = kernels.get(name, 0.0) + t / 5 / 1e3      # ms per call
    return frames, lst, step, cost, kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    res = {}
    for name, (x, truth) in (("dense_legacy", dense_capture()[::2]), ("long_range", coded_capture())):
        frames, lst, step, cost, kernels = timed(x, a.reps)
        got = {(int(r["channel"]), bytes(r["bytes"][: int(r["len"])])) for r in lst if r["status"] == 0 and r["crc_ok"]}
        prim = lst[lst["depth"] == 0]
        res[name] = dict(frames=len(frames), entries=len(lst), primaries=len(prim), primaries_crc_ok=int(prim["crc_ok"].sum()),
                         step_ms_median=float(np.median(step)), ble_coded_ms_median=float(np.median(cost)),
                         ble_coded_ms_min=float(np.min(cost)), ble_coded_ms_max=float(np.max(cost)), reps=a.reps,
                         kernel_ms_per_call={k: round(v, 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])})
        if name == "long_range":
            res[name].update(injected=len(truth), recovered=sum((t.channel, t.data) in got for t in truth))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    res["gpu"] = q.stdout.strip()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
