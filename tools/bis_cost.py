"""Cost of snrx_ble_bis: host wall time around RxEngine.ble_bis() (the call builds the aux list, the periodic list, then
the BIGs and their subevents, and ends in a stream synchronise) on two 0.98-s ble_wb40 captures:
  * the dense capture of tools/aux_cost.py (legacy traffic on all 40 channels and 1M / 2M extended advertising, no BIGs),
  * a capture of BIGs (synth.broadcast_iso_schedule: 4 BIGs, ISO_Interval 7.5 and 10 ms, 2..4 BIS, NSE 2..6),
with RxEngine.ble_periodic() timed the same way for comparison, the median, minimum and maximum of --reps calls, and a
torch.profiler run of five ble_bis calls on each capture (device time per kernel and call).  Prints one JSON line with the
card's name and power limit.

    python tools/bis_cost.py [--reps 20] [--out results/bis_cost.json]
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


def bis_capture(seconds: float = 0.98, seed: int = 9990):
    rng = np.random.default_rng(seed)
    n_ch = int(round(seconds * chanplan.NB_RATE))
    n_ch -= n_ch % chanplan.BLE_WINDOW
    streams, prim, bises, syncs, aux, bigs = synth.broadcast_iso_schedule(n_ch, rng, n_bigs=4, iso_intervals=(6, 8), num_bis=(2, 4),
                                                                          nse=(2, 6))
    x = synth.wideband_mix(streams)
    x = x + synth._awgn(len(x), np.random.default_rng(seed + 999), 4.0 * chanplan.WB_DECIM / 10 ** 2.5).astype(np.complex64)
    return x.astype(np.complex64), bises


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    res = {"reps": a.reps}
    for name, (x, truth) in (("dense_legacy", dense_capture()[::2]), ("bis", bis_capture())):
        xd = torch.from_numpy(x).cuda()
        with RxEngine("ble_wb40", max_samples=len(x)) as e:
            e.process(xd).poll()
            per, aux_t = [], []
            for k in range(a.reps + 3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                bis = e.ble_bis()
                t1 = time.perf_counter()
                e.ble_periodic()
                t2 = time.perf_counter()
                if k >= 3:
                    per.append((t1 - t0) * 1e3)
                    aux_t.append((t2 - t1) * 1e3)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    e.ble_bis()
                torch.cuda.synchronize()
            kernels = {}
            for ev in prof.key_averages():
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                if t and ("sync" in ev.key or "aux" in ev.key or "scan" in ev.key or "big" in ev.key or "bis" in ev.key):
                    kernels[ev.key.split("(")[0].replace("void snrx::", "")] = round(t / 5e3, 4)     # ms per call
            ok = {(int(r["channel"]), bytes(r["bytes"][: int(r["len"])])) for r in bis if r["status"] == 0 and r["crc_ok"]}
            res[name] = dict(entries=len(bis), bigs=len(set(bis["source"].tolist())), injected=len(truth),
                             recovered=sum((t.channel, t.data) in ok for t in truth) if truth and hasattr(truth[0], "subevent") else None,
                             ble_bis_ms_median=float(np.median(per)), ble_bis_ms_min=float(np.min(per)),
                             ble_bis_ms_max=float(np.max(per)), ble_periodic_ms_median=float(np.median(aux_t)),
                             kernel_ms=kernels)
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
