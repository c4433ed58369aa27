"""Cost of snrx_ble_aux: host wall time around RxEngine.ble_aux() (the call ends in a stream synchronise, so this is the
device time of its rounds plus their launches and read-backs) on a dense 0.98-s ble_wb40 capture that carries BLE 5
extended advertising next to legacy advertising and data traffic, with the step it follows (snrx_process + snrx_poll) timed
the same way.  Prints one JSON line with the card's name and power limit.

    python tools/aux_cost.py [--reps 20] [--out results/aux_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from snout_b200 import chanplan, synth  # noqa: E402
from snout_b200.engine import RxEngine  # noqa: E402


def capture(seconds: float = 0.98, seed: int = 9500):
    rng = np.random.default_rng(seed)
    n_ch = int(round(seconds * chanplan.NB_RATE))
    n_ch -= n_ch % chanplan.BLE_WINDOW
    streams, prim, aux = synth.ext_adv_schedule(n_ch, rng, n_events=120, max_chain=3, event_gap=2000)
    for c in range(40):                                            # legacy traffic on every channel as well
        s, _ = synth.ble_baseband(n_ch, c, np.random.default_rng(seed + c), gap=(2000, 20000))
        b = chanplan.ble_channel_bin(c)
        streams[b] = streams.get(b, 0) + s
    x = synth.wideband_mix(streams)
    x = x + synth._awgn(len(x), np.random.default_rng(seed + 999), 4.0 * chanplan.WB_DECIM / 10 ** 2.5).astype(np.complex64)
    return x.astype(np.complex64), prim, aux


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    x, prim, truth = capture()
    import torch
    xd = torch.from_numpy(x).cuda()
    res = {}
    with RxEngine("ble_wb40", max_samples=len(x)) as e:
        step, cost = [], []
        for k in range(a.reps + 3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            frames = e.process(xd).poll()
            t1 = time.perf_counter()
            aux = e.ble_aux()
            t2 = time.perf_counter()
            if k >= 3:
                step.append((t1 - t0) * 1e3)
                cost.append((t2 - t1) * 1e3)
        got = {(int(r["channel"]), bytes(r["bytes"][: int(r["len"])])) for r in aux if r["status"] == 0 and r["crc_ok"]}
        res.update(frames=len(frames), aux_entries=len(aux), aux_injected=len(truth),
                   aux_recovered=sum((t.channel, t.data) in got for t in truth), depth_max=int(aux["depth"].max()),
                   step_ms_median=float(np.median(step)), ble_aux_ms_median=float(np.median(cost)),
                   ble_aux_ms_min=float(np.min(cost)), ble_aux_ms_max=float(np.max(cost)), reps=a.reps)
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
