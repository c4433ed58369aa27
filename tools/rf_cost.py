"""Cost of the per-frame radio metrics (SNRX_F_RF_METRICS): ms per step with the flag off and on, alternated in one process.

Inputs are made on the GPU (synth.wideband_capture_gpu, 0.983 s of 96 Msps = 755 MB per capture, larger than the 126 MB L2)
and stay there; every step queues one capture while the previous one is in flight (two batches in flight), and the time
of a round of K steps comes from CUDA events around it, after the last poll.  The engines with and without the flag run
round by round in turn, so that both see the same box.

    python tools/rf_cost.py [--steps 20] [--rounds 5] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {                    # name: (engine mode, synth kind, channel-rate gap between a channel's frames)
    "ble_wb40": ("ble_wb40", "ble", None),                   # the headline capture (bench.py's dense BLE workload)
    "zb_wb16": ("zb_wb16", "zigbee", None),
    "mixed_wb56": ("mixed_wb56", "mixed", None),
    "ble_wb40_sparse": ("ble_wb40", "ble", (20000, 200000)),  # 5 .. 50 ms between the frames of a channel
}


def card() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, limit = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"name": name.strip(), "power_limit": limit.strip()}


def steps_ms(eng, x, k):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    n = 0
    eng.process(x)
    for _ in range(k - 1):
        eng.process(x)
        n += len(eng.poll(copy=False))
    n += len(eng.poll(copy=False))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k, n // k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from snout_b200 import synth
    from snout_b200.engine import RxEngine
    res = {"card": card(), "steps": a.steps, "rounds": a.rounds, "workloads": {}}
    for name, (mode, kind, gap) in WORKLOADS.items():
        if a.only and name not in a.only.split(","):
            continue
        x, truth = synth.wideband_capture_gpu(seconds=0.983, kind=kind, seed=5000, esn0_db=25.0, gap=gap)
        engines = {flag: RxEngine(mode, max_samples=len(x), max_frames=1 << 18, rf_metrics=flag) for flag in (False, True)}
        for eng in engines.values():
            steps_ms(eng, x, a.warmup)
        t = {False: [], True: []}
        frames = 0
        for _ in range(a.rounds):
            for flag, eng in engines.items():
                ms, frames = steps_ms(eng, x, a.steps)
                t[flag].append(ms)
        for eng in engines.values():
            eng.close()
        del x
        torch.cuda.empty_cache()
        off, on = sorted(t[False]), sorted(t[True])
        row = {"frames_per_step": frames, "off_ms": t[False], "on_ms": t[True], "off_median": off[len(off) // 2],
               "on_median": on[len(on) // 2], "delta_ms": on[len(on) // 2] - off[len(off) // 2]}
        res["workloads"][name] = row
        print(name, json.dumps(row), flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "rf_cost.json"), "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
