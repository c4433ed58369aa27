"""Cost of one of the on-demand BLE lists: host wall time around RxEngine.ble_<call>() (each call ends in a stream
synchronise, so this is the device time of its kernels plus their launches and read-backs) on 0.98-s ble_wb40 captures,
with the call it is compared to timed the same way right next to it, the median, minimum and maximum of --reps calls, and
a torch.profiler run of five calls on each capture (device time per kernel and call, every kernel of the window).  Prints
one JSON line with the card's name, power limit and maximum SM clock.

  --call aux       the dense capture (legacy traffic on all 40 channels and 1M / 2M extended advertising), compared to
                   the step it follows (snrx_process + snrx_poll)
  --call coded     the dense capture without its primaries' truth (no Coded packet: mostly the scan of channels 37..39)
                   and a capture of Long Range events (synth.coded_adv_schedule), compared to the step
  --call periodic  the dense capture and a capture of periodic-advertising trains (synth.periodic_adv_schedule: 8 trains,
                   Interval 6..80), compared to ble_aux
  --call bis       the dense capture and a capture of BIGs (synth.broadcast_iso_schedule: 4 BIGs, ISO_Interval 7.5 and
                   10 ms, 2..4 BIS, NSE 2..6), compared to ble_periodic

--dump DIR writes each returned list as DIR/<call>_<capture>.npy, so two builds of the library run through SNRX_LIB can be
compared byte for byte.

    python tools/list_cost.py --call periodic [--reps 20] [--dump DIR] [--out results/periodic_cost.json]
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


def _finish(streams, seed):
    x = synth.wideband_mix(streams)
    x = x + synth._awgn(len(x), np.random.default_rng(seed + 999), 4.0 * chanplan.WB_DECIM / 10 ** 2.5).astype(np.complex64)
    return x.astype(np.complex64)


def _n_ch(seconds):
    n_ch = int(round(seconds * chanplan.NB_RATE))
    return n_ch - n_ch % chanplan.BLE_WINDOW


def capture(seconds: float = 0.98, seed: int = 9500):
    """The dense capture: (iq, primary ADV_EXT_INDs, auxiliary packets)."""
    rng = np.random.default_rng(seed)
    n_ch = _n_ch(seconds)
    streams, prim, aux = synth.ext_adv_schedule(n_ch, rng, n_events=120, max_chain=3, event_gap=2000)
    for c in range(40):                                            # legacy traffic on every channel as well
        s, _ = synth.ble_baseband(n_ch, c, np.random.default_rng(seed + c), gap=(2000, 20000))
        b = chanplan.ble_channel_bin(c)
        streams[b] = streams.get(b, 0) + s
    return _finish(streams, seed), prim, aux


def coded_capture(seconds: float = 0.98, seed: int = 9900):
    streams, truth = synth.coded_adv_schedule(_n_ch(seconds), np.random.default_rng(seed), n_events=30, max_chain=2, event_gap=2000)
    return _finish(streams, seed), truth


def periodic_capture(seconds: float = 0.98, seed: int = 9800):
    streams, prim, syncs, aux = synth.periodic_adv_schedule(_n_ch(seconds), np.random.default_rng(seed), n_trains=8, intervals=(6, 80))
    return _finish(streams, seed), syncs


def bis_capture(seconds: float = 0.98, seed: int = 9990):
    streams, prim, bises, syncs, aux, bigs = synth.broadcast_iso_schedule(_n_ch(seconds), np.random.default_rng(seed), n_bigs=4,
                                                                          iso_intervals=(6, 8), num_bis=(2, 4), nse=(2, 6))
    return _finish(streams, seed), bises


def dense():
    x, _, aux = capture()
    return x, aux


def dense_legacy():                                                # the dense capture carries none of these lists' packets
    return capture()[0], None


# call: (the call it is compared to, {capture name: iq and the packets of the call's list it carries})
CALLS = {
    "aux": ("step", {"dense": dense}),
    "coded": ("step", {"dense_legacy": dense_legacy, "long_range": coded_capture}),
    "periodic": ("ble_aux", {"dense_legacy": dense_legacy, "periodic": periodic_capture}),
    "bis": ("ble_periodic", {"dense_legacy": dense_legacy, "bis": bis_capture}),
}


def measure(x, call: str, against: str, reps: int):
    """(the last list, call ms, comparison ms, device ms per call by kernel)"""
    import torch
    xd = torch.from_numpy(x).cuda()
    with RxEngine("ble_wb40", max_samples=len(x)) as e:
        fn = getattr(e, "ble_" + call)
        if against == "step":                                      # the step first: the call reads its polled batch
            first, second = (lambda: e.process(xd).poll()), fn
        else:
            e.process(xd).poll()
            first, second = fn, getattr(e, against)
        t_call, t_other = [], []
        for k in range(reps + 3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            a = first()
            t1 = time.perf_counter()
            b = second()
            t2 = time.perf_counter()
            if k >= 3:
                (t_call if first is fn else t_other).append((t1 - t0) * 1e3)
                (t_call if second is fn else t_other).append((t2 - t1) * 1e3)
        lst = a if first is fn else b
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
        kernels = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            if t:
                name = ev.key.split("(")[0].replace("void snrx::", "")
                kernels[name] = kernels.get(name, 0.0) + t / 5e3    # ms per call
    return lst, t_call, t_other, kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--call", required=True, choices=sorted(CALLS))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--dump", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    against, captures = CALLS[a.call]
    res = {"call": a.call, "reps": a.reps}
    for name, make in captures.items():
        x, truth = make()
        lst, t_call, t_other, kernels = measure(x, a.call, against, a.reps)
        ok = {(int(r["channel"]), bytes(r["bytes"][: int(r["len"])])) for r in lst if r["status"] == 0 and r["crc_ok"]}
        res[name] = {"entries": len(lst), "injected": None if truth is None else len(truth),
                     "recovered": None if truth is None else sum((t.channel, t.data) in ok for t in truth),
                     f"ble_{a.call}_ms_median": float(np.median(t_call)), f"ble_{a.call}_ms_min": float(np.min(t_call)),
                     f"ble_{a.call}_ms_max": float(np.max(t_call)), f"{against}_ms_median": float(np.median(t_other)),
                     "kernel_ms": {k: round(v, 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])}}
        if a.dump:
            os.makedirs(a.dump, exist_ok=True)
            np.save(os.path.join(a.dump, f"{a.call}_{name}.npy"), lst)
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
