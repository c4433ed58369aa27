#!/usr/bin/env python3
"""bench.py -- headline benchmark of the receive path (contract in the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic capture per GPU.  Default workload is
BASELINE.json configs[3], the configuration the metric is quoted on: a 96 Msps wideband capture
channelized into all 40 BLE channels and decoded (access-address search, de-whitening, CRC-24) on
one B200.  Rank 0 prints ONE JSON line.

  value      input-rate Msamples/s, whole job, capture resident in HBM, timed with CUDA events
  e2e        same metric through RxEngine.run() on a pinned HOST buffer (H2D + frame D2H inside)
  roofline   channelizer kernel: algorithmic 8 B/sample / its measured launch time vs MEASURED_PEAKS
  cpu_baseline  the CPU statement of the same path (oracle) timed on this box's host cores

--dump-outputs DIR writes the frame records of the last timed step (see dump_frames) so that two builds can be compared
output for output: the inputs are seeded and the same from run to run.  The benchmark writes nothing into the tree it
runs from (no bytecode caches; the CPU arm's host-tuned oracle is compiled in a temporary directory).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

WORKLOADS = {
    # name: (engine mode, BASELINE config, description)
    "ble_wb40": ("ble_wb40", "configs[3]", "BLE all 40 channels: 96 Msps wideband capture PFB-channelized into 40 GFSK receivers"),
    "zb_wb16": ("zb_wb16", "configs[2]", "Zigbee all 16 channels: 96 Msps wideband capture PFB-channelized into 16 O-QPSK receivers"),
    "mixed_wb56": ("mixed_wb56", "configs[4] (one capture)", "mixed BLE+Zigbee 96 Msps capture: 40 GFSK + 16 O-QPSK receivers"),
    "ble_nb": ("ble_nb", "configs[0]", "BLE advertising channel 37: 4 Msps cf32, 1e7 samples"),
    "zb_nb": ("zb_nb", "configs[1]", "Zigbee 802.15.4 channel 11: 4 Msps O-QPSK capture, 1e7 samples"),
}


WIDEBAND = {"ble_wb40": "ble", "zb_wb16": "zigbee", "mixed_wb56": "mixed"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_capture(workload, seconds_base, seed):
    from snout_b200 import synth
    if workload in WIDEBAND:
        base = synth.wideband_capture(seconds=seconds_base, kind=WIDEBAND[workload], seed=seed, esn0_db=25.0)
        return base.iq, len(base.truth)
    if workload == "ble_nb":
        c = synth.ble_capture(n=10_000_000, channel=37, seed=1001, esn0_db=30.0)
        return c.iq, len(c.truth)
    c = synth.zigbee_capture(n=10_000_000, channel=11, seed=2001, esn0_db=30.0)
    return c.iq, len(c.truth)


def _oracle_taps(name):
    """Prototype filters for the CPU arm, from the generator the kernels' tables come from (tools/gen_tables.py) -- the
    reference arm must not load the product library."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from gen_tables import PFB_DESIGNS, kaiser_lowpass
    return kaiser_lowpass(*PFB_DESIGNS[name])


_POOL = None


def _ref_decode_one(args):
    """One BLE channel through the UNMODIFIED btle_rx.c (oracle/_ref): the reference keeps its state in globals, so every
    worker is a process of its own."""
    import oracle
    y, ch = args
    return len(oracle.ble_decode(oracle.ble_quantize(y, 100.0), ch, impl="reference"))


def cpu_path(workload, sample, min_seconds=0.0):
    """CPU statement of the path on `sample` using every host core, repeated until at least `min_seconds`
    of CPU work have been timed; returns (seconds, samples processed, frames of one pass, cores, kind)."""
    global _POOL
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)            # torchrun exports 1 to its workers; set before libgomp loads
    import oracle
    from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor
    from snout_b200 import chanplan
    oracle.build(native=True)
    oracle.set_threads(cores)
    kind = "port"
    h = _oracle_taps("BLE_384") if workload in ("ble_wb40", "mixed_wb56") else None
    hz = _oracle_taps("ZB_384") if workload in ("zb_wb16", "mixed_wb56") else None
    bins = [chanplan.ble_channel_bin(c) for c in range(40)]
    zbins = [chanplan.zigbee_channel_bin(c) for c in range(11, 27)]
    use_ref = oracle.have_ref("btle_ref")
    if use_ref and workload in ("ble_wb40", "mixed_wb56") and _POOL is None:
        _POOL = ProcessPoolExecutor(cores)
        list(_POOL.map(_ref_decode_one, [(np.zeros(64, np.complex64), 37)] * cores))     # start the workers outside the timed region
    t0 = time.perf_counter()
    frames, done = 0, 0
    while True:
        if workload in ("zb_wb16", "mixed_wb56"):
            # CPU statement of the wideband Zigbee path: float channelizer (OpenMP) + the restated GNU Radio chain
            # and the packet sink, one channel per thread
            y = oracle.pfb(sample, hz, zbins, fast=True, native=True)
            def zone(c):
                return len(oracle.zb_receive(y[c], 11 + c))
            with ThreadPoolExecutor(cores) as ex:
                frames = sum(ex.map(zone, range(16)))
        if workload in ("ble_wb40", "mixed_wb56"):
            # channelizer: no reference counterpart (the reference retunes one 4 Msps channel at a time), CPU
            # statement = oracle/pfb_oracle.c (vectorised, OpenMP over all cores); per-channel decode = the reference's own
            # receiver() (oracle/_ref, one process per core) where it was compiled, else its port (one thread per core)
            y = oracle.pfb(sample, h, bins, fast=True, native=True)
            if use_ref:
                n_ble = sum(_POOL.map(_ref_decode_one, [(y[c], c) for c in range(40)]))
            else:
                with ThreadPoolExecutor(cores) as ex:
                    n_ble = sum(ex.map(lambda c: len(oracle.ble_decode(oracle.ble_quantize(y[c], 100.0), c, impl="port")), range(40)))
            frames = (frames if workload == "mixed_wb56" else 0) + n_ble
            kind = "port"                                  # the channelizer, where the time goes, is our own CPU statement
        elif workload == "zb_wb16":
            pass
        elif workload == "ble_nb":
            kind = "reference" if use_ref else "port"
            q = oracle.ble_quantize(sample, 128.0)
            frames = len(oracle.ble_decode(q, 37, impl=kind))
            cores = 1
        else:
            frames = len(oracle.zb_receive_serial(sample, 11))
            cores = 1
        done += len(sample)
        if time.perf_counter() - t0 >= min_seconds:
            break
    return time.perf_counter() - t0, done, frames, cores, kind


def dump_frames(out_dir, frames, budget=64_000_000):
    """Write the frame records a caller of the timed path receives (poll(): reference order, so the same computation gives
    the same files): every field as out_dir/frames_<field>.npy, float64 (integers up to 2^53 are exact), the payload bytes
    float32 [n, 132]; frames_count.npy holds the number of records.  A list larger than `budget` bytes is cut to a fixed,
    seeded sample of its records, kept in order; frames_row.npy names the records kept."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(frames)
    names = frames.dtype.names
    row_bytes = 8 + sum(4 * frames.dtype[k].itemsize if k == "bytes" else 8 for k in names)
    keep = np.arange(n)
    cap = (budget - (1 << 16)) // row_bytes                       # room for the .npy headers
    if n > cap:
        keep = np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    sub = frames[keep]
    np.save(os.path.join(out_dir, "frames_count.npy"), np.array([n], np.float64))
    np.save(os.path.join(out_dir, "frames_row.npy"), keep.astype(np.float64))
    for k in names:
        np.save(os.path.join(out_dir, f"frames_{k}.npy"), sub[k].astype(np.float32 if k == "bytes" else np.float64))


def ncu_traffic(n_samples, kernel="k_pfb_ble", stem="pfb_ncu"):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the workload's dominant kernel from the committed
    ncu --set full summary (profiles/rNN_<stem>[_vM].json), valid when it was captured on this same workload size; else None."""
    best = None
    import re
    def version(name):                   # r01_pfb_ncu_v10.json -> (1, 10), r02_pfb_ncu.json -> (2, 0): newest capture last
        m = re.match(r"r(\d+)_" + stem + r"(?:_v(\d+))?\.json$", name)
        return (int(m.group(1)), int(m.group(2) or 0)) if m else (-1, -1)
    for name in sorted(os.listdir(os.path.join(ROOT, "profiles")), key=version):
        if version(name)[0] >= 0:
            try:
                j = json.load(open(os.path.join(ROOT, "profiles", name)))
                for l in j["launches"]:
                    if kernel in l["kernel"] and abs(l["dram_read_bytes"] / (n_samples * 8) - 1) < 0.2:
                        best = (l["traffic_bytes"], name, l.get("pipe_fma_cycles_pct"))
            except Exception:
                pass
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ble_wb40", choices=sorted(WORKLOADS) + ["c5"])
    ap.add_argument("--base-seconds", type=float, default=0.1, help="length of the generated capture that is tiled")
    ap.add_argument("--tiles", type=int, default=0, help="copies of the generated capture per step (wideband); 0 = 10 (0.98 s) for "
                    "ble_wb40, 100 (9.8 s, the capture length of BASELINE configs[4]) for zb_wb16 / mixed_wb56")
    ap.add_argument("--captures", type=int, default=0, help="narrow-band workloads: captures per step (one snrx_process batch); 0 = 256, "
                    "the batch SURVEY 8d prescribes for the roofline run of configs[0] / [1] (one 80-MB capture alone is launch-latency bound)")
    ap.add_argument("--no-c5", action="store_true", help="skip the configs[4]-shaped run (time-sharded mixed captures) reported under \"c5\"")
    ap.add_argument("--c5-seconds", type=float, default=9.83, help="length of the resident mixed capture of the c5 run")
    ap.add_argument("--c5-depth", type=int, default=2, help="c5 run: shards queued at once (the library holds SNRX_LANES of them)")
    ap.add_argument("--c5-shard-units", type=int, default=2400, help="c5 run: shard body in units of 8192 channel samples (2400 = 4.9 s: 2 shards per 10-s capture; measured 480: 47.2, 960: 51.3-54.2, 2400: 56.3-58.3 Gsamples/s -- longer shards give k_zb_rx more chains per launch)")
    ap.add_argument("--taps", type=int, default=384)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work timed for cpu_baseline (bounded sample)")
    ap.add_argument("--ref-step-seconds", type=float, default=1.5, help="--impl reference: CPU work per step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame records of the last timed step to DIR/*.npy "
                    "(rank 0; --workload c5: those of the last capture's shards, copied as they are polled)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    c5_only = args.workload == "c5"
    if c5_only:
        args.workload = "mixed_wb56"
    if not args.tiles:
        args.tiles = 10 if args.workload == "ble_wb40" else 100
    mode, cfg_name, desc = WORKLOADS[args.workload]
    unit = "Msamples/s"
    metric = "input IQ Msamples/s channelized+decoded (whole job)"

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        base, n_truth = make_capture(args.workload, min(args.base_seconds, 0.05), 4000)
        times, per_step = [], 0
        for i in range(args.warmup + args.steps):
            dt, per_step, frames, cores, kind = cpu_path(args.workload, base, min_seconds=args.ref_step_seconds)
            if i >= args.warmup:
                times.append(dt)
        t = float(np.mean(times))
        v = per_step / t / 1e6
        line = {
            "impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload} ({cfg_name}): {desc}", "sample_samples": int(per_step),
                       "note": "CPU statement of the same path on all host cores: vectorised OpenMP channelizer (oracle/pfb_oracle.c, "
                               "-O3 -march=native; the reference has no channelizer, it retunes one 4 Msps channel at a time) + per channel "
                               "the reference's own receiver() (unmodified btle_rx.c, oracle/_ref, one process per core) / the restated "
                               "GNU Radio chain + packet sink for Zigbee"},
            "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": kind,
                             "sample": f"{per_step} samples per step = a {len(base)}-sample slice of the workload repeated for >= {args.ref_step_seconds} s, {frames} frames per pass"},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    from snout_b200 import _abi, dist as sdist
    from snout_b200.engine import RxEngine
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        if os.environ.get("SNRX_NCCL_CHANNELS"):
            os.environ["NCCL_MAX_NCHANNELS"] = os.environ["SNRX_NCCL_CHANNELS"]     # experiment switch; default: NCCL's choice
    rank, world, local = sdist.init_from_env()
    torch.cuda.set_device(local)
    numa = sdist.bind_to_gpu_numa(local) if world > 1 else None
    dev = torch.device("cuda", local)

    base, n_truth = make_capture(args.workload, args.base_seconds, 4000 + 37 * rank)
    tiles = args.tiles if args.workload in WIDEBAND else 1
    caps = 1 if args.workload in WIDEBAND else (args.captures or 256)
    caps_e2e = min(caps, 8)                                          # the host leg pins at most 8 captures (640 MB)
    n_cap = len(base) * tiles                                        # samples per capture
    n = n_cap * caps                                                 # samples per step
    pinned = _abi.PinnedBuffer(n_cap * caps_e2e, np.complex64)
    for i in range(tiles * caps_e2e):
        pinned.array[i * len(base):(i + 1) * len(base)] = base
    if caps > 1:
        x_dev = torch.from_numpy(base).to(dev).repeat(caps, 1)       # [captures, samples]: one snrx_process batch
        pinned_in = pinned.array.reshape(caps_e2e, n_cap)
    else:
        x_dev = torch.from_numpy(pinned.array).to(dev)               # resident input, larger than L2 for the wideband run
        pinned_in = pinned
    eng = RxEngine(mode, max_samples=n_cap, max_captures=caps, pfb_taps=args.taps if args.workload in WIDEBAND else 0, device=local,
                   channel=None, max_frames=(1 << 18) if caps == 1 else (1 << 20))

    # whole records go zero-copy from the engine's HBM frame list, which stays valid for two further process() calls ->
    # two gathers in flight.  (FrameGather(record_bytes=80) would exchange only the 80 bytes a BLE record uses; measured at
    # N=4 it does not change the step time, nor do three gathers in flight: the exchange is not bandwidth bound.)
    gather_depth = 2

    def make_gather(engine):
        """The frame exchange for `engine`: the C ABI's own (stores into every peer's HBM from the export kernel,
        include/snoutrx.h snrx_exchange_*), else copy-engine pushes through torch symmetric memory, else NCCL."""
        if world == 1:
            return None, None
        want = os.environ.get("SNRX_GATHER", "abi")
        g = sdist.AbiGather.available(engine, dev) if want == "abi" else None
        if g is not None:
            return g, "stores into the peers' HBM over NVLink from k_export_frames (snrx_exchange_* / snrx_allgather)"
        g = sdist.PeerGather.available(dev) if want in ("abi", "peer") else None
        if g is not None:
            return g, "peer-to-peer copies over NVLink (dist.PeerGather)"
        return sdist.FrameGather(dev, cap=1 << 15, depth=gather_depth), "NCCL all-gather (dist.FrameGather)"

    gather, gather_kind = make_gather(eng)

    def barrier():
        if world > 1:
            import torch.distributed as d
            d.barrier()
        torch.cuda.synchronize()

    last_polled = [None]                 # the frame list of the step run_resident collected last (a view, see poll())

    def run_resident(k, min_seconds=0.0):
        """k steps, software pipelined two deep: batch i+1 is queued before batch i is collected, so
        the GPU never waits for the host.  Returns (frames of last step, front-end ms list, launches)."""
        front, launches, nfr, done = [], 0, 0, 0
        t0 = time.perf_counter()
        pend = []
        queued = 0
        for _ in range(min(2, max(k, 1))):
            eng.process(x_dev)
            queued += 1
        while queued:
            fr = eng.poll(copy=False)
            last_polled[0] = fr
            queued -= 1
            done += 1
            nfr = len(fr)
            # queue the next batch FIRST: everything below is host bookkeeping that must not delay the GPU.  (The polled
            # batch's frame list and stats stay valid: each lane alternates two lists, include/snoutrx.h.)
            if (done + queued < k) or (time.perf_counter() - t0 < min_seconds):
                eng.process(x_dev)
                queued += 1
            st = eng.stats()
            if world > 1:
                # the one exchange of the path: this step's records go out of the engine's HBM frame list (zero copy) in an
                # asynchronous NCCL all-gather over NVLink that overlaps the next step(s)
                pend.append(gather.start(fr, *eng.polled_frames_device()[:2]))
                if len(pend) >= gather_depth:
                    nfr = sum(pend.pop(0).counts())     # collect the oldest gather in flight
            front.append(st["gpu_ms_frontend"])
            launches += st["kernel_launches"]
        while pend:
            nfr = sum(pend.pop(0).counts())
        return nfr, front, launches, done

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # warm-up: at least W steps and at least ~1.5 s under load so that nvidia-smi (100 ms period) sees the clocks.
    # With several ranks the step COUNT must be the same everywhere (every step carries a collective), so the
    # duration is turned into a count agreed by an all-reduce.
    def steps_for(seconds, t_step):
        if world == 1:
            return 0
        import torch.distributed as d
        t = torch.tensor([t_step], device=dev)
        d.all_reduce(t, op=d.ReduceOp.MAX)
        return int(min(20000, max(1, seconds / max(float(t.item()), 1e-5))))

    if world == 1:
        frames_per_step, _, _, _ = run_resident(args.warmup, min_seconds=1.5)
        t_est = 0.0
    else:
        t0 = time.perf_counter()
        run_resident(args.warmup)
        torch.cuda.synchronize()
        t_est = (time.perf_counter() - t0) / args.warmup
        frames_per_step, _, _, _ = run_resident(steps_for(1.5, t_est))
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    frames_per_step, front_ms, launches, done = run_resident(args.steps)
    ev1.record()
    barrier()
    assert done == args.steps
    if args.dump_outputs and rank == 0 and not c5_only:
        dump_frames(args.dump_outputs, last_polled[0])   # nothing is queued after the last step: the view is still valid
    ms = ev0.elapsed_time(ev1)
    # keep the load on for the clock sampler a little longer, then stop it
    if world == 1:
        run_resident(3, min_seconds=0.5)
    else:
        run_resident(steps_for(0.5, t_est))
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        import torch.distributed as d
        t = torch.tensor([ms], device=dev)
        d.all_reduce(t, op=d.ReduceOp.MAX)
        ms = float(t.item())
    value = world * n * args.steps / (ms * 1e-3) / 1e6

    # ---- end to end: pinned host buffer in, frames out, every step.  Same two-deep software pipeline a streaming
    #      caller uses (process, process, poll, ...): the H2D copy of batch i+1 overlaps the decode tail of batch i.
    def run_e2e(buf, k):
        d2h, nfr, pend, queued, done = 0, 0, [], 0, 0
        for _ in range(min(2, k)):
            eng.process(buf)
            queued += 1
        while queued:
            fr = eng.poll(copy=True)
            queued -= 1
            done += 1
            d2h += fr.nbytes + 32
            nfr = len(fr)
            if done + queued < k:
                eng.process(buf)
                queued += 1
            if world > 1:
                pend.append(gather.start(fr, *eng.polled_frames_device()[:2]))
                if len(pend) >= gather_depth:
                    pend.pop(0).counts()
        while pend:
            pend.pop(0).counts()
        torch.cuda.synchronize()
        return d2h, nfr

    def time_e2e(buf):
        run_e2e(buf, 2)
        barrier()
        t0 = time.perf_counter()
        d2h, nfr = run_e2e(buf, args.steps)
        dt = time.perf_counter() - t0
        if world > 1:
            import torch.distributed as d
            t = torch.tensor([dt], device=dev)
            d.all_reduce(t, op=d.ReduceOp.MAX)
            dt = float(t.item())
        return world * n_e2e * args.steps / dt / 1e6, d2h, nfr

    # the dominant kernel with the GPU to itself: one batch at a time, so that no other lane's back-end kernels share the SMs
    # (outside the timed region; reported beside the live figure as roofline.alone)
    alone_ms = []
    for _ in range(12):
        eng.process(x_dev).poll(copy=False)
        alone_ms.append(eng.stats()["gpu_ms_frontend"])
    alone_ms = float(np.median(alone_ms[3:]))

    # SURVEY 8(f) N1 (outside the timed region): advertising summaries + sender table of one polled batch, on the GPU
    analytics = None
    if world == 1 and eng.n_ble:
        fr = eng.process(x_dev).poll(copy=False)
        eng.adv_summary(want=False)
        t0 = time.perf_counter()
        reps = 20
        for _ in range(reps):
            eng.adv_summary(want=False)
        dt = (time.perf_counter() - t0) / reps
        n_dev = len(eng.devices(reset=True))
        analytics = {"records_per_batch": int(len(fr)), "ms_per_batch": dt * 1e3, "records_per_s": len(fr) / dt, "senders": int(n_dev),
                     "note": "snrx_ble_adv_summary (k_ble_adv_summary + k_ble_adv_devices + counter read-back), not part of value/e2e"}


    # ---- BASELINE configs[4]: long mixed BLE+Zigbee captures sharded by time segment WITH HALO, frames exchanged.  Every rank
    #      holds one resident 10-s capture standing for its 1024/N captures (SURVEY 8d: 1024 x 7.7 GB cannot be materialised) and
    #      processes it as dist.plan_job cuts it -- ~1-s bodies with the BLE / Zigbee halos of snrx_shard_t, i.e. exactly the
    #      units a multi-GPU job hands out -- two shards in flight, every shard's records exchanged with all ranks.
    def run_c5():
        from snout_b200 import stream
        # the capture is MADE on the GPU (SURVEY 8f N4, snrx_synth_wideband): a 0.98-s schedule of random BLE + 802.15.4 frames on
        # all 56 receivers, sent c5_seconds times over with fresh noise -- nothing crosses PCIe
        from snout_b200 import synth
        xc, ctruth = synth.wideband_capture_gpu(seconds=0.983, kind="mixed", seed=5000 + 37 * rank, esn0_db=25.0, device=local,
                                                repeat=max(1, int(round(args.c5_seconds / 0.983))))
        unit, pre, post = stream.shard_geometry(40, 16)
        body_units = args.c5_shard_units                        # x 8192 channel samples per shard body
        ceng = RxEngine("mixed_wb56", max_samples=(body_units * unit + pre + post) * 24, pfb_taps=args.taps, device=local,
                        max_frames=1 << 18)
        cgather, ckind = make_gather(ceng)
        units = sdist.plan_job(1, len(xc), ceng, units_per_shard=body_units)
        halo = sum(u["hi"] - u["lo"] for u in units) / len(xc) - 1.0

        def poll(stats):
            fr = ceng.poll(copy=False)
            if args.dump_outputs and c5_only and stats["polled"] >= stats["keep_from"]:
                stats["kept"].append(fr.copy())         # a shard of the last capture (the view is reused two batches later)
            stats["polled"] += 1
            stats["queued"] -= 1
            stats["frames"] += len(fr)
            stats["launches"] += ceng.stats()["kernel_launches"]
            return fr

        def one_capture(cid, pend, stats):
            for u in units:
                if stats["queued"] == args.c5_depth:
                    fr = poll(stats)
                    if world > 1:
                        pend.append(cgather.start(fr, *ceng.polled_frames_device()[:2]))
                        if len(pend) >= gather_depth:
                            stats["gathered"] += sum(pend.pop(0).counts())
                ceng.process(xc[u["lo"]: u["hi"]], shard=dict(pre_samples=u["pre_samples"], body_samples=u["body_samples"],
                                                               first_window=u["first_window"], first_capture_id=cid))
                stats["queued"] += 1

        def drain(pend, stats):
            while stats["queued"]:
                fr = poll(stats)
                if world > 1:
                    pend.append(cgather.start(fr, *ceng.polled_frames_device()[:2]))
            while pend:
                stats["gathered"] += sum(pend.pop(0).counts())

        def run(k):
            pend, stats = [], dict(queued=0, frames=0, gathered=0, launches=0, polled=0, keep_from=(k - 1) * len(units), kept=[])
            for cid in range(k):
                one_capture(cid, pend, stats)
            drain(pend, stats)
            return stats

        run(max(1, min(args.warmup, 2)))
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st = run(args.steps)
        e1.record()
        barrier()
        if args.dump_outputs and rank == 0 and c5_only:
            dump_frames(args.dump_outputs, np.concatenate(st["kept"]))
        cms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as d
            t = torch.tensor([cms], device=dev)
            d.all_reduce(t, op=d.ReduceOp.MAX)
            cms = float(t.item())
        ceng.close()
        return {"value": world * len(xc) * args.steps / (cms * 1e-3) / 1e6, "unit": unit_name, "ms_per_step": cms / args.steps,
                "steps": args.steps, "scaling": "weak",
                "config": {"workload": "c5 (configs[4]): 10-s 96 Msps mixed BLE+Zigbee captures sharded by time segment with halo, "
                                       "frames exchanged over NVLink; one resident capture per GPU stands for its 1024/N captures",
                           "samples_per_step_per_gpu": int(len(xc)), "shards_per_capture": len(units), "frames_sent_per_capture": len(ctruth),
                           "data": "generated on the GPU by snrx_synth_wideband (GFSK / O-QPSK bursts, x24 synthesis filterbank, AWGN 25 dB)",
                           "shard_body_samples": int(body_units * unit * 24), "halo_overhead": round(halo, 4),
                           "frames_per_step": int(st["frames"] / args.steps), "frame_exchange": ckind,
                           "frames_received_per_step_all_ranks": int(st["gathered"] / args.steps) if world > 1 else None},
                "gpu_launches": int(st["launches"]),
                "note": "a step = one capture = shards_per_capture snrx_process calls (snrx_shard_t halos: BLE 128 / 2048, Zigbee "
                        "102400 / 16512 channel samples), two in flight; H2D excluded (resident data), as SURVEY 8d specifies for C5"}

    unit_name = unit
    c5 = None
    if c5_only or (not args.no_c5 and args.workload == "ble_wb40"):
        c5 = run_c5()

    n_e2e = n_cap * caps_e2e
    e2e, d2h, _ = time_e2e(pinned_in)
    # narrow band: the latency of ONE capture (what a single `snout scan` sees), beside the batched throughput
    single = None
    if caps > 1:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            eng.process(x_dev[0]).poll(copy=False)
        single = {"ms_per_capture": (time.perf_counter() - t0) / 10 * 1e3, "value": n_cap * 10 / (time.perf_counter() - t0) / 1e6, "unit": unit,
                  "note": "one capture per snrx_process, resident, not pipelined: launch latency bound"}
    # the same capture as an 8-bit digitiser delivers it (interleaved int8 I,Q = the HackRF transfer format the
    # reference consumes, btle_rx.c:204,489-498) through snrx_process_sc8: a quarter of the PCIe bytes
    e2e_sc8 = None
    if args.workload in WIDEBAND or args.workload == "ble_nb":
        peak_amp = float(np.abs(pinned.array[: len(base)]).max())
        pinned8 = _abi.PinnedBuffer((n_e2e, 2), np.int8)
        q = np.clip(np.rint(base.view(np.float32).reshape(-1, 2) * (100.0 / peak_amp)), -128, 127).astype(np.int8)
        for i in range(tiles * caps_e2e):
            pinned8.array[i * len(base):(i + 1) * len(base)] = q
        pinned8_in = pinned8.array.reshape(caps_e2e, n_cap, 2) if caps > 1 else pinned8
        if args.workload in WIDEBAND:                      # keep the per-channel int8 amplitude of the cf32 run
            eng.close()
            eng = RxEngine(mode, max_samples=n_cap, pfb_taps=args.taps, device=local, max_frames=1 << 18,
                           quant_scale=100.0 * 1.28 * peak_amp)
            gather, _ = make_gather(eng)
        v8, d2h8, nfr8 = time_e2e(pinned8_in)
        e2e_sc8 = {"value": v8, "unit": unit, "h2d_bytes_per_step": int(n_e2e * 2), "d2h_bytes_per_step": int(d2h8 / args.steps),
                   "frames_per_step": int(nfr8),
                   "note": "same capture quantised to interleaved int8 I,Q (full scale = 1.28 x peak), RxEngine.run via snrx_process_sc8"}

    if rank != 0:
        return 0
    peak, peak_src = peaks()
    fms = float(np.mean(front_ms))
    achieved = n * 8 / (fms * 1e-3) / 1e9
    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": f"synthetic: {args.base_seconds}s seeded GFSK capture with AWGN, tiled x{tiles}; random frames on every channel",
        "config": {"workload": f"{args.workload} ({cfg_name}): {desc}", "samples_per_step_per_gpu": int(n), "captures_per_step": int(caps),
                   "single_capture": single,
                   "input_bytes_per_step_per_gpu": int(n * 8), "pfb_taps": args.taps if args.workload in WIDEBAND else None,
                   "l2": "input (%.0f MB) larger than L2; no flush needed" % (n * 8 / 1e6),
                   "frames_per_step": int(frames_per_step), "frame_exchange": gather_kind, "timed": "K x (process + poll), two batches in flight, frames land in pinned host memory; CUDA events on the engine stream"},
        "frames_per_s": frames_per_step * args.steps / (ms * 1e-3),
        "gpu_launches": int(launches),
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": unit, "h2d_bytes_per_step": int(n_e2e * 8), "d2h_bytes_per_step": int(d2h / args.steps),
                "note": "RxEngine.process/poll on a pinned host cf32 buffer, two batches in flight: chunked H2D overlapped with the channelizer, frames copied out"},
        "e2e_sc8": e2e_sc8,
        "analytics": analytics,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_src,
                     "kernel": {"ble_wb40": "k_pfb_ble (channelizer+slicer)", "zb_wb16": "k_pfb_zb_warp (channelizer+discriminator)",
                                "mixed_wb56": "k_pfb_ble (channelizer+slicer; the Zigbee front end runs after it on the tail stream)",
                                "ble_nb": "k_ble_slice_nb", "zb_nb": "k_zb_quad"}[mode],
                     "algorithmic_bytes_per_launch": int(n * 8), "kernel_ms": fms,
                     "alone": {"kernel_ms": alone_ms, "achieved": n * 8 / (alone_ms * 1e-3) / 1e9, "frac": n * 8 / (alone_ms * 1e-3) / 1e9 / peak,
                               "note": "same launch with one batch queued at a time (no other lane's kernels on the SMs); measured after the timed region"},
                     "step_frac": n * 8 / (ms / args.steps * 1e-3) / 1e9 / peak,
                     "binding_unit": "fp32 FMA pipe / issue slots" if args.workload in WIDEBAND else "hbm",
                     "note": "frac = 8 B per input sample (one cf32 read) / the dominant kernel's launch time vs the measured HBM copy "
                             "bandwidth; step_frac = the same bytes / the whole step.  The wideband kernels are bound by the FP32 pipe "
                             "and issue slots, not by bytes (DESIGN.md 3, 6): the HBM fraction is reported because the contract asks "
                             "for it, the binding unit is named beside it"},
        "c5": c5,
    }
    if c5_only:                    # --workload c5: the sharded run is the headline, the single-capture mixed run is context
        single = {k: line[k] for k in ("value", "ms_per_step", "frames_per_s", "gpu_launches")}
        single["config"] = line["config"]
        line.update(value=c5["value"], ms_per_step=c5["ms_per_step"], gpu_launches=c5["gpu_launches"], config=c5["config"],
                    frames_per_s=c5["config"]["frames_per_step"] * args.steps / (c5["ms_per_step"] * args.steps * 1e-3))
        line["mixed_wb56_single_capture"] = single
        line["c5"] = {"note": c5["note"]}
    tr = ncu_traffic(n) if mode == "ble_wb40" else ncu_traffic(n, "k_pfb_zb_warp", "zb_wb16_ncu") if mode == "zb_wb16" else None
    if tr:
        line["roofline"]["traffic"] = tr[0]
        line["roofline"]["traffic_source"] = f"profiles/{tr[1]} (ncu --set full, dram read+write of one launch)"
        if mode == "zb_wb16":
            line["roofline"]["traffic_note"] = "includes the 2.5 GB discriminator stream f the kernel writes (4 B per channel sample, 16 channels)"
        if tr[2] and mode == "ble_wb40":
            line["roofline"]["fp32_fma_pipe_cycles_active_pct"] = tr[2]
            line["roofline"]["note"] = ("8 B per input sample (one cf32 read). The binding unit is the FP32 FMA pipe: ncu "
                                        "sm__pipe_fma_cycles_active of the same launch, committed in profiles/; see DESIGN.md 3, 6")
    if world == 1 and not args.no_cpu_baseline:
        sample = base                                  # the whole generated capture (0.1 s wideband / 1e7 samples narrow band)
        dt, done, frames, cores, kind = cpu_path(args.workload, sample, min_seconds=args.cpu_seconds)
        line["cpu_baseline"] = {"value": done / dt / 1e6, "unit": unit, "cores": cores, "kind": kind,
                                "sample": f"{done} samples = a {len(sample)}-sample slice of the same capture repeated for "
                                          f"{dt:.1f} s of CPU work, {frames} frames per pass"}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
