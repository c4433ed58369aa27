#!/usr/bin/env python3
"""A/B of prebuilt builds of libsnoutrx.so in one GPU session, alternated through SNRX_LIB (snout_b200/_abi.py).

Each round runs, for every build (the order rotates from round to round):
  bench.py --no-cpu-baseline --no-c5 for ble_wb40 and mixed_wb56   -> ms_per_step, roofline.alone.kernel_ms, roofline.kernel_ms
  tools/ab_serial.py                                                -> front-end and batch time, one batch alone and two in flight
and prints the median and the max-min spread of every number per build, with the card's name, power limit and maximum SM
clock read in the same session.  With --dump it also writes bench.py --dump-outputs of ble_wb40 and mixed_wb56 for every build
and compares each build's frame records with the first build's.

usage: python tools/ab_lib.py [--rounds 3] [--steps 10] [--warmup 3] [--dump] [--out DIR] NAME=path/to/libsnoutrx.so ...
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = ("ble_wb40", "mixed_wb56")


def run(cmd, lib):
    env = dict(os.environ, SNRX_LIB=os.path.abspath(lib), PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable] + cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} with {lib} failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
    return r.stdout


def bench(lib, wl, args, dump=None):
    cmd = ["bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup), "--workload", wl,
           "--no-cpu-baseline", "--no-c5"]
    if dump:
        cmd += ["--dump-outputs", dump]
    line = json.loads([l for l in run(cmd, lib).splitlines() if l.startswith("{")][-1])
    return {f"{wl}.ms_per_step": line["ms_per_step"], f"{wl}.kernel_ms": line["roofline"]["kernel_ms"],
            f"{wl}.alone_kernel_ms": line["roofline"]["alone"]["kernel_ms"], f"{wl}.frames": line["config"]["frames_per_step"]}


def serial(lib):
    out = run(["tools/ab_serial.py"], lib)
    m = re.search(r"serial: frontend ([\d.]+) ms, batch ([\d.]+) ms \| two in flight: frontend ([\d.]+) ms, wall/step ([\d.]+) ms", out)
    if not m:
        raise RuntimeError(f"unexpected ab_serial output:\n{out}")
    return {"serial.frontend_ms": float(m[1]), "serial.batch_ms": float(m[2]), "piped.frontend_ms": float(m[3]),
            "piped.wall_ms": float(m[4])}


def compare_dumps(a, b):
    """Frame records of two --dump-outputs directories: count, and the kept rows (all, or the same seeded sample of a long
    list) where any field differs"""
    fields = sorted(f[len("frames_"):-len(".npy")] for f in os.listdir(a) if f.startswith("frames_") and f.endswith(".npy"))
    ca, cb = np.load(os.path.join(a, "frames_count.npy"))[0], np.load(os.path.join(b, "frames_count.npy"))[0]
    if ca != cb:
        return {"count": [int(ca), int(cb)], "equal": False}
    bad = np.zeros(len(np.load(os.path.join(a, "frames_row.npy"))), bool)
    diff_fields = []
    for f in fields:
        x, y = np.load(os.path.join(a, f"frames_{f}.npy")), np.load(os.path.join(b, f"frames_{f}.npy"))
        d = np.atleast_2d(x != y).reshape(len(x), -1).any(axis=1) if x.shape == y.shape else np.ones(len(x), bool)
        if d.any():
            diff_fields.append(f)
        bad |= d
    rows = np.nonzero(bad)[0]
    return {"count": int(ca), "equal": not rows.size, "rows_differing": rows[:50].tolist(), "n_rows_differing": int(rows.size),
            "fields_differing": diff_fields}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("libs", nargs="+", metavar="NAME=PATH")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump", action="store_true")
    ap.add_argument("--out", default=None, help="write the per-round numbers and the summary as JSON here")
    args = ap.parse_args()
    libs = [tuple(s.split("=", 1)) for s in args.libs]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print(f"GPU: {gpu}", flush=True)
    res = {name: [] for name, _ in libs}
    for r in range(args.rounds):
        for k in range(len(libs)):
            name, lib = libs[(k + r) % len(libs)]
            row = {}
            for wl in WORKLOADS:
                row.update(bench(lib, wl, args))
            row.update(serial(lib))
            res[name].append(row)
            print(f"round {r} {name}: " + ", ".join(f"{k} {v:.4f}" if isinstance(v, float) else f"{k} {v}" for k, v in row.items()),
                  flush=True)
    summary = {}
    if args.rounds:
        print(f"\nmedian [min, max] over {args.rounds} rounds; {gpu}")
    for name, _ in libs if args.rounds else []:
        summary[name] = {}
        for key in res[name][0]:
            v = np.array([row[key] for row in res[name]], float)
            summary[name][key] = {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}
        print(f"  {name:>8}: " + ", ".join(f"{k} {s['median']:.4f} [{s['min']:.4f}, {s['max']:.4f}]" for k, s in summary[name].items()))
    base = libs[0][0]
    for name, _ in libs[1:] if args.rounds else []:
        for key in ("ble_wb40.ms_per_step", "ble_wb40.alone_kernel_ms", "mixed_wb56.ms_per_step", "mixed_wb56.alone_kernel_ms",
                    "serial.frontend_ms", "piped.wall_ms"):
            a, b = summary[base][key], summary[name][key]
            spread = max(a["max"] - a["min"], b["max"] - b["min"])
            print(f"  {name} vs {base}: {key} {b['median']:.4f} vs {a['median']:.4f} ms = {100 * (b['median'] / a['median'] - 1):+.1f} %, "
                  f"difference {a['median'] - b['median']:.4f} ms, larger spread {spread:.4f} ms")
    dumps = {}
    if args.dump:
        tmp = tempfile.mkdtemp(prefix="ab_lib_dump_")
        for wl in WORKLOADS:
            for name, lib in libs:
                bench(lib, wl, argparse.Namespace(steps=2, warmup=1), dump=os.path.join(tmp, f"{wl}_{name}"))
            for name, _ in libs[1:]:
                dumps[f"{wl}: {name} vs {base}"] = c = compare_dumps(os.path.join(tmp, f"{wl}_{base}"), os.path.join(tmp, f"{wl}_{name}"))
                print(f"  dump {wl}: {name} vs {base}: {json.dumps(c)}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": gpu, "rounds": res, "summary": summary, "dumps": dumps}, f, indent=1)


if __name__ == "__main__":
    main()
