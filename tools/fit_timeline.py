"""Device timeline of cold fits (config 2 by default), from torch.profiler's CUDA activities.

Runs fits the way bench.py does (drop_caches + fit, every fit rebuilds mirror and summaries),
profiles --fits of them after its own warm-up and prints one JSON line per fit: device time per
category (head, build kernels, step kernels, tail kernels), the idle time on the stream inside
the fit and since the previous fit, and the card's name and power limit.

  python tools/fit_timeline.py [--config c2] [--fits 10] [--out FILE]

Run it on its own: tracing slows the host, so its gaps are upper bounds for a bench run.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (configs and tolerances of the benchmark)

PKG = "3d-point-cloud-multiday-imagery_b200"

BUILD = ("raster_", "mirror_", "group_summary", "super_summary")
STEP = ("lloyd_step_kernel",)


def category(name, before_steps):
    if any(b in name for b in BUILD):
        return "build"
    if any(s in name for s in STEP):
        return "steps"
    return "head" if before_steps else "tail"


def short(name):
    n = name.split("(")[0].replace("void ", "").replace("mdkm::", "")
    return n.split("<")[0]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(bench.CONFIGS))
    ap.add_argument("--fits", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile, record_function

    pkg = importlib.import_module(PKG)
    D, H, W, k, iters = bench.CONFIGS[args.config]
    tol = bench.TOL.get(args.config, 0.0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(0, stream=stream, pinned_results=True)
    hm = pkg.make_stack(D, H, W, seed=args.seed, device="cuda:0")
    n = eng.unproject(hm, stack_shape=(D, H, W), pix_begin=0)
    del hm
    torch.cuda.empty_cache()
    idx = np.sort(np.random.RandomState(args.seed).choice(eng.n_points_global, k, replace=False))
    init = eng.gather_points(idx).astype(np.float64)
    labels = torch.empty(n, dtype=torch.int32, device="cuda:0")

    def one_fit():
        eng.drop_caches()
        return eng.fit(init, max_iter=iters, tol=tol, labels_out=labels)

    for _ in range(args.warmup):
        one_fit()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(args.fits + 1):  # (fit 0: only the start of the gap before fit 1)
            with record_function(f"fit_{i}"):
                r = one_fit()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)["traceEvents"]

    fits = sorted((e for e in trace if e.get("cat") == "user_annotation" and e.get("name", "").startswith("fit_")),
                  key=lambda e: e["ts"])
    dev = sorted((e for e in trace if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")), key=lambda e: e["ts"])
    starts = [f["ts"] for f in fits] + [float("inf")]
    per_fit = [[e for e in dev if starts[i] <= e["ts"] < starts[i + 1]] for i in range(len(fits))]
    gpu = card()
    lines = []
    for i in range(1, len(fits)):
        ev, prev = per_fit[i], per_fit[i - 1]
        if not ev:
            continue
        first_step = next((j for j, e in enumerate(ev) if any(s in e["name"] for s in STEP)), len(ev))
        cats = {"head": 0.0, "build": 0.0, "steps": 0.0, "tail": 0.0}
        kernels = {}
        for j, e in enumerate(ev):
            c = category(e["name"], j < first_step)
            cats[c] += e["dur"]
            key = f"{c}:{short(e['name'])}"
            kernels[key] = kernels.get(key, 0.0) + e["dur"]
        idle_in, end = 0.0, ev[0]["ts"] + ev[0]["dur"]
        idle_by_cat = {"head": 0.0, "build": 0.0, "steps": 0.0, "tail": 0.0}
        for j, e in enumerate(ev[1:], 1):
            gap = max(0.0, e["ts"] - end)
            idle_in += gap
            idle_by_cat[category(e["name"], j < first_step)] += gap  # (the gap before an event)
            end = max(end, e["ts"] + e["dur"])
        since_prev = ev[0]["ts"] - max(e["ts"] + e["dur"] for e in prev) if prev else None
        line = {
            "fit": i, "config": args.config, "n_iter": r["n_iter"], "gpu": gpu,
            "span_us": round(end - ev[0]["ts"], 1),
            "device_us": {c: round(v, 1) for c, v in cats.items()},
            "idle_in_fit_us": round(idle_in, 1),
            "idle_before_us": {c: round(v, 1) for c, v in idle_by_cat.items()},
            "idle_since_previous_fit_us": None if since_prev is None else round(since_prev, 1),
            "events": len(ev),
            "per_kernel_us": {kk: round(v, 1) for kk, v in sorted(kernels.items())},
        }
        lines.append(json.dumps(line))
    for ln in lines:
        print(ln)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
