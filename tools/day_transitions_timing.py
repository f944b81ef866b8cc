#!/usr/bin/env python
"""Cost of the day-pair transition counts (``transitions=`` / ``return_transitions``) on one GPU.

Configs 2 (10 x 2048 x 2048 float32 stack, k = 16, 9 consecutive pairs) and 4 (12 x 4096 x 4096,
k = 1024, 11 pairs) of bench.py by default, every fit cold, no cluster map bound (so the final pass
also writes the internal map).  In one process, blocks of fits without and with transitions
alternate, so that drift of the card or the host hits both alike.  Reported per config:

* ``kernel_us``: ``day_transitions_kernel`` alone, its device time in a torch.profiler trace of a
  few fits with transitions (a separate run of fits, after the timed blocks), per launch, and the
  map bytes it reads (2 days x H*W x element size x pairs) over that time;
* ``fit_ms``: whole fits without and with transitions, CUDA events on the handle's stream;
* ``added_ms``: the medians' difference.

It also checks, once per config, that the counts equal a bincount of the cluster map of the same
fit (on the device, torch.bincount).  The card's name and power limit are read in the same run.

  python tools/day_transitions_timing.py [--configs c2 c4] [--rounds 4] [--fits 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (configs and tolerances of the benchmark)

PKG = "3d-point-cloud-multiday-imagery_b200"


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "runs": xs}


def run_config(pkg, cfg, args):
    import torch
    from torch.profiler import ProfilerActivity, profile

    D, H, W, k, iters = bench.CONFIGS[cfg]
    tol = bench.TOL.get(cfg, 0.0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(0, stream=stream, pinned_results=True)
    hm = pkg.make_stack(D, H, W, seed=0, device="cuda")
    n = eng.unproject(hm)
    del hm
    torch.cuda.empty_cache()
    init = eng.gather_points(np.sort(np.random.RandomState(0).choice(n, k, replace=False))).astype(np.float64)
    labels_dev = torch.empty(n, dtype=torch.int32, device="cuda")
    pairs = np.stack([np.arange(D - 1), np.arange(1, D)], axis=1)

    def fit(with_trans, cmap=None):
        eng.drop_caches()
        return eng.fit(init, max_iter=iters, tol=tol, labels_out=labels_dev, cluster_map_out=cmap,
                       transitions=pairs if with_trans else None)

    # correctness once: the counts of a fit against a bincount of that fit's map
    elem = torch.uint8 if k <= 255 else torch.uint16
    cmap = torch.empty(D * H * W, dtype=elem, device="cuda")
    r = fit(True, cmap)
    torch.cuda.synchronize()
    m = (cmap.view(torch.int16).to(torch.int64) & 0xFFFF) if elem == torch.uint16 else cmap.to(torch.int64)
    m = m.view(D, H * W)
    ok = True
    for p, (a, b) in enumerate(pairs):
        ref = torch.bincount(m[a] * (k + 1) + m[b], minlength=(k + 1) ** 2).cpu().numpy().reshape(k + 1, k + 1)
        ok &= bool(np.array_equal(ref, r["transitions"][p]))
    del m, cmap
    torch.cuda.empty_cache()

    variants = (False, True)
    for v in variants:  # warm-up
        for _ in range(2):
            fit(v)
    fit_ms = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(args.fits):
                fit(v)
            e1.record(stream)
            torch.cuda.synchronize()
            fit_ms[v].append(e0.elapsed_time(e1) / args.fits)

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.fits):
            fit(True)
        torch.cuda.synchronize()
    kern = [e for e in prof.events() if "day_transitions_kernel" in e.name]
    names = sorted({e.name for e in kern})
    kernel_us = [e.device_time for e in kern] if kern and hasattr(kern[0], "device_time") else \
        [e.cuda_time for e in kern]
    eng.close()
    map_bytes = 2 * H * W * (1 if k <= 255 else 2) * len(pairs)
    kmed = float(np.median(kernel_us)) if kernel_us else float("nan")
    added = float(np.median(fit_ms[True]) - np.median(fit_ms[False]))
    return {
        "config": cfg, "shape": [D, H, W], "k": k, "iters": iters, "points": n, "pairs": len(pairs),
        "counts_equal_bincount": ok, "rounds": args.rounds, "fits_per_round": args.fits,
        "kernel": names, "kernel_us": summary(kernel_us) if kernel_us else None, "map_bytes_read": map_bytes,
        "kernel_GB_per_s": map_bytes / (kmed * 1e-6) / 1e9 if kernel_us else None,
        "fit_ms": {"without": summary(fit_ms[False]), "with_transitions": summary(fit_ms[True])},
        "added_ms": added,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["c2", "c4"], choices=sorted(bench.CONFIGS))
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--fits", type=int, default=5, help="fits per setting and round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    pkg = importlib.import_module(PKG)
    out = {"card": card(), "results": [run_config(pkg, c, args) for c in args.configs],
           "note": "kernel_us: day_transitions_kernel device time per launch (torch.profiler). "
                   "fit_ms: whole cold fits, labels to the device, no cluster map bound. "
                   "added_ms: median with transitions - median without."}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
