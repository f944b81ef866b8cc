#!/usr/bin/env python
"""Cost of the region overlaps between days (``region_overlaps=`` / ``return_region_overlaps``) on
one GPU.

Settings, each at connectivity 4 and 8:
* config 2 of bench.py (10 x 2048 x 2048, k = 16): the 9 consecutive pairs;
* the one-GPU config-3 shape (20 x 1024 x 8192, k = 64): the 19 consecutive pairs;
* the worst case at the config-2 geometry: 10 days of a one-pixel checkerboard, every other day
  shifted by one pixel (k = 2), at connectivity 4 -- every pixel is its own region and every
  pixel of every pair a row.
Centroids come from one fit of the bench's k; the overlaps are then taken by ``predict`` calls.

Reported per setting, from a torch.profiler trace of ``--calls`` predicts with regions and
overlaps (device time of each kernel, summed per call, median over the calls):
* ``kernels_us`` and ``overlap_us``: the bound, insert, mark, scan and emit kernels;
* ``floor_us``: the bound and insert passes each reading 8 B per pixel and pair, at the
  device-to-device copy rate measured in the same run (a 2 GiB torch copy), and ``over_floor``;
* ``rows`` (M) and the bounds (the run starts the bound pass counts, recomputed here with torch
  from the returned region map: total and largest pair), and whether M equals the distinct keys;
* ``predict_ms``: whole predicts with regions, without and with overlaps (CUDA events, rounds
  alternating), and their difference.
The card's name, power limit and max SM clock are read in the same run.

  python tools/region_overlaps_timing.py [--settings c2 c3 checker] [--calls 5] [--out FILE]
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
import bench  # noqa: E402  (configs of the benchmark)

PKG = "3d-point-cloud-multiday-imagery_b200"
KERNELS = ("overlap_bound_kernel", "overlap_insert_kernel", "overlap_mark_kernel", "overlap_scan_kernel",
           "overlap_emit_kernel")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def copy_rate_GBps():
    import torch

    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(10):
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2 * (1 << 31) / (float(np.median(ts)) * 1e-3) / 1e9


def kernel_times(prof, calls):
    out = {}
    for base in KERNELS:
        t = [getattr(e, "device_time", None) or e.cuda_time for e in prof.events() if base in e.name]
        if t:
            out[base] = float(np.sum(t) / calls)
    return out


def bounds_and_keys(rmap, D, H, W, pairs):
    """Per pair: the run starts the bound pass counts, and the distinct (id_a, id_b) keys."""
    import torch

    ids = rmap.view(D, H * W).to(torch.int64)
    x0 = (torch.arange(H * W, device=rmap.device) % W) == 0
    bounds, keys = [], []
    for a, b in pairs:
        k = (ids[a] << 32) | ids[b]
        nz = (ids[a] > 0) & (ids[b] > 0)
        left = torch.roll(k, 1)
        bounds.append(int((nz & (x0 | (k != left))).sum()))
        keys.append(int(torch.unique(k[nz]).numel()))
    return bounds, keys


def run_setting(eng, name, D, H, W, k, centers, conn, args, rate):
    import torch
    from torch.profiler import ProfilerActivity, profile

    stream = torch.cuda.current_stream()
    pairs = [(d, d + 1) for d in range(D - 1)]
    rmap = torch.empty(D * H * W, dtype=torch.int32, device="cuda")

    def predict(with_overlaps):
        return eng.predict(centers, want_labels=False, regions=conn, region_map_out=rmap,
                           region_overlaps=pairs if with_overlaps else None)

    rows = predict(True)[-1]
    torch.cuda.synchronize()
    bounds, keys = bounds_and_keys(rmap, D, H, W, pairs)
    per_pair = np.bincount(rows[:, 0], minlength=len(pairs)).tolist()
    predict(False)
    ms = {False: [], True: []}
    for _ in range(args.rounds):
        for v in (False, True):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(args.calls):
                predict(v)
            e1.record(stream)
            torch.cuda.synchronize()
            ms[v].append(e0.elapsed_time(e1) / args.calls)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.calls):
            predict(True)
        torch.cuda.synchronize()
    kt = kernel_times(prof, args.calls)
    overlap_us = sum(kt.values())
    floor_us = 2 * 8 * H * W * len(pairs) / (rate * 1e9) * 1e6
    return {
        "setting": name, "shape": [D, H, W], "k": k, "connectivity": conn, "pairs": len(pairs),
        "rows": int(rows.shape[0]), "rows_per_pair_max": int(max(per_pair)),
        "bound_total": int(sum(bounds)), "bound_max": int(max(bounds)),
        "rows_equal_distinct_keys": per_pair == keys,
        "kernels_us": kt, "overlap_us": overlap_us, "floor_us": floor_us,
        "over_floor": overlap_us / floor_us if floor_us else None,
        "predict_ms": {"regions": float(np.median(ms[False])), "regions_and_overlaps": float(np.median(ms[True])),
                       "added": float(np.median(ms[True]) - np.median(ms[False]))},
    }


def run_config(pkg, cfg, args, rate):
    import torch

    D, H, W, k, iters = bench.CONFIGS[cfg]
    eng = pkg.Engine(0)
    hm = pkg.make_stack(D, H, W, seed=0, device="cuda")
    n = eng.unproject(hm)
    del hm
    torch.cuda.empty_cache()
    rs = np.random.RandomState(0)
    init = eng.gather_points(np.sort(rs.choice(n, k, replace=False))).astype(np.float64)
    centers = eng.fit(init, max_iter=iters, tol=0.0, want_labels=False)["centers"]
    res = []
    for conn in (4, 8):
        res.append(run_setting(eng, cfg, D, H, W, k, centers, conn, args, rate))
        print(json.dumps(res[-1]), flush=True)
    eng.close()
    torch.cuda.empty_cache()
    return res


def run_checker(pkg, args, rate):
    """One-pixel checkerboards, every other day shifted by one pixel: labels by nearest z level."""
    import torch

    D, H, W = bench.CONFIGS["c2"][:3]
    yy = torch.arange(H, device="cuda").view(H, 1)
    xx = torch.arange(W, device="cuda").view(1, W)
    days = [((yy + xx + d) % 2).float() * 260.0 - 130.0 for d in range(D)]
    hm = torch.stack(days).contiguous()
    eng = pkg.Engine(0)
    eng.unproject(hm)
    del hm, days
    torch.cuda.empty_cache()
    centers = np.array([[W / 2.0, H / 2.0, -130.0], [W / 2.0, H / 2.0, 130.0]])
    res = [run_setting(eng, "checker", D, H, W, 2, centers, 4, args, rate)]
    print(json.dumps(res[-1]), flush=True)
    eng.close()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--settings", nargs="+", default=["c2", "c3", "checker"], choices=["c2", "c3", "checker"])
    ap.add_argument("--calls", type=int, default=5, help="predicts per round and in the trace")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    pkg = importlib.import_module(PKG)
    rate = copy_rate_GBps()
    results = []
    for s in args.settings:
        results += run_checker(pkg, args, rate) if s == "checker" else run_config(pkg, s, args, rate)
    out = {"card": card(), "copy_rate_GB_per_s": rate, "results": results,
           "note": "kernels_us: device time per predict (torch.profiler), summed over the launches of one call. "
                   "floor_us: bound and insert passes reading 8 B per pixel and pair each, at the measured copy rate. "
                   "predict_ms: whole predicts with regions (region map on the device), medians of rounds."}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
