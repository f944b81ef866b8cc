#!/usr/bin/env python
"""Cost of the object tracks (``tracks=`` / ``return_tracks``) on one GPU.

Settings (connectivity 4, min_iou 0.5):
* config 2 of bench.py (10 x 2048 x 2048, k = 16);
* the one-GPU config-3 shape (20 x 1024 x 8192, k = 64);
* the many-small-regions worst case at the config-2 geometry: 10 identical days of a one-pixel
  checkerboard (k = 2) -- every pixel is a region, every pixel of every consecutive pair an
  overlap row and a link, and every track a 10-region chain.
Centroids come from one fit of the bench's k; the tracks are then taken by ``predict`` calls with
the region map and the track map in CUDA tensors.

Reported per setting:
* ``kernels_us``: device time per predict (torch.profiler) of the link, numbering, table and map
  kernels of the tracks.  The numbering kernels of the tracks are the second launch of
  ``region_number_kernel`` / ``region_resolve_kernel`` in each predict (the first labels the
  regions); ``link_number_table_us`` sums the tracks' kernels without the map pass;
* ``map_floor_us``: the map pass reading 4 B and writing 4 B per pixel at the device-to-device
  copy rate measured in the same run (a 2 GiB torch copy), and ``map_over_floor``;
* ``predict_ms``: whole predicts (CUDA events, rounds alternating) with regions alone, with regions
  and the consecutive overlaps, and with regions and tracks (device track map), and what the tracks
  add over each of the first two.
The card's name, power limit and max SM clock are read in the same run.

  python tools/tracks_timing.py [--settings c2 c3 checker] [--calls 5] [--rounds 3] [--out FILE]
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
OWN = ("track_init_kernel", "track_link_kernel", "track_table_kernel", "track_map_kernel")
SHARED = ("region_number_kernel", "region_resolve_kernel")  # the second launch of each predict is the tracks'


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
    """Device µs per predict of the tracks' kernels."""
    ev = [e for e in prof.events() if e.device_type.name == "CUDA"]
    out = {}
    for base in OWN:
        t = [getattr(e, "device_time", None) or e.cuda_time for e in ev if base in e.name]
        if t:
            out[base] = float(np.sum(t) / calls)
    for base in SHARED:
        es = sorted((e for e in ev if base in e.name), key=lambda e: e.time_range.start)
        t = [getattr(e, "device_time", None) or e.cuda_time for e in es[1::2]]
        if t:
            out[base + " (tracks)"] = float(np.sum(t) / calls)
    return out


def run_setting(eng, name, D, H, W, k, centers, args, rate):
    import torch
    from torch.profiler import ProfilerActivity, profile

    stream = torch.cuda.current_stream()
    pairs = [(d, d + 1) for d in range(D - 1)]
    rmap = torch.empty(D * H * W, dtype=torch.int32, device="cuda")
    tmap = torch.empty(D * H * W, dtype=torch.int32, device="cuda")
    variants = {
        "regions": dict(),
        "regions_and_overlaps": dict(region_overlaps=pairs),
        "regions_and_tracks": dict(tracks=args.min_iou, track_map_out=tmap),
    }

    def predict(v):
        return eng.predict(centers, want_labels=False, regions=4, region_map_out=rmap, **variants[v])

    out = predict("regions_and_tracks")
    tracks, region_tracks = out[-2], out[-1]
    for v in variants:
        predict(v)
    ms = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:
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
            predict("regions_and_tracks")
        torch.cuda.synchronize()
    kt = kernel_times(prof, args.calls)
    map_us = kt.get("track_map_kernel", 0.0)
    floor_us = 8 * D * H * W / (rate * 1e9) * 1e6
    med = {v: float(np.median(t)) for v, t in ms.items()}
    return {
        "setting": name, "shape": [D, H, W], "k": k, "connectivity": 4, "min_iou": args.min_iou,
        "regions": int(region_tracks.shape[0]), "tracks": int(tracks.shape[0]),
        "branched": int(tracks[:, 6].sum()), "longest": int(tracks[:, 3].max()) if tracks.shape[0] else 0,
        "kernels_us": kt,
        "link_number_table_us": sum(v for n, v in kt.items() if n != "track_map_kernel"),
        "map_us": map_us, "map_floor_us": floor_us, "map_over_floor": map_us / floor_us if floor_us else None,
        "predict_ms": dict(med, added_over_regions=med["regions_and_tracks"] - med["regions"],
                           added_over_overlaps=med["regions_and_tracks"] - med["regions_and_overlaps"]),
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
    res = run_setting(eng, cfg, D, H, W, k, centers, args, rate)
    print(json.dumps(res), flush=True)
    eng.close()
    torch.cuda.empty_cache()
    return [res]


def run_checker(pkg, args, rate):
    """Identical one-pixel checkerboards on every day: labels by nearest z level."""
    import torch

    D, H, W = bench.CONFIGS["c2"][:3]
    yy = torch.arange(H, device="cuda").view(H, 1)
    xx = torch.arange(W, device="cuda").view(1, W)
    day = ((yy + xx) % 2).float() * 260.0 - 130.0
    hm = day.expand(D, H, W).contiguous()
    eng = pkg.Engine(0)
    eng.unproject(hm)
    del hm, day
    torch.cuda.empty_cache()
    centers = np.array([[W / 2.0, H / 2.0, -130.0], [W / 2.0, H / 2.0, 130.0]])
    res = run_setting(eng, "checker", D, H, W, 2, centers, args, rate)
    print(json.dumps(res), flush=True)
    eng.close()
    torch.cuda.empty_cache()
    return [res]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--settings", nargs="+", default=["c2", "c3", "checker"], choices=["c2", "c3", "checker"])
    ap.add_argument("--calls", type=int, default=5, help="predicts per round and in the trace")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-iou", type=float, default=0.5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    pkg = importlib.import_module(PKG)
    rate = copy_rate_GBps()
    results = []
    for s in args.settings:
        results += run_checker(pkg, args, rate) if s == "checker" else run_config(pkg, s, args, rate)
    out = {"card": card(), "copy_rate_GB_per_s": rate, "results": results,
           "note": "kernels_us: device time per predict (torch.profiler). map_floor_us: the track map pass reading "
                   "4 B and writing 4 B per pixel at the measured copy rate. predict_ms: whole predicts with regions "
                   "(region map on the device), medians of rounds."}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
