#!/usr/bin/env python
"""Cost of the connected regions of the cluster map (``regions=`` / ``return_regions``) on one GPU.

Config 2 of bench.py (10 x 2048 x 2048 float32 stack) with k = 16 (uint8 map) and k = 300 (uint16
map), and the one-GPU config-3 shape (20 x 1024 x 8192, k = 64), each at connectivity 4 and 8.
Centroids come from one fit of the bench's k (k = 300: points drawn from the cloud); the regions
are then taken by ``predict`` calls, whose cluster map is the one the fit's labels describe.

Reported per (config, k, connectivity), from a torch.profiler trace of ``--calls`` predicts with
regions (device time of each kernel, median over the calls):

* ``label_us``: the four labelling kernels (tile, border, number, resolve), and each of them;
* ``stats_us``: the pass over the points and the table kernel;
* ``floor_us``: reading the map once and writing the int32 region map once (5 B/pixel at uint8,
  6 at uint16) at the device-to-device copy rate measured in the same run (a 2 GiB torch copy,
  read + write bytes over its time), and ``label_over_floor``;
* ``predict_ms``: whole predicts without and with regions, CUDA events, and their difference.

It also checks, once per setting, the region count against scipy.ndimage.label on the cluster map
the same call returned (first two days).  The card's name and power limit are read in the same run.

  python tools/regions_timing.py [--configs c2 c3] [--calls 5] [--out FILE]
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
LABEL = ("region_tile_kernel", "region_border_kernel", "region_number_kernel", "region_resolve_kernel")
STATS = ("region_stats_kernel", "region_finish_kernel")


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
    """{kernel base name: median per-call device time (us)} from a trace of `calls` predicts."""
    out = {}
    for base in LABEL + STATS:
        ev = [e for e in prof.events() if base in e.name]
        if not ev:
            continue
        t = [getattr(e, "device_time", None) or e.cuda_time for e in ev]
        out[base] = float(np.sum(t) / calls)
    return out


def run_setting(pkg, eng, cfg, H, W, D, k, centers, conn, args, rate):
    import torch
    from scipy import ndimage
    from torch.profiler import ProfilerActivity, profile

    stream = torch.cuda.current_stream()
    elem = 1 if k <= 255 else 2
    cmap = torch.empty(D * H * W, dtype=torch.uint8 if elem == 1 else torch.int16, device="cuda")
    rmap = torch.empty(D * H * W, dtype=torch.int32, device="cuda")
    cm = cmap if elem == 1 else cmap.view(torch.uint16)
    out = eng.predict(centers, want_labels=False, cluster_map_out=cm, regions=conn, region_map_out=rmap)
    torch.cuda.synchronize()
    table = out[2]
    # the region count of the first two days against scipy on the returned map
    st = ndimage.generate_binary_structure(2, 1 if conn == 4 else 2)
    m = cmap.view(torch.int16).to(torch.int32) & 0xFFFF if elem == 2 else cmap.to(torch.int32)
    m2 = m[:2 * H * W].view(2, H, W).cpu().numpy()
    ref = sum(ndimage.label(m2[d] == v, structure=st)[1] for d in range(2) for v in np.unique(m2[d]) if v)
    ok = int(np.sum(table[:, 0] < 2)) == int(ref)
    del m, m2

    def predict(with_regions):
        return eng.predict(centers, want_labels=False, cluster_map_out=cm,
                           regions=conn if with_regions else None, region_map_out=rmap if with_regions else None)

    for v in (False, True):
        predict(v)
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
    label_us = sum(kt.get(b, 0.0) for b in LABEL)
    stats_us = sum(kt.get(b, 0.0) for b in STATS)
    floor_us = D * H * W * (elem + 4) / (rate * 1e9) * 1e6
    return {
        "config": cfg, "shape": [D, H, W], "k": k, "map_bytes_per_pixel": elem, "connectivity": conn,
        "regions": int(table.shape[0]), "region_count_equals_scipy_first_two_days": ok,
        "kernels_us": kt, "label_us": label_us, "stats_us": stats_us, "floor_us": floor_us,
        "label_over_floor": label_us / floor_us if floor_us else None,
        "predict_ms": {"without": float(np.median(ms[False])), "with_regions": float(np.median(ms[True])),
                       "added": float(np.median(ms[True]) - np.median(ms[False]))},
    }


def run_config(pkg, cfg, ks, args, rate):
    import torch

    D, H, W, k0, iters = bench.CONFIGS[cfg]
    eng = pkg.Engine(0)
    hm = pkg.make_stack(D, H, W, seed=0, device="cuda")
    n = eng.unproject(hm)
    del hm
    torch.cuda.empty_cache()
    rs = np.random.RandomState(0)
    init = eng.gather_points(np.sort(rs.choice(n, k0, replace=False))).astype(np.float64)
    fitted = eng.fit(init, max_iter=iters, tol=0.0, want_labels=False)["centers"]
    res = []
    for k in ks:
        centers = fitted if k == k0 else eng.gather_points(np.sort(rs.choice(n, k, replace=False))).astype(np.float64)
        for conn in (4, 8):
            res.append(run_setting(pkg, eng, cfg, H, W, D, k, centers, conn, args, rate))
            print(json.dumps(res[-1]), flush=True)
    eng.close()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["c2", "c3"], choices=["c2", "c3"])
    ap.add_argument("--calls", type=int, default=5, help="predicts per round and in the trace")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    pkg = importlib.import_module(PKG)
    rate = copy_rate_GBps()
    ks = {"c2": [16, 300], "c3": [64]}
    results = []
    for c in args.configs:
        results += run_config(pkg, c, ks[c], args, rate)
    out = {"card": card(), "copy_rate_GB_per_s": rate, "results": results,
           "note": "kernels_us: device time per predict (torch.profiler), summed over the launches of one call. "
                   "floor_us: map read once + int32 region map written once at the measured copy rate. "
                   "predict_ms: whole predicts (cluster map and region map to the device), medians of rounds."}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
