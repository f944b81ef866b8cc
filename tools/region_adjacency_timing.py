#!/usr/bin/env python
"""Cost of the region adjacency within a day (``region_adjacency=`` / ``return_region_adjacency``) on
one GPU.

Settings, each at connectivity 4 and 8:
* config 2 of bench.py (10 x 2048 x 2048, k = 16);
* the one-GPU config-3 shape (20 x 1024 x 8192, k = 64);
* the worst case at the config-2 geometry: 10 days of a one-pixel checkerboard (k = 2), at
  connectivity 4 -- every pixel is its own region and every edge of every day a row.
Centroids come from one fit of the bench's k; the adjacency is then taken by ``predict`` calls.

Reported per setting, from a torch.profiler trace of ``--calls`` predicts with regions and
adjacency (device time of each kernel, summed per call):
* ``kernels_us`` and ``adjacency_us``: the bound, insert, mark, scan, emit and finish kernels;
* ``floor_us``: the bound and insert passes each reading 4 B of ids per pixel, at the
  device-to-device copy rate measured in the same run (a 2 GiB torch copy), and ``over_floor``;
* ``rows`` (M), the bound in total (the run starts the bound pass counts, recomputed here with
  torch from the returned region map), and whether the rows equal those ``torch.unique`` finds on
  that map (the keys, their counts and their first edges);
* ``predict_ms``: whole predicts with a device region map, without and with adjacency (CUDA
  events, rounds alternating), and their difference.
The card's name, power limit and max SM clock are read in the same run.

  python tools/region_adjacency_timing.py [--settings c2 c3 checker] [--calls 5] [--out FILE]
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
KERNELS = ("adjacency_bound_kernel", "adjacency_insert_kernel", "overlap_mark_kernel", "overlap_scan_kernel",
           "adjacency_emit_kernel", "adjacency_finish_kernel")


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


def reference_rows(rmap, D, H, W):
    """The adjacency rows of the region map with torch.unique (as tests/test_region_adjacency.py
    does with numpy), and the run starts the bound pass counts."""
    import torch

    ids = rmap.view(D, H, W).to(torch.int64)
    px = torch.arange(H * W, device=rmap.device, dtype=torch.int64).view(H, W)
    out, bound = [], 0
    for d in range(D):
        day = ids[d]
        for a, b, x0 in ((day[:, :-1], day[:, 1:], px[:, :-1] % W == 0), (day[:-1, :], day[1:, :], px[:-1, :] % W == 0)):
            k = torch.where((a > 0) & (b > 0) & (a != b), torch.minimum(a, b) << 32 | torch.maximum(a, b), 0)
            left = torch.cat([torch.zeros_like(k[:, :1]), k[:, :-1]], dim=1)
            bound += int(((k != 0) & (x0 | (k != left))).sum())
        a = torch.cat([day[:, :-1].reshape(-1), day[:-1, :].reshape(-1)])
        b = torch.cat([day[:, 1:].reshape(-1), day[1:, :].reshape(-1)])
        e = torch.cat([(2 * px[:, :-1]).reshape(-1), (2 * px[:-1, :] + 1).reshape(-1)])
        m = (a > 0) & (b > 0) & (a != b)
        a, b, e = a[m], b[m], e[m]
        key = torch.minimum(a, b) << 32 | torch.maximum(a, b)
        u, inv, cnt = torch.unique(key, return_inverse=True, return_counts=True)
        first = torch.full_like(u, 2 * H * W).scatter_reduce(0, inv, e, reduce="amin")
        o = torch.argsort(first)
        u, first, cnt = u[o], first[o], cnt[o]
        out.append(torch.stack([torch.full_like(u, d), u >> 32, u & 0xFFFFFFFF, cnt, (first >> 1) // W,
                                (first >> 1) % W], dim=1))
    return torch.cat(out).cpu().numpy(), bound


def run_setting(eng, name, D, H, W, k, centers, conn, args, rate):
    import torch
    from torch.profiler import ProfilerActivity, profile

    stream = torch.cuda.current_stream()
    rmap = torch.empty(D * H * W, dtype=torch.int32, device="cuda")

    def predict(with_adjacency):
        return eng.predict(centers, want_labels=False, regions=conn, region_map_out=rmap,
                           region_adjacency=with_adjacency)

    rows = predict(True)[-2]
    torch.cuda.synchronize()
    ref, bound = reference_rows(rmap, D, H, W)
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
    adjacency_us = sum(kt.values())
    floor_us = 2 * 4 * H * W * D / (rate * 1e9) * 1e6
    return {
        "setting": name, "shape": [D, H, W], "k": k, "connectivity": conn,
        "rows": int(rows.shape[0]), "bound_total": bound,
        "rows_equal_torch_unique": bool(rows.shape == ref.shape and np.array_equal(rows, ref)),
        "kernels_us": kt, "adjacency_us": adjacency_us, "floor_us": floor_us,
        "over_floor": adjacency_us / floor_us if floor_us else None,
        "predict_ms": {"regions": float(np.median(ms[False])), "regions_and_adjacency": float(np.median(ms[True])),
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
    """One-pixel checkerboards: labels by nearest z level."""
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
                   "floor_us: bound and insert passes reading 4 B of ids per pixel each, at the measured copy rate. "
                   "predict_ms: whole predicts with regions (region map on the device), medians of rounds."}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
