#!/usr/bin/env python
"""Cost of the per-day cluster statistics (``day_stats=True`` / ``return_day_stats``) on one GPU.

Configs 2 (10 x 2048 x 2048 float32 stack, k = 16) and 4 (12 x 4096 x 4096, k = 1024) of bench.py
by default, every fit cold.  In one process, blocks of fits without and with statistics
alternate, so that drift of the card or the host hits both alike.  Reported per config and
setting:

* ``final_ms``: the FINAL phase of mdkm_profile_* (CUDA events around the final pass; with
  statistics also the clear of the slots), per fit;
* ``fit_ms``: whole fits, CUDA events on the handle's stream around each block;
* ``e2e_ms``: the end-to-end call (``fuse_multiday_kmeans`` from pinned host rasters, labels and
  cloud to the host) without and with ``return_day_stats``, host clock, alternating.

It also checks, once per config, that the counts equal a bincount of the returned labels.  The
card's name and power limit are read in the same run.

  python tools/day_stats_timing.py [--configs c2 c4] [--rounds 4] [--fits 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

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

    D, H, W, k, iters = bench.CONFIGS[cfg]
    tol = bench.TOL.get(cfg, 0.0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(0, stream=stream, pinned_results=True)
    hm = pkg.make_stack(D, H, W, seed=0, device="cuda")
    torch.cuda.synchronize()
    hm_host = torch.empty(hm.shape, dtype=torch.float32, pin_memory=True)
    hm_host.copy_(hm)
    n = eng.unproject(hm)
    del hm
    torch.cuda.empty_cache()
    init = eng.gather_points(np.sort(np.random.RandomState(0).choice(n, k, replace=False))).astype(np.float64)
    labels_dev = torch.empty(n, dtype=torch.int32, device="cuda")

    def fit(stats):
        eng.drop_caches()
        return eng.fit(init, max_iter=iters, tol=tol, labels_out=labels_dev, day_stats=stats)

    r = fit(True)
    torch.cuda.synchronize()
    seg = eng.segment_offsets
    day = np.repeat(np.arange(len(seg) - 1), np.diff(seg))
    ref = np.bincount(day * k + labels_dev.cpu().numpy(), minlength=D * k).reshape(D, k)
    counts_ok = bool(np.array_equal(ref, r["day_counts"]))
    del ref, day

    variants = (False, True)
    for v in variants:  # warm-up
        for _ in range(2):
            fit(v)
    res = {v: {"final_ms": [], "fit_ms": []} for v in variants}
    for _ in range(args.rounds):
        for v in variants:
            eng.profile(True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(args.fits):
                fit(v)
            e1.record(stream)
            torch.cuda.synchronize()
            ph = eng.profile_phases()
            eng.profile(False)
            res[v]["final_ms"].append(ph["final"][0] / args.fits)
            res[v]["fit_ms"].append(e0.elapsed_time(e1) / args.fits)

    def e2e(stats):
        return pkg.fuse_multiday_kmeans(hm_host, n_clusters=k, init=init, max_iter=iters, tol=tol, engine=eng,
                                        return_day_stats=stats)

    e2e_ms = {v: [] for v in variants}
    for v in variants:
        e2e(v)
    for _ in range(args.rounds):
        for v in variants:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.e2e):
                e2e(v)
            e2e_ms[v].append((time.perf_counter() - t0) * 1e3 / args.e2e)
    eng.close()
    name = {False: "without", True: "with_stats"}
    return {
        "config": cfg, "shape": [D, H, W], "k": k, "iters": iters, "points": n, "slots": D * k,
        "counts_equal_bincount": counts_ok, "rounds": args.rounds, "fits_per_round": args.fits,
        "final_ms": {name[v]: summary(res[v]["final_ms"]) for v in variants},
        "fit_ms": {name[v]: summary(res[v]["fit_ms"]) for v in variants},
        "e2e_ms": {name[v]: summary(e2e_ms[v]) for v in variants},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["c2", "c4"], choices=sorted(bench.CONFIGS))
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--fits", type=int, default=5, help="fits per setting and round")
    ap.add_argument("--e2e", type=int, default=3, help="end-to-end calls per setting and round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    pkg = importlib.import_module(PKG)
    out = {"card": card(), "results": [run_config(pkg, c, args) for c in args.configs],
           "note": "final_ms: the FINAL phase (with statistics: the clear of the slots + the final pass). "
                   "fit_ms: whole cold fits, labels to the device. "
                   "e2e_ms: fuse_multiday_kmeans from pinned host rasters, host clock."}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
