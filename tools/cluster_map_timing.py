#!/usr/bin/env python
"""Cost of the cluster map (``cluster_map_out`` / ``return_cluster_map``) on one GPU.

Config 2 of bench.py by default (10 x 2048 x 2048 float32 stack, k = 16, 20 iterations, every
fit cold).  Blocks of fits without a map, with a device uint8 map and with a host uint8 map
alternate, so that drift of the card or the host hits every variant alike.  Reported per variant:

* ``final_ms``: the FINAL phase of mdkm_profile_* (the clear of the map and the final labelling
  pass, CUDA events), per fit;
* ``fit_ms``: whole fits, CUDA events on the handle's stream around each block;
* the end-to-end call (``fuse_multiday_kmeans`` from pinned host rasters, labels and cloud to the
  host) with and without ``return_cluster_map``, host clock, alternating.

It also checks, once, that the map of a config-2 fit equals the one built on the host from the
validity mask and the returned labels.  The card's name and power limit are read in the same run.

  python tools/cluster_map_timing.py [--config c2] [--rounds 4] [--fits 5] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(bench.CONFIGS))
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--fits", type=int, default=5, help="fits per variant and round")
    ap.add_argument("--e2e", type=int, default=3, help="end-to-end calls per variant and round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    pkg = importlib.import_module(PKG)
    D, H, W, k, iters = bench.CONFIGS[args.config]
    tol = bench.TOL.get(args.config, 0.0)
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
    map_dev = torch.empty(D * H * W, dtype=torch.uint8, device="cuda")
    map_host = np.empty(D * H * W, dtype=np.uint8)
    outs = {"none": None, "device": map_dev, "host": map_host}

    def fit(variant):
        eng.drop_caches()
        return eng.fit(init, max_iter=iters, tol=tol, labels_out=labels_dev, cluster_map_out=outs[variant])

    # the map of one fit against the validity mask and the labels (host reference)
    fit("host")
    hv = hm_host.numpy().reshape(-1)
    valid = np.isfinite(hv) & (np.abs(hv) <= 144.0)
    ref = np.zeros(D * H * W, dtype=np.uint8)
    ref[valid] = labels_dev.cpu().numpy() + 1
    map_ok = bool(np.array_equal(ref, map_host))
    fit("device")
    torch.cuda.synchronize()
    map_ok = map_ok and bool(np.array_equal(ref, map_dev.cpu().numpy()))
    del ref, hv, valid

    for v in outs:  # warm-up
        for _ in range(2):
            fit(v)
    res = {v: {"final_ms": [], "fit_ms": []} for v in outs}
    for _ in range(args.rounds):
        for v in outs:
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

    def e2e(with_map):
        return pkg.fuse_multiday_kmeans(hm_host, n_clusters=k, init=init, max_iter=iters, tol=tol, engine=eng,
                                        return_cluster_map=with_map)

    e2e_ms = {"without_map": [], "with_map": []}
    for with_map in (False, True):
        e2e(with_map)
    for _ in range(args.rounds):
        for with_map in (False, True):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.e2e):
                e2e(with_map)
            e2e_ms["with_map" if with_map else "without_map"].append((time.perf_counter() - t0) * 1e3 / args.e2e)
    eng.close()

    def summary(xs):
        return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "runs": xs}

    out = {
        "card": card(), "config": args.config, "shape": [D, H, W], "k": k, "iters": iters, "points": n,
        "map_bytes": D * H * W, "map_equals_host_reference": map_ok,
        "rounds": args.rounds, "fits_per_round": args.fits,
        "final_ms": {v: summary(res[v]["final_ms"]) for v in outs},
        "fit_ms": {v: summary(res[v]["fit_ms"]) for v in outs},
        "e2e_ms": {v: summary(x) for v, x in e2e_ms.items()},
        "note": "final_ms: the FINAL phase (map clear + final pass; for 'host' the copy is outside it). "
                "fit_ms: whole cold fits, labels to the device; 'host' includes the map's device-to-host copy. "
                "e2e_ms: fuse_multiday_kmeans from pinned host rasters, host clock.",
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
