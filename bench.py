#!/usr/bin/env python
"""bench.py -- k-means points*iterations/s of the multi-day fusion path on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + what the last step returned

A "step" is one complete Lloyd fit (BASELINE.json configs[1]: a 10-day 2048x2048 height-map
stack per GPU, ~41.9 M pixels, k = 16, 20 iterations, tol = 0) over points already resident
in HBM, labels written to a device buffer; `value` = points * iterations of all ranks / device
time (CUDA events, max over ranks).  `e2e` is the same metric through the public Python API
with pinned HOST rasters in and host labels / centroids / fused cloud out.  One JSON line is
printed by rank 0.  Sub-records of `roofline` say what the numbers are made of: the phases of a
fit, the share of group-iterations settled without reading a point, the streaming path with
settling disabled, and a cloud on which neither settling nor pruning can help (brute force).
With `--dump-outputs DIR`, rank 0 writes what its last timed fit and its last end-to-end call
returned as `DIR/<name>.npy` (float32 / float64, per-point arrays at a fixed seeded sample of
points), so that two builds can be compared output for output on identical inputs.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "3d-point-cloud-multiday-imagery_b200"

METRIC = "kmeans_points_iters_per_sec"
UNIT = "points*iters/s"
ALGO_BYTES_PER_POINT_ITER = 16.0  # SURVEY.md 8(d): 12 B xyz read + 4 B label write
ALGO_BYTES_PER_PIXEL_UNPROJECT = 16.0  # SURVEY.md 8(d): 4 B height read + 12 B xyz write, once

CONFIGS = {
    # name: (days per GPU, H, W, k, iters)
    "c1": (3, 512, 512, 8, 20),
    "c2": (10, 2048, 2048, 16, 20),
    # one rank's share of config 3 as whole "days" of 1024 rows (single-GPU profiling aid; the
    # real config 3 -- row bands of a 20 x 8192 x 8192 stack -- is the `config3` sub-record of
    # every multi-GPU line, see run_config3)
    "c3": (20, 1024, 8192, 64, 20),
    "c4": (12, 4096, 4096, 1024, 10),
    "c5": (30, 4096, 4096, 32, 300),
}
# relative tolerance of the convergence test (sklearn's tol); config 5 is the time-to-solution run
TOL = {"c5": 1e-4}
C3 = {"D": 20, "H": 8192, "W": 8192, "k": 64, "iters": 20, "n_buildings": 1024}
# --dump-outputs: per-point arrays of more points than this are written at a seeded sample of this
# many points (config 2: ~29 MB in all instead of ~1.1 GB)
DUMP_POINTS = 1 << 20


def workload_name(cfg, n_gpus):
    D, H, W, k, it = CONFIGS[cfg]
    tol = TOL.get(cfg, 0.0)
    iters = f"{it} Lloyd iters, tol=0" if tol == 0 else f"max_iter={it}, tol={tol:g} (time to solution)"
    return (f"{cfg}: synthetic {D}-day {H}x{W} height-map stack per GPU (~{D*H*W*0.975/1e6:.1f}M pts/GPU), "
            f"k={k}, {iters}, {n_gpus} GPU(s)")


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_ev = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_ev.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self._stop_ev.set()
        if self.is_alive():
            self.join(timeout=2)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def measured_traffic(cfg):
    """DRAM bytes per Lloyd iteration from the committed ncu --set full capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))[cfg]
        return float(t["dram_bytes_per_iteration"]), t.get("source", "")
    except Exception:
        return None, None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------
# reference arm: scikit-learn, the implementation the reference calls (core.py:227-228)
# ---------------------------------------------------------------------------------------
def use_all_host_threads():
    """sklearn's Lloyd loop runs on OpenMP threads; torchrun exports OMP_NUM_THREADS=1 to its
    workers, so the thread count is set explicitly (threadpoolctl -> omp_set_num_threads) to the
    cores this process may run on.  Returns (limiter kept alive by the caller, cores)."""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)
    try:
        from threadpoolctl import threadpool_limits

        return threadpool_limits(limits=cores), cores
    except Exception:
        return None, cores


def cpu_workload(pkg, cfg, seed=0):
    """The FULL workload of `cfg` on the host: the same generator, every day, every point."""
    from oracle import unproject_oracle as UO

    D, H, W, k, iters = CONFIGS[cfg]
    D_fit = D if D * H * W <= (1 << 26) else max(1, (1 << 26) // (H * W))  # f64 + sklearn's own copy must fit the host
    P = UO.unproject_stack(pkg.make_stack(D_fit, H, W, seed=seed).numpy())
    if D_fit == D:
        sample = f"the full {D}-day {H}x{W} stack ({P.shape[0]} pts), k={k}, {iters} iters, float64"
    else:
        sample = f"the first {D_fit} of {D} days of the {H}x{W} stack ({P.shape[0]} pts), k={k}, {iters} iters, float64"
    init = pkg.init_from_points(P.astype(np.float32), k, seed)
    return P, init, k, iters, sample


def time_cpu_reference(P, init, iters, repeats, tol=0.0):
    """Returns (best pts*it/s, kind, cores).  sklearn when importable, else the C port."""
    from oracle import sklearn_ref

    if sklearn_ref.available():
        best = 0.0
        for _ in range(repeats):
            r = sklearn_ref.fit(P, init, max_iter=iters, tol=tol)
            best = max(best, P.shape[0] * r["n_iter"] / r["wall_s"])
        return best, "reference", sklearn_ref.n_threads()
    from oracle import c_oracle, kmeans_oracle as KO

    P32 = P.astype(np.float32)
    x, y, z = (np.ascontiguousarray(P32[:, i]) for i in range(3))
    best = 0.0
    for _ in range(repeats):
        c = init.copy()
        t0 = time.perf_counter()
        for _it in range(iters):
            _, sums, counts, _ = c_oracle.lloyd_step_f32soa(x, y, z, c)
            KO.average_centers(sums, counts)
            c = sums
        best = max(best, P.shape[0] * iters / (time.perf_counter() - t0))
    return best, "port", c_oracle.num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    limiter, _ = use_all_host_threads()
    pkg = importlib.import_module(PKG)
    P, init, k, iters, sample = cpu_workload(pkg, args.config)
    from oracle import sklearn_ref

    kind = "reference" if sklearn_ref.available() else "port"
    tol = TOL.get(args.config, 0.0)
    for _ in range(args.warmup):
        time_cpu_reference(P, init, iters, 1, tol)
    t0 = time.perf_counter()
    secs = 0.0
    cores = 1
    for _ in range(args.steps):
        v, kind, cores = time_cpu_reference(P, init, iters, 1, tol)  # v = points * n_iter / wall of that fit
        secs += 1.0 / v
    wall = time.perf_counter() - t0
    value = args.steps / secs  # harmonic mean of the fits' rates = total point-iterations / total fit time
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(args.config, args.gpus), "sample": sample,
                   "implementation": "sklearn.cluster.KMeans(algorithm='lloyd', n_init=1, init=array) float64"
                   if kind == "reference" else "oracle/lloyd_oracle.c (C port, OpenMP)",
                   "note": "one GPU's share of the workload, whatever --gpus says: the CPU arm does not shard"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    del limiter
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------
def dump_sample(n, seed):
    """Sorted indices of the points whose per-point outputs --dump-outputs writes: every point,
    or DUMP_POINTS of them drawn with `seed` (the same draw for the same arguments)."""
    if n <= DUMP_POINTS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).choice(n, DUMP_POINTS, replace=False))


def fit_outputs(prefix, labels, centroids, inertia, n_iter):
    """What a fit returns, as the float arrays --dump-outputs writes (labels < k fit float32 exactly)."""
    return {prefix + "labels": np.asarray(labels).astype(np.float32),
            prefix + "centroids": np.asarray(centroids, dtype=np.float64),
            prefix + "inertia": np.array([inertia], dtype=np.float64),
            prefix + "n_iter": np.array([n_iter], dtype=np.float64)}


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def all_ranks_equal(t, world, dist):
    """True when the byte pattern of tensor `t` (CUDA) is identical on every rank."""
    import torch

    if world == 1:
        return True
    flat = t.contiguous().view(torch.uint8).reshape(-1)
    parts = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(parts, flat)
    return all(bool(torch.equal(parts[0], p)) for p in parts[1:])


def check_n_rank_equals_1_rank(pkg, eng, rank, world, local, seed):
    """Untimed: a config-1-size stack (3 x 512 x 512, k = 8, 20 iterations) clustered by the N
    ranks together (row-band shards, the exchange path the timed runs use) and by ONE rank alone.
    Sums are integers, so centroids must agree bit for bit, and so must n_iter, inertia (fixed
    order per rank, summed by NCCL: compared to 1e-12) and every rank's labels."""
    import torch
    import torch.distributed as dist

    D, H, W, k, iters = CONFIGS["c1"]
    hm = pkg.make_stack(D, H, W, seed=seed + 101, device=f"cuda:{local}")  # same bytes on every rank
    with pkg.Engine(local) as solo:
        n_all = solo.unproject(hm)
        init = solo.gather_points(np.sort(np.random.RandomState(seed).choice(n_all, k, replace=False))).astype(np.float64)
        ref = solo.fit(init, max_iter=iters, tol=0.0)
        ref_labels = ref["labels"].copy()
        cloud_all = solo.get_cloud(False).copy()
    b, e = pkg.shard_range(D * H * W, rank, world, align=W)
    n_loc = eng.unproject(hm.reshape(-1)[b:e], stack_shape=(D, H, W), pix_begin=b)
    r = eng.fit(init, max_iter=iters, tol=0.0)
    sizes = torch.zeros(world, dtype=torch.int64, device=f"cuda:{local}")
    sizes[rank] = n_loc
    dist.all_reduce(sizes)
    off = int(sizes[:rank].sum().item())
    ok = (r["centers"].tobytes() == ref["centers"].tobytes() and r["n_iter"] == ref["n_iter"]
          and int(sizes.sum().item()) == n_all
          and np.array_equal(r["labels"], ref_labels[off:off + n_loc])
          and np.array_equal(eng.get_cloud(False), cloud_all[off:off + n_loc])
          and abs(r["inertia"] - ref["inertia"]) <= 1e-12 * abs(ref["inertia"]))
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=f"cuda:{local}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item()), {"points": n_all, "n_iter": ref["n_iter"]}


def run_config3(pkg, eng, rank, world, local, seed, steps):
    """BASELINE.json configs[2] as it is written: a 20-day 8192 x 8192 stack (1.34 G pixels), k = 64,
    20 iterations, sharded over the ranks by ROW BANDS (contiguous pixel ranges cut on row
    boundaries, so a rank's range starts and ends inside days), generated per shard on the device."""
    import torch
    import torch.distributed as dist

    D, H, W, k, iters = C3["D"], C3["H"], C3["W"], C3["k"], C3["iters"]
    b, e = pkg.shard_range(D * H * W, rank, world, align=W)
    hm = pkg.make_stack_range(D, H, W, b, e - b, seed=seed, device=f"cuda:{local}", n_buildings=C3["n_buildings"])
    n_loc = eng.unproject(hm, stack_shape=(D, H, W), pix_begin=b)
    del hm
    torch.cuda.empty_cache()
    n_total = eng.n_points_global
    init = eng.gather_points(np.sort(np.random.RandomState(seed).choice(n_total, k, replace=False))).astype(np.float64)
    labels = torch.empty(n_loc, dtype=torch.int32, device=f"cuda:{local}")
    stream = torch.cuda.current_stream()

    def one_fit():
        eng.drop_caches()
        return eng.fit(init, max_iter=iters, tol=0.0, labels_out=labels)

    for _ in range(3):
        r = one_fit()
    eng.profile(True)
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    its = 0
    for _ in range(steps):
        r = one_fit()
        its += r["n_iter"]
    e1.record(stream)
    dist.barrier()
    torch.cuda.synchronize()
    ph = eng.profile_phases()
    eng.profile(False)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    same = all_ranks_equal(torch.from_numpy(r["centers"]).to(f"cuda:{local}"), world, dist)
    ms_fit = float(ms.item()) / steps
    del labels
    torch.cuda.empty_cache()
    return {
        "workload": f"c3: synthetic {D}-day {H}x{W} stack ({n_total} pts), k={k}, {iters} Lloyd iters, tol=0, "
                    f"row-band shards over {world} GPUs (every fit cold: mirror + summaries rebuilt)",
        "points_total": n_total, "points_rank0": n_loc, "value": n_total * its / (float(ms.item()) * 1e-3), "unit": UNIT,
        "ms_per_fit": ms_fit, "n_iter": r["n_iter"], "steps": steps,
        "step_kernel_ms": ph["step"][0] / max(1, ph["step"][1]),
        "build_ms_per_fit": ph["build"][0] / steps, "final_ms_per_fit": ph["final"][0] / steps,
        "settled_frac": 1.0 - r["worklist_groups"] / max(1, r["groups"] * r["n_iter"]),
        "cross_rank_bitwise": bool(same), "exchange": "nvlink_p2p" if eng.p2p else "nccl",
    }


def run_mine(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module(PKG)

    D, H, W, k, iters = CONFIGS[args.config]
    tol = TOL.get(args.config, 0.0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(local, stream=stream, pinned_results=True)
    pkg.init_engine_comm(eng, rank, world)

    # ---- multi-GPU correctness, untimed: N ranks == 1 rank, bit for bit ----------------------
    n_vs_1 = None
    if world > 1:
        n_vs_1, n_vs_1_info = check_n_rank_equals_1_rank(pkg, eng, rank, world, local, args.seed)

    # synthetic stack of this rank's days, generated on the device (seed differs per rank)
    hm = pkg.make_stack(D, H, W, seed=args.seed + rank, device=dev)
    torch.cuda.synchronize()
    hm_host = torch.empty(hm.shape, dtype=torch.float32, pin_memory=True)
    hm_host.copy_(hm)
    torch.cuda.synchronize()
    pix0 = rank * D * H * W
    # unprojection from device-resident rasters, timed on its own (kernels only, CUDA events)
    n_local = eng.unproject(hm, stack_shape=(D * world, H, W), pix_begin=pix0)  # warm-up (module load, allocations)
    eng.profile(True)
    for _ in range(4):
        n_local = eng.unproject(hm, stack_shape=(D * world, H, W), pix_begin=pix0)
    un_ms, un_px = eng.profile_phases()["unproject"]
    eng.profile(False)
    del hm
    torch.cuda.empty_cache()

    # identical initial centroids on every rank: k points of the global cloud (gather_points is
    # a collective with global indices, so every rank makes the same call)
    n_total = eng.n_points_global
    idx = np.sort(np.random.RandomState(args.seed).choice(n_total, k, replace=False))
    init_np = eng.gather_points(idx).astype(np.float64)
    labels_dev = torch.empty(n_local, dtype=torch.int32, device=dev)  # the fit's int32 labels land here

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_fit():
        # every timed fit starts cold: the per-cloud acceleration structures (tile-ordered mirror,
        # group summaries) are rebuilt inside the timed region, nothing is carried over
        if not args.keep_caches:
            eng.drop_caches()
        return eng.fit(init_np, max_iter=iters, tol=tol, labels_out=labels_dev)

    # ---- kernel-resident number: K fits over resident points --------------------------------
    for _ in range(args.warmup):
        r = one_fit()
    eng.profile_read()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    n_iter_sum = 0
    for _ in range(args.steps):
        r = one_fit()
        n_iter_sum += r["n_iter"]
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    _, _, launches = eng.profile_read()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = n_total * n_iter_sum / (ms_total * 1e-3)
    # every rank must hold the same centroids / n_iter / inertia after the timed fits
    cross = None
    if world > 1:
        sig = torch.from_numpy(np.concatenate([r["centers"].reshape(-1), [float(r["n_iter"]), r["inertia"]]])).to(dev)
        cross = all_ranks_equal(sig, world, dist)
    # what the last timed fit returned, taken before later fits overwrite labels_dev
    dumps = None
    if args.dump_outputs and rank == 0:
        sel = dump_sample(n_local, args.seed)
        labels_sel = labels_dev[torch.from_numpy(sel).to(dev)].cpu().numpy()
        dumps = {"point_index": sel.astype(np.float64),
                 **fit_outputs("", labels_sel, r["centers"], r["inertia"], r["n_iter"])}

    # ---- the phases of a fit and the dominant kernel, timed alone with CUDA events ------------
    eng.profile(True)
    n_prof = 3
    for _ in range(n_prof):
        r = one_fit()
    ph = eng.profile_phases()
    eng.profile(False)
    peak, peak_src = measured_peak()
    step_avg_ms = ph["step"][0] / max(ph["step"][1], 1)
    step_src = "CUDA-event spans around the batches of step launches (mdkm_profile_*)"
    if world > 1:
        # with several ranks the spans of the profiling loop also contain the wait for the slowest rank's
        # per-cloud build (the ranks restart every fit from their hosts): take the iteration time from the
        # timed region instead -- what is left of a fit after this rank's build and final pass
        fit_ms = ms_total / max(args.steps, 1)
        step_avg_ms = max(fit_ms - ph["build"][0] / n_prof - ph["final"][0] / n_prof, 0.0) / max(n_iter_sum / max(args.steps, 1), 1)
        step_src = "(timed fit - this rank's build and final-pass spans) / iterations"
    achieved = ALGO_BYTES_PER_POINT_ITER * n_local / (step_avg_ms * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic(args.config)
    dram_gbs = (traffic / (step_avg_ms * 1e-3) / 1e9) if traffic else None
    sm_clock = (clocks.get("sm_mhz") or 1965) * 1e6
    fma_peak = 148 * 128 * sm_clock  # FP32 FMA lanes x clock (CUDA cores; contraction depth 3)
    settled = 1.0 - r["worklist_groups"] / max(1, r["groups"] * r["n_iter"])
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_src,
        "dram_gbs": dram_gbs, "dram_frac": (dram_gbs / peak) if dram_gbs else None,
        "kernel": "lloyd_step_kernel = one Lloyd iteration (deferred centroid update of the previous iteration in the prologue, classification pass, grid barrier, per-point pass)",
        "avg_launch_ms": step_avg_ms, "avg_launch_source": step_src,
        "algorithmic_bytes_per_launch": ALGO_BYTES_PER_POINT_ITER * n_local, "peak_source": peak_src,
        "note": "achieved = 16 B x points / measured iteration time. frac > 1 is NOT an HBM utilisation: groups whose "
                "bounding box one centroid owns are settled from cached summaries without reading their points "
                "(settled_frac of all group-iterations), an exact pruning; `stream_all` below is the same kernel with "
                "settling disabled (every point read every iteration) and `bruteforce` a cloud where no pruning applies",
        "settled_frac": settled,
        "worklist_groups_per_iter": r["worklist_groups"] / max(1, r["n_iter"]), "groups": r["groups"],
        "fma_bound_points_iters_per_s": fma_peak / (3 * k),
        "phases_ms_per_fit": {"build_mirror_and_summaries": ph["build"][0] / n_prof,
                              "step_kernels": step_avg_ms * (n_iter_sum / max(args.steps, 1)) if world > 1 else ph["step"][0] / n_prof,
                              "final_labels_inertia": ph["final"][0] / n_prof,
                              "fit_total": ms_total / args.steps},
        "unproject": {
            "kernels": "unproject_fused_kernel (one pass: validity, rank, decoupled look-back, x/y/z runs) on device-resident rasters",
            "ms": un_ms / 4, "pixels": un_px // 4,
            "achieved": ALGO_BYTES_PER_PIXEL_UNPROJECT * (un_px / 4) / (un_ms / 4 * 1e-3) / 1e9 if un_ms > 0 else None,
            "frac": (ALGO_BYTES_PER_PIXEL_UNPROJECT * (un_px / 4) / (un_ms / 4 * 1e-3) / 1e9 / peak) if un_ms > 0 else None,
            "unit": "GB/s", "algorithmic_bytes_per_pixel": ALGO_BYTES_PER_PIXEL_UNPROJECT},
    }

    # ---- the streaming path: settling disabled, every point read and assigned per iteration -----
    if not args.no_stream_all:
        eng.settle_groups(False)
        try:
            for _ in range(2):
                one_fit()
            eng.profile(True)
            t_e0, t_e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            t_e0.record(stream)
            for _ in range(3):
                rs = one_fit()
            t_e1.record(stream)
            barrier()
            ph_s = eng.profile_phases()
            eng.profile(False)
        finally:
            eng.settle_groups(True)
        s_ms = ph_s["step"][0] / max(ph_s["step"][1], 1)
        s_gbs = ALGO_BYTES_PER_POINT_ITER * n_local / (s_ms * 1e-3) / 1e9
        roofline["stream_all"] = {
            "what": "same cloud, same kernel, MDKM_OPT_SETTLE_GROUPS=0: every group on the worklist, every point "
                    "fetched (1-D TMA) and assigned in every iteration; candidate pruning per group still applies",
            "avg_launch_ms": s_ms, "achieved": s_gbs, "frac": s_gbs / peak, "unit": "GB/s",
            "points_iters_per_s": n_local / (s_ms * 1e-3),
            "fit_ms": t_e0.elapsed_time(t_e1) / 3,
            "identical_results": bool(rs["centers"].tobytes() == r["centers"].tobytes() and rs["n_iter"] == r["n_iter"]),
            "worklist_groups_per_iter": rs["worklist_groups"] / max(1, rs["n_iter"]),
        }

    # ---- end to end through the public API: pinned host rasters in, host results out ------------
    def one_e2e():
        return pkg.fuse_multiday_kmeans(hm_host, n_clusters=k, init=init_np, max_iter=iters, tol=tol,
                                        engine=eng, stack_shape=(D * world, H, W), pix_begin=pix0)

    e2e = None
    if not args.no_e2e:
        for _ in range(max(1, args.warmup - 1)):
            res = one_e2e()
        barrier()
        t0 = time.perf_counter()
        its = 0
        for _ in range(args.steps):
            res = one_e2e()
            its += res.n_iter
        barrier()
        wall = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if dumps is not None:
            dumps.update(fit_outputs("e2e_", res.labels[sel], res.centroids, res.inertia, res.n_iter))
            dumps["e2e_fused_cloud"] = res.fused_cloud[sel].astype(np.float32)
        if world > 1:
            dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        e2e = {"value": n_total * its / float(wall.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(hm_host.numel() * 4 + init_np.nbytes),
               "d2h_bytes_per_step": int(res.labels.nbytes + res.centroids.nbytes + res.fused_cloud.nbytes),
               "ms_per_step": 1e3 * float(wall.item()) / args.steps,
               "returns": "labels int32[N], centroids f64[K,3], fused cloud f32[N,3]"}
        # what the host allows: the same byte counts as raw pinned copies, both directions at once,
        # all ranks together (no kernels at all) -- the end-to-end call cannot be faster than this
        d2h_n, h2d_n = e2e["d2h_bytes_per_step"], e2e["h2d_bytes_per_step"]
        fl_src = torch.empty(d2h_n, dtype=torch.uint8, device=dev)
        fl_dst = torch.empty(d2h_n, dtype=torch.uint8, pin_memory=True)
        fl_in = torch.empty(hm_host.numel() * 4, dtype=torch.uint8, device=dev)
        s_a, s_b = torch.cuda.Stream(), torch.cuda.Stream()

        def raw_copies():
            with torch.cuda.stream(s_a):
                fl_dst.copy_(fl_src, non_blocking=True)
            with torch.cuda.stream(s_b):
                fl_in.copy_(hm_host.view(torch.uint8).reshape(-1), non_blocking=True)
            s_a.synchronize()
            s_b.synchronize()

        raw_copies()
        barrier()
        t0 = time.perf_counter()
        for _ in range(5):
            raw_copies()
        barrier()
        fl = torch.tensor([(time.perf_counter() - t0) / 5], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(fl, op=dist.ReduceOp.MAX)
        e2e["floor_ms_raw_pinned_copies"] = 1e3 * float(fl.item())
        e2e["floor_note"] = (f"{d2h_n} B device->host + {h2d_n} B host->device per rank as plain pinned cudaMemcpyAsync, "
                             f"all {world} rank(s) at once, no kernels: the host's PCIe / memory path sets this")
        e2e["ms_over_floor"] = e2e["ms_per_step"] / e2e["floor_ms_raw_pinned_copies"]
        del fl_src, fl_dst, fl_in
        torch.cuda.empty_cache()

    # ---- brute force: a cloud on which neither settling nor candidate pruning can help -----------
    # (x, y squeezed to a thousandth of the z range: every x-y tile of the mirror spans all the
    # clusters, every centroid is a candidate of every group -> k distance evaluations per point)
    if world == 1 and not args.no_bruteforce:
        cloud = torch.empty((n_local, 3), dtype=torch.float32, device=dev)
        eng.get_cloud(napari_order=False, out=cloud)
        cloud[:, 0] *= 1.0 / 8192.0
        cloud[:, 1] *= 1.0 / 8192.0
        eng.set_points(cloud)
        del cloud
        torch.cuda.empty_cache()
        init_b = eng.gather_points(idx).astype(np.float64)
        b_iters = min(iters, 10)
        for _ in range(2):
            eng.fit(init_b, max_iter=b_iters, tol=0.0, labels_out=labels_dev)
        eng.profile(True)
        for _ in range(2):
            rb = eng.fit(init_b, max_iter=b_iters, tol=0.0, labels_out=labels_dev)
        ph_b = eng.profile_phases()
        eng.profile(False)
        b_ms = ph_b["step"][0] / max(ph_b["step"][1], 1)
        b_rate = n_local / (b_ms * 1e-3)
        roofline["bruteforce"] = {
            "what": f"the same {n_local} points with x, y scaled by 1/8192 (clusters are z-slabs): no group can be settled, "
                    f"all k={k} centroids are candidates of every group",
            "avg_launch_ms": b_ms, "points_iters_per_s": b_rate,
            "hbm_achieved": ALGO_BYTES_PER_POINT_ITER * b_rate / 1e9, "hbm_frac": ALGO_BYTES_PER_POINT_ITER * b_rate / 1e9 / peak,
            "fma_achieved_per_s": 3.0 * k * b_rate, "fma_peak_per_s": fma_peak, "fma_frac": 3.0 * k * b_rate / fma_peak,
            "binding": "hbm" if peak * 1e9 / ALGO_BYTES_PER_POINT_ITER < fma_peak / (3 * k) else "fp32_fma",
            "settled_frac": 1.0 - rb["worklist_groups"] / max(1, rb["groups"] * rb["n_iter"]),
            "n_refined": rb["n_refined"],
        }

    # ---- BASELINE.json configs[2] as written (multi-GPU lines only) -----------------------------
    c3 = None
    if world > 1 and not args.no_c3 and args.config == "c2":
        c3 = run_config3(pkg, eng, rank, world, local, args.seed, steps=max(3, min(args.steps, 10)))

    # ---- CPU baseline (rank 0, N = 1 only): the reference's sklearn path on the same workload ---
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        limiter, _ = use_all_host_threads()
        P, init_c, _, it_c, sample = cpu_workload(pkg, args.config, args.seed)
        time_cpu_reference(P[: P.shape[0] // 10], init_c, 2, 1, tol)  # threads up, pages touched
        v, kind, cores = time_cpu_reference(P, init_c, it_c, 1, tol)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
        del limiter, P

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.config, world), "points_total": n_total,
                       "iters_per_step": n_iter_sum / args.steps, "l2_policy": "inputs_exceed_l2 "
                       f"({n_local * 12 / 1e6:.0f} MB of xyz per GPU vs 126 MB L2; a cold fit reads them three times "
                       "-- build, summaries, final pass -- and the iterations read the summaries and boundary groups)",
                       "per_cloud_structures": "kept across fits" if args.keep_caches else
                       "rebuilt inside every timed fit (mirror + group summaries)",
                       "outputs_in_timed_region": "int32 labels [N] into a device buffer, centroids, inertia, n_iter",
                       "exchange": ("none" if world == 1 else
                                    "in-kernel NVLink peer exchange of K*4+8 int64 per iteration (CUDA IPC), no NCCL"
                                    if eng.p2p else "ncclAllReduce of K*4+8 int64 per iteration")},
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "e2e": e2e,
            "gpu_launches": launches,
        }
        if world > 1:
            line["cross_rank_bitwise"] = bool(cross)
            line["n_rank_equals_1_rank"] = {"ok": bool(n_vs_1), **n_vs_1_info,
                                            "what": "c1-size stack: N-rank fit vs 1-rank fit -- centroids bitwise, "
                                                    "n_iter, labels, cloud, inertia to 1e-12"}
            line["config3"] = c3
        if dumps is not None:
            write_outputs(args.dump_outputs, dumps)
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    if world > 1 and (cross is False or n_vs_1 is False):
        return 3  # a multi-GPU result that differs from the single-GPU one is a failed run
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 40; 5 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mine", choices=["mine", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-stream-all", action="store_true")
    ap.add_argument("--no-bruteforce", action="store_true")
    ap.add_argument("--no-c3", action="store_true")
    ap.add_argument("--keep-caches", action="store_true",
                    help="re-use the mirror / group summaries across fits (default: rebuilt by every fit)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what rank 0's last timed fit and end-to-end call returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what this repo's CUDA path returned: not with --impl reference")
        if args.steps is None:  # keep the default CPU run to a few minutes
            args.steps = 5
        return run_reference(args)
    if args.steps is None:
        args.steps = 40
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least three warm-up steps
    return run_mine(args)


if __name__ == "__main__":
    sys.exit(main())
