"""`DeviceGroup`: several B200s driven from ONE process, one host thread per device.

The reference calls the path in-process, from a napari worker thread
(``members/rafael/disparity/widget.py:116-147``), so a multi-GPU drop-in cannot ask its caller
to re-launch under ``torchrun``.  A ``DeviceGroup`` owns one ``Engine`` (one libmdkm handle, one
rank) per device and runs the ranks on a thread each -- every C-ABI call releases the GIL, so
the devices work concurrently.  The ranks are wired exactly like the one-process-per-GPU setup
of ``dist.py``: an NCCL communicator for the one-off collectives (``ncclCommInitRank`` called
from the threads with a shared unique id) and peer-mapped exchange buffers for the in-kernel
NVLink exchange of the K x 4 partial sums (plain peer pointers here, no CUDA IPC).  Results are
bit-identical to one GPU because the exchanged sums are integers.
"""
from __future__ import annotations

import copy
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, List, Optional, Sequence

import numpy as np

from .dist import shard_range


class DeviceGroup:
    """``DeviceGroup([0, 1, 2, 3])``; use as a context manager or call ``close()``."""

    def __init__(self, devices: Sequence[int], p2p: bool = True, engine_factory: Optional[Callable] = None,
                 make_unique_id: Optional[Callable[[], bytes]] = None):
        if len(devices) < 1 or len(set(devices)) != len(devices):
            raise ValueError("devices must be a non-empty list of distinct CUDA device indices")
        if engine_factory is None:
            from .engine import Engine

            engine_factory = Engine
            make_unique_id = Engine.make_unique_id
        self.devices = [int(d) for d in devices]
        self.world = len(self.devices)
        self._pool = ThreadPoolExecutor(max_workers=self.world, thread_name_prefix="mdkm-rank")
        self.engines: List = []
        try:
            self.engines = self.map(lambda r: engine_factory(self.devices[r]))
            if self.world > 1:
                uid = make_unique_id()
                self.map(lambda r: self.engines[r].init_comm(self.world, r, uid))  # blocks until all ranks joined
                if p2p and self.world <= 8:
                    self.map(lambda r: self.engines[r].p2p_handle())               # allocates the exchange buffers
                    ptrs = [e.p2p_buffer() for e in self.engines]
                    ok = self.map(lambda r: self.engines[r].p2p_open_ptrs(ptrs))
                    if not all(ok):  # all ranks or none
                        self.map(lambda r: self.engines[r].p2p_close())
            else:
                self.engines[0].init_comm(1, 0, None)
        except Exception:
            self.close()
            raise

    # -- plumbing -------------------------------------------------------------------------
    def map(self, fn: Callable[[int], object]) -> list:
        """Run ``fn(rank)`` for every rank concurrently (one thread per rank); re-raises the first error."""
        futs = [self._pool.submit(fn, r) for r in range(self.world)]
        out, err = [], None
        for f in futs:
            try:
                out.append(f.result())
            except Exception as e:  # noqa: BLE001 - collect, so that no thread is left behind
                out.append(None)
                err = err or e
        if err is not None:
            raise err
        return out

    @property
    def p2p(self) -> bool:
        return self.world > 1 and all(getattr(e, "p2p", False) for e in self.engines)

    def close(self):
        for e in self.engines:
            try:
                e.close()
            except Exception:  # noqa: BLE001
                pass
        self.engines = []
        self._pool.shutdown(wait=True)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- the fused path -------------------------------------------------------------------
    def fuse(self, height_maps, valid_masks=None, *, run_kmeans: Callable, max_abs_height=144.0, detrend=False,
             disparity_scale=None, ground_level=False, return_cloud=True, raster_layout=None, maps=None):
        """Shard a HOST stack over the devices by row bands (whole days when ``detrend`` or
        ``ground_level`` need them), unproject, cluster, and assemble labels / cloud in the
        reference's point order.  ``run_kmeans(engine, labels_out) -> dict`` is ``api._run_kmeans``
        bound to the k-means arguments; it runs on every rank (the collectives inside pair up).
        ``maps`` (``{keyword: dtype}``, e.g. ``{"cluster_map_out": np.uint8}``): also build these
        ``[D,H,W]`` pixel maps; every rank writes its row band of each in place
        (``run_kmeans(engine, labels_out, cluster_map_out=band, ...)``), and each is returned as
        ``extra`` under its keyword without "_out" (``extra["cluster_map"]``).
        Returns ``(result dict of rank 0, labels, cloud or None, height_norm or None, extra)``."""
        hm = height_maps
        if type(hm).__module__.startswith("torch"):
            if hm.is_cuda:
                raise ValueError("a DeviceGroup shards HOST rasters; pass a CPU tensor or a numpy array")
            hm = hm.numpy()
        hm = np.asarray(hm)
        gt = raster_layout == "gtiff3"
        shp = hm.shape[:-1] if gt else hm.shape
        if len(shp) == 2:
            shp = (1,) + tuple(shp)
        if len(shp) != 3:
            raise ValueError("height_maps must be [D,H,W] or [H,W]")
        D, H, W = (int(v) for v in shp)
        per_px = 3 if gt else 1
        flat = np.ascontiguousarray(hm).reshape(-1)
        mflat = None
        if valid_masks is not None:
            m = valid_masks.numpy() if type(valid_masks).__module__.startswith("torch") else np.asarray(valid_masks)
            mflat = np.ascontiguousarray(m).reshape(-1)
        whole_days = bool(detrend or ground_level)
        spans = [shard_range(D * H * W, r, self.world, align=(H * W if whole_days else W)) for r in range(self.world)]

        def unproject(r):
            b, e = spans[r]
            eng = self.engines[r]
            n = eng.unproject(flat[b * per_px:e * per_px].reshape((-1, 3) if gt else (-1,)),
                              None if mflat is None else mflat[b:e], max_abs_height=max_abs_height, detrend=detrend,
                              disparity_scale=disparity_scale, stack_shape=(D, H, W), pix_begin=b,
                              raster_layout=raster_layout)
            lv = eng.ground_level(True) if ground_level else None
            return n, eng.segment_offsets, lv

        ups = self.map(unproject)
        counts = [u[0] for u in ups]
        offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        n_total = int(offs[-1])
        labels = np.empty(n_total, dtype=np.int32)
        cloud = np.empty((n_total, 3), dtype=np.float32) if return_cloud else None
        whole = {kw: np.empty(D * H * W, dtype=dtype) for kw, dtype in (maps or {}).items()}

        def cluster(r):
            eng = self.engines[r]
            a, b = int(offs[r]), int(offs[r + 1])
            if cloud is not None and b > a:
                eng.get_cloud(napari_order=True, out=cloud[a:b], wait=False)  # overlaps the Lloyd loop
            res = run_kmeans(eng, labels[a:b], **{kw: m[spans[r][0]:spans[r][1]] for kw, m in whole.items()})
            eng.wait()
            return res

        results = self.map(cluster)
        hn = None
        extra = {"devices": list(self.devices), "shard_points": counts,
                 "exchange": "nvlink_p2p" if self.p2p else ("nccl" if self.world > 1 else "none")}
        if ground_level:
            hn = np.concatenate([u[2][2] for u in ups]) if n_total else np.zeros(0, dtype=np.float32)
            extra["h_min"] = np.concatenate([u[2][0] for u in ups])
            extra["h_max"] = np.concatenate([u[2][1] for u in ups])
        # day offsets of the whole cloud: a day cut by a shard boundary appears in two ranks
        day_counts = np.zeros(D, dtype=np.int64)
        for r, (b, e) in enumerate(spans):
            if e > b:
                d_first = b // (H * W)
                seg = np.diff(ups[r][1])
                day_counts[d_first:d_first + seg.shape[0]] += seg
        extra["segment_offsets"] = np.concatenate([[0], np.cumsum(day_counts)]).astype(np.int64)
        for kw, m in whole.items():
            extra[kw.removesuffix("_out")] = m.reshape(D, H, W)
        return results[0], labels, cloud, hn, extra


def clone_random_state(random_state, n: int) -> list:
    """``n`` generators that will produce the same draws (every rank draws what scikit-learn would)."""
    if isinstance(random_state, np.random.RandomState):
        return [copy.deepcopy(random_state) for _ in range(n)]
    return [random_state] * n  # None / int: each rank builds its own RandomState(seed)
