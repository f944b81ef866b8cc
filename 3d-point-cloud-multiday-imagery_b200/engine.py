"""`Engine`: one libmdkm handle (one B200, one rank) with numpy / torch friendly methods.

Thin by design: every method is one C-ABI call (include/mdkm.h); arrays are passed as raw
host or device pointers.  torch is only used to recognise CUDA tensors and to exchange the
NCCL unique id between ranks.
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, byref, c_double, c_float, c_int, c_int64, c_ubyte, c_void_p

import numpy as np

from . import _cabi as C


def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


def _as_buffer(a, dtype=None):
    """-> (pointer:int, mem_kind, keepalive, shape, np_dtype) for numpy arrays / torch tensors."""
    if _is_torch(a):
        import torch

        t = a
        if dtype is not None:
            want = {np.float32: torch.float32, np.int16: torch.int16, np.uint8: torch.uint8,
                    np.float64: torch.float64, np.int32: torch.int32}[dtype]
            if t.dtype == torch.bool and want == torch.uint8:
                t = t.to(torch.uint8)
            elif t.dtype != want:
                t = t.to(want)
        t = t.contiguous()
        mem = C.MEM_DEVICE if t.is_cuda else C.MEM_HOST
        return t.data_ptr(), mem, t, tuple(t.shape), None
    arr = np.asarray(a)
    if dtype is not None and arr.dtype != np.dtype(dtype):
        arr = arr.astype(dtype)
    arr = np.ascontiguousarray(arr)
    return arr.ctypes.data, C.MEM_HOST, arr, arr.shape, arr.dtype


def check_min_iou(value, what="tracks"):
    """``value`` as the float min_iou of object tracks: a real number in (0, 1] (not a bool, not
    NaN).  Raises ``ValueError`` otherwise."""
    if isinstance(value, (bool, np.bool_)) or not isinstance(value, (int, float, np.integer, np.floating)):
        raise ValueError(f"{what} must be a real number in (0, 1], got {value!r}")
    v = float(value)
    if not (0.0 < v <= 1.0):
        raise ValueError(f"{what} must be a real number in (0, 1], got {value!r}")
    return v


def _as_out_buffer(a, dtype, n_elems, what):
    """-> (pointer:int, mem_kind) of a caller-supplied OUTPUT array.  The library writes through
    the raw pointer, so anything that would make numpy / torch hand over a temporary copy (wrong
    dtype, non-contiguous view) is rejected instead of silently losing the result.  ``dtype``: one
    dtype, or a tuple of the dtypes the output may have."""
    dts = tuple(np.dtype(d) for d in (dtype if isinstance(dtype, tuple) else (dtype,)))
    names = " or ".join(d.name for d in dts)
    if _is_torch(a):
        import torch

        tmap = {np.dtype(np.float32): torch.float32, np.dtype(np.int32): torch.int32,
                np.dtype(np.uint8): torch.uint8, np.dtype(np.uint16): torch.uint16}
        if a.dtype not in [tmap[d] for d in dts]:
            raise ValueError(f"{what} must be {names}, got {a.dtype}")
        if not a.is_contiguous():
            raise ValueError(f"{what} must be contiguous")
        if a.numel() != n_elems:
            raise ValueError(f"{what} must hold {n_elems} elements, got {a.numel()}")
        return a.data_ptr(), (C.MEM_DEVICE if a.is_cuda else C.MEM_HOST)
    if not isinstance(a, np.ndarray):
        raise ValueError(f"{what} must be a numpy array or a torch tensor")
    if a.dtype not in dts:
        raise ValueError(f"{what} must be {names}, got {a.dtype}")
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError(f"{what} must be C-contiguous")
    if not a.flags["WRITEABLE"]:
        raise ValueError(f"{what} must be writeable")
    if a.size != n_elems:
        raise ValueError(f"{what} must hold {n_elems} elements, got {a.size}")
    return a.ctypes.data, C.MEM_HOST


def _day_pairs(pairs) -> np.ndarray:
    """Day pairs ``[P,2]`` as int32, clipped so that the library refuses out-of-range days."""
    return np.ascontiguousarray(np.clip(np.asarray(pairs, dtype=np.int64).reshape(-1, 2), -1, 2**31 - 1),
                                dtype=np.int32)


class Engine:
    """Owns one ``mdkm_handle``.  Use as a context manager or call ``close()``."""

    def __init__(self, device: int = 0, stream=None, pinned_results: bool = False):
        """``pinned_results``: result arrays (labels, cloud) are views of page-locked buffers
        owned by the engine and REUSED by the next call -- fastest device->host path; copy them
        if they must outlive the next call."""
        self._lib = C.load()
        self.pinned_results = bool(pinned_results)
        self._pinned = {}
        self._h = c_void_p()
        sptr = None
        if stream is not None:
            sptr = c_void_p(int(getattr(stream, "cuda_stream", stream)))
        rc = self._lib.mdkm_create(byref(self._h), int(device), sptr)
        if rc != C.MDKM_OK:
            self._h = c_void_p()
            raise C.MdkmError(rc, "mdkm_create failed (needs a visible sm_100 GPU; there is no CPU fallback)")
        self.device = int(device)
        self.n_ranks = 1
        self.rank = 0
        self.p2p = False
        self._stream_ptr = int(self._lib.mdkm_get_stream(self._h) or 0)
        self._ext_stream = None
        self._raster = None  # (D, H, W, pix_begin, pix_count) of the last unproject

    # -- ordering against torch's streams ----------------------------------------------------
    # The handle enqueues on its own stream.  A CUDA tensor handed to it may still be being
    # produced on torch's current stream (including the .to() / .contiguous() copies made just
    # above), and a device-resident output may be consumed there right after the call: the two
    # streams are ordered with events.  Every library call that READS a caller's device buffer
    # returns only after the handle's stream has consumed it (they all end in a stream
    # synchronisation), so temporaries may be released as soon as the call is back -- no
    # record_stream, which would tie a tensor's release to a stream this engine may already have
    # destroyed.
    def _torch_streams(self):
        import torch

        if self._ext_stream is None:
            self._ext_stream = torch.cuda.ExternalStream(self._stream_ptr, device=self.device)
        return self._ext_stream, torch.cuda.current_stream(self.device)

    def _after_torch(self, *tensors):
        """The handle's stream waits for what torch's current stream has enqueued so far."""
        ext, cur = self._torch_streams()
        if cur.cuda_stream != self._stream_ptr:
            ext.wait_stream(cur)

    def _before_torch(self):
        """torch's current stream waits for what the handle has enqueued so far."""
        ext, cur = self._torch_streams()
        if cur.cuda_stream != self._stream_ptr:
            cur.wait_stream(ext)

    # -- lifetime ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._ext_stream = None  # wraps the handle's stream, which dies with the handle
            self._lib.mdkm_destroy(self._h)
            self._h = c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _result_buffer(self, name, shape, dtype):
        """numpy result array; page-locked and cached when ``pinned_results``."""
        if not self.pinned_results:
            return np.empty(shape, dtype=dtype)
        import torch

        n = int(np.prod(shape))
        t = self._pinned.get(name)
        tdt = {np.dtype(np.float32): torch.float32, np.dtype(np.int32): torch.int32}[np.dtype(dtype)]
        if t is None or t.numel() < n or t.dtype != tdt:
            t = torch.empty(max(n, 1), dtype=tdt, pin_memory=True)
            self._pinned[name] = t
        return t.numpy()[:n].reshape(shape)

    def _check(self, rc: int):
        if rc != C.MDKM_OK:
            msg = self._lib.mdkm_last_error(self._h)
            raise C.MdkmError(rc, msg.decode() if msg else "")

    # -- multi-GPU ---------------------------------------------------------------------
    def init_comm(self, n_ranks: int, rank: int, unique_id: bytes | None):
        buf = None
        if n_ranks > 1:
            assert unique_id is not None and len(unique_id) == C.NCCL_UNIQUE_ID_BYTES
            buf = (c_ubyte * C.NCCL_UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self._lib.mdkm_comm_init(self._h, int(n_ranks), int(rank), buf))
        self.n_ranks, self.rank = int(n_ranks), int(rank)

    def p2p_handle(self) -> bytes:
        """CUDA IPC handle of this rank's partial-sum exchange buffer (64 bytes)."""
        buf = (c_ubyte * C.IPC_HANDLE_BYTES)()
        self._check(self._lib.mdkm_comm_p2p_handle(self._h, buf))
        return bytes(buf)

    def p2p_open(self, handles: bytes) -> bool:
        """Map every rank's exchange buffer (handles in rank order).  False: NCCL stays in use."""
        assert len(handles) == C.IPC_HANDLE_BYTES * self.n_ranks
        buf = (c_ubyte * len(handles)).from_buffer_copy(handles)
        rc = self._lib.mdkm_comm_p2p_open(self._h, buf)
        self.p2p = rc == C.MDKM_OK
        return self.p2p

    def p2p_close(self):
        """Back to the NCCL exchange (the communicator is kept).  No-op when nothing is open."""
        self._check(self._lib.mdkm_comm_p2p_close(self._h))
        self.p2p = False

    def p2p_buffer(self) -> int:
        """Device pointer of this rank's exchange buffer (in-process ranks; after p2p_handle)."""
        out = c_void_p()
        self._check(self._lib.mdkm_comm_p2p_buffer(self._h, byref(out)))
        return int(out.value)

    def p2p_open_ptrs(self, buffers) -> bool:
        """In-process variant of ``p2p_open``: the ranks' exchange-buffer pointers in rank order."""
        assert len(buffers) == self.n_ranks
        arr = (c_void_p * len(buffers))(*[c_void_p(int(b)) for b in buffers])
        rc = self._lib.mdkm_comm_p2p_open_ptrs(self._h, arr)
        self.p2p = rc == C.MDKM_OK
        return self.p2p

    def set_option(self, option: int, value: int):
        self._check(self._lib.mdkm_set_option(self._h, int(option), int(value)))

    def raster_mirror(self, on: bool):
        """``False``: test hook -- raster clouds use the generic (histogram + scatter) build of the
        tile-ordered mirror instead of the run-table build.  Results are identical."""
        self.set_option(C.OPT_RASTER_MIRROR, 1 if on else 0)

    def settle_groups(self, on: bool):
        """``False``: measurement mode -- every point goes through the per-point pass in every
        iteration (no group is settled from its cached summary).  Results are identical."""
        self.set_option(C.OPT_SETTLE_GROUPS, 1 if on else 0)

    @staticmethod
    def make_unique_id() -> bytes:
        lib = C.load()
        buf = (c_ubyte * C.NCCL_UNIQUE_ID_BYTES)()
        rc = lib.mdkm_comm_unique_id(buf)
        if rc != C.MDKM_OK:
            raise C.MdkmError(rc, "mdkm_comm_unique_id failed (libnccl.so.2 not loadable)")
        return bytes(buf)

    # -- data ----------------------------------------------------------------------------
    def unproject(self, height_maps, valid_masks=None, *, max_abs_height=144.0, detrend=False,
                  disparity_scale=None, pix_begin=0, stack_shape=None, stream_cloud=None,
                  raster_layout=None):
        """Height rasters -> resident XYZ cloud (plugin.py:148-171).  Returns the point count.

        ``raster_layout="gtiff3"``: ``height_maps`` is float32 ``[D,H,W,3]``, the pixel layout of
        the reference's ``5-out-F.tif`` (``tiff_io.load_height_rasters``): band 0 height, band 2
        ``final_defined``.
        ``stream_cloud``: None, or "napari" / "xyz" to also stream the cloud to the host while
        the stack is still being uploaded; the call then returns ``(n, cloud[n,3])`` and the
        array is complete after ``wait()``.

        ``height_maps``: float32 ``[D,H,W]`` (NaN = nodata) or, with ``disparity_scale``
        (the reference uses -1/16), int16 OpenCV fixed-point disparity.  For a sharded
        stack pass this rank's flat slice plus ``stack_shape=(D,H,W)`` and ``pix_begin``.
        """
        is_i16 = disparity_scale is not None
        ptr, mem, keep, shape, _ = _as_buffer(height_maps, np.int16 if is_i16 else np.float32)
        gtiff3 = raster_layout == "gtiff3"
        if gtiff3:
            # the reference's 5-out-F.tif pixels: [..., 3] float32 = height, unused, final_defined
            if is_i16 or shape[-1] != 3 or (stack_shape is None and len(shape) < 3):
                raise ValueError("raster_layout='gtiff3' needs float32 [D,H,W,3] (or [H,W,3]; [n,3] with stack_shape)")
            shape = tuple(shape[:-1])
        elif raster_layout is not None:
            raise ValueError("raster_layout must be None or 'gtiff3'")
        if stack_shape is None:
            if len(shape) == 2:
                shape = (1,) + tuple(shape)
            if len(shape) != 3:
                raise ValueError("height_maps must be [D,H,W] or [H,W]")
            D, H, W = shape
            count = D * H * W
        else:
            D, H, W = stack_shape
            count = int(np.prod(shape))
        mptr, keep_m = None, None
        if valid_masks is not None:
            mptr, mmem, keep_m, mshape, _ = _as_buffer(valid_masks, np.uint8)
            if int(np.prod(mshape)) != count:
                raise ValueError("valid_masks must match height_maps")
            if mmem != mem:
                raise ValueError("height_maps and valid_masks must live in the same memory space")
        if mem == C.MEM_DEVICE:
            self._after_torch(keep, keep_m)
        n = c_int64(0)
        cloud_buf = None
        if stream_cloud is not None:
            cloud_buf = self._result_buffer("cloud", (max(count, 1), 3), np.float32)
            self._check(self._lib.mdkm_bind_cloud_output(
                self._h, c_void_p(cloud_buf.ctypes.data), int(count), 1 if stream_cloud == "napari" else 0))
        self._check(self._lib.mdkm_unproject(
            self._h, c_void_p(ptr), C.HM_I16 if is_i16 else (C.HM_F32_GTIFF3 if gtiff3 else C.HM_F32),
            float(disparity_scale) if is_i16 else 1.0, c_void_p(mptr) if mptr else None,
            int(D), int(H), int(W), int(pix_begin), int(count), float(max_abs_height),
            1 if detrend else 0, mem, byref(n)))
        del keep, keep_m
        self._raster = (int(D), int(H), int(W), int(pix_begin), int(count))
        if stream_cloud is not None:
            return int(n.value), cloud_buf[: int(n.value)]
        return int(n.value)

    def set_points(self, points, layout="aos") -> int:
        """Load an ``[N,3]`` (x,y,z) float32 cloud (or SoA ``[3,N]`` with layout="soa")."""
        ptr, mem, keep, shape, _ = _as_buffer(points, np.float32)
        if layout == "aos":
            if len(shape) != 2 or shape[1] != 3:
                raise ValueError("points must be [N,3]")
            n = shape[0]
            lay = C.POINTS_AOS
        else:
            if len(shape) != 2 or shape[0] != 3:
                raise ValueError("SoA points must be [3,N]")
            n = shape[1]
            lay = C.POINTS_SOA
        if mem == C.MEM_DEVICE:
            self._after_torch(keep)
        self._raster = None
        self._check(self._lib.mdkm_set_points(self._h, c_void_p(ptr), int(n), lay, mem))
        del keep
        return int(n)

    @property
    def n_points(self) -> int:
        return int(self._lib.mdkm_num_points(self._h))

    @property
    def n_points_global(self) -> int:
        """Points over all ranks (== ``n_points`` without a communicator)."""
        n = int(self._lib.mdkm_num_points_global(self._h))
        if n < 0:
            self._check(C.STATUS_BY_NAME["MDKM_ERR_STATE"])
        return n

    def gather_points(self, idx) -> np.ndarray:
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        out = np.empty((idx.shape[0], 3), dtype=np.float32)
        self._check(self._lib.mdkm_gather_points(
            self._h, idx.ctypes.data_as(POINTER(c_int64)), int(idx.shape[0]),
            out.ctypes.data_as(POINTER(c_float))))
        return out

    def get_cloud(self, napari_order=True, out=None, wait=True):
        """Resident cloud as float32 ``[N,3]``; (z,y,x) columns when ``napari_order``.

        ``wait=False`` only enqueues the copy (it overlaps later calls such as ``fit``); the
        array is complete after ``wait()``."""
        n = self.n_points
        if out is None:
            out = self._result_buffer("cloud", (n, 3), np.float32)
        ptr, mem = _as_out_buffer(out, np.float32, n * 3, "out")
        if mem == C.MEM_DEVICE:
            self._after_torch(out)  # earlier work on torch's stream may still use the buffer
        fn = self._lib.mdkm_get_cloud if wait else self._lib.mdkm_get_cloud_async
        self._check(fn(self._h, c_void_p(ptr), 1 if napari_order else 0, mem))
        if mem == C.MEM_DEVICE:
            self._before_torch()
        return out

    def wait(self):
        """Block until every asynchronous result copy of this engine has completed."""
        self._check(self._lib.mdkm_wait(self._h))

    @property
    def raster_range(self):
        """``(D, H, W, pix_begin, pix_count)`` of the last ``unproject``, or None when the resident
        cloud came from ``set_points`` (or there is none)."""
        return self._raster

    def _pixel_map(self, out, dtype, what):
        """-> (pointer, memory kind, capacity) of the caller's pixel map ``out`` (one element per pixel
        of the last unprojected range), or (None, host, 0) without one."""
        if out is None:
            return None, C.MEM_HOST, 0
        cap = self._raster[4] if self._raster is not None else (out.numel() if _is_torch(out) else np.size(out))
        ptr, mem = _as_out_buffer(out, dtype, cap, what)
        if mem == C.MEM_DEVICE:
            self._after_torch(out)  # earlier work on torch's stream may still use the buffer
        return ptr, mem, cap

    def _bind_cluster_map(self, out):
        """Bind ``out`` (uint8 / uint16, one element per pixel of the last unprojected range) as the
        cluster map of the next fit / predict.  -> its memory kind."""
        ptr, mem, n_pix = self._pixel_map(out, (np.uint8, np.uint16), "cluster_map_out")
        elem = out.element_size() if _is_torch(out) else out.itemsize
        self._check(self._lib.mdkm_bind_cluster_map(self._h, c_void_p(ptr), int(elem), int(n_pix), mem))
        return mem

    @property
    def n_days(self) -> int:
        """Days of the stack of the last ``unproject`` (its ``stack_shape``), 1 after ``set_points``:
        the rows of ``day_counts`` / ``day_means``."""
        return self._raster[0] if self._raster is not None else 1

    def _bind_day_stats(self, k):
        """Bind fresh ``day_counts`` int64 ``[D,k]`` / ``day_means`` float64 ``[D,k,3]`` arrays to the
        next fit / predict.  -> (counts, means)."""
        d = self.n_days
        counts = np.empty((d, k), dtype=np.int64)
        means = np.empty((d, k, 3), dtype=np.float64)
        self._check(self._lib.mdkm_bind_day_stats(self._h, c_void_p(counts.ctypes.data), c_void_p(means.ctypes.data),
                                                  int(d), int(k)))
        return counts, means

    def _bind_day_transitions(self, pairs, k):
        """Bind the day pairs ``pairs`` (``[P,2]`` global days) and a fresh int64 ``[P,k+1,k+1]``
        array to the next fit / predict.  -> the array."""
        pr = _day_pairs(pairs)
        counts = np.empty((pr.shape[0], k + 1, k + 1), dtype=np.int64)
        self._check(self._lib.mdkm_bind_day_transitions(self._h, c_void_p(pr.ctypes.data), int(pr.shape[0]),
                                                        c_void_p(counts.ctypes.data), int(k)))
        return counts

    def _bind_regions(self, connectivity, out):
        """Bind connected regions (``connectivity`` 4 or 8) and the optional int32 region map ``out``
        (one element per pixel of the last unprojected range) to the next fit / predict.  -> the
        map's memory kind (host without a map)."""
        if connectivity not in (4, 8) or isinstance(connectivity, bool):
            raise ValueError(f"regions must be 4 or 8 (the connectivity), got {connectivity!r}")
        ptr, mem, cap = self._pixel_map(out, np.int32, "region_map_out")
        self._check(self._lib.mdkm_bind_regions(self._h, int(connectivity), c_void_p(ptr), int(cap), mem))
        return mem

    def _region_table(self):
        """The regions of the last fit / predict that had them -> (table int64 ``[R,7]``, means
        float64 ``[R,3]``)."""
        n = c_int64(0)
        self._check(self._lib.mdkm_region_count(self._h, byref(n)))
        table = np.empty((n.value, 7), dtype=np.int64)
        means = np.empty((n.value, 3), dtype=np.float64)
        self._check(self._lib.mdkm_region_table(self._h, c_void_p(table.ctypes.data), c_void_p(means.ctypes.data),
                                                int(n.value)))
        return table, means

    def _bind_region_overlaps(self, pairs):
        """Bind the day pairs ``pairs`` (``[P,2]`` global days) of region overlaps to the next fit /
        predict."""
        pr = _day_pairs(pairs)
        self._check(self._lib.mdkm_bind_region_overlaps(self._h, c_void_p(pr.ctypes.data), int(pr.shape[0])))

    def _region_overlap_table(self):
        """The region overlaps of the last fit / predict that had them -> int64 ``[M,6]``."""
        n = c_int64(0)
        self._check(self._lib.mdkm_region_overlap_count(self._h, byref(n)))
        rows = np.empty((n.value, 6), dtype=np.int64)
        self._check(self._lib.mdkm_region_overlap_table(self._h, c_void_p(rows.ctypes.data), int(n.value)))
        return rows

    def _bind_tracks(self, min_iou, out):
        """Bind object tracks (``min_iou`` in (0, 1]) and the optional int32 track map ``out`` (one
        element per pixel of the last unprojected range) to the next fit / predict.  -> the map's
        memory kind (host without a map)."""
        iou = check_min_iou(min_iou)
        ptr, mem, cap = self._pixel_map(out, np.int32, "track_map_out")
        self._check(self._lib.mdkm_bind_tracks(self._h, iou, c_void_p(ptr), int(cap), mem))
        return mem

    def _track_table(self):
        """The tracks of the last fit / predict that had them -> (table int64 ``[T,7]``, region
        tracks int32 ``[R]``)."""
        n, r = c_int64(0), c_int64(0)
        self._check(self._lib.mdkm_track_count(self._h, byref(n)))
        self._check(self._lib.mdkm_region_count(self._h, byref(r)))
        table = np.empty((n.value, 7), dtype=np.int64)
        region_tracks = np.empty(r.value, dtype=np.int32)
        self._check(self._lib.mdkm_track_table(self._h, c_void_p(table.ctypes.data),
                                               c_void_p(region_tracks.ctypes.data), int(n.value), int(r.value)))
        return table, region_tracks

    def _region_adjacency_table(self):
        """The region adjacency of the last fit / predict that had it -> (rows int64 ``[M,6]``,
        region boundaries int64 ``[R,4]``)."""
        n, r = c_int64(0), c_int64(0)
        self._check(self._lib.mdkm_region_adjacency_count(self._h, byref(n)))
        self._check(self._lib.mdkm_region_count(self._h, byref(r)))
        rows = np.empty((n.value, 6), dtype=np.int64)
        boundaries = np.empty((r.value, 4), dtype=np.int64)
        self._check(self._lib.mdkm_region_adjacency_table(self._h, c_void_p(rows.ctypes.data),
                                                          c_void_p(boundaries.ctypes.data), int(n.value), int(r.value)))
        return rows, boundaries

    def _bind_outputs(self, k, cluster_map_out=None, day_stats=False, transitions=None, regions=None,
                      region_map_out=None, region_overlaps=None, tracks=None, track_map_out=None,
                      region_adjacency=False):
        """Bind the optional outputs of the next fit / predict (the keywords of ``fit``) -> (whether
        a pixel map is device memory, (counts, means) or None, transitions or None).  When one
        binding is refused none is left behind: the statistics and transition arrays live only in
        this call, and a binding that outlived them would have the next fit / predict write into
        freed memory."""
        if region_map_out is not None and regions is None:
            raise ValueError("region_map_out needs regions=4 or regions=8")
        if region_overlaps is not None and regions is None:
            raise ValueError("region_overlaps needs regions=4 or regions=8")
        if tracks is not None and regions is None:
            raise ValueError("tracks needs regions=4 or regions=8")
        if track_map_out is not None and tracks is None:
            raise ValueError("track_map_out needs tracks=min_iou")
        if region_adjacency and regions is None:
            raise ValueError("region_adjacency needs regions=4 or regions=8")
        try:
            map_mem = self._bind_cluster_map(cluster_map_out) if cluster_map_out is not None else None
            stats = self._bind_day_stats(k) if day_stats else None
            trans = self._bind_day_transitions(transitions, k) if transitions is not None else None
            reg_mem = self._bind_regions(regions, region_map_out) if regions is not None else None
            if region_overlaps is not None:
                self._bind_region_overlaps(region_overlaps)
            trk_mem = self._bind_tracks(tracks, track_map_out) if tracks is not None else None
            if region_adjacency:
                self._check(self._lib.mdkm_bind_region_adjacency(self._h, 1))
        except BaseException:
            self._lib.mdkm_bind_cluster_map(self._h, None, 1, 0, C.MEM_HOST)
            self._lib.mdkm_bind_day_stats(self._h, None, None, 0, 0)
            self._lib.mdkm_bind_day_transitions(self._h, None, 0, None, 0)
            self._lib.mdkm_bind_regions(self._h, 0, None, 0, C.MEM_HOST)
            self._lib.mdkm_bind_region_overlaps(self._h, None, 0)
            self._lib.mdkm_bind_tracks(self._h, 0.0, None, 0, C.MEM_HOST)
            self._lib.mdkm_bind_region_adjacency(self._h, 0)
            raise
        return C.MEM_DEVICE in (map_mem, reg_mem, trk_mem), stats, trans

    def _read_outputs(self, stats, trans, regions, region_overlaps, tracks, region_adjacency=False) -> dict:
        """The optional results of the last fit / predict that were asked for, in ``predict``'s order:
        day_counts, day_means, transitions, regions, region_means, region_overlaps, tracks, region_tracks,
        region_adjacency, region_boundaries."""
        out = {}
        if stats is not None:
            out["day_counts"], out["day_means"] = stats
        if trans is not None:
            out["transitions"] = trans
        if regions is not None:
            out["regions"], out["region_means"] = self._region_table()
        if region_overlaps is not None:
            out["region_overlaps"] = self._region_overlap_table()
        if tracks is not None:
            out["tracks"], out["region_tracks"] = self._track_table()
        if region_adjacency:
            out["region_adjacency"], out["region_boundaries"] = self._region_adjacency_table()
        return out

    @property
    def segment_offsets(self) -> np.ndarray:
        """Point offsets of the cloud's segments (one per day), int64 ``[n_segments + 1]``."""
        ns = int(self._lib.mdkm_num_segments(self._h))
        if ns < 0:
            raise C.MdkmError(C.STATUS_BY_NAME["MDKM_ERR_STATE"], "no points resident")
        out = np.zeros(ns + 1, dtype=np.int64)
        self._check(self._lib.mdkm_segment_offsets(self._h, out.ctypes.data_as(POINTER(c_int64))))
        return out

    def ground_level(self, want_height_norm=True):
        """plugin.py:181-192 per day.  Returns (h_min[S], h_max[S], height_norm[N] or None)."""
        n = self.n_points
        ns = int(self._lib.mdkm_num_segments(self._h))
        hn = self._result_buffer("height_norm", (n,), np.float32) if want_height_norm else None
        lo = np.zeros(max(ns, 1), dtype=np.float64)
        hi = np.zeros(max(ns, 1), dtype=np.float64)
        self._check(self._lib.mdkm_ground_level(
            self._h, c_void_p(hn.ctypes.data) if hn is not None else None, C.MEM_HOST,
            lo.ctypes.data_as(POINTER(c_double)), hi.ctypes.data_as(POINTER(c_double))))
        return lo[:ns], hi[:ns], hn

    # -- k-means -------------------------------------------------------------------------
    def fit(self, init, max_iter=300, tol=1e-4, want_labels=True, labels_out=None, cluster_map_out=None,
            day_stats=False, transitions=None, regions=None, region_map_out=None, region_overlaps=None,
            tracks=None, track_map_out=None, region_adjacency=False):
        """One Lloyd run from explicit centroids.  Returns dict(labels, centers, n_iter, inertia, ...).

        ``cluster_map_out``: optional uint8 (k <= 255) or uint16 array / tensor, host or CUDA, with
        one element per pixel of the last ``unproject``'s range; it receives the labels on the
        pixel grid (label + 1 where a pixel produced a point, 0 elsewhere), written by the final
        pass.  A CUDA output is ordered against torch's current stream like ``labels_out``.

        ``day_stats=True``: the result also has ``day_counts`` (int64 ``[D,k]``, points of day d with
        label j) and ``day_means`` (float64 ``[D,k,3]``, their mean (x, y, z) in the clustered frame,
        NaN where the count is 0), accumulated by the final pass; D is ``n_days`` (global days of the
        stack), and with several ranks both are summed over all of them.

        ``transitions``: day pairs ``[P,2]`` (global days of the stack); the result also has
        ``transitions``, int64 ``[P,k+1,k+1]``: ``[p,s,t]`` pixels with state s on day a and t on
        day b of pair p, state = label + 1 where the pixel produced a point, 0 where it did not
        (the cluster map's value).  Binned on the GPU from the map the final pass writes; needs a
        cloud from ``unproject`` whose ranks together hold the whole stack, and with several ranks
        every rank receives the counts of the whole stack.

        ``regions``: 4 or 8, the connectivity of the connected regions of the cluster map (maximal
        connected sets of pixels of one day with the same label), numbered 1..R in the raster
        order (day, y, x) of their first pixel.  The result also has ``regions``, int64 ``[R,7]``
        rows (day, cluster, pixels, y_min, x_min, y_max, x_max), and ``region_means``, float64
        ``[R,3]``, the mean (x, y, z) of each region's points in the clustered frame (computed like
        ``day_means``).  ``region_map_out``: optional int32 array / tensor, host or CUDA, with one
        element per pixel of the last ``unproject``'s range; it receives the region ids, 0 where a
        pixel has no point.  Labelled on the GPU after the fit; same cover rule as
        ``transitions``, and with several ranks every rank receives the whole stack's regions.

        ``region_overlaps``: day pairs ``[P,2]`` (global days; needs ``regions``, else
        ``ValueError`` before any GPU work); the result also has ``region_overlaps``, int64
        ``[M,6]`` rows (pair, region_a, region_b, pixels, y_first, x_first): one for every pair of
        regions (r of day a, s of day b) that share at least one pixel, with the number of shared
        pixels and the first shared pixel, sorted by pair and then by that pixel's raster order.
        Counted on the GPU from the region map; with several ranks every rank builds the same
        rows.

        ``tracks``: min_iou, a real number in (0, 1] (needs ``regions``, else ``ValueError`` before
        any GPU work): object tracks over the stack.  Region r of day d and region s of day d+1 are
        linked when they have the same cluster and share at least one pixel with
        ``shared / (pixels_r + pixels_s - shared) >= min_iou`` (FP64); a track is a connected
        component of the links, numbered 1..T in the order of its smallest region id.  With
        ``min_iou > 0.5`` every track is a chain with one region per day over its days.  The result
        also has ``tracks``, int64 ``[T,7]`` rows (cluster, first_day, last_day, regions, pixels,
        first_region, branched), and ``region_tracks``, int32 ``[R]``, the track of region r at
        index r - 1.  ``track_map_out``: optional int32 array / tensor, host or CUDA, like
        ``region_map_out``; it receives the track id of every pixel, 0 where no point.  Built on
        the GPU from the region map and the overlaps of consecutive days; the caller's own
        ``region_overlaps`` stay as they are without tracks.

        ``region_adjacency=True`` (needs ``regions``, else ``ValueError`` before any GPU work): the
        result also has ``region_adjacency``, int64 ``[M,6]`` rows (day, region_a, region_b, edges,
        y_first, x_first): one for every pair of regions a < b of one day joined by at least one
        edge between 4-neighbouring pixels, with the number of such edges (their shared border) and
        the upper or left pixel of their first edge, sorted by that edge (index 2 (y W + x) +
        direction, 0 to the right and 1 downwards, within the day).  Corner contacts have no row.
        And ``region_boundaries``, int64 ``[R,4]`` (perimeter, region_edges, background_edges,
        border_edges) of region r at index r - 1: the sides of its pixels facing another region,
        a pixel without a point and the raster edge, and their sum.  Counted on the GPU from the
        region map; with several ranks every rank builds the same rows."""
        init = np.ascontiguousarray(init, dtype=np.float64)
        if init.ndim != 2 or init.shape[1] != 3:
            raise ValueError("init must be [K,3]")
        k = init.shape[0]
        n = self.n_points
        lab_ptr, lab_mem, labels = None, C.MEM_HOST, None
        if labels_out is not None:
            lab_ptr, lab_mem = _as_out_buffer(labels_out, np.int32, n, "labels_out")
            labels = labels_out
            if lab_mem == C.MEM_DEVICE:
                self._after_torch(labels_out)
        elif want_labels:
            labels = self._result_buffer("labels", (n,), np.int32)
            lab_ptr = labels.ctypes.data
        centers = np.empty((k, 3), dtype=np.float64)
        n_iter = c_int(0)
        inertia = c_double(0.0)
        dev_maps, stats, trans = self._bind_outputs(
            k, cluster_map_out=cluster_map_out, day_stats=day_stats, transitions=transitions, regions=regions,
            region_map_out=region_map_out, region_overlaps=region_overlaps, tracks=tracks, track_map_out=track_map_out,
            region_adjacency=region_adjacency)
        self._check(self._lib.mdkm_fit(
            self._h, int(k), init.ctypes.data_as(POINTER(c_double)), int(max_iter), float(tol),
            c_void_p(lab_ptr) if lab_ptr else None, lab_mem,
            centers.ctypes.data_as(POINTER(c_double)), byref(n_iter), byref(inertia)))
        if lab_mem == C.MEM_DEVICE or dev_maps:
            self._before_torch()
        nref, nrel, tols = c_int64(0), c_int64(0), c_double(0)
        self._lib.mdkm_fit_stats(self._h, byref(nref), byref(nrel), byref(tols))
        work, groups = c_int64(0), c_int64(0)
        self._lib.mdkm_fit_worklist(self._h, byref(work), byref(groups))
        out = {
            "labels": labels, "centers": centers, "n_iter": int(n_iter.value),
            "inertia": float(inertia.value), "n_refined": int(nref.value),
            "n_relocations": int(nrel.value), "tol_scaled": float(tols.value),
            "worklist_groups": int(work.value), "groups": int(groups.value),
        }
        out.update(self._read_outputs(stats, trans, regions, region_overlaps, tracks, region_adjacency))
        return out

    def lloyd_step(self, centroids, want_labels=True):
        """Single E-step + sums (test hook).  Returns (labels, sums[K,3], counts[K], n_refined)."""
        c = np.ascontiguousarray(centroids, dtype=np.float64)
        k = c.shape[0]
        n = self.n_points
        labels = np.empty(n, dtype=np.int32) if want_labels else None
        sums = np.empty((k, 3), dtype=np.float64)
        counts = np.empty(k, dtype=np.int64)
        self._check(self._lib.mdkm_lloyd_step(
            self._h, int(k), c.ctypes.data_as(POINTER(c_double)),
            c_void_p(labels.ctypes.data) if labels is not None else None, C.MEM_HOST,
            sums.ctypes.data_as(POINTER(c_double)), counts.ctypes.data_as(POINTER(c_int64))))
        nref = c_int64(0)
        self._lib.mdkm_fit_stats(self._h, byref(nref), None, None)
        return labels, sums, counts, int(nref.value)

    def predict(self, centroids, want_labels=True, cluster_map_out=None, day_stats=False, transitions=None,
                regions=None, region_map_out=None, region_overlaps=None, tracks=None, track_map_out=None,
                region_adjacency=False):
        """E-step only (KMeans.predict): returns (labels int32[N] or None, inertia).
        ``cluster_map_out``: as in ``fit``.  ``day_stats=True``: returns
        (labels, inertia, day_counts, day_means) instead, as in ``fit``.  ``transitions``: day
        pairs as in ``fit``; their counts are appended to the returned tuple.  ``regions`` /
        ``region_map_out``: as in ``fit``; the table and the means are appended after that.
        ``region_overlaps``: as in ``fit``; the rows are appended after that.  ``tracks`` /
        ``track_map_out``: as in ``fit``; the track table and the region tracks are appended after
        that.  ``region_adjacency``: as in ``fit``; the rows and the region boundaries are appended
        last."""
        c = np.ascontiguousarray(centroids, dtype=np.float64)
        if c.ndim != 2 or c.shape[1] != 3:
            raise ValueError("centroids must be [K,3]")
        labels = self._result_buffer("labels", (self.n_points,), np.int32) if want_labels else None
        inertia = c_double(0.0)
        dev_maps, stats, trans = self._bind_outputs(
            c.shape[0], cluster_map_out=cluster_map_out, day_stats=day_stats, transitions=transitions, regions=regions,
            region_map_out=region_map_out, region_overlaps=region_overlaps, tracks=tracks, track_map_out=track_map_out,
            region_adjacency=region_adjacency)
        self._check(self._lib.mdkm_predict(
            self._h, int(c.shape[0]), c.ctypes.data_as(POINTER(c_double)),
            c_void_p(labels.ctypes.data) if labels is not None else None, C.MEM_HOST, byref(inertia)))
        if dev_maps:
            self._before_torch()
        results = self._read_outputs(stats, trans, regions, region_overlaps, tracks, region_adjacency)
        return (labels, float(inertia.value)) + tuple(results.values())

    def kmeans_plusplus(self, n_clusters: int, random_state):
        """k-means++ seeding (sklearn/_kmeans.py:180-278); RNG draws come from ``random_state``
        (a ``numpy.random.RandomState``) in scikit-learn's order, distances run on the GPU."""
        k = int(n_clusters)
        n = self.n_points_global
        n_local_trials = 2 + int(np.log(k))
        # RandomState.choice(n, p=w/w.sum()) (sklearn/_kmeans.py:228): one uniform draw inverted
        # through cdf = cumsum(p)/cdf[-1] with searchsorted(side="right") -- reproduced bit for bit
        # for any n from the closed form of that running sum (_npdraw.py), without an n-sized array.
        from ._npdraw import choice_uniform

        first = choice_uniform(random_state, n)
        rv = np.ascontiguousarray(
            [random_state.uniform(size=n_local_trials) for _ in range(k - 1)], dtype=np.float64
        ).reshape(max(k - 1, 0), n_local_trials)
        centers = np.empty((k, 3), dtype=np.float64)
        idx = np.empty(k, dtype=np.int64)
        self._check(self._lib.mdkm_kmeans_plusplus(
            self._h, k, first, rv.ctypes.data_as(POINTER(c_double)) if k > 1 else None, n_local_trials,
            centers.ctypes.data_as(POINTER(c_double)), idx.ctypes.data_as(POINTER(c_int64))))
        return centers, idx

    def drop_caches(self):
        """Forget the tile-ordered mirror and the group summaries of the resident cloud (the next
        fit rebuilds them)."""
        self._check(self._lib.mdkm_drop_caches(self._h))

    # -- profiling -----------------------------------------------------------------------
    def profile(self, on: bool):
        self._check(self._lib.mdkm_profile_enable(self._h, 1 if on else 0))

    def profile_phases(self):
        """{phase: (ms, count)} of the kernel groups since the last read (see mdkm_profile_phase)."""
        out = {}
        for name, ph in (("unproject", C.PHASE_UNPROJECT), ("build", C.PHASE_BUILD), ("step", C.PHASE_STEP),
                         ("final", C.PHASE_FINAL)):
            ms, cnt = c_double(0), c_int64(0)
            self._check(self._lib.mdkm_profile_phase(self._h, ph, byref(ms), byref(cnt)))
            out[name] = (float(ms.value), int(cnt.value))
        return out

    def profile_read(self):
        ms, ns, nl = c_double(0), c_int(0), c_int(0)
        self._check(self._lib.mdkm_profile_read(self._h, byref(ms), byref(ns), byref(nl)))
        return float(ms.value), int(ns.value), int(nl.value)
