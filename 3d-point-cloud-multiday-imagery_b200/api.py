"""Public Python API: the drop-in for the reference's multi-day point-cloud fusion step.

The reference has no such routine of its own (SURVEY.md F1); the signature below is
assembled from the three anchors it does have:

* the plugin contract ``SatellitePlugin.run(...) -> List[Layer]`` (``interface.py:10-47``,
  ``Layer = (ndarray, params, type)`` at ``interface.py:5-7``),
* the unprojection tail of ``HeightMapExtractor.run``
  (``members/rafael/disparity/plugin.py:147-233``), whose Points layer this module
  reproduces (napari (z, y, x) column order, ``plugin.py:192``; layer params ``:220-233``),
* scikit-learn's ``KMeans`` call convention as the reference uses it
  (``members/jasraj/land_use_classification/core.py:227-228``): ``n_clusters``, ``init``,
  ``n_init``, ``max_iter=300``, ``tol=1e-4``, ``random_state``; results named like
  ``labels_ / cluster_centers_ / inertia_ / n_iter_``.

Everything numeric happens in libmdkm.so (sm_100a CUDA kernels); this file only validates
arguments, draws the host-side random numbers scikit-learn would draw, and packs results.
"""
from __future__ import annotations

import traceback
from dataclasses import dataclass, field
from typing import Any, Dict, List, Literal, Optional, Tuple

import numpy as np

from .engine import Engine, check_min_iou

LayerType = Literal["image", "labels", "points", "shapes"]
Layer = Tuple[np.ndarray, Dict[str, Any], LayerType]  # interface.py:5-7

MAX_ABS_HEIGHT = 144.0  # MAX_DISP / 2 (constants.py:54, plugin.py:151)
MAX_REGION_OVERLAP_PAIRS = 8192  # day pairs of one call's region overlaps (mdkm_bind_region_overlaps)


@dataclass
class FusionResult:
    """What the fused k-means returns (names follow scikit-learn's fitted attributes)."""

    labels: np.ndarray           # int32 [N], np.where order per day, days concatenated
    centroids: np.ndarray        # float64 [K,3] as (x, y, z)
    fused_cloud: Optional[np.ndarray]  # float32 [N,3] in napari (z, y, x) order, or None
    n_iter: int
    inertia: float
    n_points: int
    n_refined: int = 0           # point-iterations decided by the FP64 refine (near-ties)
    n_relocations: int = 0
    height_norm: Optional[np.ndarray] = None  # plugin.py:184-188 'height' property, if requested
    extra: Dict[str, Any] = field(default_factory=dict)
    # labels on the pixel grid (return_cluster_map=True): label + 1 where a pixel produced a point,
    # 0 elsewhere; uint8 (k <= 255) or uint16, [D,H,W] -- or this rank's flat pixel range
    cluster_map: Optional[np.ndarray] = None
    # per-day composition (return_day_stats=True), rows = global days of the stack: points of day d
    # with label j (int64 [D,K]) and their mean (x, y, z) in the clustered frame (float64 [D,K,3],
    # NaN where the count is 0); summed over all ranks
    day_counts: Optional[np.ndarray] = None
    day_means: Optional[np.ndarray] = None
    # from-to counts of day pairs (return_transitions): transitions[p, s, t] = pixels with state s on
    # day a and t on day b of transition_pairs[p] = (a, b), state = label + 1 or 0 (no point);
    # int64 [P,K+1,K+1] and int64 [P,2], over the whole stack on every rank
    transitions: Optional[np.ndarray] = None
    transition_pairs: Optional[np.ndarray] = None
    # connected regions of the cluster map (return_regions): one row per region, numbered 1..R in
    # the raster order (day, y, x) of its first pixel -- int64 [R,7] (day, cluster, pixels, y_min,
    # x_min, y_max, x_max) and float64 [R,3] mean (x, y, z) in the clustered frame, over the whole
    # stack on every rank; region_map (return_region_map): int32 region id per pixel, 0 where no
    # point, [D,H,W] or this rank's flat pixel range like cluster_map
    regions: Optional[np.ndarray] = None
    region_means: Optional[np.ndarray] = None
    region_map: Optional[np.ndarray] = None
    # region overlaps of day pairs (return_region_overlaps): one row per pair of regions (r of day a,
    # s of day b) with a shared pixel -- int64 [M,6] (pair, region_a, region_b, pixels, y_first,
    # x_first), sorted by pair, then by the first shared pixel -- and the pairs, int64 [P,2]; over
    # the whole stack on every rank
    region_overlaps: Optional[np.ndarray] = None
    region_overlap_pairs: Optional[np.ndarray] = None
    # object tracks (return_tracks): regions of consecutive days linked by IoU >= track_min_iou and
    # the same cluster, numbered 1..T by their smallest region id -- int64 [T,7] (cluster,
    # first_day, last_day, regions, pixels, first_region, branched) and the track of every region,
    # int32 [R] (region r at index r - 1), over the whole stack on every rank; track_map
    # (return_track_map): int32 track id per pixel, 0 where no point, shaped like region_map
    tracks: Optional[np.ndarray] = None
    region_tracks: Optional[np.ndarray] = None
    track_map: Optional[np.ndarray] = None
    # region adjacency within a day (return_region_adjacency): one row per pair of regions a < b of
    # one day that share an edge -- int64 [M,6] (day, region_a, region_b, edges, y_first, x_first),
    # sorted by their first edge -- and per region int64 [R,4] (perimeter, region_edges,
    # background_edges, border_edges); over the whole stack on every rank
    region_adjacency: Optional[np.ndarray] = None
    region_boundaries: Optional[np.ndarray] = None

    # scikit-learn style aliases
    @property
    def labels_(self):
        return self.labels

    @property
    def cluster_centers_(self):
        return self.centroids

    @property
    def inertia_(self):
        return self.inertia

    @property
    def n_iter_(self):
        return self.n_iter


def _check_random_state(seed):
    if seed is None or isinstance(seed, (int, np.integer)):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError("random_state must be None, an int or a numpy RandomState")


def _label_mapping(l1, l2, k):
    """The map label-of-l1 -> label-of-l2 by first occurrence, and whether every point obeys it
    (the loop of sklearn/cluster/_k_means_common.pyx:314-330 on one shard)."""
    mapping = np.full(k, -1, dtype=np.int64)
    if l1.shape[0]:
        uniq, first = np.unique(l1, return_index=True)
        mapping[uniq] = l2[first]
    return mapping, bool(np.array_equal(mapping[l1], l2))


def _merge_label_mappings(mappings, oks) -> bool:
    """Do the shards' maps describe ONE map?  (labels equal up to a permutation, over all shards)"""
    merged = np.full(mappings[0].shape[0], -1, dtype=np.int64)
    for m in mappings:
        m = np.asarray(m, dtype=np.int64)
        both = (m >= 0) & (merged >= 0)
        if np.any(m[both] != merged[both]):
            return False
        merged = np.where(m >= 0, m, merged)
    return bool(all(oks))


def _is_same_clustering(l1, l2, k, gather=None) -> bool:
    """sklearn/cluster/_k_means_common.pyx:314-330 (labels equal up to a permutation).  With
    sharded labels ``gather(mapping, ok) -> (mappings, oks)`` collects every rank's shard map
    (a collective: all ranks call it), and the verdict is the same on every rank."""
    mapping, ok = _label_mapping(l1, l2, k)
    if gather is None:
        return ok
    return _merge_label_mappings(*gather(mapping, ok))


def _random_seeds(rs, n: int, k: int) -> np.ndarray:
    """``random_state.choice(n, size=k, replace=False, p=w / w.sum())`` with unit weights
    (sklearn/_kmeans.py:1014-1021), reproduced bit for bit for any ``n`` without the n-sized
    probability vector (``_npdraw.py``)."""
    from ._npdraw import choice_uniform_without_replacement

    return choice_uniform_without_replacement(rs, n, k)


def cluster_map_dtype(n_clusters: int):
    """Element type of a cluster map for ``n_clusters`` labels (0 is the background)."""
    return np.uint8 if int(n_clusters) <= 255 else np.uint16


# The pixel-map outputs of ``Engine.fit``; the FusionResult field of each is its name without "_out".
PIXEL_MAP_OUTPUTS = ("cluster_map_out", "region_map_out", "track_map_out")


def _pixel_map_dtype(kw, n_clusters):
    """Element type of the pixel map output ``kw``: labels + 1 for the cluster map, int32 ids otherwise."""
    return cluster_map_dtype(n_clusters) if kw == "cluster_map_out" else np.int32


def transition_pairs(spec, n_days: int, what: str = "transitions") -> np.ndarray:
    """The day pairs ``return_transitions`` asks for, as int64 ``[P,2]``: ``True`` -> the
    consecutive pairs ``(d, d+1)``; a sequence of ``(a, b)`` -> those pairs in that order (they
    may skip days, run backwards, repeat, or have ``a == b``).  Raises ``ValueError`` for a day
    outside ``[0, n_days)`` or when there is no pair.  ``what``: the output the pairs are for, as
    the messages name it ("region overlaps" for ``return_region_overlaps``)."""
    arg = "return_" + what.replace(" ", "_")
    if isinstance(spec, (bool, np.bool_)):
        if not spec:
            raise ValueError(f"{arg}=False asks for no pairs")
        d = np.arange(max(int(n_days) - 1, 0), dtype=np.int64)
        pairs = np.stack([d, d + 1], axis=1)
    else:
        pairs = np.asarray(spec)
        if pairs.size == 0:
            pairs = pairs.reshape(0, 2)
        if pairs.ndim != 2 or pairs.shape[1] != 2 or not (np.issubdtype(pairs.dtype, np.integer)):
            raise ValueError(f"{arg} must be True or a sequence of (day_a, day_b) integer pairs")
        pairs = pairs.astype(np.int64)
    if pairs.shape[0] == 0:
        raise ValueError(f"no day pair to count {what} of (the stack has {n_days} day(s))")
    bad = (pairs < 0) | (pairs >= n_days)
    if bad.any():
        p = int(np.argmax(bad.any(axis=1)))
        raise ValueError(f"{what[:-1]} pair {p} = {tuple(int(v) for v in pairs[p])}: days must be in [0, {n_days})")
    return pairs


def _asks_for_pairs(spec) -> bool:
    """Does a ``return_transitions`` / ``return_region_overlaps`` value ask for pairs (not None / False)?"""
    return spec is not None and not (isinstance(spec, (bool, np.bool_)) and not spec)


def requested_connectivity(return_regions, connectivity=4, return_region_map=False):
    """The connectivity ``return_regions`` / ``return_region_map`` ask for: None (no regions) or
    4 / 8.  The region map implies the regions.  Raises ``ValueError`` for a connectivity other
    than 4 or 8."""
    if not (return_regions or return_region_map):
        return None
    if isinstance(connectivity, (bool, np.bool_)) or connectivity not in (4, 8):
        raise ValueError(f"region_connectivity must be 4 or 8, got {connectivity!r}")
    return int(connectivity)


def requested_min_iou(return_tracks, min_iou=0.5, return_track_map=False):
    """The min_iou ``return_tracks`` / ``return_track_map`` ask for: None (no tracks) or a float in
    (0, 1].  The track map implies the tracks.  Raises ``ValueError`` for a value that is not a
    real number in (0, 1] (NaN and bools included)."""
    if not (return_tracks or return_track_map):
        return None
    return check_min_iou(min_iou, "track_min_iou")


def _stack_days(height_maps, stack_shape, raster_layout) -> int:
    """D of the stack ``fuse_multiday_kmeans`` is given (before anything reaches the GPU)."""
    if stack_shape is not None:
        return int(stack_shape[0])
    shp = tuple(height_maps.shape)
    if raster_layout == "gtiff3":
        shp = shp[:-1]
    return 1 if len(shp) == 2 else int(shp[0])


def _run_kmeans(eng: Engine, *, n_clusters, init, n_init, max_iter, tol, random_state, want_labels=True,
                labels_out=None, gather_mappings=None, **outputs):
    """KMeans.fit driver (sklearn/_kmeans.py:1436-1563): init, n_init restarts, best inertia.

    ``labels_out``: optional int32 array that receives this rank's labels of the best run.
    ``outputs``: the optional outputs of ``Engine.fit`` (``cluster_map_out``, ``day_stats``,
    ``transitions``, ``regions``, ...); the result has the best run's -- every run returns fresh
    arrays, so the best run's stay with it.  With restarts every run writes its pixel maps
    (``PIXEL_MAP_OUTPUTS``) into device scratch tensors; the best run's are kept by swapping and
    copied out once at the end.
    ``gather_mappings``: with a multi-rank engine, the collective that lets the ranks agree on
    sklearn's "same clustering up to a permutation" test (see ``_is_same_clustering``); when it is
    missing the test is skipped on multi-rank engines (the inertia comparison alone decides)."""
    n = eng.n_points_global  # with a communicator: every rank draws the same seeds
    k = int(n_clusters)
    if k < 1:
        raise ValueError("n_clusters must be >= 1")
    if n < k:
        raise ValueError(f"n_samples={n} should be >= n_clusters={k}.")
    rs = _check_random_state(random_state)
    init_is_array = not isinstance(init, str)
    if init_is_array:
        init_arr = np.ascontiguousarray(init, dtype=np.float64)
        if init_arr.shape != (k, 3):
            raise ValueError(f"The shape of the initial centers {init_arr.shape} does not match (n_clusters, 3)")
        n_init = 1  # sklearn/_kmeans.py:905-913: explicit init => single run
    elif init not in ("k-means++", "random"):
        raise ValueError("init must be 'k-means++', 'random' or an array of shape (n_clusters, 3)")
    if n_init == "auto":
        n_init = 1 if init == "k-means++" else 10  # sklearn/_kmeans.py:896-903
    if eng.n_ranks > 1 and gather_mappings is None:
        from .dist import torch_gather_mappings

        gather_mappings = torch_gather_mappings(eng)  # None unless torch.distributed spans the ranks
    single = int(n_init) == 1
    best = None
    scratch = {}  # pixel-map keyword -> [this run's map, the best run's map]
    for kw in PIXEL_MAP_OUTPUTS:
        if outputs.get(kw) is not None and not single:
            import torch

            # (a copy of the best map per improvement would cost a device->host transfer each time)
            tdt = getattr(torch, np.dtype(_pixel_map_dtype(kw, k)).name)
            run_map = torch.empty(eng.raster_range[4], dtype=tdt, device=f"cuda:{eng.device}")
            scratch[kw] = [run_map, torch.empty_like(run_map)]
    for _ in range(int(n_init)):
        if init_is_array:
            centers0 = init_arr
        elif init == "random":
            centers0 = eng.gather_points(_random_seeds(rs, n, k)).astype(np.float64)
        else:
            centers0, _ = eng.kmeans_plusplus(k, rs)
        r = eng.fit(centers0, max_iter=max_iter, tol=tol, want_labels=want_labels,
                    labels_out=labels_out if (single and want_labels) else None,
                    **dict(outputs, **{kw: maps[0] for kw, maps in scratch.items()}))
        # sklearn/_kmeans.py:1534-1541: a run replaces the best one when its inertia is lower AND it
        # is not the same clustering up to a permutation.  The inertia is global, so every rank
        # takes the same branch and the (collective) permutation test pairs up.
        better = best is not None and r["inertia"] < best["inertia"]
        same = False
        if better and want_labels and (eng.n_ranks == 1 or gather_mappings is not None):
            same = _is_same_clustering(r["labels"], best["labels"], k, gather_mappings if eng.n_ranks > 1 else None)
        if best is None or (better and not same):
            best = r
            if not single and r["labels"] is not None:
                best = dict(r, labels=r["labels"].copy())  # result buffers are reused by the next run
            for maps in scratch.values():
                maps.reverse()  # this run's map becomes the best one
    if labels_out is not None and want_labels and not single:
        labels_out[...] = best["labels"]
        best = dict(best, labels=labels_out)
    for kw, (_, best_map) in scratch.items():
        _copy_map_out(best_map, outputs[kw])
    return best


def _copy_map_out(src, out):
    """Device map ``src`` (flat torch tensor) -> the caller's ``out`` (numpy array or torch tensor).
    16-bit maps are moved as int16: the bits are the same and every torch build copies int16."""
    import torch

    wide = src.dtype == torch.uint16
    s = src.view(torch.int16) if wide else src
    if type(out).__module__.startswith("torch"):
        o = out.view(torch.int16) if wide else out
        o.view(-1).copy_(s)
    else:
        host = s.cpu().numpy()
        out.reshape(-1)[...] = host.view(np.uint16) if wide else host


def fuse_multiday_kmeans(height_maps, valid_masks=None, *, n_clusters=8, init="k-means++", n_init=1,
                         max_iter=300, tol=1e-4, random_state=None, max_abs_height=MAX_ABS_HEIGHT,
                         detrend=False, disparity_scale=None, ground_level=False, return_cloud=True,
                         device=0, devices=None, engine=None, stack_shape=None,
                         pix_begin=0, raster_layout=None, return_cluster_map=False,
                         return_day_stats=False, return_transitions=False, return_regions=False,
                         region_connectivity=4, return_region_map=False,
                         return_region_overlaps=False, return_tracks=False, track_min_iou=0.5,
                         return_track_map=False, return_region_adjacency=False) -> FusionResult:
    """Unproject a multi-day height-map stack into one XYZ cloud and cluster it (Lloyd).

    height_maps : float32 ``[D,H,W]`` (NaN = nodata), numpy or torch (CPU or CUDA); or int16
        OpenCV fixed-point disparity with ``disparity_scale=-1/16`` (plugin.py:147-148).
    valid_masks : optional bool/uint8 ``[D,H,W]`` (``final_defined`` of disparity.py:203-204).
    n_clusters, init, n_init, max_iter, tol, random_state : as sklearn.cluster.KMeans.
    detrend : apply the per-day plane fit of plugin.py:161-171 to z before clustering.
    ground_level : per day, shift z so that its 2nd percentile is 0 and return the 'height'
        colour property (plugin.py:181-192), before clustering -- with ``detrend=True`` this
        is the reference's whole per-pair tail, applied to every day of the stack.
    raster_layout : "gtiff3" when ``height_maps`` is ``[D,H,W,3]`` float32 in the pixel layout of the
        reference's ``5-out-F.tif`` (see ``fuse_height_rasters``).
    engine : reuse an existing ``Engine`` (keeps device buffers, and with
        ``Engine(pinned_results=True)`` page-locked result buffers, across calls); with a
        multi-rank engine pass this rank's flat slice plus ``stack_shape`` / ``pix_begin``.
        A ``DeviceGroup`` is accepted too (see ``devices``).
    devices : several CUDA devices used from THIS process (``[0, 1, 2, 3]``): the host stack is
        sharded over them by row bands, one host thread drives each device, the devices exchange
        their K x 4 partial sums over NVLink inside the Lloyd kernel, and the results are
        assembled in the reference's point order -- bit-identical to one device.  This is how the
        in-process caller of the reference (a napari worker thread, widget.py:116-147) gets more
        than one GPU without ``torchrun``.
    return_cluster_map : also return ``cluster_map``, the labels on the input pixel grid (a
        napari Labels layer): ``label + 1`` at each pixel that produced a point, 0 at the others;
        uint8 for ``n_clusters <= 255``, else uint16.  ``[D,H,W]`` for a whole stack; this rank's
        flat ``[pix_count]`` slice for a pre-sharded call (``stack_shape`` / ``pix_begin``), as
        ``labels`` is this rank's shard.  The map is written on the GPU by the final labelling pass.
    return_day_stats : also return ``day_counts`` (int64 ``[D,K]``: points of day d with label j) and
        ``day_means`` (float64 ``[D,K,3]``: their mean (x, y, z) in the clustered coordinates, like
        ``centroids``; NaN where the count is 0).  Rows are the global days of the stack, also for a
        pre-sharded call, and the numbers are summed over all ranks.  They come from integer sums on
        the fixed-point frame accumulated by the final labelling pass, so they are bitwise the same
        for any number of GPUs.
    return_transitions : ``True`` (the consecutive pairs ``(d, d+1)``) or a sequence of day pairs
        ``(a, b)``: also return ``transitions``, int64 ``[P,K+1,K+1]``, the from-to matrix of every
        pair -- ``transitions[p, s, t]`` is the number of pixels with state s on day a and t on day
        b, where a pixel's state is ``label + 1`` when it produced a point that day and 0 when it
        did not (row 0 / column 0: pixels that gained / lost their point) -- and
        ``transition_pairs`` (int64 ``[P,2]``).  Binned on the GPU from the cluster map the final
        labelling pass writes (the map itself need not be returned).  A pre-sharded call needs
        ranks that together hold the whole stack; every rank receives the global counts.
        Out-of-range days raise ``ValueError`` before any GPU work.
    return_regions : also return the connected regions of the cluster map -- maximal sets of
        pixels of one day with the same label that are connected (``region_connectivity`` 4: edge
        neighbours, as ``scipy.ndimage.label``; 8: edge and corner neighbours), numbered 1..R over
        the whole stack in the raster order (day, y, x) of each region's first pixel: ``regions``,
        int64 ``[R,7]`` rows (day, cluster, pixels, y_min, x_min, y_max, x_max; inclusive bounds),
        and ``region_means``, float64 ``[R,3]``, the mean (x, y, z) of each region's points in the
        clustered coordinates (computed like ``day_means``: bitwise the same on any number of
        GPUs).  Labelled on the GPU from the cluster map; a pre-sharded call needs ranks that
        together hold the whole stack, and every rank receives the whole table.
    return_region_map : also return ``region_map``, int32, the region id of every pixel that
        produced a point and 0 elsewhere; ``[D,H,W]``, or this rank's flat slice for a pre-sharded
        call, like ``cluster_map``.  Implies ``return_regions``.  A connectivity other than 4 or 8
        raises ``ValueError`` before any GPU work.
    return_region_overlaps : ``True`` (the consecutive pairs ``(d, d+1)``) or a sequence of day
        pairs ``(a, b)``, as for ``return_transitions``: also return ``region_overlaps``, int64
        ``[M,6]`` rows (pair, region_a, region_b, pixels, y_first, x_first) -- one for every pair
        of regions (r of day a, s of day b) that share at least one pixel, with the number of
        shared pixels and the first shared pixel, sorted by pair and then by the raster order of
        that pixel -- and ``region_overlap_pairs`` (int64 ``[P,2]``).  Region ids are those of
        ``regions``; r and s may have different clusters.  Implies ``return_regions``.  Counted on
        the GPU from the region map; every rank of a pre-sharded call receives the same rows.
        Out-of-range days, or more than ``MAX_REGION_OVERLAP_PAIRS``
        (8192) pairs, raise ``ValueError`` before any GPU work.
    return_region_adjacency : also return which regions of one day touch and each region's
        perimeter.  ``region_adjacency``, int64 ``[M,6]`` rows (day, region_a, region_b, edges,
        y_first, x_first): one for every pair of regions a < b of one day joined by at least one
        edge between 4-neighbouring pixels, with the number of such edges (the length of their
        shared border) and the upper or left pixel of their first edge, sorted by that edge (index
        ``2 (y W + x) + direction`` within the day, direction 0 to the right, 1 downwards).
        Regions that touch only at a corner have no row.  ``region_boundaries``, int64 ``[R,4]``
        (perimeter, region_edges, background_edges, border_edges; region r at index r - 1): the
        sides of a region's pixels facing another region, a pixel without a point and the raster
        edge, and their sum (``4 pixels = perimeter + 2 x inner edges``).  Implies
        ``return_regions``; counted on the GPU from the region map, and every rank of a
        pre-sharded call receives the same rows.
    return_tracks : also return object tracks -- which region is the same object over the stack.
        Region r of day d and region s of day d+1 are linked when they have the same cluster and
        share at least one pixel with ``shared / (pixels_r + pixels_s - shared) >= track_min_iou``
        (FP64); a track is a connected component of the links (a region without links is a track
        of its own), numbered 1..T in the order of its smallest region id, and does not bridge a
        day without the object.  ``tracks``, int64 ``[T,7]`` rows (cluster, first_day, last_day,
        regions, pixels, first_region, branched: 1 when a region of the track has two or more
        links to one neighbouring day), and ``region_tracks``, int32 ``[R]`` (the track of region r
        at index r - 1).  With ``track_min_iou > 0.5`` every track is a chain with one region per
        day over ``[first_day, last_day]``: two regions of day d+1 cannot both overlap more than
        half of one region of day d.  Implies ``return_regions``; built on the GPU, with no map
        copy to the host, and every rank of a pre-sharded call receives the same tracks.
    track_min_iou : the IoU a link needs, a real number in (0, 1] (default 0.5); anything else,
        NaN and bools included, raises ``ValueError`` before any GPU work.
    return_track_map : also return ``track_map``, int32, the track id of every pixel that produced
        a point and 0 elsewhere (a napari Labels layer in which an object keeps its colour across
        days); shaped like ``region_map``.  Implies ``return_tracks``.
    Returns a FusionResult; ``fused_cloud`` is float32 ``[N,3]`` in napari (z,y,x) order.
    """
    from .group import DeviceGroup

    pairs = ov_pairs = None
    if _asks_for_pairs(return_transitions):
        pairs = transition_pairs(return_transitions, _stack_days(height_maps, stack_shape, raster_layout))
    if _asks_for_pairs(return_region_overlaps):
        ov_pairs = transition_pairs(return_region_overlaps, _stack_days(height_maps, stack_shape, raster_layout),
                                    "region overlaps")
        if ov_pairs.shape[0] > MAX_REGION_OVERLAP_PAIRS:
            raise ValueError(f"return_region_overlaps asks for {ov_pairs.shape[0]} pairs, at most "
                             f"{MAX_REGION_OVERLAP_PAIRS} are allowed")
    min_iou = requested_min_iou(return_tracks, track_min_iou, return_track_map)
    conn = requested_connectivity(return_regions or ov_pairs is not None or min_iou is not None
                                  or return_region_adjacency, region_connectivity, return_region_map)
    outputs = {"day_stats": return_day_stats, "transitions": pairs, "regions": conn, "region_overlaps": ov_pairs,
               "tracks": min_iou, "region_adjacency": bool(return_region_adjacency)}
    wanted = (return_cluster_map, return_region_map, return_track_map)
    maps = [kw for kw, want in zip(PIXEL_MAP_OUTPUTS, wanted) if want]
    if devices is not None or isinstance(engine, DeviceGroup):
        if stack_shape is not None or pix_begin:
            raise ValueError("stack_shape / pix_begin describe a pre-sharded stack; a device group shards by itself")
        return _fuse_on_group(height_maps, valid_masks, group=engine if isinstance(engine, DeviceGroup) else None,
                              devices=devices, n_clusters=n_clusters, init=init, n_init=n_init, max_iter=max_iter,
                              tol=tol, random_state=random_state, max_abs_height=max_abs_height, detrend=detrend,
                              disparity_scale=disparity_scale, ground_level=ground_level, return_cloud=return_cloud,
                              raster_layout=raster_layout, outputs=outputs, maps=maps)
    own = engine is None
    eng = engine or Engine(device)
    try:
        # without ground levelling the cloud is final as soon as a slab is unprojected: it is
        # streamed back while the rest of the stack is still being uploaded
        stream = "napari" if (return_cloud and not ground_level) else None
        n = eng.unproject(height_maps, valid_masks, max_abs_height=max_abs_height, detrend=detrend,
                          disparity_scale=disparity_scale, stack_shape=stack_shape, pix_begin=pix_begin,
                          stream_cloud=stream, raster_layout=raster_layout)
        cloud = None
        if stream is not None:
            n, cloud = n
        hn = None
        extra = {"segment_offsets": eng.segment_offsets}
        if ground_level:
            lo, hi, hn = eng.ground_level(True)
            extra["h_min"], extra["h_max"] = lo, hi
        # otherwise its device->host copy is issued now and overlaps the Lloyd loop
        if return_cloud and cloud is None:
            cloud = eng.get_cloud(napari_order=True, wait=False)
        for kw in maps:
            D, H, W, _, count = eng.raster_range
            shape = (D, H, W) if stack_shape is None else (count,)
            outputs[kw] = np.empty(shape, dtype=_pixel_map_dtype(kw, n_clusters))
        r = _run_kmeans(eng, n_clusters=n_clusters, init=init, n_init=n_init, max_iter=max_iter,
                        tol=tol, random_state=random_state, **outputs)
        eng.wait()
        return _fusion_result(r, outputs, {kw: outputs[kw] for kw in maps}, labels=r["labels"], fused_cloud=cloud,
                              n_points=n, height_norm=hn, extra=extra)
    finally:
        if own:
            eng.close()


def _fusion_result(r, outputs, maps, **fields) -> FusionResult:
    """The FusionResult of the k-means result ``r`` of a call with the ``Engine.fit`` keywords
    ``outputs`` and the pixel maps ``maps`` (keyword -> array).  ``fields``: labels, fused_cloud,
    n_points, height_norm and extra."""
    return FusionResult(centroids=r["centers"], n_iter=r["n_iter"], inertia=r["inertia"], n_refined=r["n_refined"],
                        n_relocations=r["n_relocations"],
                        day_counts=r.get("day_counts"), day_means=r.get("day_means"),
                        transitions=r.get("transitions"), transition_pairs=outputs["transitions"],
                        regions=r.get("regions"), region_means=r.get("region_means"),
                        region_overlaps=r.get("region_overlaps"), region_overlap_pairs=outputs["region_overlaps"],
                        tracks=r.get("tracks"), region_tracks=r.get("region_tracks"),
                        region_adjacency=r.get("region_adjacency"), region_boundaries=r.get("region_boundaries"),
                        **{kw.removesuffix("_out"): m for kw, m in maps.items()}, **fields)


def _fuse_on_group(height_maps, valid_masks, *, group, devices, n_clusters, init, n_init, max_iter, tol,
                   random_state, outputs, maps, **unproject_kw) -> FusionResult:
    """``fuse_multiday_kmeans`` on several devices of this process (``group.DeviceGroup``):
    ``outputs`` are the ``Engine.fit`` keywords of every rank, ``maps`` the keywords of the pixel
    maps to build."""
    import threading

    from .group import DeviceGroup, clone_random_state

    own = group is None
    grp = group or DeviceGroup(devices)
    try:
        if random_state is None:  # every rank must draw the same numbers
            random_state = int(np.random.RandomState().randint(0, 2**31 - 1))
        states = clone_random_state(random_state, grp.world)
        # thread all-gather of the shards' label maps (see _is_same_clustering)
        barrier = threading.Barrier(grp.world)
        slots = [None] * grp.world

        def gather_for(rank):
            def gather(mapping, ok):
                slots[rank] = (mapping, ok)
                barrier.wait()
                got = list(slots)
                barrier.wait()  # nobody overwrites a slot before everybody has read it
                return [g[0] for g in got], [g[1] for g in got]
            return gather

        def run(eng, labels_out, **map_bands):
            r = eng.rank
            return _run_kmeans(eng, n_clusters=n_clusters, init=init, n_init=n_init, max_iter=max_iter, tol=tol,
                               random_state=states[r], labels_out=labels_out,
                               gather_mappings=gather_for(r) if grp.world > 1 else None, **outputs, **map_bands)

        res, labels, cloud, hn, extra = grp.fuse(height_maps, valid_masks, run_kmeans=run,
                                                 maps={kw: _pixel_map_dtype(kw, n_clusters) for kw in maps},
                                                 **unproject_kw)
        return _fusion_result(res, outputs, {kw: extra.pop(kw.removesuffix("_out")) for kw in maps}, labels=labels,
                              fused_cloud=cloud, n_points=int(labels.shape[0]), height_norm=hn, extra=extra)
    finally:
        if own:
            grp.close()


def fuse_height_rasters(paths, **kwargs) -> FusionResult:
    """``fuse_multiday_kmeans`` on the reference's own per-pair height rasters: the
    ``5-out-F.tif`` files its stereo stage writes (disparity.py:213-224; 3-band Float32 GTiff,
    band 0 = -disparity/16, band 2 = final_defined).  The pixels go to the GPU as they are in
    the files; validity (band 2) and the |h| <= 144 test are applied there."""
    from .tiff_io import load_height_rasters

    stack = load_height_rasters(list(paths))
    return fuse_multiday_kmeans(stack, raster_layout="gtiff3", **kwargs)


def kmeans_points(points, *, n_clusters=8, init="k-means++", n_init=1, max_iter=300, tol=1e-4,
                  random_state=None, return_cloud=False, device=0,
                  engine: Optional[Engine] = None) -> FusionResult:
    """Lloyd k-means of an already unprojected ``[N,3]`` (x,y,z) float32 cloud."""
    own = engine is None
    eng = engine or Engine(device)
    try:
        n = eng.set_points(points)
        r = _run_kmeans(eng, n_clusters=n_clusters, init=init, n_init=n_init, max_iter=max_iter,
                        tol=tol, random_state=random_state)
        cloud = eng.get_cloud(napari_order=True) if return_cloud else None
        return FusionResult(labels=r["labels"], centroids=r["centers"], fused_cloud=cloud,
                            n_iter=r["n_iter"], inertia=r["inertia"], n_points=n,
                            n_refined=r["n_refined"], n_relocations=r["n_relocations"])
    finally:
        if own:
            eng.close()


def to_layers(result: FusionResult, prefix: str = "Multi-day") -> List[Layer]:
    """napari layers for a FusionResult, mirroring plugin.py:220-233.

    One Points layer with the fused cloud coloured by cluster (or by the reference's
    'height' property when it was computed) and one with the K centroids; when the result has a
    ``cluster_map``, a Labels layer with it (0 = no point at that pixel), and when it has a
    ``region_map``, a Labels layer with the region ids, and when it has a ``track_map``, a Labels
    layer with the track ids (one object keeps its colour from day to day).
    """
    if result.fused_cloud is None:
        raise ValueError("result has no fused_cloud (return_cloud=False)")
    props: Dict[str, Any] = {"cluster": result.labels}
    face = "cluster"
    if result.height_norm is not None:
        props["height"] = result.height_norm  # plugin.py:186-188
        face = "height"                       # plugin.py:231: the reference colours by 'height'
    layers: List[Layer] = [(
        result.fused_cloud,
        {
            "name": f"{prefix} 3D Point Cloud",
            "size": 2,
            "properties": props,
            "scale": (1, 1, 1),
            "opacity": 0.8,
            "face_colormap": "turbo",
            "face_color": face,
        },
        "points",
    )]
    c = result.centroids
    layers.append((
        np.stack([c[:, 2], c[:, 1], c[:, 0]], axis=1),
        {"name": f"{prefix} Cluster Centroids", "size": 12, "scale": (1, 1, 1),
         "properties": {"cluster": np.arange(c.shape[0])}, "face_color": "cluster",
         "face_colormap": "turbo", "symbol": "cross"},
        "points",
    ))
    if result.cluster_map is not None:
        layers.append((result.cluster_map, {"name": f"{prefix} Cluster Map", "opacity": 0.7}, "labels"))
    if result.region_map is not None:
        layers.append((result.region_map, {"name": f"{prefix} Regions", "opacity": 0.7}, "labels"))
    if result.track_map is not None:
        layers.append((result.track_map, {"name": f"{prefix} Tracks", "opacity": 0.7}, "labels"))
    return layers


class MultiDayFusionPlugin:
    """``SatellitePlugin``-shaped wrapper (interface.py:10-47) around the fused path.

    ``run`` never raises: like ``HeightMapExtractor.run`` (plugin.py:236-241) it returns a
    single 100x100 image layer named ``"Error: ..."`` on failure, so the napari worker thread
    (widget.py:116-147) sees the same convention.
    """

    requires_image = False  # plugin.py:30

    def __init__(self, n_clusters=8, device=0, devices=None, log_path=None, **kmeans_kwargs):
        """``log_path``: where the traceback of a failed run is appended, like the reference's
        ``data/TEMP/log.txt`` (plugin.py:48, 236-240); None = only printed.
        ``devices``: several GPUs of this process (see ``fuse_multiday_kmeans``)."""
        self.n_clusters = n_clusters
        self.device = device
        self.devices = devices
        self.log_path = log_path
        self.kmeans_kwargs = kmeans_kwargs

    @property
    def name(self) -> str:
        return "Multi-day 3D Point Cloud (B200 k-means fusion)"

    @property
    def requires_viewer(self) -> bool:
        return False

    def run(self, image, viewer=None, valid_masks=None) -> List[Layer]:
        try:
            res = fuse_multiday_kmeans(image, valid_masks, n_clusters=self.n_clusters, device=self.device,
                                       devices=self.devices, **self.kmeans_kwargs)
            return to_layers(res)
        except Exception as e:  # noqa: BLE001 - reference convention, plugin.py:236-241
            traceback.print_exc()
            if self.log_path is not None:
                try:  # plugin.py:238-239: f.writelines(f"Error: {e}\n{traceback}") into TEMP/log.txt
                    with open(self.log_path, "a") as f:
                        f.writelines(f"Error: {str(e)}\n{traceback.format_exc()}")
                except OSError:
                    pass
            return [(np.ones((100, 100)), {"name": f"Error: {str(e)}"}, "image")]
