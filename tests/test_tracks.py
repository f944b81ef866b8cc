"""Object tracks (``return_tracks`` / ``tracks=``): regions of consecutive days linked when they have
the same cluster and ``shared / (pixels_r + pixels_s - shared) >= min_iou`` in FP64, a track being
a connected component of the links, numbered 1..T by its smallest region id -- int64 [T,7]
(cluster, first_day, last_day, regions, pixels, first_region, branched), the track of every
region (int32 [R]) and an optional int32 track map.

The oracle is a numpy / scipy restatement on the region map and region table the same call
returns: the overlaps of (d, d+1) with ``np.unique`` on packed keys, the FP64 rule,
``scipy.sparse.csgraph.connected_components`` renumbered by smallest region id, and the table from
``np.minimum.at`` / ``np.maximum.at`` / ``np.add.at``.  The region map itself is checked against
``scipy.ndimage.label`` (restated from ``test_regions.py``).  Every GPU case also checks that asking
for tracks changes nothing else the call returns.

Label patterns are drawn with ``predict`` as in ``test_regions.py``: centroids that share x and y
and differ only in z make a pixel's label its nearest z level."""
import importlib
import math

import numpy as np
import pytest
from scipy import ndimage
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from oracle import unproject_oracle as UO

PKG = "3d-point-cloud-multiday-imagery_b200"
synth = importlib.import_module(PKG + ".synth")
api = importlib.import_module(PKG + ".api")
C = importlib.import_module(PKG + "._cabi")

IOUS = [1e-9, 0.5, float(np.nextafter(0.5, 1.0)), 1.0]


# ---------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------
def ref_region_map(cmap, conn):
    """scipy.ndimage.label per (day, value), ids renumbered by first raster pixel."""
    cmap = np.asarray(cmap)
    st = ndimage.generate_binary_structure(2, 1 if conn == 4 else 2)
    tmp = np.zeros(cmap.shape, dtype=np.int64)
    nxt = 0
    for d in range(cmap.shape[0]):
        for v in np.unique(cmap[d]):
            if v == 0:
                continue
            lab, n = ndimage.label(cmap[d] == v, structure=st)
            tmp[d][lab > 0] = lab[lab > 0] + nxt
            nxt += n
    flat = tmp.ravel()
    ids, first = np.unique(flat, return_index=True)
    keep = ids > 0
    ids, first = ids[keep], first[keep]
    order = np.argsort(first, kind="stable")
    remap = np.zeros(nxt + 1, dtype=np.int64)
    remap[ids[order]] = np.arange(1, ids.size + 1)
    return remap[flat].reshape(cmap.shape).astype(np.int32)


def ref_links(rmap, regions, min_iou):
    """The links (r, s) (0-based region indices) of consecutive days under the FP64 rule."""
    rmap = np.asarray(rmap)
    D = rmap.shape[0]
    flat = rmap.reshape(D, -1).astype(np.int64)
    rs = []
    for d in range(D - 1):
        a, b = flat[d], flat[d + 1]
        both = (a > 0) & (b > 0)
        keys, shared = np.unique((a[both] << 32) | b[both], return_counts=True)
        r, s = (keys >> 32) - 1, (keys & 0xFFFFFFFF) - 1
        iou = shared.astype(np.float64) / (regions[r, 2] + regions[s, 2] - shared).astype(np.float64)
        ok = (regions[r, 1] == regions[s, 1]) & (iou >= min_iou)
        rs.append(np.stack([r[ok], s[ok]], axis=1))
    return np.concatenate(rs) if rs else np.zeros((0, 2), np.int64)


def ref_tracks(rmap, regions, min_iou):
    """(tracks int64 [T,7], region_tracks int32 [R]) of the region map and its table."""
    R = regions.shape[0]
    links = ref_links(rmap, regions, min_iou)
    g = coo_matrix((np.ones(links.shape[0]), (links[:, 0], links[:, 1])), shape=(R, R))
    n, comp = connected_components(g, directed=False)
    first = np.full(n, R, np.int64)
    np.minimum.at(first, comp, np.arange(R))
    order = np.argsort(first, kind="stable")
    renum = np.empty(n, np.int64)
    renum[order] = np.arange(n)
    tid = renum[comp]
    fwd = np.bincount(links[:, 0], minlength=R)
    bwd = np.bincount(links[:, 1], minlength=R)
    t = np.zeros((n, 7), np.int64)
    t[:, 0] = regions[first[order], 1]
    t[:, 1] = np.iinfo(np.int64).max
    np.minimum.at(t[:, 1], tid, regions[:, 0])
    np.maximum.at(t[:, 2], tid, regions[:, 0])
    np.add.at(t[:, 3], tid, 1)
    np.add.at(t[:, 4], tid, regions[:, 2])
    t[:, 5] = first[order] + 1
    np.maximum.at(t[:, 6], tid, ((fwd > 1) | (bwd > 1)).astype(np.int64))
    return t, (tid + 1).astype(np.int32)


def check_tracks(tracks, region_tracks, rmap, regions, min_iou, tmap=None):
    """Bit for bit against the oracle, and the consequences the semantics promise."""
    ref_t, ref_rt = ref_tracks(rmap, regions, min_iou)
    assert tracks.dtype == np.int64 and tracks.ndim == 2 and tracks.shape[1] == 7
    assert region_tracks.dtype == np.int32 and region_tracks.shape == (regions.shape[0],)
    assert tracks.shape == ref_t.shape and tracks.tobytes() == ref_t.tobytes()
    assert region_tracks.tobytes() == ref_rt.tobytes()
    R, T = regions.shape[0], tracks.shape[0]
    assert T <= R
    if R:
        assert np.all(regions[:, 1] == tracks[region_tracks - 1, 0])  # one cluster per track
    if min_iou > 0.5:  # chains: one region per day over [first_day, last_day]
        assert np.all(tracks[:, 6] == 0)
        assert np.array_equal(tracks[:, 3], tracks[:, 2] - tracks[:, 1] + 1)
        days = np.unique(region_tracks.astype(np.int64) * (1 << 20) + regions[:, 0])
        assert days.size == R
    if tmap is not None:
        rmap = np.asarray(rmap)
        want = np.where(rmap > 0, np.concatenate([[0], region_tracks])[np.clip(rmap, 0, None)], 0)
        assert tmap.dtype == np.int32 and tmap.tobytes() == want.astype(np.int32).tobytes()


def levels(k):
    return np.linspace(-130.0, 130.0, k) if k > 1 else np.array([5.0])


def draw(labels_map, k):
    """Heights whose nearest level is the wanted label (-1: NaN, no point)."""
    z = levels(k)
    return np.where(labels_map >= 0, z[np.clip(labels_map, 0, k - 1)], np.nan).astype(np.float32)


def level_centroids(k, H, W):
    return np.stack([np.full(k, W / 2.0), np.full(k, H / 2.0), levels(k)], axis=1)


def _device_out(n, where):
    import torch

    buf = torch.full((n + 4,), -7, dtype=torch.int32, device="cuda")
    return buf[:n] if where == "aligned" else buf[1:n + 1]


def predict_checked(engine, labels_map, k, conn, min_iou, pairs=None, device_map=None, unproject=True):
    """predict on the drawn map with regions (and the caller's overlaps ``pairs``), without and with
    tracks: everything else bitwise equal, the region map against scipy, the tracks and the track
    map against the oracle.  ``device_map``: "aligned" / "offset" -- region and track maps in CUDA
    tensors (16-byte aligned, or 4 bytes past that), so the ids are read from the caller's map."""
    D, H, W = labels_map.shape
    hm = draw(labels_map, k)
    if unproject:
        engine.unproject(hm)
    c = level_centroids(k, H, W)
    dt = np.uint8 if k <= 255 else np.uint16
    trans = [(0, D - 1)]
    extra = {} if pairs is None else {"region_overlaps": pairs}
    cmap0 = np.empty(hm.shape, dt)
    rmap0 = np.empty(hm.shape, np.int32)
    base = engine.predict(c, cluster_map_out=cmap0, day_stats=True, transitions=trans, regions=conn,
                          region_map_out=rmap0, **extra)
    base = (base[0].copy(),) + base[1:]
    cmap = np.empty(hm.shape, dt)
    if device_map is not None:
        import torch

        rdev, tdev = _device_out(hm.size, device_map), _device_out(hm.size, device_map)
        out = engine.predict(c, cluster_map_out=cmap, day_stats=True, transitions=trans, regions=conn,
                             region_map_out=rdev, tracks=min_iou, track_map_out=tdev, **extra)
        torch.cuda.synchronize()
        rmap = rdev.cpu().numpy().reshape(hm.shape)
        tmap = tdev.cpu().numpy().reshape(hm.shape)
    else:
        rmap = np.full(hm.shape, -7, np.int32)
        tmap = np.full(hm.shape, -7, np.int32)
        out = engine.predict(c, cluster_map_out=cmap, day_stats=True, transitions=trans, regions=conn,
                             region_map_out=rmap, tracks=min_iou, track_map_out=tmap, **extra)
    assert len(out) == len(base) + 2
    assert np.array_equal(out[0], base[0]) and out[1] == base[1]
    for x, y in zip(out[2:-2], base[2:]):
        assert x.tobytes() == y.tobytes()
    assert cmap.tobytes() == cmap0.tobytes() and rmap.tobytes() == rmap0.tobytes()
    assert np.array_equal(cmap.astype(np.int64) - 1, np.where(labels_map >= 0, labels_map, -1))
    assert rmap.tobytes() == ref_region_map(cmap, conn).tobytes()
    table = out[5]
    tracks, region_tracks = out[-2:]
    check_tracks(tracks, region_tracks, rmap, table, min_iou, tmap)
    return tracks, region_tracks, table, tmap


def square_days(D, H, W, boxes, label=1, bg=0):
    """D days of background ``bg`` with one box per day: boxes[d] = (y0, x0, h, w[, label]) or None."""
    m = np.full((D, H, W), bg, np.int64)
    for d, b in enumerate(boxes):
        if b is not None:
            y0, x0, h, w = b[:4]
            m[d, y0:y0 + h, x0:x0 + w] = b[4] if len(b) > 4 else label
    return m


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def test_oracle_on_a_hand_drawn_stack():
    # day 0: regions 1 (cluster 0, 4 px) and 2 (cluster 1, 2 px); day 1: 3 (cluster 0, 3 px), 4
    # (cluster 1, 3 px); day 2: 5 (cluster 0, 6 px)
    r = np.array([[[1, 1, 2], [1, 1, 2]],
                  [[3, 3, 4], [3, 4, 4]],
                  [[5, 5, 5], [5, 5, 5]]], np.int32)
    regions = np.array([[0, 0, 4], [0, 1, 2], [1, 0, 3], [1, 1, 3], [2, 0, 6]], np.int64)
    t, rt = ref_tracks(r, regions, 0.5)
    # 1-3: 3 / 4 = 0.75; 2-4: 2 / 3; 3-5: 3 / 6 = 0.5 (links: exactly the threshold); 4-5: clusters differ
    assert rt.tolist() == [1, 2, 1, 2, 1]
    assert t.tolist() == [[0, 0, 2, 3, 13, 1, 0], [1, 0, 1, 2, 5, 2, 0]]
    t, rt = ref_tracks(r, regions, float(np.nextafter(0.5, 1.0)))
    assert rt.tolist() == [1, 2, 1, 2, 3]
    t, rt = ref_tracks(r[:1], regions[:2], 0.5)
    assert rt.tolist() == [1, 2] and t[:, 3].tolist() == [1, 1]


def test_oracle_marks_splits_and_merges():
    r = np.array([[[1, 1, 1, 1]], [[2, 0, 0, 3]], [[4, 4, 4, 4]]], np.int32)
    regions = np.array([[0, 0, 4], [1, 0, 1], [1, 0, 1], [2, 0, 4]], np.int64)
    t, rt = ref_tracks(r, regions, 0.25)
    assert rt.tolist() == [1, 1, 1, 1] and t.tolist() == [[0, 0, 2, 4, 10, 1, 1]]
    t, rt = ref_tracks(r, regions, 0.3)
    assert rt.tolist() == [1, 2, 3, 4] and np.all(t[:, 6] == 0)


def test_requested_min_iou():
    assert api.requested_min_iou(False) is None
    assert api.requested_min_iou(False, float("nan")) is None  # not asked for: not looked at
    assert api.requested_min_iou(True) == 0.5
    assert api.requested_min_iou(False, 1, True) == 1.0
    assert api.requested_min_iou(True, np.float32(0.25)) == 0.25
    for bad in (0.0, -0.1, 1.0 + 1e-12, float("nan"), float("inf"), True, np.bool_(True), "0.5", None, [0.5]):
        with pytest.raises(ValueError, match="track_min_iou must be a real number in \\(0, 1\\]"):
            api.requested_min_iou(True, bad)


class NoEngine:  # any use of the engine would raise AttributeError instead
    pass


@pytest.mark.parametrize("bad", [0.0, 1.5, float("nan"), True, "x"])
def test_bad_min_iou_raises_before_any_gpu_work(pkg, bad):
    hm = np.zeros((2, 4, 4), dtype=np.float32)
    with pytest.raises(ValueError, match="track_min_iou"):
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_tracks=True, track_min_iou=bad)
    with pytest.raises(ValueError, match="track_min_iou"):
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_track_map=True, track_min_iou=bad)
    with pytest.raises(AttributeError):  # without tracks it is not looked at
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), track_min_iou=bad)


def test_tracks_imply_regions(pkg):
    hm = np.zeros((2, 4, 4), dtype=np.float32)
    for kw in ({"return_tracks": True}, {"return_track_map": True}):
        with pytest.raises(ValueError, match="region_connectivity"):
            pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), region_connectivity=6, **kw)


def test_engine_refuses_before_binding(pkg):
    bind = pkg.Engine._bind_outputs
    with pytest.raises(ValueError, match="tracks needs regions"):
        bind(NoEngine(), 3, None, False, None, None, None, None, 0.5)
    with pytest.raises(ValueError, match="track_map_out needs tracks"):
        bind(NoEngine(), 3, None, False, None, 4, None, None, None, np.empty(4, np.int32))


def test_fusion_result_and_layers():
    r = api.FusionResult(labels=np.zeros(1, np.int32), centroids=np.zeros((1, 3)), fused_cloud=np.zeros((1, 3)),
                         n_iter=1, inertia=0.0, n_points=1)
    assert r.tracks is None and r.region_tracks is None and r.track_map is None
    r.tracks = np.zeros((3, 7), np.int64)
    assert [t for _, _, t in api.to_layers(r)] == ["points", "points"]
    r.track_map = np.zeros((2, 3, 3), np.int32)
    layers = api.to_layers(r)
    assert [t for _, _, t in layers] == ["points", "points", "labels"]
    assert layers[-1][1]["name"] == "Multi-day Tracks" and layers[-1][0] is r.track_map


# ---------------------------------------------------------------------------------------
# GPU: drawn patterns
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_a_square_that_persists(engine, conn):
    m = square_days(5, 40, 50, [(10, 12, 9, 11)] * 5)
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, conn, 0.5)
    assert tracks.shape[0] == 2  # the background and the square, one chain each
    assert np.all(tmap[:, 12, 14] == tmap[0, 12, 14])
    # region 1 is day 0's background (first pixel (0, 0)), region 2 day 0's square
    assert tracks[tmap[0, 12, 14] - 1].tolist() == [1, 0, 4, 5, 5 * 99, 2, 0]


@pytest.mark.gpu
def test_a_square_that_shifts_until_the_iou_falls(engine):
    # shifts 1, 2, 3, 4 between the days: IoU 30/42, 24/48 = 0.5 (links), 18/54, 12/60
    xs = [5, 6, 8, 11, 15]
    m = square_days(5, 20, 40, [(7, x, 6, 6) for x in xs])
    for iou, want in ((0.5, [1, 1, 1, 2, 3]), (0.3, [1, 1, 1, 1, 2]), (0.75, [1, 2, 3, 4, 5])):
        tracks, rt, regions, tmap = predict_checked(engine, m, 2, 4, iou)
        ids = [tmap[d, 7, xs[d]] for d in range(5)]
        first = {}
        assert [first.setdefault(i, len(first) + 1) for i in ids] == want


@pytest.mark.gpu
def test_split_then_merge(engine):
    boxes = [(5, 5, 10, 10), None, (5, 5, 10, 10)]
    m = square_days(3, 24, 24, boxes)
    m[1, 5:15, 5:9] = 1
    m[1, 5:15, 11:15] = 1  # two 10 x 4 halves: IoU 40 / 100 with the whole square each
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, 8, 0.3)
    t = tracks[tmap[0, 6, 6] - 1]
    assert t[3] == 4 and t[6] == 1 and t[1] == 0 and t[2] == 2
    assert tmap[1, 6, 6] == tmap[1, 6, 12] == tmap[2, 6, 6] == tmap[0, 6, 6]
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, 8, 0.6)
    assert len({tmap[0, 6, 6], tmap[1, 6, 6], tmap[1, 6, 12], tmap[2, 6, 6]}) == 4
    assert np.all(tracks[:, 6] == 0)


@pytest.mark.gpu
def test_a_change_of_cluster_breaks_the_track(engine):
    m = square_days(4, 30, 30, [(4, 4, 8, 8, 1), (4, 4, 8, 8, 1), (4, 4, 8, 8, 2), (4, 4, 8, 8, 1)])
    tracks, rt, regions, tmap = predict_checked(engine, m, 3, 4, 0.5)
    ids = [tmap[d, 5, 5] for d in range(4)]
    assert ids[0] == ids[1] and len(set(ids[1:])) == 3
    assert tracks[ids[0] - 1][[1, 2, 3]].tolist() == [0, 1, 2]


@pytest.mark.gpu
def test_no_bridge_over_a_missing_day(engine):
    m = square_days(4, 30, 30, [(4, 4, 8, 8), (4, 4, 8, 8), None, (4, 4, 8, 8)])
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, 4, 0.5)
    assert tmap[0, 5, 5] == tmap[1, 5, 5] != tmap[3, 5, 5]
    assert tracks[tmap[3, 5, 5] - 1][[1, 2, 3]].tolist() == [3, 3, 1]


@pytest.mark.gpu
def test_an_empty_day_and_one_pixel_regions(engine):
    m = np.zeros((4, 17, 19), np.int64)
    m[2] = -1  # no point on day 2
    m[:, 3, 4] = 1  # a one-pixel region on days 0, 1 and 3
    m[2, 3, 4] = -1
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, 4, 1.0)
    assert tmap[0, 3, 4] == tmap[1, 3, 4] != tmap[3, 3, 4] and np.all(tmap[2] == 0)
    assert tracks[tmap[0, 3, 4] - 1].tolist()[1:5] == [0, 1, 2, 2]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 33, 65), (2, 1, 70), (3, 70, 1), (2, 1, 1), (3, 31, 17)])
def test_border_regions_and_odd_sizes(engine, shape):
    rs = np.random.RandomState(sum(shape))
    D, H, W = shape
    m = np.zeros(shape, np.int64)
    m[:, 0, :] = 1  # the top row, the left column: regions on the border of every day
    m[:, :, 0] = 1
    m[:, -1, -1] = 1
    m[rs.rand(*shape) < 0.15] = -1
    for conn in (4, 8):
        for iou in (0.5, 1.0):
            predict_checked(engine, m, 2, conn, iou)


@pytest.mark.gpu
def test_the_exact_threshold(engine):
    # two 2-pixel regions that share 1: IoU 1 / 3, the correctly rounded FP64 quotient
    m = np.zeros((2, 5, 8), np.int64)
    m[0, 2, 2:4] = 1
    m[1, 2, 3:5] = 1
    third = 1.0 / 3.0
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, 4, third)
    assert tmap[0, 2, 2] == tmap[1, 2, 4]
    tracks, rt, regions, tmap = predict_checked(engine, m, 2, 4, float(np.nextafter(third, 2.0)))
    assert tmap[0, 2, 2] != tmap[1, 2, 4]


def random_stack(D, H, W, k, seed):
    """Blobby labels that mostly persist from day to day, with holes and labels above 255 for
    k > 255 (a uint16 map)."""
    rs = np.random.RandomState(seed)
    n = min(k, 4)
    lo = rs.randint(0, n, size=(max(H // 4, 1) + 1, max(W // 4, 1) + 1))
    day = np.kron(lo, np.ones((4, 4), np.int64))[:H, :W]
    out = []
    for _ in range(D):
        out.append(day.copy())
        flip = rs.rand(H, W) < 0.08
        day = np.where(flip, rs.randint(0, n, size=(H, W)), np.roll(day, rs.randint(-1, 2), axis=1))
    m = np.stack(out)
    if k > 255:
        m = m + (m % 2) * (k - 4)
    m[rs.rand(*m.shape) < 0.1] = -1
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("k", [2, 16, 300])
@pytest.mark.parametrize("D", [1, 2, 10])
def test_random_label_maps(engine, D, k, conn):
    m = random_stack(D, 37, 53, k, 100 * D + k + conn)
    for i, iou in enumerate(IOUS):
        tracks, rt, regions, tmap = predict_checked(engine, m, k, conn, iou, unproject=i == 0)
        if D == 1:  # nothing to link: every region is a track of its own
            assert tracks.shape[0] == regions.shape[0]
            assert np.array_equal(rt, np.arange(1, regions.shape[0] + 1, dtype=np.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["aligned", "offset"])
def test_device_maps(engine, where):
    """Region ids read from the caller's CUDA map, the track map written into a CUDA tensor; 4 bytes
    past alignment the map pass takes its scalar head and tail."""
    m = random_stack(3, 50, 97, 4, 5)
    for conn in (4, 8):
        predict_checked(engine, m, 4, conn, 0.5, device_map=where)


@pytest.mark.gpu
def test_host_region_map_and_device_track_map(engine):
    import torch

    m = random_stack(3, 41, 59, 3, 6)
    hm = draw(m, 3)
    engine.unproject(hm)
    c = level_centroids(3, 41, 59)
    rmap = np.empty(hm.shape, np.int32)
    tdev = _device_out(hm.size, "offset")
    out = engine.predict(c, regions=4, region_map_out=rmap, tracks=0.5, track_map_out=tdev)
    torch.cuda.synchronize()
    check_tracks(out[-2], out[-1], rmap, out[2], 0.5, tdev.cpu().numpy().reshape(hm.shape))
    out2 = engine.predict(c, regions=4, tracks=0.5)  # no maps at all: the same tracks
    assert out2[-2].tobytes() == out[-2].tobytes() and out2[-1].tobytes() == out[-1].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("pairs", [[(0, 2), (3, 1), (2, 2)], [(0, 1), (1, 2), (2, 3)], [(2, 3), (0, 1), (0, 1)]])
def test_with_the_callers_overlaps(engine, pairs):
    """The caller's rows and their count are those of a call without tracks, whether their pairs are
    other pairs, exactly the consecutive ones, or some of them (repeated)."""
    m = random_stack(4, 40, 60, 3, 7)
    predict_checked(engine, m, 3, 8, 0.5, pairs=pairs)  # (the rows come from the count: compared there)


# ---------------------------------------------------------------------------------------
# GPU: fits
# ---------------------------------------------------------------------------------------
def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter and a.n_refined == b.n_refined
    for name in ("cluster_map", "day_counts", "day_means", "transitions", "regions", "region_means", "region_map",
                 "region_overlaps"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None)
        if x is not None:
            assert x.tobytes() == y.tobytes()


def fuse_checked(pkg, hm, *, k, iou=0.5, conn=4, overlaps=True, **kw):
    """The call without and with tracks: everything else bitwise equal; the tracks against the
    oracle on the returned region map, which is checked against scipy."""
    common = dict(n_clusters=k, return_cluster_map=True, return_day_stats=True, return_transitions=True,
                  return_region_map=True, region_connectivity=conn, return_region_overlaps=overlaps, **kw)
    plain = pkg.fuse_multiday_kmeans(hm, **common)
    res = pkg.fuse_multiday_kmeans(hm, return_track_map=True, track_min_iou=iou, **common)
    assert plain.tracks is None and plain.region_tracks is None and plain.track_map is None
    same_result(plain, res)
    assert res.region_map.tobytes() == ref_region_map(res.cluster_map, conn).tobytes()
    check_tracks(res.tracks, res.region_tracks, res.region_map, res.regions, iou, res.track_map)
    return res


def stack(D, H, W, seed):
    return synth.make_stack(D, H, W, seed=seed, n_buildings=6).numpy()


def seeds(hm, k, seed):
    return synth.init_from_points(UO.unproject_stack(hm).astype(np.float32), k, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("iou", [0.2, 0.5, 0.8])
def test_synthetic_stack(pkg, engine, iou):
    hm = stack(4, 130, 170, 3)
    res = fuse_checked(pkg, hm, k=9, iou=iou, conn=8, init="k-means++", random_state=1, max_iter=20, engine=engine)
    assert res.tracks.shape[0] < res.regions.shape[0]  # something persists


@pytest.mark.gpu
def test_detrend_and_ground_level(pkg, engine):
    hm = stack(3, 90, 140, 4)
    fuse_checked(pkg, hm, k=7, conn=8, overlaps=[(2, 0)], init="k-means++", random_state=2, max_iter=20,
                 detrend=True, ground_level=True, engine=engine)


@pytest.mark.gpu
def test_restarts_keep_the_returned_runs_tracks(pkg, engine):
    hm = stack(3, 60, 130, 9)
    fuse_checked(pkg, hm, k=12, conn=8, overlaps=False, init="k-means++", n_init=3, random_state=11, max_iter=15,
                 engine=engine)


@pytest.mark.gpu
def test_restarts_return_the_best_run_not_the_last(engine, monkeypatch):
    hm = stack(3, 60, 130, 9)
    engine.unproject(hm)
    runs = []
    fit = engine.fit

    def fit_and_record(init, **kw):
        if len(runs) == 2:
            kw["max_iter"] = 1
        r = fit(init, **kw)
        runs.append(r)
        return r

    monkeypatch.setattr(engine, "fit", fit_and_record)
    rmap = np.empty(hm.shape, np.int32)
    tmap = np.empty(hm.shape, np.int32)
    best = api._run_kmeans(engine, n_clusters=12, init="k-means++", n_init=3, max_iter=15, tol=1e-4, random_state=11,
                           regions=8, region_map_out=rmap, tracks=0.5, track_map_out=tmap)
    assert len(runs) == 3
    won = [i for i, r in enumerate(runs) if r["tracks"] is best["tracks"]]
    assert won and won[0] != 2
    assert best["tracks"].tobytes() != runs[2]["tracks"].tobytes()
    check_tracks(best["tracks"], best["region_tracks"], rmap, best["regions"], 0.5, tmap)


@pytest.mark.gpu
def test_relocation(engine):
    hm = stack(3, 80, 120, 10)
    init = seeds(hm, 8, 2)
    init[5] = [1e5, -1e5, 1e4]  # far outside the cloud: empty after the first E-step
    engine.unproject(hm)
    kw = dict(max_iter=30, tol=0.0, day_stats=True, regions=8, region_overlaps=[(0, 1), (2, 0)])
    rmap = np.empty(hm.shape, np.int32)
    tmap = np.empty(hm.shape, np.int32)
    r1 = engine.fit(init, region_map_out=rmap, tracks=0.5, track_map_out=tmap, **kw)
    labels1 = r1["labels"].copy()
    r0 = engine.fit(init, **kw)
    assert r1["n_relocations"] >= 1 and "tracks" not in r0
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    assert r1["inertia"] == r0["inertia"] and r1["n_iter"] == r0["n_iter"]
    for name in ("day_counts", "day_means", "regions", "region_means", "region_overlaps"):
        assert r1[name].tobytes() == r0[name].tobytes()
    check_tracks(r1["tracks"], r1["region_tracks"], rmap, r1["regions"], 0.5, tmap)


@pytest.mark.gpu
def test_predict_on_a_second_stack(engine):
    hm = stack(2, 50, 140, 12)
    engine.unproject(hm)
    centers = engine.fit(seeds(hm, 9, 3), max_iter=10, regions=4, tracks=0.5)["centers"]
    hm2 = stack(4, 30, 91, 13)
    engine.unproject(hm2)  # drops the tracks of the fit
    with pytest.raises(C.MdkmError):
        engine._track_table()
    cmap = np.empty(hm2.shape, np.uint8)
    rmap = np.empty(hm2.shape, np.int32)
    tmap = np.empty(hm2.shape, np.int32)
    out = engine.predict(centers, cluster_map_out=cmap, regions=8, region_map_out=rmap, tracks=0.6,
                         track_map_out=tmap)
    labels, inertia, table, rmeans, tracks, region_tracks = out
    assert rmap.tobytes() == ref_region_map(cmap, 8).tobytes()
    check_tracks(tracks, region_tracks, rmap, table, 0.6, tmap)


# ---------------------------------------------------------------------------------------
# GPU: errors and the lifecycle
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_errors(pkg, engine):
    ERR_STATE, ERR_INVALID = C.STATUS_BY_NAME["MDKM_ERR_STATE"], C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    bind = engine._lib.mdkm_bind_tracks
    hm = stack(3, 30, 60, 17)
    init = seeds(hm, 5, 1)
    fresh = pkg.Engine(0)
    try:  # no resident cloud; nothing computed yet
        assert bind(fresh._h, 0.5, None, 0, C.MEM_HOST) == ERR_STATE
        with pytest.raises(C.MdkmError) as ei:
            fresh._track_table()
        assert ei.value.code == ERR_STATE
    finally:
        fresh.close()
    engine.set_points(UO.unproject_stack(hm).astype(np.float32))  # no raster
    assert bind(engine._h, 0.5, None, 0, C.MEM_HOST) == ERR_STATE
    engine.unproject(hm)
    with pytest.raises(C.MdkmError) as ei:  # count / table before any computation
        engine._track_table()
    assert ei.value.code == ERR_STATE
    small = np.empty(hm.size - 1, np.int32)
    big = np.empty(hm.size, np.int32)
    for iou, ptr, cap, mem in ((0.0, big.ctypes.data, big.size, C.MEM_HOST), (-0.5, None, 0, C.MEM_HOST),
                               (1.0000001, None, 0, C.MEM_HOST), (math.nan, None, 0, C.MEM_HOST),
                               (math.inf, None, 0, C.MEM_HOST), (0.5, small.ctypes.data, small.size, C.MEM_HOST),
                               (0.5, big.ctypes.data, big.size, 7)):
        assert bind(engine._h, iou, ptr, cap, mem) == ERR_INVALID
    assert bind(engine._h, 1.0, big.ctypes.data, big.size, C.MEM_HOST) == C.MDKM_OK
    assert bind(engine._h, 0.0, None, 0, C.MEM_HOST) == C.MDKM_OK  # cleared
    r = engine.fit(init, max_iter=5, regions=4)
    assert "tracks" not in r
    with pytest.raises(C.MdkmError):
        engine._track_table()
    # Python: bad values, tracks without regions, a map without tracks
    for bad in (0.0, 2.0, math.nan, True, "0.5"):
        with pytest.raises(ValueError):
            engine.fit(init, max_iter=5, regions=4, tracks=bad)
    with pytest.raises(ValueError):
        engine.fit(init, max_iter=5, tracks=0.5)
    with pytest.raises(ValueError):
        engine.predict(init, regions=4, track_map_out=big)
    # tracks without regions at the C ABI: MDKM_ERR_STATE from the fit / predict
    for call in (lambda: engine.fit(init, max_iter=5), lambda: engine.predict(init)):
        assert bind(engine._h, 0.5, None, 0, C.MEM_HOST) == C.MDKM_OK
        with pytest.raises(C.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_STATE
    r = engine.fit(init, max_iter=5)  # the binding was consumed by the refused call
    # short capacities; either output may be left out
    r = engine.fit(init, max_iter=5, regions=4, tracks=0.5)
    T, R = r["tracks"].shape[0], r["regions"].shape[0]
    assert 0 < T < R
    t = np.empty((T, 7), np.int64)
    rt = np.empty(R, np.int32)
    tab = engine._lib.mdkm_track_table
    assert tab(engine._h, t.ctypes.data, rt.ctypes.data, T - 1, R) == ERR_INVALID
    assert tab(engine._h, t.ctypes.data, rt.ctypes.data, T, R - 1) == ERR_INVALID
    assert tab(engine._h, t.ctypes.data, None, T, 0) == C.MDKM_OK
    assert tab(engine._h, None, rt.ctypes.data, 0, R) == C.MDKM_OK
    assert t.tobytes() == r["tracks"].tobytes() and rt.tobytes() == r["region_tracks"].tobytes()
    # a fit without regions keeps the tracks; one with regions but without tracks drops them
    engine.fit(init, max_iter=5)
    assert engine._track_table()[0].tobytes() == r["tracks"].tobytes()
    engine.fit(init, max_iter=5, regions=8)
    with pytest.raises(C.MdkmError) as ei:
        engine._track_table()
    assert ei.value.code == ERR_STATE
    # tracks alone leave the caller without overlaps
    engine.fit(init, max_iter=5, regions=8, tracks=0.5)
    with pytest.raises(C.MdkmError) as ei:
        engine._region_overlap_table()
    assert ei.value.code == ERR_STATE
    # the binding is dropped by unproject
    assert bind(engine._h, 0.5, None, 0, C.MEM_HOST) == C.MDKM_OK
    engine.unproject(hm)
    engine.fit(init, max_iter=5, regions=4)
    with pytest.raises(C.MdkmError):
        engine._track_table()


@pytest.mark.gpu
def test_a_refused_binding_leaves_none_behind(engine):
    hm = stack(2, 40, 60, 21)
    engine.unproject(hm)
    init = seeds(hm, 5, 1)
    with pytest.raises(ValueError):  # short track map: refused after the regions and overlaps were bound
        engine.fit(init, max_iter=5, day_stats=True, regions=4, region_overlaps=[(0, 1)], tracks=0.5,
                   track_map_out=np.empty(5, np.int32))
    r = engine.fit(init, max_iter=5)
    assert "regions" not in r and "day_counts" not in r
    for table in (engine._region_table, engine._region_overlap_table, engine._track_table):
        with pytest.raises(C.MdkmError):
            table()
    r = engine.fit(init, max_iter=5, regions=4)  # nothing left bound: regions alone
    assert "regions" in r and "tracks" not in r
    with pytest.raises(C.MdkmError):
        engine._track_table()


@pytest.mark.gpu
def test_plugin_passes_the_options(pkg, monkeypatch):
    hm = stack(3, 64, 80, 13)
    seen = []
    to_layers = api.to_layers
    monkeypatch.setattr(api, "to_layers", lambda res: seen.append(res) or to_layers(res))
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_track_map=True, track_min_iou=0.6, init="k-means++",
                                    random_state=0, max_iter=10)
    layers = plug.run(hm)
    assert [t for _, _, t in layers] == ["points", "points", "labels"]
    assert layers[-1][1]["name"].endswith("Tracks")
    (res,) = seen
    assert res.region_map is None and res.regions is not None and res.track_map.shape == hm.shape
    assert np.array_equal(np.unique(res.track_map[res.track_map > 0]), np.unique(res.region_tracks))
    assert res.tracks.shape[0] == res.region_tracks.max()


# ---------------------------------------------------------------------------------------
# GPU: two devices
# ---------------------------------------------------------------------------------------
def _two_gpus():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 300])
def test_device_group_equals_one_device(pkg, k):
    _two_gpus()
    hm = stack(3, 31, 77, 18)
    kw = dict(n_clusters=k, init="k-means++", random_state=7, max_iter=10, return_region_map=True,
              region_connectivity=8, return_track_map=True, return_region_overlaps=[(2, 0)])
    one = pkg.fuse_multiday_kmeans(hm, device=0, **kw)
    two = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], **kw)
    assert np.array_equal(one.labels, two.labels)
    for name in ("tracks", "region_tracks", "track_map", "region_overlaps"):
        assert getattr(two, name).tobytes() == getattr(one, name).tobytes()
    check_tracks(one.tracks, one.region_tracks, one.region_map, one.regions, 0.5, one.track_map)


@pytest.mark.gpu
def test_pre_sharded_ranks_receive_the_same_tracks(pkg):
    _two_gpus()
    from concurrent.futures import ThreadPoolExecutor

    hm = stack(3, 30, 70, 19)
    flat = hm.reshape(-1)
    cut = 30 * 70 + 517  # inside day 1
    init = seeds(hm, 6, 4)
    kw = dict(n_clusters=6, init=init, max_iter=10, return_region_map=True, return_track_map=True)
    one = pkg.fuse_multiday_kmeans(hm, **kw)
    uid = pkg.Engine.make_unique_id()
    engines = [pkg.Engine(r) for r in range(2)]
    try:
        with ThreadPoolExecutor(2) as ex:
            list(ex.map(lambda r: engines[r].init_comm(2, r, uid), range(2)))
            spans = [(0, cut), (cut, flat.size)]
            res = list(ex.map(lambda r: pkg.fuse_multiday_kmeans(
                flat[spans[r][0]:spans[r][1]], engine=engines[r], stack_shape=hm.shape, pix_begin=spans[r][0],
                **kw), range(2)))
    finally:
        for e in engines:
            e.close()
    for r, (b, e) in zip(res, spans):
        assert r.tracks.tobytes() == one.tracks.tobytes()
        assert r.region_tracks.tobytes() == one.region_tracks.tobytes()
        assert r.track_map.tobytes() == one.track_map.reshape(-1)[b:e].tobytes()
    check_tracks(one.tracks, one.region_tracks, one.region_map, one.regions, 0.5, one.track_map)
