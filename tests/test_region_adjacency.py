"""Region adjacency within a day (``return_region_adjacency`` / ``region_adjacency=``): one row per
unordered pair of distinct regions a < b of one day joined by at least one edge between
4-neighbouring pixels -- int64 (day, region_a, region_b, edges, y_first, x_first), sorted by the
first edge (index 2 (y W + x) + direction within the day) -- and per region int64 (perimeter,
region_edges, background_edges, border_edges).

The oracle is a numpy restatement on the region map the same call returns: the horizontal and
vertical neighbour pairs of two different non-zero ids with their edge indices, the packed
min << 32 | max keys, ``np.unique`` with first index and counts, ordered by (day, first edge); the
boundaries count each pixel's four sides by what lies across them.  The region map itself is
checked against ``scipy.ndimage.label`` (restated from ``test_regions.py``), and every GPU case
checks that asking for adjacency changes nothing else.

Label patterns are drawn with ``predict`` as in ``test_regions.py``: centroids that share x and y
and differ only in z make a pixel's label its nearest z level."""
import importlib

import numpy as np
import pytest
from scipy import ndimage

from oracle import unproject_oracle as UO

PKG = "3d-point-cloud-multiday-imagery_b200"
synth = importlib.import_module(PKG + ".synth")
api = importlib.import_module(PKG + ".api")
C = importlib.import_module(PKG + "._cabi")


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


def neighbour_pairs(day):
    """(a, b, edge index) of every edge of one [H,W] day: horizontal edges, then vertical ones."""
    H, W = day.shape
    day = day.astype(np.int64)
    px = np.arange(H * W, dtype=np.int64).reshape(H, W)
    a = np.concatenate([day[:, :-1].ravel(), day[:-1, :].ravel()])
    b = np.concatenate([day[:, 1:].ravel(), day[1:, :].ravel()])
    e = np.concatenate([2 * px[:, :-1].ravel(), 2 * px[:-1, :].ravel() + 1])
    return a, b, e


def ref_adjacency(rmap):
    """int64 [M,6] rows of the region map ``rmap`` [D,H,W]."""
    rmap = np.asarray(rmap)
    D, H, W = rmap.shape
    out = []
    for d in range(D):
        a, b, e = neighbour_pairs(rmap[d])
        m = (a > 0) & (b > 0) & (a != b)
        a, b, e = a[m], b[m], e[m]
        order = np.argsort(e, kind="stable")
        keys = (np.minimum(a, b) << 32 | np.maximum(a, b))[order]
        e = e[order]
        u, first, cnt = np.unique(keys, return_index=True, return_counts=True)
        o = np.argsort(first, kind="stable")
        u, fe, cnt = u[o], e[first[o]], cnt[o]
        t = np.empty((u.size, 6), dtype=np.int64)
        t[:, 0] = d
        t[:, 1] = u >> 32
        t[:, 2] = u & 0xFFFFFFFF
        t[:, 3] = cnt
        t[:, 4] = (fe >> 1) // W
        t[:, 5] = (fe >> 1) % W
        out.append(t)
    return np.concatenate(out) if out else np.zeros((0, 6), np.int64)


def ref_boundaries(rmap, R):
    """int64 [R,4] (perimeter, region, background, border sides) and the inner edges [R] of every
    region: each pixel's four sides counted by what lies across them."""
    rmap = np.asarray(rmap).astype(np.int64)
    side = np.zeros((R + 1, 4), np.int64)  # region, background, border, inner
    for day in rmap:
        P = np.pad(day, 1, constant_values=-1)
        c = P[1:-1, 1:-1]
        for n in (P[:-2, 1:-1], P[2:, 1:-1], P[1:-1, :-2], P[1:-1, 2:]):
            own = c > 0
            for j, cls in enumerate(((n > 0) & (n != c), n == 0, n == -1, n == c)):
                side[:, j] += np.bincount(c[own & cls], minlength=R + 1)
    out = np.empty((R, 4), np.int64)
    out[:, 1:] = side[1:, :3]
    out[:, 0] = out[:, 1:].sum(axis=1)
    return out, side[1:, 3] // 2


def check_adjacency(rows, bnd, rmap, regions, cmap=None):
    """The rows and boundaries bit for bit against the oracle, and the consequences the semantics
    promise."""
    rmap = np.asarray(rmap)
    R = regions.shape[0]
    assert rows.dtype == np.int64 and rows.ndim == 2 and rows.shape[1] == 6
    assert bnd.dtype == np.int64 and bnd.shape == (R, 4)
    ref = ref_adjacency(rmap)
    assert rows.shape == ref.shape and rows.tobytes() == ref.tobytes()
    ref_b, inner = ref_boundaries(rmap, R)
    assert bnd.tobytes() == ref_b.tobytes()
    # invariants
    assert np.array_equal(bnd[:, 0], bnd[:, 1:].sum(axis=1))
    re = np.bincount(rows[:, 1], weights=rows[:, 3], minlength=R + 1)[1:]
    re += np.bincount(rows[:, 2], weights=rows[:, 3], minlength=R + 1)[1:]
    assert np.array_equal(re.astype(np.int64), bnd[:, 1])
    assert np.array_equal(4 * regions[:, 2], bnd[:, 0] + 2 * inner)
    assert np.all(rows[:, 1] < rows[:, 2]) and np.all(rows[:, 3] > 0)
    ra, rb = rows[:, 1] - 1, rows[:, 2] - 1
    assert np.all(regions[ra, 1] != regions[rb, 1])
    assert np.array_equal(regions[ra, 0], rows[:, 0]) and np.array_equal(regions[rb, 0], rows[:, 0])
    H, W = rmap.shape[1:]
    e = 2 * (rows[:, 4] * W + rows[:, 5])  # (the first edge's direction is not in the row: order by pixel)
    key = rows[:, 0] * (2 * H * W) + e
    assert np.all(np.diff(key) >= 0)
    if cmap is not None:  # edges by cluster pair = differently labelled neighbour pairs of the cluster map
        k = int(max(cmap.max(), 1))
        got = np.zeros((k + 1, k + 1), np.int64)
        ca, cb = regions[ra, 1] + 1, regions[rb, 1] + 1
        np.add.at(got, (np.minimum(ca, cb), np.maximum(ca, cb)), rows[:, 3])
        want = np.zeros_like(got)
        for day in np.asarray(cmap):
            a, b, _ = neighbour_pairs(day)
            m = (a > 0) & (b > 0) & (a != b)
            np.add.at(want, (np.minimum(a[m], b[m]), np.maximum(a[m], b[m])), 1)
        assert np.array_equal(got, want)


def levels(k):
    return np.linspace(-130.0, 130.0, k) if k > 1 else np.array([5.0])


def draw(labels_map, k):
    """Heights whose nearest level is the wanted label (-1: NaN, no point)."""
    z = levels(k)
    return np.where(labels_map >= 0, z[np.clip(labels_map, 0, k - 1)], np.nan).astype(np.float32)


def level_centroids(k, H, W):
    return np.stack([np.full(k, W / 2.0), np.full(k, H / 2.0), levels(k)], axis=1)


def predict_checked(engine, labels_map, k, conn, device_map=None, overlaps=None, tracks=None):
    """predict on the drawn map with regions, without and with adjacency: everything else bitwise
    equal, the region map against scipy, the adjacency against the oracle.  ``device_map``:
    "aligned" / "offset" -- the region map in a CUDA tensor (its start 16-byte aligned, or 4 bytes
    past that).  ``overlaps`` / ``tracks``: also asked for, in both calls."""
    D, H, W = labels_map.shape
    hm = draw(labels_map, k)
    engine.unproject(hm)
    c = level_centroids(k, H, W)
    dt = np.uint8 if k <= 255 else np.uint16
    extra = dict(region_overlaps=overlaps, tracks=tracks)
    cmap0 = np.empty(hm.shape, dt)
    rmap0 = np.empty(hm.shape, np.int32)
    base = engine.predict(c, cluster_map_out=cmap0, day_stats=True, regions=conn, region_map_out=rmap0, **extra)
    base = (base[0].copy(),) + base[1:]
    cmap = np.empty(hm.shape, dt)
    if device_map is not None:
        import torch

        buf = torch.full((hm.size + 4,), -7, dtype=torch.int32, device="cuda")
        rdev = buf[:hm.size] if device_map == "aligned" else buf[1:hm.size + 1]
        out = engine.predict(c, cluster_map_out=cmap, day_stats=True, regions=conn, region_map_out=rdev,
                             region_adjacency=True, **extra)
        torch.cuda.synchronize()
        rmap = rdev.cpu().numpy().reshape(hm.shape)
    else:
        rmap = np.full(hm.shape, -7, np.int32)
        out = engine.predict(c, cluster_map_out=cmap, day_stats=True, regions=conn, region_map_out=rmap,
                             region_adjacency=True, **extra)
    assert len(out) == len(base) + 2
    assert np.array_equal(out[0], base[0]) and out[1] == base[1]
    for x, y in zip(out[2:-2], base[2:]):
        assert x.tobytes() == y.tobytes()
    assert cmap.tobytes() == cmap0.tobytes() and rmap.tobytes() == rmap0.tobytes()
    assert np.array_equal(cmap.astype(np.int64) - 1, np.where(labels_map >= 0, labels_map, -1))
    assert rmap.tobytes() == ref_region_map(cmap, conn).tobytes()
    table = out[4]
    rows, bnd = out[-2:]
    check_adjacency(rows, bnd, rmap, table, cmap)
    return rows, bnd, rmap, table


# ---------------------------------------------------------------------------------------
# patterns
# ---------------------------------------------------------------------------------------
def nested_squares(H, W, n):
    """Concentric square rings of alternating labels 0 / 1 around the centre."""
    yy, xx = np.mgrid[0:H, 0:W]
    ring = np.minimum(np.minimum(yy, H - 1 - yy), np.minimum(xx, W - 1 - xx)) // n
    return (ring % 2).astype(np.int64)


def checker(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    return ((yy + xx) % 2).astype(np.int64)


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def test_oracle_on_a_hand_drawn_stack():
    r = np.array([[[1, 1, 0, 2],
                   [1, 3, 3, 2]],
                  [[4, 0, 5, 5],
                   [0, 6, 5, 5]]], np.int32)
    rows = ref_adjacency(r)
    # day 0: 1|3 at (1,0)->(1,1) edge 2*4+0 = 8, 1/3 at (0,1)->(1,1) edge 2*1+1 = 3 (first); 3|2 at (1,2) edge 12,
    # 2/2 inner; day 1: 4 and 6 meet only at a corner, 6|5 at (1,1) edge 10
    assert rows.tolist() == [[0, 1, 3, 2, 0, 1], [0, 2, 3, 1, 1, 2], [1, 5, 6, 1, 1, 1]]
    bnd, inner = ref_boundaries(r, 6)
    assert bnd.tolist() == [[8, 2, 1, 5], [6, 1, 1, 4], [6, 3, 1, 2], [4, 0, 2, 2], [8, 1, 1, 6], [4, 1, 2, 1]]
    assert inner.tolist() == [2, 1, 1, 0, 4, 0]
    regions = np.array([[0, 0, 3], [0, 1, 2], [0, 2, 2], [1, 0, 1], [1, 1, 4], [1, 0, 1]], np.int64)
    check_adjacency(rows, bnd, r, regions)
    assert ref_adjacency(np.zeros((2, 3, 3), np.int32)).shape == (0, 6)


def test_oracle_on_a_full_day():
    r = np.ones((1, 5, 7), np.int32)
    bnd, inner = ref_boundaries(r, 1)
    assert bnd.tolist() == [[24, 0, 0, 24]] and inner.tolist() == [5 * 6 + 4 * 7]


class NoEngine:  # any use of the engine would raise AttributeError instead
    pass


def test_adjacency_implies_regions(pkg):
    """return_region_adjacency asks for regions: a bad connectivity is refused, as with return_regions;
    without adjacency it is not looked at."""
    hm = np.zeros((2, 4, 4), dtype=np.float32)
    with pytest.raises(ValueError, match="region_connectivity"):
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_region_adjacency=True, region_connectivity=6)
    with pytest.raises(AttributeError):  # past the option checks, at the engine
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_region_adjacency=False, region_connectivity=6)


def test_engine_refuses_adjacency_without_regions_before_binding(pkg):
    with pytest.raises(ValueError, match="region_adjacency needs regions"):
        pkg.Engine._bind_outputs(NoEngine(), 3, region_adjacency=True)


def test_fusion_result_has_no_adjacency_by_default():
    r = api.FusionResult(labels=np.zeros(1, np.int32), centroids=np.zeros((1, 3)), fused_cloud=np.zeros((1, 3)),
                         n_iter=1, inertia=0.0, n_points=1)
    assert r.region_adjacency is None and r.region_boundaries is None
    r.region_adjacency = np.zeros((3, 6), np.int64)
    assert [t for _, _, t in api.to_layers(r)] == ["points", "points"]


# ---------------------------------------------------------------------------------------
# GPU: drawn patterns
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_nested_squares(engine, conn):
    H, W = 97, 131
    m = np.stack([nested_squares(H, W, 3), nested_squares(H, W, 1), np.roll(nested_squares(H, W, 5), 2, axis=1)])
    rows, bnd, _, table = predict_checked(engine, m, 2, conn)
    # every ring touches the ring inside it and the ring outside it
    day0 = rows[rows[:, 0] == 0]
    n0 = int(np.sum(table[:, 0] == 0))
    assert day0.shape[0] == n0 - 1


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_diagonal_contacts_only(engine, conn):
    """Regions of different clusters that touch only at corners have no row, under 4 and 8."""
    H, W = 40, 52
    m = np.full((2, H, W), -1, np.int64)
    yy, xx = np.mgrid[0:H, 0:W]
    m[0][(yy % 2 == 0) & (xx % 2 == 0)] = ((yy // 2 + xx // 2) % 3)[(yy % 2 == 0) & (xx % 2 == 0)]
    m[0][(yy % 2 == 1) & (xx % 2 == 1)] = 2 - ((yy // 2 + xx // 2) % 3)[(yy % 2 == 1) & (xx % 2 == 1)]
    m[1, 10:20, 10:20] = 0
    m[1, 20:30, 20:30] = 1
    rows, bnd, _, table = predict_checked(engine, m, 3, conn)
    assert rows.shape == (0, 6) and np.all(bnd[:, 1] == 0)


@pytest.mark.gpu
def test_one_pixel_checkerboard_under_connectivity_8(engine):
    """Under 8-connectivity the two colours of a checkerboard are one region each; every edge of the
    day lies between them."""
    H, W = 63, 90
    m = np.stack([checker(H, W), 1 - checker(H, W)])
    rows, bnd, _, table = predict_checked(engine, m, 2, 8)
    assert table.shape[0] == 4
    assert rows[:, 3].tolist() == [H * (W - 1) + (H - 1) * W] * 2


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 96, 128), (2, 61, 67), (3, 160, 257)])
def test_one_pixel_checkerboard(engine, shape):
    """Every pixel a region and every edge a row: the largest bound, hash tables at full load."""
    D, H, W = shape
    m = np.stack([checker(H, W) if d % 2 == 0 else 1 - checker(H, W) for d in range(D)])
    rows, _, _, _ = predict_checked(engine, m, 2, 4)
    assert rows.shape[0] == D * (H * (W - 1) + (H - 1) * W)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_border_regions_a_full_day_and_an_empty_day(engine, conn):
    H, W = 50, 75
    full = np.full((H, W), 1, np.int64)
    border = np.full((H, W), -1, np.int64)
    border[0, :] = 0
    border[:, -1] = 1
    border[-1, 5:40] = 2
    border[20:30, 0:3] = 2
    border[25, 3:10] = 0
    m = np.stack([full, border, np.full((H, W), -1, np.int64), full * 2])
    rows, bnd, _, table = predict_checked(engine, m, 3, conn)
    for r in np.nonzero(table[:, 2] == H * W)[0]:
        assert bnd[r].tolist() == [2 * (H + W), 0, 0, 2 * (H + W)]
    assert not np.any(table[:, 0] == 2)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 1, 1), (3, 1, 70), (2, 70, 1), (2, 33, 65), (2, 17, 6), (2, 9, 131)])
def test_tiny_and_odd_days(engine, shape):
    rs = np.random.RandomState(sum(shape))
    k = 3 if np.prod(shape) > 8 else 2
    m = rs.randint(-1, k, size=shape).astype(np.int64)
    m[0, 0, 0] = 0
    for conn in (4, 8):
        predict_checked(engine, m, k, conn)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("k", [3, 17, 300])
def test_random_labels(engine, k, conn):
    rs = np.random.RandomState(k + conn)
    m = rs.randint(0, min(k, 5), size=(4, 45, 77)).astype(np.int64)
    if k > 255:
        m = m + rs.randint(0, 2, size=m.shape) * (k - 5)  # labels above 255: a uint16 map
    m[rs.rand(*m.shape) < 0.2] = -1
    m[2] = -1  # a day without a point
    predict_checked(engine, m, k, conn)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["aligned", "offset"])
def test_device_region_map(engine, where):
    """The ids are read from the caller's CUDA map; 4 bytes off alignment they take the scalar loads."""
    rs = np.random.RandomState(5)
    for shape in ((3, 50, 96), (2, 41, 75)):
        m = rs.randint(-1, 4, size=shape).astype(np.int64)
        for conn in (4, 8):
            predict_checked(engine, m, 4, conn, device_map=where)


@pytest.mark.gpu
def test_long_borders_cross_the_warp_spans(engine):
    """Large uniform areas: runs of one key across many 128-pixel groups and warp spans."""
    H, W = 300, 700
    a = np.zeros((H, W), np.int64)
    a[:, 350:] = 1
    a[150:, :] = 2
    a[10:20, 100:600] = -1
    rows, _, _, _ = predict_checked(engine, a[None], 3, 4)
    assert rows.shape[0] == 3


@pytest.mark.gpu
@pytest.mark.parametrize("where", [None, "offset"])
def test_with_overlaps_and_tracks(engine, where):
    rs = np.random.RandomState(8)
    m = rs.randint(0, 3, size=(4, 37, 59)).astype(np.int64)
    m[rs.rand(*m.shape) < 0.1] = -1
    predict_checked(engine, m, 3, 8, device_map=where, overlaps=[(0, 1), (3, 2)], tracks=0.3)


# ---------------------------------------------------------------------------------------
# GPU: fits
# ---------------------------------------------------------------------------------------
def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter and a.n_refined == b.n_refined
    for name in ("cluster_map", "day_counts", "day_means", "transitions", "regions", "region_means", "region_map",
                 "region_overlaps", "tracks", "region_tracks", "track_map"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None)
        if x is not None:
            assert x.tobytes() == y.tobytes()


def fuse_checked(pkg, hm, *, k, conn=4, **kw):
    """The call without and with adjacency: everything else bitwise equal; the adjacency against the
    oracle on the returned region map, which is checked against scipy."""
    common = dict(n_clusters=k, return_cluster_map=True, return_day_stats=True, return_transitions=True,
                  return_region_map=True, region_connectivity=conn, return_region_overlaps=True,
                  return_track_map=True, **kw)
    plain = pkg.fuse_multiday_kmeans(hm, **common)
    res = pkg.fuse_multiday_kmeans(hm, return_region_adjacency=True, **common)
    assert plain.region_adjacency is None and plain.region_boundaries is None
    same_result(plain, res)
    assert res.region_map.tobytes() == ref_region_map(res.cluster_map, conn).tobytes()
    check_adjacency(res.region_adjacency, res.region_boundaries, res.region_map, res.regions, res.cluster_map)
    return res


def stack(D, H, W, seed):
    return synth.make_stack(D, H, W, seed=seed, n_buildings=6).numpy()


def seeds(hm, k, seed):
    return synth.init_from_points(UO.unproject_stack(hm).astype(np.float32), k, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_synthetic_stack(pkg, engine, conn):
    hm = stack(4, 130, 170, 3)
    res = fuse_checked(pkg, hm, k=9, conn=conn, init="k-means++", random_state=1, max_iter=20, engine=engine)
    assert res.region_adjacency.shape[0] > 9


@pytest.mark.gpu
def test_restarts_keep_the_best_runs_table(pkg, engine):
    hm = stack(3, 60, 130, 9)
    fuse_checked(pkg, hm, k=12, conn=8, init="k-means++", n_init=3, random_state=11, max_iter=15, detrend=True,
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
    best = api._run_kmeans(engine, n_clusters=12, init="k-means++", n_init=3, max_iter=15, tol=1e-4, random_state=11,
                           regions=8, region_map_out=rmap, region_adjacency=True)
    assert len(runs) == 3
    won = [i for i, r in enumerate(runs) if r["region_adjacency"] is best["region_adjacency"]]
    assert won and won[0] != 2
    check_adjacency(best["region_adjacency"], best["region_boundaries"], rmap, best["regions"])


@pytest.mark.gpu
def test_relocation(engine):
    hm = stack(3, 80, 120, 10)
    init = seeds(hm, 8, 2)
    init[5] = [1e5, -1e5, 1e4]  # far outside the cloud: empty after the first E-step
    engine.unproject(hm)
    kw = dict(max_iter=30, tol=0.0, day_stats=True, regions=8)
    cmap = np.empty(hm.shape, np.uint8)
    rmap = np.empty(hm.shape, np.int32)
    r1 = engine.fit(init, cluster_map_out=cmap, region_map_out=rmap, region_adjacency=True, **kw)
    labels1 = r1["labels"].copy()
    r0 = engine.fit(init, **kw)
    assert r1["n_relocations"] >= 1 and "region_adjacency" not in r0
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    for name in ("day_counts", "day_means", "regions", "region_means"):
        assert r1[name].tobytes() == r0[name].tobytes()
    assert rmap.tobytes() == ref_region_map(cmap, 8).tobytes()
    check_adjacency(r1["region_adjacency"], r1["region_boundaries"], rmap, r1["regions"], cmap)


@pytest.mark.gpu
def test_predict_on_a_second_stack(engine):
    hm = stack(2, 50, 140, 12)
    engine.unproject(hm)
    centers = engine.fit(seeds(hm, 9, 3), max_iter=10, regions=4, region_adjacency=True)["centers"]
    hm2 = stack(4, 30, 91, 13)
    engine.unproject(hm2)  # drops the adjacency of the fit
    with pytest.raises(C.MdkmError):
        engine._region_adjacency_table()
    cmap = np.empty(hm2.shape, np.uint8)
    rmap = np.empty(hm2.shape, np.int32)
    labels, inertia, table, rmeans, rows, bnd = engine.predict(centers, cluster_map_out=cmap, regions=8,
                                                               region_map_out=rmap, region_adjacency=True)
    assert rmap.tobytes() == ref_region_map(cmap, 8).tobytes()
    check_adjacency(rows, bnd, rmap, table, cmap)


@pytest.mark.gpu
def test_adjacency_without_a_region_map(pkg, engine):
    """No region map bound: the rows come from the internal whole-stack map."""
    hm = stack(3, 60, 80, 15)
    kw = dict(n_clusters=5, init="k-means++", random_state=6, max_iter=10, engine=engine, region_connectivity=8)
    a = pkg.fuse_multiday_kmeans(hm, return_region_map=True, return_region_adjacency=True, **kw)
    b = pkg.fuse_multiday_kmeans(hm, return_region_adjacency=True, **kw)
    assert b.region_map is None and b.regions is not None
    assert a.region_adjacency.tobytes() == b.region_adjacency.tobytes()
    assert a.region_boundaries.tobytes() == b.region_boundaries.tobytes()
    check_adjacency(b.region_adjacency, b.region_boundaries, a.region_map, b.regions)


# ---------------------------------------------------------------------------------------
# GPU: errors and the lifecycle
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_errors(pkg, engine):
    ERR_STATE, ERR_INVALID = C.STATUS_BY_NAME["MDKM_ERR_STATE"], C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    lib = engine._lib
    bind = lib.mdkm_bind_region_adjacency
    hm = stack(3, 30, 60, 17)
    init = seeds(hm, 5, 1)
    fresh = pkg.Engine(0)
    try:  # no resident cloud; nothing computed yet
        assert bind(fresh._h, 1) == ERR_STATE
        with pytest.raises(C.MdkmError) as ei:
            fresh._region_adjacency_table()
        assert ei.value.code == ERR_STATE
    finally:
        fresh.close()
    engine.set_points(UO.unproject_stack(hm).astype(np.float32))  # no raster
    assert bind(engine._h, 1) == ERR_STATE
    engine.unproject(hm)
    from ctypes import byref, c_int64

    n = c_int64(-1)
    assert lib.mdkm_region_adjacency_count(engine._h, byref(n)) == ERR_STATE  # before any computation
    assert bind(engine._h, 0) == C.MDKM_OK  # cleared
    r = engine.fit(init, max_iter=5, regions=4)
    assert "region_adjacency" not in r
    assert lib.mdkm_region_adjacency_count(engine._h, byref(n)) == ERR_STATE
    # adjacency without regions: ValueError in Python, MDKM_ERR_STATE from the C fit / predict
    with pytest.raises(ValueError):
        engine.fit(init, max_iter=5, region_adjacency=True)
    for call in (lambda: engine.fit(init, max_iter=5), lambda: engine.predict(init)):
        assert bind(engine._h, 1) == C.MDKM_OK
        with pytest.raises(C.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_STATE
    r = engine.fit(init, max_iter=5)  # the binding was consumed by the refused call
    assert lib.mdkm_region_adjacency_count(engine._h, byref(n)) == ERR_STATE
    # short capacities
    r = engine.fit(init, max_iter=5, regions=4, region_adjacency=True)
    M, R = r["region_adjacency"].shape[0], r["regions"].shape[0]
    assert M > 0 and R > 0
    assert lib.mdkm_region_adjacency_count(engine._h, byref(n)) == C.MDKM_OK and n.value == M
    t = np.empty((M, 6), np.int64)
    b = np.empty((R, 4), np.int64)
    assert lib.mdkm_region_adjacency_table(engine._h, t.ctypes.data, None, M - 1, 0) == ERR_INVALID
    assert lib.mdkm_region_adjacency_table(engine._h, None, b.ctypes.data, 0, R - 1) == ERR_INVALID
    assert lib.mdkm_region_adjacency_table(engine._h, t.ctypes.data, None, M, 0) == C.MDKM_OK
    assert lib.mdkm_region_adjacency_table(engine._h, None, b.ctypes.data, 0, R) == C.MDKM_OK
    assert t.tobytes() == r["region_adjacency"].tobytes() and b.tobytes() == r["region_boundaries"].tobytes()
    # a fit without regions keeps the table; one with regions but without adjacency drops it
    engine.fit(init, max_iter=5)
    assert engine._region_adjacency_table()[0].tobytes() == r["region_adjacency"].tobytes()
    engine.fit(init, max_iter=5, regions=8)
    with pytest.raises(C.MdkmError) as ei:
        engine._region_adjacency_table()
    assert ei.value.code == ERR_STATE
    # the binding is dropped by unproject
    assert bind(engine._h, 1) == C.MDKM_OK
    engine.unproject(hm)
    engine.fit(init, max_iter=5, regions=4)
    with pytest.raises(C.MdkmError):
        engine._region_adjacency_table()


@pytest.mark.gpu
def test_plugin_passes_the_option(pkg, monkeypatch):
    hm = stack(3, 64, 80, 13)
    seen = []
    to_layers = api.to_layers
    monkeypatch.setattr(api, "to_layers", lambda res: seen.append(res) or to_layers(res))
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_region_adjacency=True, return_region_map=True,
                                    init="k-means++", random_state=0, max_iter=10)
    layers = plug.run(hm)
    assert [t for _, _, t in layers] == ["points", "points", "labels"]
    (res,) = seen
    check_adjacency(res.region_adjacency, res.region_boundaries, res.region_map, res.regions)


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
              region_connectivity=8, return_region_adjacency=True)
    one = pkg.fuse_multiday_kmeans(hm, device=0, **kw)
    two = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], **kw)
    assert np.array_equal(one.labels, two.labels)
    assert two.region_adjacency.tobytes() == one.region_adjacency.tobytes()
    assert two.region_boundaries.tobytes() == one.region_boundaries.tobytes()
    check_adjacency(one.region_adjacency, one.region_boundaries, one.region_map, one.regions)


@pytest.mark.gpu
def test_pre_sharded_ranks_receive_the_same_rows(pkg):
    _two_gpus()
    from concurrent.futures import ThreadPoolExecutor

    hm = stack(3, 30, 70, 19)
    flat = hm.reshape(-1)
    cut = 30 * 70 + 517  # inside day 1
    init = seeds(hm, 6, 4)
    kw = dict(n_clusters=6, init=init, max_iter=10, return_region_map=True, return_region_adjacency=True)
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
    for r in res:
        assert r.region_adjacency.tobytes() == one.region_adjacency.tobytes()
        assert r.region_boundaries.tobytes() == one.region_boundaries.tobytes()
    check_adjacency(one.region_adjacency, one.region_boundaries, one.region_map, one.regions)
