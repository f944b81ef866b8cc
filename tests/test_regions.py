"""Connected regions of the cluster map (``return_regions`` / ``regions=``): maximal 4- or
8-connected sets of pixels of one day with the same label, numbered 1..R in the raster order
(day, y, x) of each region's first pixel, with a table (day, cluster, pixels, y_min, x_min, y_max,
x_max) and the mean (x, y, z) of each region's points.

The oracle is ``scipy.ndimage.label`` per (day, cluster value), renumbered by each component's
first raster pixel; its table comes from ``np.bincount`` / ``np.minimum.at`` / ``np.maximum.at``.
Every GPU case compares the region map bit for bit with the oracle run on the cluster map the same
call returns, the table exactly, the pixels summed per (day, cluster) with ``day_counts``, and
everything else with the same call without regions.

Label patterns are drawn with ``predict``: centroids that share x and y and differ only in z make
a pixel's label its nearest z level, so heights drawn from the levels (NaN for background) give
any map.  The labelling works on 32 x 32 tiles; the patterns cross their borders and corners."""
import importlib
import math

import numpy as np
import pytest
from scipy import ndimage

from oracle import unproject_oracle as UO

PKG = "3d-point-cloud-multiday-imagery_b200"
synth = importlib.import_module(PKG + ".synth")
api = importlib.import_module(PKG + ".api")
C = importlib.import_module(PKG + "._cabi")

QUANT_BITS = 22  # common.cuh: |quantised coordinate| < 2^22


# ---------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------
def ref_region_map(cmap, conn):
    """The oracle: scipy.ndimage.label per (day, value), ids renumbered by first raster pixel."""
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


def ref_table(rmap, cmap):
    """int64 [R,7]: day, cluster, pixels, y_min, x_min, y_max, x_max of every region."""
    rmap, cmap = np.asarray(rmap), np.asarray(cmap)
    D, H, W = rmap.shape
    R = int(rmap.max()) if rmap.size else 0
    flat = rmap.ravel()
    sel = flat > 0
    idx = np.nonzero(sel)[0]
    r = flat[sel].astype(np.int64) - 1
    day, rem = np.divmod(idx, H * W)
    y, x = np.divmod(rem, W)
    t = np.zeros((R, 7), dtype=np.int64)
    t[:, 3] = t[:, 4] = np.iinfo(np.int64).max
    t[:, 5] = t[:, 6] = -1
    t[:, 2] = np.bincount(r, minlength=R)
    first = np.full(R, np.iinfo(np.int64).max)
    np.minimum.at(first, r, idx)
    t[:, 0] = first // (H * W)
    t[:, 1] = cmap.ravel()[first].astype(np.int64) - 1
    np.minimum.at(t[:, 3], r, y)
    np.minimum.at(t[:, 4], r, x)
    np.maximum.at(t[:, 5], r, y)
    np.maximum.at(t[:, 6], r, x)
    assert np.array_equal(np.sort(first), first), "ids are not in first-pixel order"
    return t


def frame_exponents(P):
    """compute_frame (mdkm.cu) as test_day_stats.py restates it: the fixed-point scale exponents."""
    P32 = np.asarray(P, dtype=np.float32)
    e = np.zeros(3)
    for d in range(3):
        lo, hi = float(P32[:, d].min()), float(P32[:, d].max())
        mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
        o = float(np.float32(float(np.rint(mid)) if abs(mid) > 0.25 * half else 0.0))
        hr = max(abs(lo - o), abs(hi - o)) * (1.0 + 1e-6) + 1e-30
        e[d] = min(100, max(-100, math.floor(math.log2(((1 << QUANT_BITS) - 2) / hr))))
    return e


def check_regions(table, means, rmap, cmap, conn, P=None, valid=None, day_counts=None, exact=False):
    """The region map against the oracle on ``cmap``, the table exactly, the pixels against
    day_counts, and the means (points ``P`` of the ``valid`` pixels, np.where order) exactly on
    dyadic clouds or within half a grid step."""
    cmap = np.asarray(cmap)
    ref = ref_region_map(cmap, conn)
    assert rmap.dtype == np.int32 and rmap.shape == cmap.shape
    assert rmap.tobytes() == ref.tobytes()
    R = int(ref.max()) if ref.size else 0
    assert table.dtype == np.int64 and table.shape == (R, 7)
    assert means.dtype == np.float64 and means.shape == (R, 3)
    assert table.tobytes() == ref_table(ref, cmap).tobytes()
    if day_counts is not None:
        k = day_counts.shape[1]
        per = np.zeros(day_counts.size, dtype=np.int64)
        np.add.at(per, table[:, 0] * k + table[:, 1], table[:, 2])
        np.testing.assert_array_equal(per.reshape(day_counts.shape), day_counts)
    if P is not None and R:
        P = np.asarray(P, dtype=np.float64)
        r = ref.ravel()[np.asarray(valid).ravel()].astype(np.int64) - 1
        assert r.shape[0] == P.shape[0] and np.all(r >= 0)
        cnt = np.bincount(r, minlength=R).astype(np.float64)
        if exact:
            P16 = P * 16.0
            assert np.array_equal(P16, np.rint(P16))
            refm = np.stack([np.bincount(r, weights=P16[:, d], minlength=R) / (16.0 * cnt) for d in range(3)], 1)
            assert refm.tobytes() == means.tobytes()
        else:
            half = 2.0 ** -(frame_exponents(P) + 1)
            for d in range(3):
                refm = np.bincount(r, weights=P[:, d], minlength=R) / cnt
                assert np.all(np.abs(means[:, d] - refm) <= half[d] * 1.001 + 1e-13 * np.abs(refm))


def levels(k):
    """k distinct z levels inside the valid height range."""
    return np.linspace(-130.0, 130.0, k) if k > 1 else np.array([5.0])


def draw(labels_map, k):
    """Heights whose nearest level is the wanted label (-1: NaN, no point)."""
    z = levels(k)
    hm = np.where(labels_map >= 0, z[np.clip(labels_map, 0, k - 1)], np.nan).astype(np.float32)
    return hm


def level_centroids(k, H, W):
    return np.stack([np.full(k, W / 2.0), np.full(k, H / 2.0), levels(k)], axis=1)


def predict_checked(engine, labels_map, k, conn, device_map=False):
    """predict on the drawn map with and without regions: everything else equal, the region map
    and table against the oracle on the returned cluster map, whose values are the drawn labels."""
    D, H, W = labels_map.shape
    hm = draw(labels_map, k)
    engine.unproject(hm)
    c = level_centroids(k, H, W)
    dt = np.uint8 if k <= 255 else np.uint16
    cmap0 = np.empty(hm.shape, dt)
    lab0, in0, cnt0, mean0 = engine.predict(c, cluster_map_out=cmap0, day_stats=True)
    lab0 = lab0.copy()
    cmap = np.empty(hm.shape, dt)
    if device_map:
        import torch

        rdev = torch.full(hm.shape, -7, dtype=torch.int32, device="cuda")
        lab, inertia, cnt, mean, table, means = engine.predict(c, cluster_map_out=cmap, day_stats=True, regions=conn,
                                                               region_map_out=rdev)
        torch.cuda.synchronize()
        rmap = rdev.cpu().numpy()
    else:
        rmap = np.full(hm.shape, -7, np.int32)
        lab, inertia, cnt, mean, table, means = engine.predict(c, cluster_map_out=cmap, day_stats=True, regions=conn,
                                                               region_map_out=rmap)
    assert np.array_equal(lab, lab0) and inertia == in0
    assert cmap.tobytes() == cmap0.tobytes() and cnt.tobytes() == cnt0.tobytes() and mean.tobytes() == mean0.tobytes()
    assert np.array_equal(cmap.astype(np.int64) - 1, np.where(labels_map >= 0, labels_map, -1))
    valid = UO.valid_mask(hm)
    check_regions(table, means, rmap, cmap, conn, UO.unproject_stack(hm), valid, cnt)
    return table, rmap


# ---------------------------------------------------------------------------------------
# patterns
# ---------------------------------------------------------------------------------------
def spiral(H, W):
    """A one-pixel-wide spiral of label 0 on a background of label 1 (one long chain)."""
    m = np.ones((H, W), np.int64)
    top, left, bottom, right = 0, 0, H - 1, W - 1
    while top <= bottom and left <= right:
        m[top, left:right + 1] = 0
        m[top:bottom + 1, right] = 0
        if top + 2 <= bottom:
            m[bottom, left:right + 1] = 0
        if left + 2 <= right:
            m[top + 2:bottom + 1, left] = 0
        top, left, bottom, right = top + 2, left + 2, bottom - 2, right - 2
        if top <= bottom:
            m[top - 1, left] = 0 if left <= right else m[top - 1, left - 1]
    return m


def serpentine(H, W):
    m = np.full((H, W), -1, np.int64)
    m[::2, :] = 0
    for r in range(1, H, 2):
        m[r, W - 1 if (r // 2) % 2 == 0 else 0] = 0
    return m


def comb(H, W):
    m = np.full((H, W), 1, np.int64)
    m[0, :] = 0
    m[:, ::3] = 0
    m[H - 1, 1::3] = -1
    return m


def checker(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    return ((yy + xx) % 2).astype(np.int64)


def staircase(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    m = np.full((H, W), -1, np.int64)
    m[(xx - yy) % 7 == 0] = 0
    m[(xx + yy) % 5 == 0] = 1
    return m


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def test_oracle_on_hand_drawn_maps():
    c = np.array([[[1, 2, 1, 2], [2, 1, 2, 1], [1, 2, 1, 2], [2, 1, 2, 1]]], np.uint8)
    assert ref_region_map(c, 4).max() == 16 and ref_region_map(c, 8).max() == 2
    m = np.array([[[0, 1, 1, 0, 2],
                   [1, 0, 1, 0, 2],
                   [1, 1, 0, 3, 0]],
                  [[3, 3, 0, 0, 0],
                   [0, 0, 0, 0, 0],
                   [0, 0, 0, 0, 3]]], np.uint8)
    r4 = ref_region_map(m, 4)
    assert r4.tolist() == [[[0, 1, 1, 0, 2], [3, 0, 1, 0, 2], [3, 3, 0, 4, 0]],
                           [[5, 5, 0, 0, 0], [0, 0, 0, 0, 0], [0, 0, 0, 0, 6]]]
    r8 = ref_region_map(m, 8)
    assert r8.tolist() == [[[0, 1, 1, 0, 2], [1, 0, 1, 0, 2], [1, 1, 0, 3, 0]],
                           [[4, 4, 0, 0, 0], [0, 0, 0, 0, 0], [0, 0, 0, 0, 5]]]
    t = ref_table(r8, m)
    assert t.tolist() == [[0, 0, 6, 0, 0, 2, 2], [0, 1, 2, 0, 4, 1, 4], [0, 2, 1, 2, 3, 2, 3],
                          [1, 2, 2, 0, 0, 0, 1], [1, 2, 1, 2, 4, 2, 4]]


def test_one_cluster_matches_scipy_numbering():
    rs = np.random.RandomState(0)
    m = (rs.rand(1, 40, 50) < 0.5).astype(np.uint8)
    lab, n = ndimage.label(m[0])
    assert ref_region_map(m, 4)[0].tolist() == lab.tolist() and n == ref_region_map(m, 4).max()


def test_region_connectivity_normalisation():
    assert api.requested_connectivity(False) is None
    assert api.requested_connectivity(False, 8) is None
    assert api.requested_connectivity(True) == 4
    assert api.requested_connectivity(True, 8) == 8
    assert api.requested_connectivity(False, 8, True) == 8
    assert api.requested_connectivity(np.True_, np.int64(4)) == 4
    for bad in (6, 0, True, None, "4", 4.5):
        with pytest.raises(ValueError):
            api.requested_connectivity(True, bad)


def test_bad_connectivity_raises_before_any_gpu_work(pkg):
    class NoEngine:  # any use of the engine would raise AttributeError instead
        pass

    for kw in (dict(return_regions=True, region_connectivity=6), dict(return_region_map=True, region_connectivity=2)):
        with pytest.raises(ValueError):
            pkg.fuse_multiday_kmeans(np.zeros((2, 4, 4), dtype=np.float32), engine=NoEngine(), **kw)


def test_fusion_result_has_no_regions_by_default():
    r = api.FusionResult(labels=np.zeros(1, np.int32), centroids=np.zeros((1, 3)), fused_cloud=np.zeros((1, 3)),
                         n_iter=1, inertia=0.0, n_points=1)
    assert r.regions is None and r.region_means is None and r.region_map is None
    assert [t for _, _, t in api.to_layers(r)] == ["points", "points"]
    r.region_map = np.zeros((1, 1, 1), np.int32)
    layers = api.to_layers(r, prefix="P")
    assert [t for _, _, t in layers] == ["points", "points", "labels"] and layers[-1][1]["name"] == "P Regions"


# ---------------------------------------------------------------------------------------
# GPU: controlled label patterns
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("name", ["spiral", "serpentine", "comb", "checker", "staircase"])
def test_patterns(engine, name, conn):
    H, W = 97, 131
    f = {"spiral": spiral, "serpentine": serpentine, "comb": comb, "checker": checker, "staircase": staircase}[name]
    m = np.stack([f(H, W), f(H, W)[::-1, ::-1].copy(), np.where(f(H, W) >= 0, 1 - f(H, W), -1)])
    m[m > 1] = 1
    predict_checked(engine, m, 2, conn)


@pytest.mark.gpu
def test_checkerboard_connectivities_differ(engine):
    m = checker(64, 64)[None]
    t4, _ = predict_checked(engine, m, 2, 4)
    t8, _ = predict_checked(engine, m, 2, 8)
    assert t4.shape[0] == 64 * 64 and t8.shape[0] == 2


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 16, 300])
def test_one_cluster_everywhere_and_an_empty_day(engine, k):
    m = np.full((3, 70, 45), k - 1, np.int64)
    m[1] = -1
    t, rmap = predict_checked(engine, m, k, 8)
    assert t[:, :3].tolist() == [[0, k - 1, 70 * 45], [2, k - 1, 70 * 45]]
    assert (rmap[1] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("k", [2, 16, 300])
@pytest.mark.parametrize("D", [1, 3, 10])
def test_random_holes_and_labels(engine, k, conn, D):
    rs = np.random.RandomState(k * 10 + D)
    m = rs.randint(0, k, size=(D, 45, 77)).astype(np.int64)
    if k > 16:
        m = (m % 4) + rs.randint(0, 2, size=m.shape) * (k - 4)  # a few labels, some of them above 255
    m[rs.rand(*m.shape) < 0.5] = -1
    predict_checked(engine, m, k, conn)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 1, 70), (2, 70, 1), (1, 1, 1), (3, 33, 65), (2, 64, 32), (1, 31, 97)])
def test_odd_shapes(engine, shape):
    rs = np.random.RandomState(sum(shape))
    k = 3 if np.prod(shape) > 8 else 1  # (predict needs at least k points)
    m = rs.randint(-1, k, size=shape).astype(np.int64)
    m[0].flat[0] = k - 1
    for conn in (4, 8):
        predict_checked(engine, m, k, conn)


@pytest.mark.gpu
def test_device_region_map_in_place(engine):
    rs = np.random.RandomState(5)
    m = rs.randint(-1, 4, size=(2, 50, 90)).astype(np.int64)
    for conn in (4, 8):
        predict_checked(engine, m, 4, conn, device_map=True)


# ---------------------------------------------------------------------------------------
# GPU: fits
# ---------------------------------------------------------------------------------------
def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter and a.n_refined == b.n_refined
    for name in ("cluster_map", "day_counts", "day_means", "transitions"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None)
        if x is not None:
            assert x.tobytes() == y.tobytes()


def fuse_checked(pkg, hm, masks=None, *, k, conn=4, exact=False, P=None, **kw):
    """The call without and with regions: everything else bitwise equal; regions checked against the
    oracle on the returned cluster map."""
    plain = pkg.fuse_multiday_kmeans(hm, masks, n_clusters=k, return_cluster_map=True, return_day_stats=True, **kw)
    res = pkg.fuse_multiday_kmeans(hm, masks, n_clusters=k, return_cluster_map=True, return_day_stats=True,
                                   return_region_map=True, region_connectivity=conn, **kw)
    assert plain.regions is None and plain.region_map is None
    same_result(plain, res)
    valid = UO.valid_mask(UO.height_from_disparity(hm) if exact else hm, masks)
    if P is None:
        P = res.fused_cloud[:, ::-1]  # the clustered cloud, (x, y, z)
    check_regions(res.regions, res.region_means, res.region_map, res.cluster_map, conn, P, valid, res.day_counts,
                  exact=exact)
    return res


def stack(D, H, W, seed):
    return synth.make_stack(D, H, W, seed=seed, n_buildings=6).numpy()


def seeds(hm, k, seed):
    return synth.init_from_points(UO.unproject_stack(hm).astype(np.float32), k, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_synthetic_stack(pkg, engine, conn):
    hm = stack(3, 130, 170, 3)
    res = fuse_checked(pkg, hm, k=9, conn=conn, init="k-means++", random_state=1, max_iter=20, engine=engine)
    assert res.regions.shape[0] > 9


@pytest.mark.gpu
def test_detrend_and_ground_level(pkg, engine):
    hm = stack(2, 90, 140, 4)
    fuse_checked(pkg, hm, k=7, conn=8, init="k-means++", random_state=2, max_iter=20, detrend=True,
                 ground_level=True, engine=engine)


@pytest.mark.gpu
def test_dyadic_means_are_exact(pkg, engine):
    rs = np.random.RandomState(9)
    H, W = 70, 110
    yy, xx = np.mgrid[0:H, 0:W]
    disp = (16 * 20.0 * (np.sin(xx / 9.0) * np.cos(yy / 7.0))[None] + rs.randint(-8, 9, size=(3, H, W)))
    disp = disp.astype(np.int16)
    mask = rs.rand(3, H, W) < 0.95
    P = UO.unproject_stack(UO.height_from_disparity(disp), mask)
    fuse_checked(pkg, disp, mask, k=6, conn=4, exact=True, P=P, init="k-means++", random_state=3, max_iter=20,
                 disparity_scale=-1.0 / 16.0, engine=engine)


@pytest.mark.gpu
def test_restarts_keep_the_returned_runs_regions(pkg, engine):
    hm = stack(3, 60, 130, 9)
    fuse_checked(pkg, hm, k=12, conn=8, init="k-means++", n_init=3, random_state=11, max_iter=15, engine=engine)


@pytest.mark.gpu
def test_restarts_with_a_device_region_map(pkg, engine):
    import torch

    hm = stack(2, 50, 70, 10)
    engine.unproject(hm)
    out = torch.zeros(hm.size, dtype=torch.int32, device="cuda")
    cmap = np.empty(hm.shape, np.uint8)
    r = api._run_kmeans(engine, n_clusters=5, init="k-means++", n_init=3, max_iter=10, tol=1e-4, random_state=4,
                        cluster_map_out=cmap, regions=4, region_map_out=out)
    torch.cuda.synchronize()
    check_regions(r["regions"], r["region_means"], out.cpu().numpy().reshape(hm.shape), cmap, 4)


@pytest.mark.gpu
def test_relocation(engine):
    hm = stack(3, 80, 120, 10)
    init = seeds(hm, 8, 2)
    init[5] = [1e5, -1e5, 1e4]  # far outside the cloud: empty after the first E-step
    engine.unproject(hm)
    cmap = np.empty(hm.shape, np.uint8)
    rmap = np.empty(hm.shape, np.int32)
    r1 = engine.fit(init, max_iter=30, tol=0.0, cluster_map_out=cmap, day_stats=True, regions=8, region_map_out=rmap)
    labels1 = r1["labels"].copy()
    r0 = engine.fit(init, max_iter=30, tol=0.0, day_stats=True)
    assert r1["n_relocations"] >= 1
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    assert r1["inertia"] == r0["inertia"] and r1["n_iter"] == r0["n_iter"]
    check_regions(r1["regions"], r1["region_means"], rmap, cmap, 8, UO.unproject_stack(hm), UO.valid_mask(hm),
                  r1["day_counts"])


@pytest.mark.gpu
def test_predict_on_a_second_stack(engine):
    hm = stack(2, 50, 140, 12)
    engine.unproject(hm)
    centers = engine.fit(seeds(hm, 9, 3), max_iter=10, regions=4)["centers"]
    hm2 = stack(4, 30, 91, 13)
    engine.unproject(hm2)  # drops the regions of the fit
    with pytest.raises(C.MdkmError):
        engine._region_table()
    cmap = np.empty(hm2.shape, np.uint8)
    rmap = np.empty(hm2.shape, np.int32)
    labels, inertia, counts, means, table, rmeans = engine.predict(centers, cluster_map_out=cmap, day_stats=True,
                                                                   regions=8, region_map_out=rmap)
    check_regions(table, rmeans, rmap, cmap, 8, UO.unproject_stack(hm2), UO.valid_mask(hm2), counts)


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_with_transitions_one_shared_map(pkg, engine, conn):
    hm = stack(3, 70, 100, 14)
    res = fuse_checked(pkg, hm, k=6, conn=conn, init="k-means++", random_state=5, max_iter=10, engine=engine,
                       return_transitions=True)
    m = res.cluster_map.reshape(3, -1).astype(np.int64)
    ref = np.bincount(m[0] * 7 + m[1], minlength=49).reshape(7, 7)
    assert np.array_equal(res.transitions[0], ref)


@pytest.mark.gpu
def test_regions_without_a_cluster_map(pkg, engine):
    """No map bound: the final pass writes the internal one."""
    hm = stack(2, 60, 80, 15)
    a = pkg.fuse_multiday_kmeans(hm, n_clusters=5, init="k-means++", random_state=6, max_iter=10, engine=engine,
                                 return_regions=True, return_cluster_map=True)
    b = pkg.fuse_multiday_kmeans(hm, n_clusters=5, init="k-means++", random_state=6, max_iter=10, engine=engine,
                                 return_regions=True, region_connectivity=4)
    assert b.region_map is None and b.cluster_map is None
    assert a.regions.tobytes() == b.regions.tobytes() and a.region_means.tobytes() == b.region_means.tobytes()
    check_regions(b.regions, b.region_means, ref_region_map(a.cluster_map, 4), a.cluster_map, 4)


@pytest.mark.gpu
def test_errors(pkg, engine):
    ERR_STATE, ERR_INVALID = C.STATUS_BY_NAME["MDKM_ERR_STATE"], C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    bind = engine._lib.mdkm_bind_regions
    hm = stack(3, 30, 60, 17)
    init = seeds(hm, 5, 1)
    out = np.empty(hm.size, np.int32)
    fresh = pkg.Engine(0)
    try:  # no resident cloud; no regions yet
        assert bind(fresh._h, 4, None, 0, C.MEM_HOST) == ERR_STATE
        with pytest.raises(C.MdkmError) as ei:
            fresh._region_table()
        assert ei.value.code == ERR_STATE
    finally:
        fresh.close()
    engine.set_points(UO.unproject_stack(hm).astype(np.float32))  # no raster
    assert bind(engine._h, 4, None, 0, C.MEM_HOST) == ERR_STATE
    with pytest.raises(C.MdkmError) as ei:
        engine.fit(init, max_iter=5, regions=4)
    assert ei.value.code == ERR_STATE
    engine.unproject(hm)
    for conn in (0, 1, 5, 6, -4):
        assert bind(engine._h, conn, out.ctypes.data, out.size, C.MEM_HOST) == ERR_INVALID
    assert bind(engine._h, 4, out.ctypes.data, out.size - 1, C.MEM_HOST) == ERR_INVALID
    assert bind(engine._h, 8, out.ctypes.data, out.size, 7) == ERR_INVALID
    assert bind(engine._h, 0, None, 0, C.MEM_HOST) == C.MDKM_OK
    with pytest.raises(ValueError):
        engine.fit(init, max_iter=5, regions=6)
    with pytest.raises(ValueError):
        engine.fit(init, max_iter=5, region_map_out=out)
    r = engine.fit(init, max_iter=5)
    assert "regions" not in r
    # a short table capacity
    r = engine.fit(init, max_iter=5, regions=4)
    R = r["regions"].shape[0]
    t = np.empty((R, 7), np.int64)
    m = np.empty((R, 3), np.float64)
    assert engine._lib.mdkm_region_table(engine._h, t.ctypes.data, m.ctypes.data, R - 1) == ERR_INVALID
    assert engine._lib.mdkm_region_table(engine._h, t.ctypes.data, m.ctypes.data, R) == C.MDKM_OK
    assert t.tobytes() == r["regions"].tobytes()
    # a fit without regions keeps the last ones
    engine.fit(init, max_iter=5)
    assert engine._region_table()[0].tobytes() == r["regions"].tobytes()
    # one handle without a communicator holding part of the stack: ERR_STATE, and the handle still works
    flat = hm.reshape(-1)
    HW = 30 * 60
    engine.unproject(flat[HW + 100:2 * HW + 50], stack_shape=hm.shape, pix_begin=HW + 100)
    for call in (lambda: engine.fit(init, max_iter=5, regions=8), lambda: engine.predict(init, regions=4)):
        with pytest.raises(C.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_STATE
    engine.predict(init)
    # the binding is dropped by unproject
    engine.unproject(hm)
    assert bind(engine._h, 4, None, 0, C.MEM_HOST) == C.MDKM_OK
    engine.unproject(hm)
    r = engine.fit(init, max_iter=5)
    assert "regions" not in r
    with pytest.raises(C.MdkmError):
        engine._region_table()
    r = engine.fit(init, max_iter=5, regions=4, region_map_out=out)
    cm = np.zeros(hm.size, np.uint8)
    cm[UO.valid_mask(hm).ravel()] = r["labels"] + 1
    check_regions(r["regions"], r["region_means"], out.reshape(hm.shape), cm.reshape(hm.shape), 4)


@pytest.mark.gpu
def test_a_refused_binding_leaves_none_behind(engine):
    hm = stack(2, 40, 60, 21)
    engine.unproject(hm)
    init = seeds(hm, 5, 1)
    with pytest.raises(C.MdkmError):  # day 2 does not exist: refused after the regions were... not yet bound
        engine.fit(init, max_iter=5, transitions=[(0, 2)], regions=4)
    with pytest.raises(ValueError):  # short region map: refused after the other bindings
        engine.fit(init, max_iter=5, day_stats=True, regions=4, region_map_out=np.empty(5, np.int32))
    r = engine.fit(init, max_iter=5)
    assert "regions" not in r and "day_counts" not in r


@pytest.mark.gpu
def test_plugin_passes_the_options(pkg, monkeypatch):
    hm = stack(2, 64, 80, 13)
    seen = []
    to_layers = api.to_layers
    monkeypatch.setattr(api, "to_layers", lambda res: seen.append(res) or to_layers(res))
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_region_map=True, region_connectivity=8,
                                    return_cluster_map=True, init="k-means++", random_state=0, max_iter=10)
    layers = plug.run(hm)
    assert [t for _, _, t in layers] == ["points", "points", "labels", "labels"]
    assert layers[-1][1]["name"] == "Multi-day Regions"
    (res,) = seen
    check_regions(res.regions, res.region_means, res.region_map, res.cluster_map, 8)


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
              region_connectivity=8)
    one = pkg.fuse_multiday_kmeans(hm, device=0, return_cluster_map=True, return_day_stats=True, **kw)
    two = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], **kw)
    assert np.array_equal(one.labels, two.labels)
    assert two.region_map.tobytes() == one.region_map.tobytes()
    assert two.regions.tobytes() == one.regions.tobytes() and two.region_means.tobytes() == one.region_means.tobytes()
    check_regions(one.regions, one.region_means, one.region_map, one.cluster_map, 8, day_counts=one.day_counts)


@pytest.mark.gpu
def test_pre_sharded_ranks_receive_the_whole_table(pkg):
    _two_gpus()
    from concurrent.futures import ThreadPoolExecutor

    hm = stack(3, 30, 70, 19)
    flat = hm.reshape(-1)
    cut = 30 * 70 + 517
    init = seeds(hm, 6, 4)
    one = pkg.fuse_multiday_kmeans(hm, n_clusters=6, init=init, max_iter=10, return_region_map=True)
    uid = pkg.Engine.make_unique_id()
    engines = [pkg.Engine(r) for r in range(2)]
    try:
        with ThreadPoolExecutor(2) as ex:
            list(ex.map(lambda r: engines[r].init_comm(2, r, uid), range(2)))
            spans = [(0, cut), (cut, flat.size)]
            res = list(ex.map(lambda r: pkg.fuse_multiday_kmeans(
                flat[spans[r][0]:spans[r][1]], n_clusters=6, init=init, max_iter=10, engine=engines[r],
                stack_shape=hm.shape, pix_begin=spans[r][0], return_region_map=True), range(2)))
    finally:
        for e in engines:
            e.close()
    for r in res:
        assert r.regions.tobytes() == one.regions.tobytes() and r.region_means.tobytes() == one.region_means.tobytes()
    assert np.concatenate([r.region_map for r in res]).tobytes() == one.region_map.tobytes()
