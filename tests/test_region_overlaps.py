"""Region overlaps between days (``return_region_overlaps`` / ``region_overlaps=``): for every
requested pair of days (a, b), one row per pair of regions (r of day a, s of day b) that share at
least one pixel -- int64 (pair, region_a, region_b, pixels, y_first, x_first) -- sorted by pair,
then by the raster order of the first shared pixel.

The oracle is a numpy restatement per pair on the region map the same call returns: the packed
(id_a, id_b) keys of the pixels where both ids are non-zero, ``np.unique`` with first index and
counts, ordered by first index.  The region map itself is checked against ``scipy.ndimage.label``
(restated from ``test_regions.py``).  Every GPU case also checks the rows against the transition
counts when those are asked for, and that asking for overlaps changes nothing else.

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


def ref_overlaps(rmap, pairs):
    """int64 [M,6] rows of the day pairs on the region map ``rmap`` [D,H,W]."""
    rmap = np.asarray(rmap)
    D, H, W = rmap.shape
    flat = rmap.reshape(D, -1).astype(np.int64)
    out = []
    for p, (a, b) in enumerate(np.asarray(pairs).reshape(-1, 2)):
        ra, rb = flat[a], flat[b]
        idx = np.nonzero((ra > 0) & (rb > 0))[0]
        keys = (ra[idx] << 32) | rb[idx]
        u, first, cnt = np.unique(keys, return_index=True, return_counts=True)
        order = np.argsort(first, kind="stable")
        u, px, cnt = u[order], idx[first[order]], cnt[order]
        t = np.empty((u.size, 6), dtype=np.int64)
        t[:, 0] = p
        t[:, 1] = u >> 32
        t[:, 2] = u & 0xFFFFFFFF
        t[:, 3] = cnt
        t[:, 4] = px // W
        t[:, 5] = px % W
        out.append(t)
    return np.concatenate(out) if out else np.zeros((0, 6), np.int64)


def check_overlaps(rows, rmap, pairs, regions, transitions=None):
    """The rows bit for bit against the oracle, and the consequences the semantics promise."""
    rmap = np.asarray(rmap)
    pairs = np.asarray(pairs).reshape(-1, 2)
    D = rmap.shape[0]
    flat = rmap.reshape(D, -1)
    assert rows.dtype == np.int64 and rows.ndim == 2 and rows.shape[1] == 6
    ref = ref_overlaps(rmap, pairs)
    assert rows.shape == ref.shape and rows.tobytes() == ref.tobytes()
    by_pair = [rows[rows[:, 0] == p] for p in range(pairs.shape[0])]
    cluster = np.concatenate([[-1], regions[:, 1]])
    for p, (a, b) in enumerate(pairs):
        t = by_pair[p]
        if a == b:  # every region of day a with itself, in id order
            ids = np.nonzero(regions[:, 0] == a)[0] + 1
            assert np.array_equal(t[:, 1], ids) and np.array_equal(t[:, 2], ids)
            assert np.array_equal(t[:, 3], regions[ids - 1, 2])
            _, first = np.unique(flat[a], return_index=True)
            first = first[1:] if flat[a][first[0]] == 0 else first
            assert np.array_equal(t[:, 4] * rmap.shape[2] + t[:, 5], first)
        # a region's pixels that have a point on day b, summed over its rows
        has_b = flat[b] > 0
        want = np.bincount(flat[a][has_b], minlength=regions.shape[0] + 1)[1:]
        got = np.bincount(t[:, 1], weights=t[:, 3], minlength=regions.shape[0] + 1)[1:].astype(np.int64)
        assert np.array_equal(got[regions[:, 0] == a], want[regions[:, 0] == a])
        for q, (c, d) in enumerate(pairs):  # (b, a) rows are (a, b) rows with columns 1 and 2 swapped
            if c == b and d == a:
                u = by_pair[q]
                assert np.array_equal(u[:, [2, 1, 3, 4, 5]], t[:, 1:])
        if transitions is not None:
            k = transitions.shape[1] - 1
            T = np.zeros((k, k), dtype=np.int64)
            np.add.at(T, (cluster[t[:, 1]], cluster[t[:, 2]]), t[:, 3])
            assert np.array_equal(T, transitions[p, 1:, 1:])


def levels(k):
    return np.linspace(-130.0, 130.0, k) if k > 1 else np.array([5.0])


def draw(labels_map, k):
    """Heights whose nearest level is the wanted label (-1: NaN, no point)."""
    z = levels(k)
    return np.where(labels_map >= 0, z[np.clip(labels_map, 0, k - 1)], np.nan).astype(np.float32)


def level_centroids(k, H, W):
    return np.stack([np.full(k, W / 2.0), np.full(k, H / 2.0), levels(k)], axis=1)


def predict_checked(engine, labels_map, k, conn, pairs, device_map=None):
    """predict on the drawn map with regions and transitions, without and with overlaps: everything
    else equal, the region map against scipy, the overlaps against the oracle and the transitions.
    ``device_map``: "aligned" / "offset" -- the region map in a CUDA tensor (its start 16-byte
    aligned, or 4 bytes past that)."""
    D, H, W = labels_map.shape
    hm = draw(labels_map, k)
    engine.unproject(hm)
    c = level_centroids(k, H, W)
    dt = np.uint8 if k <= 255 else np.uint16
    cmap0 = np.empty(hm.shape, dt)
    rmap0 = np.empty(hm.shape, np.int32)
    base = engine.predict(c, cluster_map_out=cmap0, day_stats=True, transitions=pairs, regions=conn,
                          region_map_out=rmap0)
    base = (base[0].copy(),) + base[1:]
    cmap = np.empty(hm.shape, dt)
    if device_map is not None:
        import torch

        buf = torch.full((hm.size + 4,), -7, dtype=torch.int32, device="cuda")
        rdev = buf[:hm.size] if device_map == "aligned" else buf[1:hm.size + 1]
        out = engine.predict(c, cluster_map_out=cmap, day_stats=True, transitions=pairs, regions=conn,
                             region_map_out=rdev, region_overlaps=pairs)
        torch.cuda.synchronize()
        rmap = rdev.cpu().numpy().reshape(hm.shape)
    else:
        rmap = np.full(hm.shape, -7, np.int32)
        out = engine.predict(c, cluster_map_out=cmap, day_stats=True, transitions=pairs, regions=conn,
                             region_map_out=rmap, region_overlaps=pairs)
    assert len(out) == len(base) + 1
    lab, inertia, cnt, mean, trans, table, means, rows = out
    assert np.array_equal(lab, base[0]) and inertia == base[1]
    for x, y in zip((cnt, mean, trans, table, means), base[2:]):
        assert x.tobytes() == y.tobytes()
    assert cmap.tobytes() == cmap0.tobytes() and rmap.tobytes() == rmap0.tobytes()
    assert np.array_equal(cmap.astype(np.int64) - 1, np.where(labels_map >= 0, labels_map, -1))
    assert rmap.tobytes() == ref_region_map(cmap, conn).tobytes()
    check_overlaps(rows, rmap, pairs, table, trans)
    return rows, rmap, table


# ---------------------------------------------------------------------------------------
# patterns
# ---------------------------------------------------------------------------------------
def spiral(H, W):
    """A one-pixel-wide spiral of label 0 on a background of label 1 (test_regions.py)."""
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


def checker(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    return ((yy + xx) % 2).astype(np.int64)


def stripes(H, W, s, vertical):
    yy, xx = np.mgrid[0:H, 0:W]
    return (((xx if vertical else yy) // s) % 2).astype(np.int64)


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def test_oracle_on_a_hand_drawn_pair():
    r = np.array([[[1, 1, 0, 2],
                   [1, 1, 2, 2]],
                  [[3, 4, 4, 4],
                   [0, 3, 5, 0]]], np.int32)
    rows = ref_overlaps(r, [(0, 1), (1, 0), (0, 0)])
    assert rows.tolist() == [[0, 1, 3, 2, 0, 0], [0, 1, 4, 1, 0, 1], [0, 2, 4, 1, 0, 3], [0, 2, 5, 1, 1, 2],
                             [1, 3, 1, 2, 0, 0], [1, 4, 1, 1, 0, 1], [1, 4, 2, 1, 0, 3], [1, 5, 2, 1, 1, 2],
                             [2, 1, 1, 4, 0, 0], [2, 2, 2, 3, 0, 3]]
    regions = np.array([[0, 0, 4], [0, 1, 3], [1, 0, 2], [1, 1, 3], [1, 2, 1]], np.int64)
    check_overlaps(rows, r, [(0, 1), (1, 0), (0, 0)], regions)
    assert ref_overlaps(np.zeros((2, 3, 3), np.int32), [(0, 1)]).shape == (0, 6)


def test_pair_normalisation_names_the_option():
    assert api.transition_pairs(True, 4, "region overlaps").tolist() == [[0, 1], [1, 2], [2, 3]]
    assert api.transition_pairs([(3, 1), (2, 2), (3, 1)], 4, "region overlaps").tolist() == [[3, 1], [2, 2], [3, 1]]
    with pytest.raises(ValueError, match="^return_region_overlaps=False asks for no pairs$"):
        api.transition_pairs(False, 4, "region overlaps")
    with pytest.raises(ValueError, match="^return_region_overlaps must be True or a sequence"):
        api.transition_pairs([(0.5, 1)], 4, "region overlaps")
    with pytest.raises(ValueError, match=r"^no day pair to count region overlaps of \(the stack has 1 day\(s\)\)$"):
        api.transition_pairs(True, 1, "region overlaps")
    with pytest.raises(ValueError, match=r"^region overlap pair 1 = \(0, 4\): days must be in \[0, 4\)$"):
        api.transition_pairs([(0, 1), (0, 4)], 4, "region overlaps")
    # the messages of return_transitions are as they were
    with pytest.raises(ValueError, match="^return_transitions=False asks for no pairs$"):
        api.transition_pairs(False, 4)
    with pytest.raises(ValueError, match=r"^no day pair to count transitions of \(the stack has 1 day\(s\)\)$"):
        api.transition_pairs(True, 1)
    with pytest.raises(ValueError, match=r"^transition pair 0 = \(-1, 0\): days must be in \[0, 4\)$"):
        api.transition_pairs([(-1, 0)], 4)


class NoEngine:  # any use of the engine would raise AttributeError instead
    pass


@pytest.mark.parametrize("spec", [[(0, 2)], [(-1, 0)], [(0, 1), (1, 5)], True, [(0.0, 1.0)], []])
def test_bad_pairs_raise_before_any_gpu_work(pkg, spec):
    hm = np.zeros((2, 4, 4), dtype=np.float32)
    with pytest.raises(ValueError):
        pkg.fuse_multiday_kmeans(hm[:1] if spec is True else hm, engine=NoEngine(), return_region_overlaps=spec)


def test_too_many_pairs_raise_before_any_gpu_work(pkg):
    hm = np.zeros((2, 4, 4), dtype=np.float32)
    n = api.MAX_REGION_OVERLAP_PAIRS
    with pytest.raises(ValueError, match=f"{n + 1} pairs, at most {n}"):
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_region_overlaps=[(0, 1)] * (n + 1))
    with pytest.raises(AttributeError):  # the limit itself passes the option checks
        pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_region_overlaps=[(0, 1)] * n)


def test_overlaps_imply_regions(pkg):
    """return_region_overlaps asks for regions: a bad connectivity is refused, as with return_regions;
    without overlaps (False / None) it is not looked at."""
    hm = np.zeros((2, 4, 4), dtype=np.float32)
    for spec in (True, [(1, 0)]):
        with pytest.raises(ValueError, match="region_connectivity"):
            pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_region_overlaps=spec, region_connectivity=6)
    for spec in (False, None):
        with pytest.raises(AttributeError):  # past the option checks, at the engine
            pkg.fuse_multiday_kmeans(hm, engine=NoEngine(), return_region_overlaps=spec, region_connectivity=6)


def test_engine_refuses_overlaps_without_regions_before_binding(pkg):
    with pytest.raises(ValueError, match="region_overlaps needs regions"):
        pkg.Engine._bind_outputs(NoEngine(), 3, None, False, None, None, None, [(0, 1)])


def test_fusion_result_has_no_overlaps_by_default():
    r = api.FusionResult(labels=np.zeros(1, np.int32), centroids=np.zeros((1, 3)), fused_cloud=np.zeros((1, 3)),
                         n_iter=1, inertia=0.0, n_points=1)
    assert r.region_overlaps is None and r.region_overlap_pairs is None
    r.region_overlaps = np.zeros((3, 6), np.int64)
    assert [t for _, _, t in api.to_layers(r)] == ["points", "points"]


# ---------------------------------------------------------------------------------------
# GPU: drawn patterns
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_spiral_against_a_shifted_spiral(engine, conn):
    H, W = 97, 131
    s = spiral(H, W)
    m = np.stack([s, np.roll(s, 1, axis=1), np.roll(s, (3, -2), axis=(0, 1))])
    predict_checked(engine, m, 2, conn, [(0, 1), (1, 2), (2, 0), (1, 0), (0, 0)])


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_horizontal_against_vertical_stripes(engine, conn):
    H, W, s = 100, 150, 7
    m = np.stack([stripes(H, W, s, False), stripes(H, W, s, True)])
    rows, _, table = predict_checked(engine, m, 2, conn, [(0, 1), (1, 0)])
    n_a, n_b = -(-H // s), -(-W // s)
    assert int(np.sum(table[:, 0] == 0)) == n_a and int(np.sum(table[:, 0] == 1)) == n_b
    assert rows.shape[0] == 2 * n_a * n_b


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
def test_one_region_against_many(engine, conn):
    rs = np.random.RandomState(3)
    H, W = 130, 90
    b = rs.randint(0, 5, size=(H, W))
    b[rs.rand(H, W) < 0.2] = -1
    m = np.stack([np.full((H, W), 2, np.int64), b])
    rows, _, table = predict_checked(engine, m, 5, conn, [(0, 1), (1, 0), (1, 1)])
    assert np.all(rows[rows[:, 0] == 0][:, 1] == 1)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 64, 64), (2, 61, 67), (3, 160, 257)])
def test_checkerboard_against_its_shift(engine, shape):
    """Every pixel is a region and every pixel a row: the largest bound, hash tables at full load."""
    D, H, W = shape
    c = checker(H, W)
    m = np.stack([c if d % 2 == 0 else np.roll(c, 1, axis=1) for d in range(D)])
    pairs = [(d, d + 1) for d in range(D - 1)] + [(D - 1, 0)]
    rows, _, _ = predict_checked(engine, m, 2, 4, pairs)
    assert rows.shape[0] == len(pairs) * H * W


@pytest.mark.gpu
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("k", [3, 300])
def test_random_labels_odd_sizes_and_an_empty_day(engine, k, conn):
    rs = np.random.RandomState(k + conn)
    m = rs.randint(0, min(k, 4), size=(4, 45, 77)).astype(np.int64)
    if k > 255:
        m = m + rs.randint(0, 2, size=m.shape) * (k - 4)  # labels above 255: a uint16 map
    m[rs.rand(*m.shape) < 0.3] = -1
    m[2] = -1  # a day without a point
    predict_checked(engine, m, k, conn, [(0, 1), (1, 2), (2, 3), (3, 0), (0, 3), (2, 2), (1, 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 1, 1), (3, 1, 70), (2, 70, 1), (2, 33, 65)])
def test_tiny_days(engine, shape):
    rs = np.random.RandomState(sum(shape))
    k = 2 if np.prod(shape) > 8 else 1
    m = rs.randint(-1, k, size=shape).astype(np.int64)
    m[:, 0, 0] = k - 1
    if shape[1] * shape[2] > 1:
        m[-1] = -1
        m[-1, 0, 0] = 0  # a day of one pixel with a point
    for conn in (4, 8):
        predict_checked(engine, m, k, conn, [(d, (d + 1) % shape[0]) for d in range(shape[0])] + [(0, 0)])


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["aligned", "offset"])
def test_device_region_map(engine, where):
    """The ids are read from the caller's CUDA map; 4 bytes off alignment they take the scalar loads."""
    rs = np.random.RandomState(5)
    m = rs.randint(-1, 4, size=(3, 50, 96)).astype(np.int64)
    for conn in (4, 8):
        predict_checked(engine, m, 4, conn, [(0, 1), (2, 1), (0, 2)], device_map=where)


@pytest.mark.gpu
def test_long_runs_cross_the_warp_spans(engine):
    """Large uniform areas: runs of one key across many 128-pixel groups and warp spans."""
    H, W = 300, 700
    a = np.zeros((H, W), np.int64)
    a[:, 350:] = 1
    b = np.zeros((H, W), np.int64)
    b[150:, :] = 1
    b[10:20, 100:600] = -1
    rows, _, _ = predict_checked(engine, np.stack([a, b]), 2, 8, [(0, 1), (1, 0)])
    assert rows.shape[0] == 8


# ---------------------------------------------------------------------------------------
# GPU: fits
# ---------------------------------------------------------------------------------------
def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter and a.n_refined == b.n_refined
    for name in ("cluster_map", "day_counts", "day_means", "transitions", "regions", "region_means", "region_map"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None)
        if x is not None:
            assert x.tobytes() == y.tobytes()


def fuse_checked(pkg, hm, *, k, pairs=True, conn=4, **kw):
    """The call without and with overlaps: everything else bitwise equal; the overlaps against the
    oracle on the returned region map, which is checked against scipy."""
    common = dict(n_clusters=k, return_cluster_map=True, return_day_stats=True, return_transitions=pairs,
                  return_region_map=True, region_connectivity=conn, **kw)
    plain = pkg.fuse_multiday_kmeans(hm, **common)
    res = pkg.fuse_multiday_kmeans(hm, return_region_overlaps=pairs, **common)
    assert plain.region_overlaps is None and plain.region_overlap_pairs is None
    same_result(plain, res)
    assert np.array_equal(res.region_overlap_pairs, res.transition_pairs)
    assert res.region_map.tobytes() == ref_region_map(res.cluster_map, conn).tobytes()
    check_overlaps(res.region_overlaps, res.region_map, res.region_overlap_pairs, res.regions, res.transitions)
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
    assert res.region_overlaps.shape[0] > 9


@pytest.mark.gpu
def test_explicit_pairs_backwards_repeated_and_skipping(pkg, engine):
    hm = stack(4, 90, 120, 4)
    pairs = [(3, 0), (1, 1), (0, 2), (3, 0), (2, 0), (0, 3)]
    res = fuse_checked(pkg, hm, k=6, pairs=pairs, conn=8, init="k-means++", random_state=2, max_iter=10,
                       engine=engine)
    ov = res.region_overlaps
    assert np.array_equal(ov[ov[:, 0] == 0][:, 1:], ov[ov[:, 0] == 3][:, 1:])


@pytest.mark.gpu
def test_detrend_and_ground_level(pkg, engine):
    hm = stack(3, 90, 140, 4)
    fuse_checked(pkg, hm, k=7, conn=8, init="k-means++", random_state=2, max_iter=20, detrend=True,
                 ground_level=True, engine=engine)


@pytest.mark.gpu
def test_restarts_keep_the_returned_runs_overlaps(pkg, engine):
    hm = stack(3, 60, 130, 9)
    fuse_checked(pkg, hm, k=12, conn=8, init="k-means++", n_init=3, random_state=11, max_iter=15, engine=engine)


@pytest.mark.gpu
def test_restarts_return_the_best_run_not_the_last(engine, monkeypatch):
    """The last of three runs is cut to one iteration, so a better run comes before it: the rows
    returned are that run's, not the last run's, and match the region map returned with them."""
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
    pairs = [(0, 1), (2, 1)]
    rmap = np.empty(hm.shape, np.int32)
    best = api._run_kmeans(engine, n_clusters=12, init="k-means++", n_init=3, max_iter=15, tol=1e-4, random_state=11,
                           regions=8, region_map_out=rmap, region_overlaps=pairs)
    assert len(runs) == 3
    inertias = [r["inertia"] for r in runs]
    won = [i for i, r in enumerate(runs) if r["region_overlaps"] is best["region_overlaps"]]
    assert won and won[0] != 2 and inertias[won[0]] < inertias[2]
    assert best["region_overlaps"].tobytes() != runs[2]["region_overlaps"].tobytes()
    check_overlaps(best["region_overlaps"], rmap, pairs, best["regions"])


@pytest.mark.gpu
def test_relocation(engine):
    hm = stack(3, 80, 120, 10)
    init = seeds(hm, 8, 2)
    init[5] = [1e5, -1e5, 1e4]  # far outside the cloud: empty after the first E-step
    engine.unproject(hm)
    pairs = [(0, 1), (2, 1), (1, 1)]
    kw = dict(max_iter=30, tol=0.0, day_stats=True, transitions=pairs, regions=8)
    cmap = np.empty(hm.shape, np.uint8)
    rmap = np.empty(hm.shape, np.int32)
    r1 = engine.fit(init, cluster_map_out=cmap, region_map_out=rmap, region_overlaps=pairs, **kw)
    labels1 = r1["labels"].copy()
    r0 = engine.fit(init, **kw)
    assert r1["n_relocations"] >= 1 and "region_overlaps" not in r0
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    assert r1["inertia"] == r0["inertia"] and r1["n_iter"] == r0["n_iter"]
    for name in ("day_counts", "day_means", "transitions", "regions", "region_means"):
        assert r1[name].tobytes() == r0[name].tobytes()
    assert rmap.tobytes() == ref_region_map(cmap, 8).tobytes()
    check_overlaps(r1["region_overlaps"], rmap, pairs, r1["regions"], r1["transitions"])


@pytest.mark.gpu
def test_predict_on_a_second_stack(engine):
    hm = stack(2, 50, 140, 12)
    engine.unproject(hm)
    centers = engine.fit(seeds(hm, 9, 3), max_iter=10, regions=4, region_overlaps=[(0, 1)])["centers"]
    hm2 = stack(4, 30, 91, 13)
    engine.unproject(hm2)  # drops the overlaps of the fit
    with pytest.raises(C.MdkmError):
        engine._region_overlap_table()
    cmap = np.empty(hm2.shape, np.uint8)
    rmap = np.empty(hm2.shape, np.int32)
    pairs = [(0, 3), (3, 0), (1, 2)]
    out = engine.predict(centers, cluster_map_out=cmap, regions=8, region_map_out=rmap, region_overlaps=pairs)
    labels, inertia, table, rmeans, rows = out
    assert rmap.tobytes() == ref_region_map(cmap, 8).tobytes()
    check_overlaps(rows, rmap, pairs, table)


@pytest.mark.gpu
def test_overlaps_without_a_region_map(pkg, engine):
    """No region map bound: the rows come from the internal whole-stack map."""
    hm = stack(3, 60, 80, 15)
    kw = dict(n_clusters=5, init="k-means++", random_state=6, max_iter=10, engine=engine, region_connectivity=8)
    a = pkg.fuse_multiday_kmeans(hm, return_region_map=True, return_region_overlaps=True, **kw)
    b = pkg.fuse_multiday_kmeans(hm, return_region_overlaps=True, **kw)
    assert b.region_map is None and b.regions is not None
    assert a.region_overlaps.tobytes() == b.region_overlaps.tobytes()
    check_overlaps(b.region_overlaps, a.region_map, b.region_overlap_pairs, b.regions)


# ---------------------------------------------------------------------------------------
# GPU: errors and the lifecycle
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_errors(pkg, engine):
    ERR_STATE, ERR_INVALID = C.STATUS_BY_NAME["MDKM_ERR_STATE"], C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    bind = engine._lib.mdkm_bind_region_overlaps
    hm = stack(3, 30, 60, 17)
    init = seeds(hm, 5, 1)
    pr = np.array([[0, 1], [2, 0]], np.int32)
    fresh = pkg.Engine(0)
    try:  # no resident cloud; nothing computed yet
        assert bind(fresh._h, pr.ctypes.data, 2) == ERR_STATE
        with pytest.raises(C.MdkmError) as ei:
            fresh._region_overlap_table()
        assert ei.value.code == ERR_STATE
    finally:
        fresh.close()
    engine.set_points(UO.unproject_stack(hm).astype(np.float32))  # no raster
    assert bind(engine._h, pr.ctypes.data, 2) == ERR_STATE
    engine.unproject(hm)
    with pytest.raises(C.MdkmError) as ei:  # count / table before any computation
        engine._region_overlap_table()
    assert ei.value.code == ERR_STATE
    for bad, np_ in (([[0, 3]], 1), ([[-1, 0]], 1), ([[0, 1]], 0), ([[0, 1]], -2)):
        b = np.array(bad, np.int32)
        assert bind(engine._h, b.ctypes.data, np_) == ERR_INVALID
    many = np.zeros((8193, 2), np.int32)
    assert bind(engine._h, many.ctypes.data, 8193) == ERR_INVALID
    assert bind(engine._h, many.ctypes.data, 8192) == C.MDKM_OK
    assert bind(engine._h, None, 0) == C.MDKM_OK  # cleared
    r = engine.fit(init, max_iter=5, regions=4)
    assert "region_overlaps" not in r
    with pytest.raises(C.MdkmError):
        engine._region_overlap_table()
    # overlaps without regions: ValueError in Python, MDKM_ERR_STATE from the C fit / predict
    with pytest.raises(ValueError):
        engine.fit(init, max_iter=5, region_overlaps=[(0, 1)])
    for call in (lambda: engine.fit(init, max_iter=5), lambda: engine.predict(init)):
        assert bind(engine._h, pr.ctypes.data, 2) == C.MDKM_OK
        with pytest.raises(C.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_STATE
    r = engine.fit(init, max_iter=5)  # the binding was consumed by the refused call
    # a short table capacity
    r = engine.fit(init, max_iter=5, regions=4, region_overlaps=pr)
    M = r["region_overlaps"].shape[0]
    assert M > 0
    t = np.empty((M, 6), np.int64)
    assert engine._lib.mdkm_region_overlap_table(engine._h, t.ctypes.data, M - 1) == ERR_INVALID
    assert engine._lib.mdkm_region_overlap_table(engine._h, t.ctypes.data, M) == C.MDKM_OK
    assert t.tobytes() == r["region_overlaps"].tobytes()
    # a fit without regions keeps the rows; one with regions but without overlaps drops them
    engine.fit(init, max_iter=5)
    assert engine._region_overlap_table().tobytes() == r["region_overlaps"].tobytes()
    engine.fit(init, max_iter=5, regions=8)
    with pytest.raises(C.MdkmError) as ei:
        engine._region_overlap_table()
    assert ei.value.code == ERR_STATE
    # the binding is dropped by unproject
    assert bind(engine._h, pr.ctypes.data, 2) == C.MDKM_OK
    engine.unproject(hm)
    engine.fit(init, max_iter=5, regions=4)
    with pytest.raises(C.MdkmError):
        engine._region_overlap_table()


@pytest.mark.gpu
def test_a_refused_binding_leaves_none_behind(engine):
    hm = stack(2, 40, 60, 21)
    engine.unproject(hm)
    init = seeds(hm, 5, 1)
    with pytest.raises(C.MdkmError):  # day 2 does not exist: the overlaps are refused after the regions
        engine.fit(init, max_iter=5, day_stats=True, transitions=[(0, 1)], regions=4, region_overlaps=[(0, 2)])
    r = engine.fit(init, max_iter=5)
    assert "regions" not in r and "day_counts" not in r and "transitions" not in r
    for table in (engine._region_table, engine._region_overlap_table):
        with pytest.raises(C.MdkmError):
            table()
    with pytest.raises(ValueError):  # short region map: refused before the overlaps are bound
        engine.fit(init, max_iter=5, regions=4, region_map_out=np.empty(5, np.int32), region_overlaps=[(0, 1)])
    r = engine.fit(init, max_iter=5, regions=4)  # nothing left bound: regions alone, no overlaps
    assert "regions" in r and "region_overlaps" not in r
    with pytest.raises(C.MdkmError):
        engine._region_overlap_table()


@pytest.mark.gpu
def test_plugin_passes_the_option(pkg, monkeypatch):
    hm = stack(3, 64, 80, 13)
    seen = []
    to_layers = api.to_layers
    monkeypatch.setattr(api, "to_layers", lambda res: seen.append(res) or to_layers(res))
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_region_overlaps=[(2, 0)], return_region_map=True,
                                    init="k-means++", random_state=0, max_iter=10)
    layers = plug.run(hm)
    assert [t for _, _, t in layers] == ["points", "points", "labels"]
    (res,) = seen
    assert res.region_overlap_pairs.tolist() == [[2, 0]]
    check_overlaps(res.region_overlaps, res.region_map, [(2, 0)], res.regions)


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
              region_connectivity=8, return_region_overlaps=[(0, 1), (2, 0), (1, 1)])
    one = pkg.fuse_multiday_kmeans(hm, device=0, **kw)
    two = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], **kw)
    assert np.array_equal(one.labels, two.labels)
    assert two.region_overlaps.tobytes() == one.region_overlaps.tobytes()
    check_overlaps(one.region_overlaps, one.region_map, one.region_overlap_pairs, one.regions)


@pytest.mark.gpu
def test_pre_sharded_ranks_receive_the_same_rows(pkg):
    _two_gpus()
    from concurrent.futures import ThreadPoolExecutor

    hm = stack(3, 30, 70, 19)
    flat = hm.reshape(-1)
    cut = 30 * 70 + 517  # inside day 1
    init = seeds(hm, 6, 4)
    kw = dict(n_clusters=6, init=init, max_iter=10, return_region_map=True, return_region_overlaps=True)
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
        assert r.region_overlaps.tobytes() == one.region_overlaps.tobytes()
    check_overlaps(one.region_overlaps, one.region_map, one.region_overlap_pairs, one.regions)
