"""Per-day cluster composition (``return_day_stats`` / ``day_stats=True``): ``day_counts[d, j]``
points of day d with label j, and ``day_means[d, j]`` their mean (x, y, z) in the clustered frame,
accumulated by the final labelling pass from integer sums on the fixed-point frame.

Every GPU case checks the counts against a bincount of the labels the same call returns, and the
means against an exact host reference: bit for bit on dyadic stacks (int16 disparities with
``disparity_scale=-1/16``: every coordinate a multiple of 2^-4, so every sum is exact), within half
a grid step of the frame (``compute_frame`` restated as in ``test_kernel_edges.py``) elsewhere.
Each case also checks that asking for the statistics changes nothing else."""
import importlib
import math

import numpy as np
import pytest

from oracle import unproject_oracle as UO

PKG = "3d-point-cloud-multiday-imagery_b200"
synth = importlib.import_module(PKG + ".synth")
api = importlib.import_module(PKG + ".api")
C = importlib.import_module(PKG + "._cabi")

QUANT_BITS = 22  # common.cuh: |quantised coordinate| < 2^22


# ---------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------
def day_of_points(seg_offsets, day0=0):
    """Global day of every point from a cloud's segment offsets (one segment per day of its range)."""
    return day0 + np.repeat(np.arange(len(seg_offsets) - 1), np.diff(seg_offsets))


def ref_counts(day, labels, D, k):
    return np.bincount(day * k + labels, minlength=D * k).reshape(D, k).astype(np.int64)


def ref_means_dyadic(P, day, labels, D, k):
    """Exact means of points whose coordinates are multiples of 2^-4: the sums of 16 * x are
    integers below 2^53 (exact in FP64), so one division gives the correctly rounded mean."""
    P16 = np.asarray(P, dtype=np.float64) * 16.0
    assert np.array_equal(P16, np.rint(P16)), "not a dyadic cloud"
    key = day * k + labels
    cnt = np.bincount(key, minlength=D * k).astype(np.float64)
    out = np.full((D * k, 3), np.nan)
    nz = cnt > 0
    for d in range(3):
        s = np.bincount(key, weights=P16[:, d], minlength=D * k)
        assert np.all(np.abs(s) < 2.0 ** 53)
        out[nz, d] = s[nz] / (16.0 * cnt[nz])
    return out.reshape(D, k, 3)


def frame_exponents(P):
    """compute_frame (mdkm.cu), restated for clouds of extent of a unit or more: per dimension the
    exponent e of the fixed-point scale 2^e (integer origin, |q| < 2^22)."""
    P32 = np.asarray(P, dtype=np.float32)
    e = np.zeros(3)
    for d in range(3):
        lo, hi = float(P32[:, d].min()), float(P32[:, d].max())
        mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
        o = float(np.float32(float(np.rint(mid)) if abs(mid) > 0.25 * half else 0.0))
        assert half == 0 or abs(mid - o) <= half, "narrow cloud: use test_kernel_edges.frame_quantum"
        hr = max(abs(lo - o), abs(hi - o)) * (1.0 + 1e-6) + 1e-30
        e[d] = min(100, max(-100, math.floor(math.log2(((1 << QUANT_BITS) - 2) / hr))))
    return e


def check_means_near(P, day, labels, D, k, means):
    """Off the grid: every point moves by at most half a grid step, so the mean does too (plus
    FP64 rounding of the two sums)."""
    P = np.asarray(P, dtype=np.float64)
    key = day * k + labels
    cnt = np.bincount(key, minlength=D * k)
    m = means.reshape(D * k, 3)
    assert np.all(np.isnan(m[cnt == 0]))
    assert not np.any(np.isnan(m[cnt > 0]))
    half = 2.0 ** -(frame_exponents(P) + 1)
    for d in range(3):
        ref = np.bincount(key, weights=P[:, d], minlength=D * k)[cnt > 0] / cnt[cnt > 0]
        tol = half[d] * 1.001 + 1e-13 * np.abs(ref)
        assert np.all(np.abs(m[cnt > 0, d] - ref) <= tol), np.max(np.abs(m[cnt > 0, d] - ref) - tol)


def check_exact(P, day, labels, D, k, counts, means):
    assert counts.dtype == np.int64 and counts.shape == (D, k)
    assert means.dtype == np.float64 and means.shape == (D, k, 3)
    np.testing.assert_array_equal(counts, ref_counts(day, labels, D, k))
    ref = ref_means_dyadic(P, day, labels, D, k)
    assert ref.tobytes() == means.tobytes() or np.array_equal(ref, means, equal_nan=True)
    assert np.array_equal(np.isnan(ref), np.isnan(means))


def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter and a.n_refined == b.n_refined
    if a.cluster_map is not None or b.cluster_map is not None:
        assert a.cluster_map.tobytes() == b.cluster_map.tobytes()


def fuse_both(pkg, hm, masks=None, **kw):
    """The same call without and with statistics (and with a cluster map in both): everything
    else bitwise equal."""
    plain = pkg.fuse_multiday_kmeans(hm, masks, return_cluster_map=True, **kw)
    with_stats = pkg.fuse_multiday_kmeans(hm, masks, return_cluster_map=True, return_day_stats=True, **kw)
    assert plain.day_counts is None and plain.day_means is None
    same_result(plain, with_stats)
    return with_stats


def dyadic_stack(D, H, W, seed, valid=0.9):
    """int16 disparities (x, y integers, z a multiple of 1/16) and a random validity mask."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = 16 * 20.0 * (np.sin(xx / 7.0) * np.cos(yy / 5.0))
    disp = (base[None] + rs.randint(-48, 49, size=(D, H, W))).astype(np.int16)
    mask = rs.rand(D, H, W) < valid
    return disp, mask


def dyadic_points(disp, mask):
    return UO.unproject_stack(UO.height_from_disparity(disp), mask)


def seeds(P, k, seed):
    return synth.init_from_points(np.asarray(P, dtype=np.float32), k, seed)


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def test_fusion_result_has_no_stats_by_default():
    r = api.FusionResult(labels=np.zeros(2, dtype=np.int32), centroids=np.zeros((1, 3)), fused_cloud=None,
                         n_iter=1, inertia=0.0, n_points=2)
    assert r.day_counts is None and r.day_means is None


def test_references_on_a_small_cloud():
    P = np.array([[0.0, 0, 0.0625], [2.0, 0, 0], [1.0, 1, 0], [5.0, 5, 5]])
    day = day_of_points(np.array([0, 2, 2, 4]), day0=1)
    assert day.tolist() == [1, 1, 3, 3]
    labels = np.array([0, 0, 1, 1])
    counts = ref_counts(day, labels, 4, 2)
    assert counts.tolist() == [[0, 0], [2, 0], [0, 0], [0, 2]]
    m = ref_means_dyadic(P, day, labels, 4, 2)
    assert m[1, 0].tolist() == [1.0, 0.0, 0.03125] and m[3, 1].tolist() == [3.0, 3.0, 2.5]
    assert np.isnan(m[0]).all() and np.isnan(m[1, 1]).all()


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 16, 17, 64, 65, 129, 257, 1024, 2048])
def test_dyadic_every_final_variant(pkg, engine, k):
    """Every final-pass variant (k <= 32, <= 64, run-time loop, bucketed) on a dyadic stack whose
    width is not a multiple of 128 (split-row groups) and whose middle day is empty."""
    D, H, W = 3, 40, 200
    disp, mask = dyadic_stack(D, H, W, k)
    mask[1] = False
    P = dyadic_points(disp, mask)
    r = fuse_both(pkg, disp, mask, n_clusters=k, init=seeds(P, k, 1), max_iter=4, tol=0.0,
                  disparity_scale=-1.0 / 16.0, engine=engine)
    day = day_of_points(r.extra["segment_offsets"])
    check_exact(P, day, r.labels, D, k, r.day_counts, r.day_means)
    assert not r.day_counts[1].any() and np.isnan(r.day_means[1]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 10])
def test_dyadic_days(pkg, engine, D):
    H, W = 24, 150
    disp, mask = dyadic_stack(D, H, W, 20 + D)
    if D > 1:
        mask[3] = False
        mask[6] = False
        mask[6, 11, 77] = True  # a day with one valid pixel
    P = dyadic_points(disp, mask)
    r = fuse_both(pkg, disp, mask, n_clusters=16, init="k-means++", random_state=D, max_iter=20,
                  disparity_scale=-1.0 / 16.0, engine=engine)
    day = day_of_points(r.extra["segment_offsets"])
    check_exact(P, day, r.labels, D, 16, r.day_counts, r.day_means)
    if D > 1:
        assert r.day_counts[6].sum() == 1 and not r.day_counts[3].any()
        j = int(np.argmax(r.day_counts[6]))
        assert r.day_means[6, j].tolist() == P[day == 6][0].tolist()


@pytest.mark.gpu
def test_float32_stack_off_grid(pkg, engine):
    hm = synth.make_stack(3, 100, 160, seed=3, n_buildings=6).numpy()
    P = UO.unproject_stack(hm)
    r = fuse_both(pkg, hm, n_clusters=16, init=seeds(P, 16, 0), max_iter=20, tol=0.0, engine=engine)
    day = day_of_points(r.extra["segment_offsets"])
    np.testing.assert_array_equal(r.day_counts, ref_counts(day, r.labels, 3, 16))
    check_means_near(P, day, r.labels, 3, 16, r.day_means)


@pytest.mark.gpu
def test_detrend_and_ground_level_use_the_clustered_cloud(pkg, engine):
    hm = synth.make_stack(3, 80, 144, seed=4, n_buildings=6).numpy()
    r = fuse_both(pkg, hm, n_clusters=10, init="k-means++", random_state=2, max_iter=25, detrend=True,
                  ground_level=True, engine=engine)
    cloud = r.fused_cloud[:, ::-1].astype(np.float64)  # napari (z, y, x) -> (x, y, z)
    day = day_of_points(r.extra["segment_offsets"])
    np.testing.assert_array_equal(r.day_counts, ref_counts(day, r.labels, 3, 10))
    check_means_near(cloud, day, r.labels, 3, 10, r.day_means)


@pytest.mark.gpu
def test_relocation_fit(engine, golden):
    g = golden("kmeans_relocate.npz")
    engine.set_points(g["X"])
    r1 = engine.fit(g["init"], max_iter=100, tol=0.0, day_stats=True)
    labels1 = r1["labels"].copy()
    r0 = engine.fit(g["init"], max_iter=100, tol=0.0)
    assert r1["n_relocations"] >= 1
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    assert r1["inertia"] == r0["inertia"] and r1["n_iter"] == r0["n_iter"] and r1["n_refined"] == r0["n_refined"]
    k = g["init"].shape[0]
    day = np.zeros(labels1.shape[0], dtype=np.int64)
    np.testing.assert_array_equal(r1["day_counts"], ref_counts(day, labels1, 1, k))
    check_means_near(g["X"], day, labels1, 1, k, r1["day_means"])


@pytest.mark.gpu
def test_restarts_keep_the_returned_runs_stats(pkg, engine):
    disp, mask = dyadic_stack(3, 60, 130, 9)
    P = dyadic_points(disp, mask)
    r = fuse_both(pkg, disp, mask, n_clusters=12, init="k-means++", n_init=3, random_state=11, max_iter=15,
                  disparity_scale=-1.0 / 16.0, engine=engine)
    check_exact(P, day_of_points(r.extra["segment_offsets"]), r.labels, 3, 12, r.day_counts, r.day_means)


@pytest.mark.gpu
def test_predict_on_a_second_stack(engine):
    disp, mask = dyadic_stack(2, 50, 140, 12)
    P = dyadic_points(disp, mask)
    engine.unproject(disp, mask, disparity_scale=-1.0 / 16.0)
    centers = engine.fit(seeds(P, 9, 3), max_iter=10)["centers"]
    disp2, mask2 = dyadic_stack(4, 30, 90, 13)
    P2 = dyadic_points(disp2, mask2)
    engine.unproject(disp2, mask2, disparity_scale=-1.0 / 16.0)
    assert engine.n_days == 4
    labels, inertia, counts, means = engine.predict(centers, day_stats=True)
    labels = labels.copy()
    labels0, inertia0 = engine.predict(centers)
    assert np.array_equal(labels, labels0) and inertia == inertia0
    check_exact(P2, day_of_points(engine.segment_offsets), labels, 4, 9, counts, means)


@pytest.mark.gpu
def test_set_points_cloud_has_one_day(engine):
    disp, mask = dyadic_stack(2, 40, 100, 14)
    P = dyadic_points(disp, mask)
    rs = np.random.RandomState(0)
    P = P[rs.permutation(P.shape[0])]  # not in raster order
    engine.set_points(P.astype(np.float32))
    assert engine.n_days == 1
    init = seeds(P, 7, 2)
    r = engine.fit(init, max_iter=20, tol=0.0, day_stats=True)
    labels = r["labels"].copy()
    r0 = engine.fit(init, max_iter=20, tol=0.0)
    assert np.array_equal(labels, r0["labels"]) and r["inertia"] == r0["inertia"]
    check_exact(P, np.zeros(P.shape[0], dtype=np.int64), labels, 1, 7, r["day_counts"], r["day_means"])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [64, 2048])
def test_many_tiny_days_global_slots(engine, k):
    """1100 days of 4 x 8 pixels: D * k slots far beyond shared memory (accumulated in global)."""
    D, H, W = 1100, 4, 8
    disp, mask = dyadic_stack(D, H, W, 15, valid=0.95)
    mask[500] = False
    P = dyadic_points(disp, mask)
    engine.unproject(disp, mask, disparity_scale=-1.0 / 16.0)
    centers = seeds(P, k, 4)
    labels, inertia, counts, means = engine.predict(centers, day_stats=True)
    labels = labels.copy()
    labels0, inertia0 = engine.predict(centers)
    assert np.array_equal(labels, labels0) and inertia == inertia0
    check_exact(P, day_of_points(engine.segment_offsets), labels, D, k, counts, means)
    r = engine.fit(centers, max_iter=3, tol=0.0, day_stats=True)
    check_exact(P, day_of_points(engine.segment_offsets), r["labels"], D, k, r["day_counts"], r["day_means"])


@pytest.mark.gpu
def test_pre_sharded_slices_across_a_day_boundary(pkg, engine):
    D, H, W = 4, 30, 70
    disp, mask = dyadic_stack(D, H, W, 16)
    P = dyadic_points(disp, mask)
    flat, mflat = disp.ravel(), mask.ravel()
    b, m, e = H * W + 517, 2 * H * W + 611, D * H * W  # slice [b, m) spans days 1-2, [m, e) days 2-3
    init = seeds(P, 8, 5)
    # a fit on one slice: global rows, zeros outside its days
    r = fuse_both(pkg, flat[b:m], mflat[b:m], n_clusters=8, init=init, max_iter=10, tol=0.0,
                  disparity_scale=-1.0 / 16.0, engine=engine, stack_shape=(D, H, W), pix_begin=b)
    valid = mflat & (np.abs(UO.height_from_disparity(flat)) <= 144.0)
    Pb = P[(np.cumsum(valid) - 1)[b:m][valid[b:m]]]
    day = day_of_points(r.extra["segment_offsets"], day0=b // (H * W))
    check_exact(Pb, day, r.labels, D, 8, r.day_counts, r.day_means)
    assert not r.day_counts[0].any() and not r.day_counts[3].any()
    # predict: the whole stack's counts are the sums of two adjacent slices' counts
    engine.unproject(disp, mask, disparity_scale=-1.0 / 16.0)
    _, _, whole, _ = engine.predict(init, want_labels=False, day_stats=True)
    parts = []
    for lo, hi in ((0, m), (m, e)):
        engine.unproject(flat[lo:hi], mflat[lo:hi], disparity_scale=-1.0 / 16.0, stack_shape=(D, H, W), pix_begin=lo)
        parts.append(engine.predict(init, want_labels=False, day_stats=True)[2])
    np.testing.assert_array_equal(parts[0] + parts[1], whole)
    assert not parts[1][:2].any() and not parts[0][3].any()


@pytest.mark.gpu
def test_errors(pkg, engine):
    fresh = pkg.Engine(0)
    try:
        cnt = np.empty((1, 4), dtype=np.int64)
        means = np.empty((1, 4, 3))
        rc = fresh._lib.mdkm_bind_day_stats(fresh._h, cnt.ctypes.data, means.ctypes.data, 1, 4)
        assert rc == C.STATUS_BY_NAME["MDKM_ERR_STATE"]
    finally:
        fresh.close()
    disp, mask = dyadic_stack(3, 30, 60, 17)
    P = dyadic_points(disp, mask)
    engine.unproject(disp, mask, disparity_scale=-1.0 / 16.0)
    cnt = np.empty((3, 4), dtype=np.int64)
    means = np.empty((3, 4, 3))
    for n_days in (1, 4):
        rc = engine._lib.mdkm_bind_day_stats(engine._h, cnt.ctypes.data, means.ctypes.data, n_days, 4)
        assert rc == C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    init = seeds(P, 5, 1)
    assert engine._lib.mdkm_bind_day_stats(engine._h, cnt.ctypes.data, means.ctypes.data, 3, 4) == C.MDKM_OK
    with pytest.raises(C.MdkmError) as ei:
        engine.fit(init, max_iter=5)  # k = 5 > k_capacity = 4
    assert ei.value.code == C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    assert engine._lib.mdkm_bind_day_stats(engine._h, cnt.ctypes.data, means.ctypes.data, 3, 4) == C.MDKM_OK
    with pytest.raises(C.MdkmError) as ei:
        engine.predict(init)
    assert ei.value.code == C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    # the failed calls consumed their bindings; the handle still works
    r = engine.fit(init, max_iter=5, day_stats=True)
    check_exact(P, day_of_points(engine.segment_offsets), r["labels"], 3, 5, r["day_counts"], r["day_means"])
    r0 = engine.fit(init, max_iter=5)
    assert r0["inertia"] == r["inertia"]


@pytest.mark.gpu
def test_plugin_passes_the_option(pkg):
    hm = synth.make_stack(2, 64, 80, seed=13, n_buildings=6).numpy()
    kw = dict(init="k-means++", random_state=0, max_iter=10)
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_day_stats=True, **kw)
    assert [t for _, _, t in plug.run(hm)] == ["points", "points"]
    res = pkg.fuse_multiday_kmeans(hm, n_clusters=5, return_day_stats=True, **kw)
    np.testing.assert_array_equal(res.day_counts, ref_counts(day_of_points(res.extra["segment_offsets"]),
                                                             res.labels, 2, 5))


@pytest.mark.gpu
def test_device_group_stats_equal_one_device(pkg):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    disp, mask = dyadic_stack(3, 50, 130, 18)
    kw = dict(n_clusters=8, init="k-means++", random_state=7, max_iter=20, return_day_stats=True,
              disparity_scale=-1.0 / 16.0)
    one = pkg.fuse_multiday_kmeans(disp, mask, device=0, **kw)
    two = pkg.fuse_multiday_kmeans(disp, mask, devices=[0, 1], **kw)
    same_result(one, two)
    assert two.day_counts.tobytes() == one.day_counts.tobytes()
    assert two.day_means.tobytes() == one.day_means.tobytes()
