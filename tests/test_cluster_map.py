"""Per-day cluster maps on the input pixel grid (``return_cluster_map`` / ``cluster_map_out``):
written on the device by the final labelling pass, label + 1 at every pixel that produced a point
and 0 elsewhere.  Every GPU case checks the map against one built on the host from the oracle's
validity mask and the labels the same call returns, and that asking for a map changes nothing
else (labels, centroids, inertia, n_iter bit for bit)."""
import importlib

import numpy as np
import pytest

from oracle import unproject_oracle as UO

PKG = "3d-point-cloud-multiday-imagery_b200"
synth = importlib.import_module(PKG + ".synth")
api = importlib.import_module(PKG + ".api")
engine_mod = importlib.import_module(PKG + ".engine")
C = importlib.import_module(PKG + "._cabi")


def ref_map(valid, labels, k):
    """The map the labels describe: np.where order over the flattened validity mask."""
    ref = np.zeros(valid.size, dtype=np.uint8 if k <= 255 else np.uint16)
    ref[valid.ravel()] = labels + 1
    return ref


def check_map(cmap, ref):
    assert cmap.dtype == ref.dtype
    assert cmap.tobytes() == ref.tobytes()


def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter


def fuse_both(pkg, hm, masks=None, **kw):
    """The same call without and with a map; the two must agree on everything else."""
    plain = pkg.fuse_multiday_kmeans(hm, masks, **kw)
    with_map = pkg.fuse_multiday_kmeans(hm, masks, return_cluster_map=True, **kw)
    assert plain.cluster_map is None
    same_result(plain, with_map)
    return with_map


def stack(D, H, W, seed):
    return synth.make_stack(D, H, W, seed=seed, n_buildings=6).numpy()


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def _result(cmap=None):
    return api.FusionResult(labels=np.array([0, 1], dtype=np.int32), centroids=np.array([[1.0, 2, 3], [4, 5, 6]]),
                            fused_cloud=np.zeros((2, 3), dtype=np.float32), n_iter=3, inertia=1.0, n_points=2,
                            cluster_map=cmap)


def test_to_layers_appends_labels_layer_only_with_a_map():
    plain = api.to_layers(_result())
    assert [t for _, _, t in plain] == ["points", "points"]
    cmap = np.array([[[1, 0], [0, 2]]], dtype=np.uint8)
    layers = api.to_layers(_result(cmap), prefix="P")
    assert [t for _, _, t in layers] == ["points", "points", "labels"]
    assert layers[2][0] is cmap and layers[2][1]["name"] == "P Cluster Map"
    for (d0, p0, t0), (d1, p1, t1) in zip(plain, layers[:2]):
        assert t0 == t1 and np.array_equal(d0, d1) and p0.keys() == p1.keys()


def test_cluster_map_dtype():
    assert api.cluster_map_dtype(255) == np.uint8 and api.cluster_map_dtype(256) == np.uint16


def test_out_buffer_accepts_map_dtypes_and_rejects_copies():
    f = engine_mod._as_out_buffer
    for dt in (np.uint8, np.uint16):
        ptr, mem = f(np.zeros(12, dtype=dt), (np.uint8, np.uint16), 12, "m")
        assert mem == C.MEM_HOST and ptr
    with pytest.raises(ValueError, match="uint8 or uint16"):
        f(np.zeros(12, dtype=np.int32), (np.uint8, np.uint16), 12, "m")
    with pytest.raises(ValueError, match="hold 12"):
        f(np.zeros(11, dtype=np.uint8), (np.uint8, np.uint16), 12, "m")
    with pytest.raises(ValueError, match="contiguous"):
        f(np.zeros((4, 6), dtype=np.uint8)[:, ::2], (np.uint8, np.uint16), 12, "m")
    import torch

    f(torch.zeros(12, dtype=torch.uint16), (np.uint8, np.uint16), 12, "m")
    with pytest.raises(ValueError, match="uint8 or uint16"):
        f(torch.zeros(12, dtype=torch.int16), (np.uint8, np.uint16), 12, "m")
    with pytest.raises(ValueError, match="contiguous"):
        f(torch.zeros(4, 6, dtype=torch.uint8)[:, ::2], (np.uint8, np.uint16), 12, "m")


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_float32_stack(pkg, engine):
    hm = stack(3, 120, 200, 1)  # W not a multiple of 16
    P = UO.unproject_stack(hm)
    init = synth.init_from_points(P.astype(np.float32), 16, 0)
    r = fuse_both(pkg, hm, n_clusters=16, init=init, max_iter=20, tol=0.0, engine=engine)
    assert r.cluster_map.shape == hm.shape
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r.labels, 16))


@pytest.mark.gpu
def test_int16_disparity_with_masks(pkg, engine):
    hm = stack(3, 90, 160, 2)
    disp = np.where(np.isfinite(hm), np.round(-hm * 16.0), -32768).astype(np.int16)
    masks = np.random.RandomState(2).rand(*hm.shape) > 0.1
    r = fuse_both(pkg, disp, masks, n_clusters=8, init="k-means++", random_state=3, max_iter=30,
                  disparity_scale=-1.0 / 16.0, engine=engine)
    valid = UO.valid_mask(UO.height_from_disparity(disp), masks)
    check_map(r.cluster_map.ravel(), ref_map(valid, r.labels, 8))


@pytest.mark.gpu
def test_gtiff3_layout(pkg, engine):
    hm = stack(2, 64, 96, 3)
    rs = np.random.RandomState(3)
    px = np.zeros(hm.shape + (3,), dtype=np.float32)
    px[..., 0] = hm
    px[..., 1] = rs.rand(*hm.shape)
    px[..., 2] = rs.rand(*hm.shape) > 0.15
    r = fuse_both(pkg, px, n_clusters=6, init="k-means++", random_state=1, max_iter=20, raster_layout="gtiff3",
                  engine=engine)
    assert r.cluster_map.shape == hm.shape
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm, px[..., 2] != 0), r.labels, 6))


@pytest.mark.gpu
def test_detrend_and_ground_level(pkg, engine):
    hm = stack(3, 80, 144, 4)
    r = fuse_both(pkg, hm, n_clusters=10, init="k-means++", random_state=2, max_iter=25, detrend=True,
                  ground_level=True, engine=engine)
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r.labels, 10))


@pytest.mark.gpu
def test_narrow_rows(pkg, engine):
    hm = stack(3, 50, 20, 5)  # fewer than 32 pixels per row
    r = fuse_both(pkg, hm, n_clusters=5, init="k-means++", random_state=4, max_iter=20, engine=engine)
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r.labels, 5))


@pytest.mark.gpu
def test_k300_gives_uint16(pkg, engine):
    hm = stack(3, 120, 200, 6)
    r = fuse_both(pkg, hm, n_clusters=300, init="random", random_state=5, max_iter=5, engine=engine)
    assert r.cluster_map.dtype == np.uint16 and r.cluster_map.max() > 255
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r.labels, 300))


@pytest.mark.gpu
def test_empty_middle_day(pkg, engine):
    hm = stack(3, 60, 100, 7)
    hm[1] = np.nan
    r = fuse_both(pkg, hm, n_clusters=8, init="k-means++", random_state=6, max_iter=20, engine=engine)
    assert not r.cluster_map[1].any() and r.cluster_map[2].any()
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r.labels, 8))


@pytest.mark.gpu
def test_row_band_mid_day_across_a_day_boundary(pkg, engine):
    D, H, W = 3, 40, 50
    hm = stack(D, H, W, 8)
    b, e = H * W + 514, 2 * H * W + 611  # starts mid-day, off a 32-pixel boundary; ends a day later
    assert b % 32 and b % (H * W) and b // (H * W) != (e - 1) // (H * W)
    valid = UO.valid_mask(hm).ravel()
    P = UO.unproject_stack(hm)[(np.cumsum(valid) - 1)[b:e][valid[b:e]]]  # the band's points
    init = synth.init_from_points(P.astype(np.float32), 7, 1)
    kw = dict(n_clusters=7, init=init, max_iter=20, tol=0.0, engine=engine, stack_shape=(D, H, W), pix_begin=b)
    r = fuse_both(pkg, hm.ravel()[b:e], **kw)
    assert r.cluster_map.shape == (e - b,)
    ref_whole = np.zeros(D * H * W, dtype=np.uint8)
    ref_whole[b:e] = ref_map(valid[b:e], r.labels, 7)
    check_map(r.cluster_map, ref_whole[b:e])
    # Engine level, and a device output of the same range
    import torch

    engine.unproject(hm.ravel()[b:e], stack_shape=(D, H, W), pix_begin=b)
    out = torch.full((e - b,), 77, dtype=torch.uint8, device="cuda:0")
    f = engine.fit(init, max_iter=20, tol=0.0, cluster_map_out=out)
    assert np.array_equal(f["labels"], r.labels)
    check_map(out.cpu().numpy(), ref_whole[b:e])


@pytest.mark.gpu
def test_restarts_keep_the_best_runs_map(pkg, engine):
    hm = stack(3, 100, 160, 9)
    r = fuse_both(pkg, hm, n_clusters=12, init="k-means++", n_init=3, random_state=11, max_iter=15, engine=engine)
    check_map(r.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r.labels, 12))
    r16 = pkg.fuse_multiday_kmeans(hm, n_clusters=300, init="random", n_init=2, random_state=12, max_iter=3,
                                   engine=engine, return_cluster_map=True)
    check_map(r16.cluster_map.ravel(), ref_map(UO.valid_mask(hm), r16.labels, 300))


@pytest.mark.gpu
def test_relocation_on_a_raster_cloud(engine):
    hm = stack(3, 80, 120, 10)
    P = UO.unproject_stack(hm)
    init = synth.init_from_points(P.astype(np.float32), 8, 2)
    init[5] = [1e5, -1e5, 1e4]  # far outside the cloud: empty after the first E-step
    engine.unproject(hm)
    out = np.full(hm.size, 99, dtype=np.uint8)
    r1 = engine.fit(init, max_iter=30, tol=0.0, cluster_map_out=out)
    labels1 = r1["labels"].copy()
    r0 = engine.fit(init, max_iter=30, tol=0.0)
    assert r1["n_relocations"] >= 1
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    assert r1["inertia"] == r0["inertia"] and r1["n_iter"] == r0["n_iter"]
    check_map(out, ref_map(UO.valid_mask(hm), labels1, 8))


@pytest.mark.gpu
def test_predict_writes_a_map(engine):
    hm = stack(2, 70, 90, 11)
    P = UO.unproject_stack(hm)
    engine.unproject(hm)
    centers = engine.fit(synth.init_from_points(P.astype(np.float32), 9, 3), max_iter=10)["centers"]
    out = np.empty(hm.shape, dtype=np.uint8)
    labels, inertia = engine.predict(centers, cluster_map_out=out)
    labels = labels.copy()
    labels0, inertia0 = engine.predict(centers)
    assert np.array_equal(labels, labels0) and inertia == inertia0
    check_map(out.ravel(), ref_map(UO.valid_mask(hm), labels, 9))


@pytest.mark.gpu
def test_device_map_used_on_torch_stream_right_after_fit(engine):
    import torch

    hm = stack(3, 120, 200, 12)
    P = UO.unproject_stack(hm)
    init = synth.init_from_points(P.astype(np.float32), 16, 4)
    engine.unproject(hm)
    host = np.empty(hm.size, dtype=np.uint8)
    engine.fit(init, max_iter=20, cluster_map_out=host)
    dev = torch.empty(hm.size, dtype=torch.uint8, device="cuda:0")
    engine.fit(init, max_iter=20, cluster_map_out=dev)
    counts = torch.bincount(dev.long(), minlength=17)  # torch's stream, no explicit synchronisation
    assert np.array_equal(counts.cpu().numpy(), np.bincount(host, minlength=17))


@pytest.mark.gpu
def test_plugin_returns_a_labels_layer(pkg):
    hm = stack(2, 64, 80, 13)
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_cluster_map=True, init="k-means++", random_state=0,
                                    max_iter=10)
    layers = plug.run(hm)
    assert [t for _, _, t in layers] == ["points", "points", "labels"], layers[0][1].get("name")
    res = pkg.fuse_multiday_kmeans(hm, n_clusters=5, init="k-means++", random_state=0, max_iter=10,
                                   return_cluster_map=True)
    check_map(layers[2][0].ravel(), res.cluster_map.ravel())
    check_map(res.cluster_map.ravel(), ref_map(UO.valid_mask(hm), res.labels, 5))


@pytest.mark.gpu
def test_device_group_map_equals_one_device(pkg):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    hm = stack(3, 96, 160, 14)
    kw = dict(n_clusters=8, init="k-means++", random_state=7, max_iter=20, return_cluster_map=True)
    one = pkg.fuse_multiday_kmeans(hm, device=0, **kw)
    two = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], **kw)
    same_result(one, two)
    assert two.cluster_map.shape == hm.shape
    check_map(two.cluster_map, one.cluster_map)


@pytest.mark.gpu
def test_errors(engine):
    hm = stack(2, 40, 60, 15)
    P = UO.unproject_stack(hm)
    engine.set_points(P.astype(np.float32))
    with pytest.raises(C.MdkmError) as ei:
        engine.fit(synth.init_from_points(P.astype(np.float32), 4, 0), max_iter=5,
                   cluster_map_out=np.empty(hm.size, dtype=np.uint8))
    assert ei.value.code == C.STATUS_BY_NAME["MDKM_ERR_STATE"]
    engine.unproject(hm)
    init = synth.init_from_points(P.astype(np.float32), 256, 0)
    with pytest.raises(C.MdkmError) as ei:
        engine.fit(init, max_iter=2, cluster_map_out=np.empty(hm.size, dtype=np.uint8))
    assert ei.value.code == C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    ok = np.empty(hm.size, dtype=np.uint16)  # the failed call consumed its binding; uint16 holds k = 256
    r = engine.fit(init, max_iter=2, cluster_map_out=ok)
    check_map(ok, ref_map(UO.valid_mask(hm), r["labels"], 256))
    small = init[:4]
    with pytest.raises(ValueError, match="hold"):
        engine.fit(small, max_iter=2, cluster_map_out=np.empty(hm.size - 1, dtype=np.uint8))
    with pytest.raises(ValueError, match="uint8 or uint16"):
        engine.fit(small, max_iter=2, cluster_map_out=np.empty(hm.size, dtype=np.int32))
    with pytest.raises(ValueError, match="contiguous"):
        engine.fit(small, max_iter=2, cluster_map_out=np.empty(2 * hm.size, dtype=np.uint8)[::2])
