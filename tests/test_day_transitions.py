"""From-to (transition) counts of day pairs (``return_transitions`` / ``transitions=``):
``T[p, s, t]`` pixels with state s on day a and t on day b of pair p = (a, b), where a pixel's state
is ``label + 1`` when it produced a point that day and 0 when it did not -- the cluster map's value.

Every GPU case compares T bit for bit with the bincount of the oracle
(``np.bincount(map[a] * (k+1) + map[b])``), on the map the same call returns or on one built from
the oracle's validity mask and the returned labels; checks the marginals against ``day_counts``;
and checks that asking for transitions changes nothing else (labels, centroids, inertia, n_iter,
n_refined, cluster map, day statistics bit for bit).

The kernel keeps the bins of a pair in a copy per warp, one copy per CTA, or global memory,
whichever is the first that does not cost a resident CTA.  At 64 registers (4 CTAs of 256
threads per SM) and 228 KB of shared memory per SM (1 KB reserved per CTA) that is per warp up to
k = 41, per CTA up to k = 118, global above: the k lists below sit on both sides of each switch."""
import importlib

import numpy as np
import pytest

from oracle import unproject_oracle as UO

PKG = "3d-point-cloud-multiday-imagery_b200"
synth = importlib.import_module(PKG + ".synth")
api = importlib.import_module(PKG + ".api")
C = importlib.import_module(PKG + "._cabi")


# ---------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------
def ref_transitions(cmap, pairs, k):
    """The oracle: one bincount per pair over the [D, H*W] map."""
    m = np.asarray(cmap).reshape(np.asarray(cmap).shape[0], -1).astype(np.int64)
    k1 = k + 1
    return np.stack([np.bincount(m[a] * k1 + m[b], minlength=k1 * k1).reshape(k1, k1) for a, b in pairs])


def ref_map(valid, labels, k):
    """The map the labels describe: np.where order over the flattened validity mask."""
    ref = np.zeros(valid.size, dtype=np.uint8 if k <= 255 else np.uint16)
    ref[valid.ravel()] = labels + 1
    return ref.reshape(valid.shape)


def check_transitions(T, cmap, pairs, k, day_counts=None):
    pairs = np.asarray(pairs)
    assert T.dtype == np.int64 and T.shape == (pairs.shape[0], k + 1, k + 1)
    assert T.tobytes() == ref_transitions(cmap, pairs, k).tobytes()
    if day_counts is not None:
        for p, (a, b) in enumerate(pairs):
            np.testing.assert_array_equal(T[p].sum(1)[1:], day_counts[a])
            np.testing.assert_array_equal(T[p].sum(0)[1:], day_counts[b])


def same_result(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert a.centroids.tobytes() == b.centroids.tobytes()
    assert a.inertia == b.inertia and a.n_iter == b.n_iter and a.n_refined == b.n_refined
    for name in ("cluster_map", "day_counts", "day_means"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None)
        if x is not None:
            assert x.tobytes() == y.tobytes()


def fuse_checked(pkg, hm, pairs, *, k, with_map=True, **kw):
    """The call without and with transitions (both with day statistics, and with a cluster map or
    without one): everything else bitwise equal, T equal to the oracle's on the returned map (or the
    map of the oracle's validity mask and the returned labels), marginals equal to day_counts."""
    plain = pkg.fuse_multiday_kmeans(hm, n_clusters=k, return_cluster_map=with_map, return_day_stats=True, **kw)
    res = pkg.fuse_multiday_kmeans(hm, n_clusters=k, return_cluster_map=with_map, return_day_stats=True,
                                   return_transitions=pairs, **kw)
    assert plain.transitions is None and plain.transition_pairs is None
    same_result(plain, res)
    cmap = res.cluster_map if with_map else ref_map(UO.valid_mask(hm), res.labels, k)
    if with_map:
        assert cmap.tobytes() == ref_map(UO.valid_mask(hm), res.labels, k).tobytes()
    check_transitions(res.transitions, cmap.reshape(hm.shape), res.transition_pairs, k, res.day_counts)
    return res


def stack(D, H, W, seed):
    return synth.make_stack(D, H, W, seed=seed, n_buildings=6).numpy()


def seeds(hm, k, seed):
    return synth.init_from_points(UO.unproject_stack(hm).astype(np.float32), k, seed)


# ---------------------------------------------------------------------------------------
# host only
# ---------------------------------------------------------------------------------------
def test_pairs_true_means_consecutive_days():
    assert api.transition_pairs(True, 4).tolist() == [[0, 1], [1, 2], [2, 3]]
    assert api.transition_pairs(np.True_, 2).tolist() == [[0, 1]]
    assert api.transition_pairs(True, 2).dtype == np.int64


def test_pairs_explicit_kept_as_given():
    p = api.transition_pairs([(3, 0), (1, 1), (0, 2), (0, 2)], 4)
    assert p.tolist() == [[3, 0], [1, 1], [0, 2], [0, 2]] and p.dtype == np.int64
    assert api.transition_pairs(np.array([[0, 0]], dtype=np.int32), 1).tolist() == [[0, 0]]


@pytest.mark.parametrize("spec, n_days", [([(0, 3)], 3), ([(-1, 0)], 3), ([(0, 1), (2, 5)], 3), (True, 1),
                                          ([], 3), ([0, 1], 3), ([(0.0, 1.0)], 3), (False, 3)])
def test_pairs_rejected(spec, n_days):
    with pytest.raises(ValueError):
        api.transition_pairs(spec, n_days)


def test_out_of_range_day_raises_before_any_gpu_work(pkg):
    class NoEngine:  # any use of the engine would raise AttributeError instead
        pass

    with pytest.raises(ValueError):
        pkg.fuse_multiday_kmeans(np.zeros((2, 4, 4), dtype=np.float32), return_transitions=[(0, 2)],
                                 engine=NoEngine())
    with pytest.raises(ValueError):
        pkg.fuse_multiday_kmeans(np.zeros((2, 4, 4), dtype=np.float32), return_transitions=[(0, 4)],
                                 engine=NoEngine(), stack_shape=(4, 2, 4))


def test_reference_on_a_small_map():
    m = np.array([[[0, 1], [2, 2]], [[1, 1], [0, 2]]], dtype=np.uint8)
    T = ref_transitions(m, [(0, 1), (1, 0)], 2)
    assert T[0].tolist() == [[0, 1, 0], [0, 1, 0], [1, 0, 1]]
    assert np.array_equal(T[1], T[0].T)


def test_fusion_result_has_no_transitions_by_default():
    r = api.FusionResult(labels=np.zeros(2, dtype=np.int32), centroids=np.zeros((1, 3)), fused_cloud=None,
                         n_iter=1, inertia=0.0, n_points=2)
    assert r.transitions is None and r.transition_pairs is None


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
PAIRS3 = [(0, 1), (1, 2), (0, 2), (2, 0), (1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 16, 41, 42, 118, 119, 255, 256, 1024, 2048])
def test_every_bin_variant(pkg, engine, k):
    """Per-warp / per-CTA / global bins and uint8 / uint16 maps, on a stack whose H*W (25 * 53) is
    odd, so that every day starts at a different offset from 16-byte alignment, with an empty
    middle day; pairs forwards, backwards, skipping a day and a == b."""
    hm = stack(3, 25, 53, k)
    hm[1] = np.nan
    fuse_checked(pkg, hm, PAIRS3, k=k, init=seeds(hm, k, 1), max_iter=4, tol=0.0, engine=engine)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 2, 3, 10])
def test_days_without_a_bound_map(pkg, engine, D):
    """Consecutive pairs (True) and no cluster map asked for: the final pass writes an internal one.
    Ten days include an empty day and a day with one valid pixel."""
    hm = stack(D, 30, 41, 30 + D)
    if D == 10:
        hm[3] = np.nan
        one = hm[6, 11, 17]
        hm[6] = np.nan
        hm[6, 11, 17] = one
    r = fuse_checked(pkg, hm, [(0, 0)] if D == 1 else True, k=9, with_map=False, init="k-means++", random_state=D,
                     max_iter=20, engine=engine)
    if D == 10:
        assert r.transitions[2].sum(0)[1:].sum() == 0 and r.transitions[5].sum(0)[1:].sum() == 1
    assert r.transition_pairs.shape == (max(D - 1, 1), 2)


@pytest.mark.gpu
def test_bound_host_device_and_no_map_agree(engine):
    import torch

    hm = stack(4, 37, 70, 5)
    init = seeds(hm, 20, 2)
    pairs = [(0, 3), (3, 1), (2, 2), (1, 2)]
    engine.unproject(hm)
    host = np.full(hm.shape, 99, dtype=np.uint8)
    r_host = engine.fit(init, max_iter=15, cluster_map_out=host, day_stats=True, transitions=pairs)
    labels = r_host["labels"].copy()
    dev = torch.empty(hm.size, dtype=torch.uint16, device="cuda:0")  # a 16-bit map for k <= 255
    r_dev = engine.fit(init, max_iter=15, cluster_map_out=dev, transitions=pairs)
    torch.cuda.synchronize()
    r_none = engine.fit(init, max_iter=15, transitions=pairs)
    r0 = engine.fit(init, max_iter=15)
    for r in (r_dev, r_none, r0):
        assert np.array_equal(r["labels"], labels) and r["centers"].tobytes() == r_host["centers"].tobytes()
        assert r["inertia"] == r_host["inertia"] and r["n_iter"] == r_host["n_iter"]
    assert host.tobytes() == ref_map(UO.valid_mask(hm), labels, 20).tobytes()
    assert np.array_equal(dev.view(torch.int16).cpu().numpy().view(np.uint16).reshape(hm.shape), host)
    check_transitions(r_host["transitions"], host, pairs, 20, r_host["day_counts"])
    assert r_dev["transitions"].tobytes() == r_host["transitions"].tobytes()
    assert r_none["transitions"].tobytes() == r_host["transitions"].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [16, 64, 1024])
def test_one_label_everywhere(engine, k):
    """Every valid pixel in one cluster (the other centroids far away): worst contention, every lane
    of every warp on the same bin or two."""
    rs = np.random.RandomState(k)
    hm = (10.0 + rs.rand(3, 256, 520)).astype(np.float32)
    hm[1, :, :100] = np.nan
    engine.unproject(hm)
    c = np.full((k, 3), 1e6)
    c[k // 2] = [260.0, 128.0, 10.5]
    labels, inertia, T = engine.predict(c, transitions=[(0, 1), (1, 2), (2, 0)])
    assert (labels == k // 2).all()
    labels0, inertia0 = engine.predict(c)
    assert inertia == inertia0
    check_transitions(T, ref_map(UO.valid_mask(hm), labels, k), [(0, 1), (1, 2), (2, 0)], k)
    assert T[0, k // 2 + 1, k // 2 + 1] == 256 * 420 and T[0, k // 2 + 1, 0] == 256 * 100


@pytest.mark.gpu
@pytest.mark.parametrize("k", [16, 100, 1024])
def test_random_labels(engine, k):
    """Noise heights and random centroids: nearly every pixel its own key within a lane."""
    rs = np.random.RandomState(100 + k)
    hm = (rs.rand(3, 96, 133) * 100.0).astype(np.float32)
    hm[rs.rand(*hm.shape) < 0.2] = np.nan
    engine.unproject(hm)
    c = np.stack([rs.rand(k) * 133, rs.rand(k) * 96, rs.rand(k) * 100], axis=1)
    pairs = [(0, 1), (2, 1), (0, 0)]
    labels, inertia, counts, means, T = engine.predict(c, day_stats=True, transitions=pairs)
    labels = labels.copy()
    assert len(np.unique(labels)) > min(k // 2, 50)
    check_transitions(T, ref_map(UO.valid_mask(hm), labels, k), pairs, k, counts)


@pytest.mark.gpu
def test_restarts_keep_the_returned_runs_transitions(pkg, engine):
    hm = stack(3, 60, 130, 9)
    fuse_checked(pkg, hm, True, k=12, init="k-means++", n_init=3, random_state=11, max_iter=15, engine=engine)


@pytest.mark.gpu
def test_relocation(engine):
    hm = stack(3, 80, 120, 10)
    init = seeds(hm, 8, 2)
    init[5] = [1e5, -1e5, 1e4]  # far outside the cloud: empty after the first E-step
    engine.unproject(hm)
    r1 = engine.fit(init, max_iter=30, tol=0.0, day_stats=True, transitions=[(0, 1), (1, 2)])
    labels1 = r1["labels"].copy()
    r0 = engine.fit(init, max_iter=30, tol=0.0, day_stats=True)
    assert r1["n_relocations"] >= 1
    assert np.array_equal(labels1, r0["labels"]) and r1["centers"].tobytes() == r0["centers"].tobytes()
    assert r1["inertia"] == r0["inertia"] and r1["n_iter"] == r0["n_iter"] and r1["n_refined"] == r0["n_refined"]
    assert r1["day_counts"].tobytes() == r0["day_counts"].tobytes()
    check_transitions(r1["transitions"], ref_map(UO.valid_mask(hm), labels1, 8), [(0, 1), (1, 2)], 8,
                      r1["day_counts"])


@pytest.mark.gpu
def test_predict_on_a_second_stack(engine):
    hm = stack(2, 50, 140, 12)
    engine.unproject(hm)
    centers = engine.fit(seeds(hm, 9, 3), max_iter=10)["centers"]
    hm2 = stack(4, 30, 91, 13)
    engine.unproject(hm2)
    pairs = [(0, 3), (1, 2), (3, 3)]
    out = np.empty(hm2.shape, dtype=np.uint8)
    labels, inertia, counts, means, T = engine.predict(centers, cluster_map_out=out, day_stats=True, transitions=pairs)
    labels = labels.copy()
    labels0, inertia0 = engine.predict(centers)
    assert np.array_equal(labels, labels0) and inertia == inertia0
    check_transitions(T, out, pairs, 9, counts)


@pytest.mark.gpu
def test_errors(pkg, engine):
    ERR_STATE, ERR_INVALID = C.STATUS_BY_NAME["MDKM_ERR_STATE"], C.STATUS_BY_NAME["MDKM_ERR_INVALID"]
    bind = engine._lib.mdkm_bind_day_transitions
    pairs = np.array([[0, 1]], dtype=np.int32)
    out = np.empty(1 << 16, dtype=np.int64)
    fresh = pkg.Engine(0)
    try:  # no resident cloud
        assert bind(fresh._h, pairs.ctypes.data, 1, out.ctypes.data, 4) == ERR_STATE
    finally:
        fresh.close()
    hm = stack(3, 30, 60, 17)
    init = seeds(hm, 5, 1)
    engine.set_points(UO.unproject_stack(hm).astype(np.float32))  # no raster
    assert bind(engine._h, pairs.ctypes.data, 1, out.ctypes.data, 4) == ERR_STATE
    engine.unproject(hm)
    for bad in ([[0, 3]], [[-1, 0]], [[0, 1], [2, 3]]):
        p = np.array(bad, dtype=np.int32)
        assert bind(engine._h, p.ctypes.data, len(bad), out.ctypes.data, 4) == ERR_INVALID
    assert bind(engine._h, pairs.ctypes.data, 0, out.ctypes.data, 4) == ERR_INVALID
    assert bind(engine._h, None, 1, out.ctypes.data, 4) == ERR_INVALID
    assert bind(engine._h, pairs.ctypes.data, 1, out.ctypes.data, 0) == ERR_INVALID
    assert bind(engine._h, pairs.ctypes.data, 1, out.ctypes.data, 46340) == ERR_INVALID  # 46341^2 >= 2^31
    assert bind(engine._h, pairs.ctypes.data, 1, out.ctypes.data, 46339) == C.MDKM_OK   # 46340^2 < 2^31
    assert bind(engine._h, pairs.ctypes.data, 2, out.ctypes.data, 32767) == ERR_INVALID  # 2 * 2^30
    # k > k_capacity: the fit / predict fails before any work, and consumes the binding
    for call in (lambda: engine.fit(init, max_iter=5), lambda: engine.predict(init)):
        assert bind(engine._h, pairs.ctypes.data, 1, out.ctypes.data, 4) == C.MDKM_OK
        with pytest.raises(C.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_INVALID
    r = engine.fit(init, max_iter=5, transitions=[(0, 1)])
    check_transitions(r["transitions"], ref_map(UO.valid_mask(hm), r["labels"], 5), [(0, 1)], 5)
    # one handle without a communicator holding part of the stack: ERR_STATE, and the handle still works
    flat = hm.reshape(-1)
    HW = 30 * 60
    engine.unproject(flat[HW + 100:2 * HW + 50], stack_shape=hm.shape, pix_begin=HW + 100)
    for call in (lambda: engine.fit(init, max_iter=5, transitions=[(1, 2)]),
                 lambda: engine.predict(init, transitions=[(1, 2)])):
        with pytest.raises(C.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_STATE
    with pytest.raises(C.MdkmError) as ei:
        pkg.fuse_multiday_kmeans(flat[:HW + 7], n_clusters=3, engine=engine, stack_shape=hm.shape,
                                 return_transitions=True)
    assert ei.value.code == ERR_STATE
    engine.predict(init)
    # the bindings are dropped by unproject / set_points
    engine.unproject(hm)
    assert bind(engine._h, pairs.ctypes.data, 1, out.ctypes.data, 4) == C.MDKM_OK
    engine.unproject(hm)
    r = engine.fit(init, max_iter=5)
    assert "transitions" not in r


@pytest.mark.gpu
def test_plugin_passes_the_option(pkg, monkeypatch):
    """The plugin's layers carry no transitions (``to_layers`` is unchanged): the result the plugin
    computed is caught on its way to ``to_layers``."""
    hm = stack(2, 64, 80, 13)
    seen = []
    to_layers = api.to_layers
    monkeypatch.setattr(api, "to_layers", lambda res: seen.append(res) or to_layers(res))
    plug = pkg.MultiDayFusionPlugin(n_clusters=5, return_transitions=[(1, 0), (0, 1)], return_cluster_map=True,
                                    init="k-means++", random_state=0, max_iter=10)
    assert [t for _, _, t in plug.run(hm)] == ["points", "points", "labels"]
    (res,) = seen
    assert res.transition_pairs.tolist() == [[1, 0], [0, 1]]
    check_transitions(res.transitions, res.cluster_map, [(1, 0), (0, 1)], 5)


@pytest.mark.gpu
def test_a_refused_binding_leaves_none_behind(engine):
    """When one output of a call is refused, none of its bindings outlives the call: a binding left
    behind would point at an array freed with the call (and, with k_capacity 5, would refuse the
    k = 6 fits below)."""
    hm = stack(2, 40, 60, 21)
    engine.unproject(hm)
    init5, init6 = seeds(hm, 5, 1), seeds(hm, 6, 1)
    with pytest.raises(ValueError):  # int32 is not a map type: refused after nothing, before the rest
        engine.fit(init5, max_iter=5, cluster_map_out=np.empty(hm.shape, np.int32), day_stats=True,
                   transitions=[(0, 1)])
    with pytest.raises(C.MdkmError):  # day 2 does not exist: refused after the map and the statistics
        engine.fit(init5, max_iter=5, cluster_map_out=np.empty(hm.shape, np.uint8), day_stats=True,
                   transitions=[(0, 2)])
    with pytest.raises(C.MdkmError):
        engine.predict(init5, day_stats=True, transitions=[(2, 0)])
    r = engine.fit(init6, max_iter=5)
    assert "transitions" not in r and "day_counts" not in r
    labels, inertia = engine.predict(init6)
    r = engine.fit(init6, max_iter=5, transitions=[(0, 1)])
    check_transitions(r["transitions"], ref_map(UO.valid_mask(hm), r["labels"], 6), [(0, 1)], 6)


@pytest.mark.gpu
@pytest.mark.parametrize("k, mode", [(41, 0), (42, 1), (118, 1), (119, 2), (255, 2)])
def test_bin_variant_chosen(engine, k, mode):
    """The k values of ``test_every_bin_variant`` sit on both sides of the run-time switches: the
    variant that ran (0: per-warp, 1: per-CTA, 2: global bins) is read from the kernel's name in a
    profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    import torch

    rs = np.random.RandomState(k)
    hm = (rs.rand(2, 40, 77) * 50).astype(np.float32)
    engine.unproject(hm)
    c = np.stack([rs.rand(k) * 77, rs.rand(k) * 40, rs.rand(k) * 50], axis=1)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        labels, _, T = engine.predict(c, transitions=[(0, 1)])
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "day_transitions_kernel" in e.name}
    assert len(names) == 1 and f"day_transitions_kernel<unsigned char, {mode}>" in names.pop(), names
    check_transitions(T, ref_map(UO.valid_mask(hm), labels.copy(), k), [(0, 1)], k)


def _two_gpus():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 300])
def test_device_group_equals_one_device(pkg, k):
    """Row bands that cut days (31 rows over two devices); the whole-stack map merged over NVLink."""
    _two_gpus()
    hm = stack(3, 31, 77, 18)
    kw = dict(n_clusters=k, init="k-means++", random_state=7, max_iter=10, return_day_stats=True,
              return_transitions=[(0, 1), (2, 1), (1, 1)])
    one = pkg.fuse_multiday_kmeans(hm, device=0, return_cluster_map=True, **kw)
    two = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], **kw)
    assert np.array_equal(one.labels, two.labels) and one.inertia == two.inertia
    assert two.transitions.tobytes() == one.transitions.tobytes()
    check_transitions(one.transitions, one.cluster_map, [(0, 1), (2, 1), (1, 1)], k, one.day_counts)
    two_map = pkg.fuse_multiday_kmeans(hm, devices=[0, 1], return_cluster_map=True, **kw)
    assert two_map.cluster_map.tobytes() == one.cluster_map.tobytes()
    assert two_map.transitions.tobytes() == one.transitions.tobytes()


@pytest.mark.gpu
def test_pre_sharded_ranks_receive_the_global_counts(pkg):
    """Two engines with a communicator, each given a flat slice that ends inside a day."""
    _two_gpus()
    from concurrent.futures import ThreadPoolExecutor

    hm = stack(3, 30, 70, 19)
    flat = hm.reshape(-1)
    cut = 30 * 70 + 517
    init = seeds(hm, 6, 4)
    one = pkg.fuse_multiday_kmeans(hm, n_clusters=6, init=init, max_iter=10, return_transitions=True,
                                   return_cluster_map=True, return_day_stats=True)
    uid = pkg.Engine.make_unique_id()
    engines = [pkg.Engine(r) for r in range(2)]
    try:
        with ThreadPoolExecutor(2) as ex:
            list(ex.map(lambda r: engines[r].init_comm(2, r, uid), range(2)))
            spans = [(0, cut), (cut, flat.size)]
            res = list(ex.map(lambda r: pkg.fuse_multiday_kmeans(
                flat[spans[r][0]:spans[r][1]], n_clusters=6, init=init, max_iter=10, engine=engines[r],
                stack_shape=hm.shape, pix_begin=spans[r][0], return_transitions=True, return_cluster_map=True),
                range(2)))
    finally:
        for e in engines:
            e.close()
    for r in res:
        assert r.transitions.tobytes() == one.transitions.tobytes()
        assert r.transition_pairs.tolist() == [[0, 1], [1, 2]]
    assert np.concatenate([r.cluster_map for r in res]).tobytes() == one.cluster_map.tobytes()
