"""CPU: the C-ABI library loads and exports every symbol include/mdkm.h declares (no compute
without a GPU), host-side argument logic, sharding arithmetic."""
import ctypes
import importlib
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "3d-point-cloud-multiday-imagery_b200"


@pytest.fixture(scope="module")
def built():
    build = importlib.import_module(PKG + ".build")
    return build.build_library()


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "mdkm.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mdkm_[a-z_0-9]+)\s*\(", txt)))


def test_header_declares_expected_entry_points():
    syms = header_symbols()
    for s in ("mdkm_create", "mdkm_destroy", "mdkm_unproject", "mdkm_set_points", "mdkm_fit",
              "mdkm_lloyd_step", "mdkm_last_error", "mdkm_comm_init", "mdkm_get_cloud"):
        assert s in syms


def test_library_exports_every_declared_symbol(built):
    lib = ctypes.CDLL(built)
    for s in header_symbols():
        assert hasattr(lib, s), f"{s} declared in include/mdkm.h but not exported by libmdkm.so"


def test_ctypes_prototypes_cover_header(built):
    cabi = importlib.import_module(PKG + "._cabi")
    assert sorted(cabi.SIGNATURES) == header_symbols()
    lib = cabi.load()
    assert lib.mdkm_version().decode().endswith("sm_100a")


def test_ctypes_constants_match_header():
    """Option / memory / dtype / phase constants of the Python binding against the enums of the header."""
    cabi = importlib.import_module(PKG + "._cabi")
    txt = open(os.path.join(ROOT, "include", "mdkm.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    enums = {}
    for body in re.findall(r"enum\s*\w*\s*\{(.*?)\}", txt, flags=re.S):
        nxt = 0
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, val = (t.strip() for t in item.split("=", 1))
                nxt = int(val, 0)
            else:
                name = item
            enums[name] = nxt
            nxt += 1
    checked = 0
    for name, val in vars(cabi).items():
        for prefix in ("OPT_", "MEM_", "HM_", "PHASE_", "POINTS_"):
            if name.startswith(prefix) and isinstance(val, int) and "MDKM_" + name in enums:
                assert enums["MDKM_" + name] == val, (name, val, enums["MDKM_" + name])
                checked += 1
    assert checked >= 12, checked
    assert enums["MDKM_OPT_DEPENDENT_LAUNCH"] == cabi.OPT_DEPENDENT_LAUNCH
    for name, code in cabi.STATUS_BY_NAME.items():
        if name in enums:
            assert enums[name] == code, name


def test_library_is_sm100a_only(built):
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", built], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def run_without_gpu(src):
    """Runs `src` in a fresh interpreter that sees no CUDA device, so that what the package does
    without a GPU is checked on machines that have one, too."""
    src = f"import sys\nsys.path.insert(0, {ROOT!r})\n" + textwrap.dedent(src)
    res = subprocess.run([sys.executable, "-c", src], cwd=ROOT, capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 0, res.stdout + res.stderr


def test_create_fails_loudly_without_gpu(built):
    run_without_gpu(f"""
        import importlib
        import numpy as np
        import pytest
        import torch

        assert not torch.cuda.is_available()
        pkg = importlib.import_module({PKG!r})
        with pytest.raises(Exception, match="MDKM_ERR_NO_DEVICE"):
            pkg.Engine(0)
        # the plugin wrapper keeps the reference's error-layer convention (plugin.py:236-241)
        layers = pkg.MultiDayFusionPlugin().run(np.zeros((1, 4, 4), dtype=np.float32))
        assert len(layers) == 1 and layers[0][2] == "image" and layers[0][1]["name"].startswith("Error:")
        assert layers[0][0].shape == (100, 100)
    """)


def test_product_never_imports_oracle():
    pkg_dir = os.path.join(ROOT, PKG)
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert not re.search(r"#include\s+[\"<].*oracle", txt), f
                assert "lloyd_oracle" not in txt and "import_module(\"oracle" not in txt, f


def test_shard_range_partitions_exactly():
    dist = importlib.import_module(PKG + ".dist")
    for total in (0, 1, 7, 100, 2048 * 2048 * 10 + 3):
        for world in (1, 2, 3, 4, 8):
            for align in (1, 2048):
                spans = [dist.shard_range(total, r, world, align) for r in range(world)]
                assert spans[0][0] == 0 and spans[-1][1] == total
                for a, b in zip(spans, spans[1:]):
                    assert a[1] == b[0]
                sizes = [e - b for b, e in spans]
                assert max(sizes) - min(sizes) <= 2 * align
                for b, e in spans[:-1]:
                    assert b % align == 0 or b == total


def test_same_clustering_helper():
    api = importlib.import_module(PKG + ".api")
    a = np.array([0, 0, 1, 2, 2, 1])
    assert api._is_same_clustering(a, np.array([2, 2, 0, 1, 1, 0]), 3)
    assert not api._is_same_clustering(a, np.array([2, 2, 0, 1, 0, 0]), 3)


def test_uniform_choice_matches_numpy_bit_for_bit():
    """scikit-learn's first k-means++ index and its init="random" seeds are numpy
    RandomState.choice(n, p=uniform) draws (sklearn/_kmeans.py:228, 1014-1021); _npdraw.py
    reproduces them from a closed form of np.cumsum(np.full(n, 1/n)), for any n."""
    nd = importlib.import_module(PKG + "._npdraw")
    rs = np.random.RandomState(0)
    ns = list(range(1, 130)) + [int(v) for v in rs.randint(130, 2_000_000, size=25)] + [2 ** 20, 2 ** 20 + 1, 3 * 2 ** 19, 10 ** 6]
    for n in ns:
        c = nd.UniformCdf(n)
        ref = np.cumsum(np.full(n, 1.0 / n))
        idx = np.unique(np.concatenate([np.arange(min(n, 40)), rs.randint(0, n, size=120), [n - 1]]))
        np.testing.assert_array_equal(np.array([c.at(int(i)) for i in idx]), ref[idx], err_msg=str(n))
        refn = ref / ref[-1]
        us = np.concatenate([rs.random_sample(30), refn[idx[:15]], np.nextafter(refn[idx[:15]], 0), np.nextafter(refn[idx[:15]], 2)])
        us = us[us < 1.0]
        np.testing.assert_array_equal(np.array([c.search(float(u)) for u in us]), refn.searchsorted(us, side="right"),
                                      err_msg=str(n))
    for n, k, seed in [(1000, 17, 0), (50, 50, 1), (12345, 300, 2), (7, 3, 3), (10, 10, 4), (300000, 1024, 5)]:
        want = np.random.RandomState(seed).choice(n, size=k, replace=False, p=np.full(n, 1.0 / n))
        got = nd.choice_uniform_without_replacement(np.random.RandomState(seed), n, k)
        np.testing.assert_array_equal(got, want)
        assert nd.choice_uniform(np.random.RandomState(seed), n) == np.random.RandomState(seed).choice(n, p=np.full(n, 1.0 / n))
    # BASELINE config sizes (no n-sized array anywhere): sane and monotone
    for n in (1342177280, 503316480):
        c = nd.UniformCdf(n)
        assert len(c._i0) < 200 and abs(c.last - 1.0) < 1e-6
        probe = [0, 1, 2, n // 3, n // 2, n - 2, n - 1]
        vals = [c.at(i) for i in probe]
        assert vals == sorted(vals) and vals[0] == 1.0 / n
        for u in (0.0, 0.25, 0.5, 0.999999):
            j = c.search(u)
            assert abs(j - u * n) <= 1e-6 * n + 2 and (j == 0 or c.at(j - 1) / c.last <= u < c.at(j) / c.last)


def test_same_clustering_over_shards():
    """sklearn's permutation test (_k_means_common.pyx:314-330) decided from per-shard label maps."""
    api = importlib.import_module(PKG + ".api")
    rs = np.random.RandomState(0)
    k = 7
    l1 = rs.randint(0, k, size=1000)
    perm = rs.permutation(k)
    for l2, want in ((perm[l1], True), (np.where(np.arange(1000) == 777, (perm[l1] + 1) % k, perm[l1]), False)):
        assert api._is_same_clustering(l1, l2, k) is want
        for cuts in ([0, 1000], [0, 400, 1000], [0, 10, 10, 600, 1000]):  # shards, one of them empty
            maps, oks = zip(*[api._label_mapping(l1[a:b], l2[a:b], k) for a, b in zip(cuts, cuts[1:])])
            assert api._merge_label_mappings(list(maps), list(oks)) is want, cuts
    # consistent inside every shard, but the shards disagree about the image of label 0
    a = api._label_mapping(np.array([0, 0, 1]), np.array([2, 2, 0]), 3)
    b = api._label_mapping(np.array([0, 2]), np.array([1, 1]), 3)
    assert a[1] and b[1] and not api._merge_label_mappings([a[0], b[0]], [True, True])


class _FakeRankEngine:
    """Host-only stand-in for Engine inside a DeviceGroup: numpy unprojection, labels = rank."""

    def __init__(self, device):
        self.device, self.p2p, self.closed = device, False, False
        self.rank, self.n_ranks = 0, 1

    def init_comm(self, world, rank, uid):
        self.n_ranks, self.rank, self.uid = world, rank, uid

    def p2p_handle(self):
        return b"\0" * 64

    def p2p_buffer(self):
        return 0x1000 + self.device

    def p2p_open_ptrs(self, ptrs):
        self.ptrs, self.p2p = list(ptrs), True
        return True

    def p2p_close(self):
        self.p2p = False

    def unproject(self, hm, mask, *, stack_shape, pix_begin, **kw):
        D, H, W = stack_shape
        ok = np.isfinite(hm) & (np.abs(hm) <= 144)
        if mask is not None:
            ok &= mask.astype(bool)
        idx = np.flatnonzero(ok) + pix_begin
        self.P = np.stack([idx % W, (idx // W) % H, hm[ok]], axis=1).astype(np.float32)
        days = idx // (H * W)
        d0, d1 = pix_begin // (H * W), (pix_begin + hm.shape[0] - 1) // (H * W)
        self.seg = np.concatenate([[0], np.cumsum([(days == d).sum() for d in range(d0, d1 + 1)])]).astype(np.int64)
        return self.P.shape[0]

    @property
    def segment_offsets(self):
        return self.seg

    def get_cloud(self, napari_order=True, out=None, wait=True):
        out[...] = self.P[:, ::-1] if napari_order else self.P

    def wait(self):
        pass

    def close(self):
        self.closed = True


def test_device_group_shards_and_assembles_in_reference_order():
    grp_mod = importlib.import_module(PKG + ".group")
    pkg = importlib.import_module(PKG)
    from oracle import unproject_oracle as UO

    D, H, W = 3, 20, 16
    hm = pkg.make_stack(D, H, W, seed=2, n_buildings=3).numpy()
    P = UO.unproject_stack(hm)
    fakes = []

    def factory(dev):
        fakes.append(_FakeRankEngine(dev))
        return fakes[-1]

    with grp_mod.DeviceGroup([5, 6, 7, 8], engine_factory=factory, make_unique_id=lambda: b"u" * 128) as grp:
        assert grp.world == 4 and grp.p2p
        engs = sorted(fakes, key=lambda f: f.rank)
        assert [f.rank for f in engs] == [0, 1, 2, 3] and all(f.uid == b"u" * 128 and f.n_ranks == 4 for f in engs)
        assert all(f.ptrs == [0x1005, 0x1006, 0x1007, 0x1008] for f in engs)

        def run(eng, labels_out):
            labels_out[...] = eng.rank
            return {"rank": eng.rank}

        res, labels, cloud, hn, extra = grp.fuse(hm, run_kmeans=run)
        assert res == {"rank": 0} and hn is None
        np.testing.assert_array_equal(cloud.astype(np.float64), UO.to_napari_points(P))  # np.where order, days merged
        assert sum(extra["shard_points"]) == P.shape[0] and labels.shape == (P.shape[0],)
        assert np.all(np.diff(labels) >= 0) and set(labels.tolist()) == {0, 1, 2, 3}      # rank order == point order
        per_day = [UO.unproject_stack(hm[d:d + 1]).shape[0] for d in range(D)]
        np.testing.assert_array_equal(extra["segment_offsets"], np.concatenate([[0], np.cumsum(per_day)]))
        # row-band shards: 60 rows over 4 ranks = 15 rows each, cut on row boundaries
        assert [len(np.unique(f.P[:, 1])) <= 16 for f in engs]
        # an error on one rank surfaces, the other ranks still finish their call
        with pytest.raises(RuntimeError, match="boom"):
            grp.map(lambda r: (_ for _ in ()).throw(RuntimeError("boom")) if r == 2 else r)
    assert all(f.closed for f in fakes)
    with pytest.raises(ValueError):
        grp_mod.DeviceGroup([0, 0], engine_factory=factory, make_unique_id=lambda: b"")


def test_to_layers_matches_reference_layer_contract():
    api = importlib.import_module(PKG + ".api")
    res = api.FusionResult(labels=np.array([0, 1], dtype=np.int32), centroids=np.array([[1.0, 2, 3], [4, 5, 6]]),
                           fused_cloud=np.zeros((2, 3), dtype=np.float32), n_iter=3, inertia=1.0, n_points=2)
    layers = api.to_layers(res)
    data, params, kind = layers[0]
    assert kind == "points" and data.shape == (2, 3)
    # same params the reference's Points layer carries (plugin.py:220-233)
    for key in ("name", "size", "properties", "scale", "opacity", "face_colormap", "face_color"):
        assert key in params
    assert params["size"] == 2 and params["opacity"] == 0.8 and params["face_colormap"] == "turbo"
    np.testing.assert_array_equal(layers[1][0], [[3, 2, 1], [6, 5, 4]])  # centroids in (z,y,x)
    assert res.labels_ is res.labels and res.cluster_centers_ is res.centroids


def test_to_layers_colours_by_height_when_levelled():
    api = importlib.import_module(PKG + ".api")
    hn = np.array([0.0, 1.0], dtype=np.float32)
    res = api.FusionResult(labels=np.array([0, 1], dtype=np.int32), centroids=np.zeros((2, 3)),
                           fused_cloud=np.zeros((2, 3), dtype=np.float32), n_iter=1, inertia=0.0, n_points=2,
                           height_norm=hn)
    params = api.to_layers(res)[0][1]
    assert params["face_color"] == "height" and params["properties"]["height"] is hn  # plugin.py:186-188, 231
    assert params["properties"]["cluster"] is res.labels
    res.height_norm = None
    assert api.to_layers(res)[0][1]["face_color"] == "cluster"


def test_output_buffers_are_validated_not_copied():
    eng = importlib.import_module(PKG + ".engine")
    ok = np.empty((5, 3), dtype=np.float32)
    ptr, mem = eng._as_out_buffer(ok, np.float32, 15, "out")
    assert ptr == ok.ctypes.data and mem == 0
    for bad, msg in ((np.empty((5, 3), dtype=np.float64), "float32"),
                     (np.empty((5, 6), dtype=np.float32)[:, ::2], "contiguous"),
                     (np.empty((4, 3), dtype=np.float32), "15 elements"),
                     ([0.0] * 15, "numpy array")):
        with pytest.raises(ValueError, match=msg):
            eng._as_out_buffer(bad, np.float32, 15, "out")
    t = __import__("torch").empty(10, dtype=__import__("torch").int32)
    assert eng._as_out_buffer(t, np.int32, 10, "labels_out")[0] == t.data_ptr()
    with pytest.raises(ValueError, match="contiguous"):
        eng._as_out_buffer(t[::2], np.int32, 5, "labels_out")
    with pytest.raises(ValueError, match="int32"):
        eng._as_out_buffer(t.float(), np.int32, 10, "labels_out")


def test_plugin_error_is_logged_like_the_reference(tmp_path, built):
    log = tmp_path / "log.txt"
    run_without_gpu(f"""
        import importlib
        import numpy as np

        pkg = importlib.import_module({PKG!r})
        layers = pkg.MultiDayFusionPlugin(log_path={str(log)!r}).run(np.zeros((1, 4, 4), dtype=np.float32))
        assert layers[0][1]["name"].startswith("Error:")
    """)
    txt = log.read_text()  # plugin.py:238-239: "Error: <e>\n<traceback>"
    assert txt.startswith("Error: ") and "Traceback (most recent call last)" in txt


def test_synthetic_stack_properties():
    pkg = importlib.import_module(PKG)
    hm = pkg.make_stack(3, 64, 96, seed=1).numpy()
    assert hm.shape == (3, 64, 96) and hm.dtype == np.float32
    assert 0.005 < np.isnan(hm).mean() < 0.05
    assert (np.abs(hm[np.isfinite(hm)]) > 144).mean() > 0.001
    assert np.array_equal(np.isnan(hm), np.isnan(pkg.make_stack(3, 64, 96, seed=1).numpy()))
