"""The start and the end of a fit: status, accumulators and table set up by one launch, the end of
the fit enqueued right behind the last batch of iterations (no host wait in between), centroids
and status written by the final pass, and the raster mirror index built in one pass."""
import importlib

import numpy as np
import pytest

from oracle import kmeans_oracle as KO, unproject_oracle as UO

pytestmark = pytest.mark.gpu

synth = importlib.import_module("3d-point-cloud-multiday-imagery_b200.synth")
LABEL_BAND = 1e-5
CENTROID_TOL = 1e-5


def same_fit(a, b):
    assert a["n_iter"] == b["n_iter"]
    assert a["centers"].tobytes() == b["centers"].tobytes()
    assert np.array_equal(a["labels"], b["labels"])
    assert a["inertia"] == b["inertia"]


@pytest.fixture(scope="module")
def raster():
    D, H, W = 3, 120, 200  # W not a multiple of 16: 8-pixel cells
    hm = synth.make_stack(D, H, W, seed=5, n_buildings=8).numpy()
    return hm, UO.unproject_stack(hm)


@pytest.mark.parametrize("k", [16, 64, 300])
def test_back_to_back_fits_equal_fresh_handles(pkg, engine, raster, k):
    """Fits of varying length on one handle (the end of each is enqueued behind its last batch)
    equal the same fits on a fresh handle, and the oracle."""
    hm, P = raster
    init = synth.init_from_points(P.astype(np.float32), k, 3)
    engine.unproject(hm)
    cases = [(m, 0.0) for m in (1, 9, 10, 11, 20)] + [(50, 0.5)]  # tol 0.5: converges in the first batch
    runs = []
    for max_iter, tol in cases:
        engine.drop_caches()
        runs.append(engine.fit(init, max_iter=max_iter, tol=tol))
    assert runs[-1]["n_iter"] < 10
    fresh = pkg.Engine(0)
    try:
        fresh.unproject(hm)
        for (max_iter, tol), r in zip(cases, runs):
            same_fit(r, fresh.fit(init, max_iter=max_iter, tol=tol))
    finally:
        fresh.close()
    for (max_iter, tol), r in zip(cases, runs):
        if tol == 0.0:
            ref = KO.kmeans_fit(P, init, max_iter=max_iter, tol=0.0)
            assert r["n_iter"] == ref["n_iter"]
            assert KO.compare_labels(P, ref["centers"], ref["labels"], r["labels"], rel_band=LABEL_BAND)["n_hard"] == 0
            assert KO.centroid_rel_err(ref["centers"], r["centers"], P.std(axis=0)) <= CENTROID_TOL


@pytest.mark.parametrize("max_iter", [10, 20])
def test_fit_relocation_at_batch_boundaries(engine, golden, max_iter):
    """An empty cluster found while the end of the fit is already enqueued: the final pass does
    nothing, the host relocates and runs the end again (as test_fit_relocation_at_any_iteration_count)."""
    from oracle import sklearn_ref

    if not sklearn_ref.available():
        pytest.skip("scikit-learn not importable")
    g = golden("kmeans_relocate.npz")
    X = g["X"].astype(np.float64)
    engine.set_points(g["X"])
    r = engine.fit(g["init"], max_iter=max_iter, tol=0.0)
    ref = sklearn_ref.fit(X, g["init"], max_iter=max_iter, tol=0.0)
    assert r["n_relocations"] >= 1
    assert r["n_iter"] == ref["n_iter"]
    assert KO.compare_labels(X, ref["centers"], ref["labels"], r["labels"], rel_band=LABEL_BAND)["n_hard"] == 0
    assert KO.centroid_rel_err(ref["centers"], r["centers"], X.std(axis=0)) <= CENTROID_TOL
    np.testing.assert_allclose(r["inertia"], ref["inertia"], rtol=1e-6)


def test_device_labels_ready_on_torch_stream(engine, raster):
    """labels_out on the device is consumed on torch's stream right after fit returns."""
    import torch

    hm, P = raster
    init = synth.init_from_points(P.astype(np.float32), 16, 4)
    engine.unproject(hm)
    host = engine.fit(init, max_iter=20, tol=0.0)
    out = torch.full((P.shape[0],), -1, dtype=torch.int32, device="cuda:0")
    engine.drop_caches()
    engine.fit(init, max_iter=20, tol=0.0, labels_out=out)
    counts = torch.bincount(out.long(), minlength=16).cpu().numpy()  # (queued at once on torch's stream)
    assert np.array_equal(out.cpu().numpy(), host["labels"])
    assert np.array_equal(counts, np.bincount(host["labels"], minlength=16))


@pytest.mark.parametrize("shape,k,rows", [
    ((3, 200, 1000), 16, (150, 450)),   # row band crossing two day boundaries, W % 16 != 0
    ((2, 300, 512), 16, (100, 600)),    # 16-pixel cells, a run list of many index tiles
    ((4, 100, 264), 64, None),
])
def test_raster_index_equals_generic_mirror(engine, shape, k, rows):
    """The one-pass raster index (several look-back tiles) gives the same fit as the generic
    histogram + scatter build of the mirror."""
    D, H, W = shape
    hm = synth.make_stack(D, H, W, seed=H + W + k, n_buildings=8).numpy()
    r0, r1 = rows if rows else (0, D * H)
    n = engine.unproject(hm.reshape(-1)[r0 * W:r1 * W], stack_shape=shape, pix_begin=r0 * W)
    full = UO.unproject_stack(hm)
    valid = UO.valid_mask(hm, None).reshape(-1)
    P = full[int(valid[: r0 * W].sum()):int(valid[: r1 * W].sum())]
    assert n == P.shape[0]
    init = synth.init_from_points(P.astype(np.float32), k, 2)
    res = {}
    for on in (True, False):
        engine.raster_mirror(on)
        try:
            engine.drop_caches()
            res[on] = engine.fit(init, max_iter=12, tol=0.0)
        finally:
            engine.raster_mirror(True)
    same_fit(res[True], res[False])
