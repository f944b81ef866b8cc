"""The assignment kernels at their edges, against exact references.

DESIGN.md section 4 promises that every label is the FP64 argmin (lowest index on exact ties)
and that the per-cluster sums are exact integers on the fixed-point grid of the frame.  Most of
the suite checks this on synthetic terrain with centroids drawn from the data, where the FP32
decision is rarely close.  The cases here are built to make the kernels decide close cases on
every variant that is picked at run time:

- every k on either side of a variant boundary (table chunks at kpad 32 / 64, private
  accumulator slices up to kpad 128, uint16 labels above 256, the bucket index from k = 33, its
  grid sizes, the largest k);
- exact ties under the bucket index, with shuffled and duplicated centroids;
- more than kCandCap (64) candidates per group, where the bucketed pass falls back to the
  brute-force one;
- frames with zero, tiny and huge extents, far origins and centroids far outside the frame;
- group tails, and more days than the mirror keeps as separate segments.

Exact references: on "dyadic" inputs (multiples of 2^-5 with |coordinate| < 2^12) every FP64
form of the squared distance is exact, so ``dyadic_argmin`` is THE argmin and labels must match
it with no tolerance.  Rasters from int16 disparities (``disparity_scale=-1/16``) are dyadic.
Elsewhere labels are compared with a 1e-12 relative near-tie band, and the sums are checked
against the quantum of the frame (``frame_quantum``, the scale ``compute_frame`` picks).
"""
import importlib
import math

import numpy as np
import pytest

from oracle import c_oracle, kmeans_oracle as KO, unproject_oracle as UO

synth = importlib.import_module("3d-point-cloud-multiday-imagery_b200.synth")
cabi = importlib.import_module("3d-point-cloud-multiday-imagery_b200._cabi")

gpu = pytest.mark.gpu
REL_BAND = 1e-12
DYADIC_STEP = 2.0 ** -5
DYADIC_LIMIT = 2.0 ** 12
QUANT_BITS = 22  # common.cuh: |quantised coordinate| < 2^22
ERR_INVALID = cabi.STATUS_BY_NAME["MDKM_ERR_INVALID"]


# ---------------------------------------------------------------------------------------
# exact references (host only)
# ---------------------------------------------------------------------------------------
def is_dyadic(A) -> bool:
    A = np.asarray(A, dtype=np.float64)
    return bool(np.all(np.abs(A) < DYADIC_LIMIT) and np.all(A / DYADIC_STEP == np.rint(A / DYADIC_STEP)))


def dyadic_argmin(P, C, chunk=4096):
    """The exact nearest centroid of every point, lowest index on exact ties.  Only for dyadic
    inputs: there every difference, square and sum below is exact in FP64."""
    P = np.asarray(P, dtype=np.float64)
    C = np.asarray(C, dtype=np.float64)
    assert is_dyadic(P) and is_dyadic(C), "dyadic_argmin needs multiples of 2^-5 below 2^12"
    out = np.empty(P.shape[0], dtype=np.int32)
    for s in range(0, P.shape[0], chunk):
        d = ((P[s:s + chunk, None, :] - C[None, :, :]) ** 2).sum(axis=2)
        out[s:s + chunk] = np.argmin(d, axis=1)  # first minimum = lowest index
    return out


def f64_argmin(P, C, chunk=2048):
    """FP64 nearest centroid by direct differences (the most accurate FP64 form)."""
    P = np.asarray(P, dtype=np.float64)
    C = np.asarray(C, dtype=np.float64)
    out = np.empty(P.shape[0], dtype=np.int32)
    for s in range(0, P.shape[0], chunk):
        d = ((P[s:s + chunk, None, :] - C[None, :, :]) ** 2).sum(axis=2)
        out[s:s + chunk] = np.argmin(d, axis=1)
    return out


def frame_quantum(P):
    """compute_frame (mdkm.cu), restated: per dimension the origin and the exponent e of the
    fixed-point scale 2^e, q = rint((x - origin) * 2^e), |q| < 2^22.  -> (origin[3], e[3])."""
    P32 = np.asarray(P, dtype=np.float32)
    origin = np.zeros(3)
    e = np.zeros(3, dtype=np.int64)
    for d in range(3):
        lo, hi = (float(P32[:, d].min()), float(P32[:, d].max())) if P32.shape[0] else (0.0, 0.0)
        mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
        o = float(np.rint(mid)) if abs(mid) > 0.25 * half else 0.0
        o = float(np.float32(o))
        if half > 0 and abs(mid - o) > half:  # narrower than a unit, away from an integer
            step = 2.0 ** math.floor(math.log2(half))
            o2 = float(np.rint(mid / step)) * step
            hr2 = max(abs(lo - o2), abs(hi - o2))
            amin = lo if lo > 0 else (-hi if hi < 0 else 0.0)
            ulp_max = 2.0 ** (math.floor(math.log2(max(abs(lo), abs(hi)))) - 23)
            if hr2 < amin and step >= ulp_max and float(np.float32(o2)) == o2:
                o = o2
        hr = max(abs(lo - o), abs(hi - o)) * (1.0 + 1e-6) + 1e-30
        e[d] = min(100, max(-100, math.floor(math.log2(((1 << QUANT_BITS) - 2) / hr))))
        origin[d] = o
    return origin, e


def check_sums(P, labels, sums, counts, k):
    """Counts exact; sums within count * 2^-(e+1) per dimension of the exact sums (one rounding
    to the grid per point) plus FP64 rounding, and bit-equal to the grid sums when every point
    lies on the grid."""
    P = np.asarray(P, dtype=np.float64)
    np.testing.assert_array_equal(counts, np.bincount(labels, minlength=k).astype(np.int64))
    origin, e = frame_quantum(P)
    order = np.argsort(labels, kind="stable")
    cuts = np.searchsorted(labels[order], np.arange(k + 1))
    for d in range(3):
        xr = P[order, d] - origin[d]  # exact: a float32 minus an integer-valued float32
        q = xr * 2.0 ** e[d]
        if np.array_equal(q, np.rint(q)):
            qs = np.add.reduceat(np.append(q.astype(np.int64), 0), cuts[:-1])[:k] * (cuts[1:] > cuts[:-1])
            want = qs.astype(np.float64) / 2.0 ** e[d] + counts.astype(np.float64) * origin[d]
            np.testing.assert_array_equal(sums[:, d], want)
            continue
        exact = np.array([math.fsum(xr[cuts[j]:cuts[j + 1]]) for j in range(k)])
        got = sums[:, d] - counts * origin[d]
        slack = 4 * np.spacing(np.abs(sums[:, d])) + 4 * np.spacing(np.abs(counts * origin[d]))
        bound = counts * 2.0 ** -(e[d] + 1) + slack
        assert np.all(np.abs(got - exact) <= bound), (d, np.max(np.abs(got - exact) - bound))


def classify(P, C, ref, labels):
    """Mismatches between two labellings under centres C: a near tie is a gap within 1e-12
    relative, or within the FP64 rounding of the ||c'||^2 - 2 x'.c' form the kernels evaluate
    (16 eps max(||x'||, ||c'||)^2, primes in the frame of compute_frame or around the mean).
    -> (n_mismatch, n_near, n_hard)."""
    P = np.asarray(P, dtype=np.float64)
    bad = np.flatnonzero(ref != labels)
    if bad.size == 0:
        return 0, 0, 0
    p, ca, cb = P[bad], C[ref[bad]], C[labels[bad]]
    da, db = ((p - ca) ** 2).sum(1), ((p - cb) ** 2).sum(1)
    m2 = np.zeros(bad.size)
    for o in (frame_quantum(P)[0], P.mean(0)):
        for v in (p, ca, cb):
            m2 = np.maximum(m2, ((v - o) ** 2).sum(1))
    near = np.abs(da - db) <= REL_BAND * np.minimum(da, db) + 16 * 2.0 ** -53 * m2
    return int(bad.size), int(near.sum()), int((~near).sum())


def check_labels_f64(P, C, labels, near_ok=False):
    """Labels against the FP64 argmin: equal where the inputs are dyadic, else no mismatch
    beyond a near tie (and none at all unless ``near_ok``)."""
    if is_dyadic(P) and is_dyadic(C):
        ref = dyadic_argmin(P, C)
        bad = np.flatnonzero(ref != labels)
        assert bad.size == 0, (bad.size, bad[:8], ref[bad[:8]], labels[bad[:8]])
        return ref
    ref = f64_argmin(P, C)
    n_bad, n_near, n_hard = classify(P, C, ref, labels)
    assert n_hard == 0, (n_bad, n_near, n_hard)
    if not near_ok:
        assert n_near == 0, (n_bad, n_near, n_hard)
    return ref


def oracle_fit(P, init, iters):
    """KO.kmeans_fit with tol = 0; for k >= 1024 the same loop (sklearn/_kmeans.py:630-758) on
    the C oracle, unless a cluster empties (the relocation path is KO's)."""
    k = init.shape[0]
    if k >= 1024:
        P32 = P.astype(np.float32)
        x, y, z = (np.ascontiguousarray(P32[:, d]) for d in range(3))
        C = init.astype(np.float64).copy()
        old = None
        strict = False
        empty = False
        for i in range(iters):
            lab, sums, counts, _ = c_oracle.lloyd_step_f32soa(x, y, z, C)
            if counts.min() == 0:
                empty = True
                break
            C_new = sums / counts[:, None]
            shift2 = float(((C_new - C) ** 2).sum())
            C = C_new
            if old is not None and np.array_equal(lab, old):
                strict = True
                break
            if shift2 <= 0.0:
                break
            old = lab
        if not empty:
            if not strict:
                lab = c_oracle.lloyd_step_f32soa(x, y, z, C, want_sums=False)[0]
            return {"labels": lab, "centers": C, "n_iter": i + 1, "inertia": KO.inertia(P, C, lab)}
    return KO.kmeans_fit(P, init, max_iter=iters, tol=0.0)


def on_grid(P) -> bool:
    """Every coordinate on the fixed-point grid of the frame: the sums are then exact."""
    o, e = frame_quantum(P)
    q = (np.asarray(P, dtype=np.float64) - o) * 2.0 ** e
    return bool(np.array_equal(q, np.rint(q)))


def check_fit(engine, P, init, iters, near_ok=False):
    """A short fit against the oracle.  Always: the same n_iter, and labels that are the FP64
    argmin under the returned centroids (the final pass) with their inertia.  On grid points
    without a relocation: the oracle's labels (near ties only) and centroids within the grid
    quantum.  Off the grid the centroids carry the quantum (up to 2^-(e+1) per dimension), which
    can move a boundary point: centroids to the suite's 1e-5 relative.  A relocation takes the
    farthest point, and with exact ties in those distances (dyadic clouds) scikit-learn's pick
    (np.argpartition) is unspecified, so then only the first two checks apply."""
    r = engine.fit(init, max_iter=iters, tol=0.0)
    ref = oracle_fit(P, init, iters)
    assert r["n_iter"] == ref["n_iter"], (r["n_iter"], ref["n_iter"])
    check_labels_f64(P, r["centers"], r["labels"], near_ok=True)
    spread = float(((P - P.mean(axis=0)) ** 2).sum())  # (FP64 rounding when the inertia is ~0)
    np.testing.assert_allclose(r["inertia"], KO.inertia(P, r["centers"], r["labels"]), rtol=1e-9, atol=1e-12 * spread)
    if r["n_relocations"]:
        return r
    if not on_grid(P):
        err = KO.centroid_rel_err(ref["centers"], r["centers"], P.std(axis=0))
        assert err <= 1e-5, err
        return r
    n_bad, n_near, n_hard = classify(P, ref["centers"], ref["labels"], r["labels"])
    assert n_hard == 0, (n_bad, n_near, n_hard)
    if not near_ok:
        assert n_near == 0, (n_bad, n_near, n_hard)
    if n_bad == 0:
        _, e = frame_quantum(P)
        q = 2.0 ** -(e.astype(np.float64) + 1)
        slack = 1e-12 * np.maximum(np.abs(ref["centers"]), np.abs(P).max(axis=0))
        dev = np.abs(r["centers"] - ref["centers"]) - (q[None, :] + slack)
        assert dev.max() <= 0, dev.max()
        np.testing.assert_allclose(r["inertia"], ref["inertia"], rtol=1e-9, atol=1e-12 * spread)
    return r


def ref_map(valid, labels, k):
    ref = np.zeros(valid.size, dtype=np.uint8 if k <= 255 else np.uint16)
    ref[valid.ravel()] = labels + 1
    return ref


def check_step_predict(engine, P, C, near_ok=False):
    """lloyd_step (pass 1 / pass 2 + FP64 re-decision, sums) and predict (final pass) against
    the references.  -> the reference labels."""
    k = C.shape[0]
    labels, sums, counts, _ = engine.lloyd_step(C)
    ref = check_labels_f64(P, C, labels, near_ok)
    check_sums(P, labels, sums, counts, k)
    plab, inertia = engine.predict(C)
    check_labels_f64(P, C, plab, near_ok)
    # dyadic inputs: every term exact; otherwise the kernel's FP64 terms are formed in its frame
    rtol = REL_BAND if is_dyadic(P) and is_dyadic(C) else 1e-9
    np.testing.assert_allclose(inertia, KO.inertia(P, C, ref), rtol=rtol, atol=1e-300)
    return ref


# ---------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------
def dyadic_raster(D, H, W, seed, valid=0.9, zspan=40.0):
    """int16 disparities (z = -d/16, so x, y integers and z a multiple of 1/16), terrain plus
    noise, a random validity mask.  -> (disparity, mask, P float64)."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = 16 * zspan * 0.5 * (np.sin(xx / 7.0) * np.cos(yy / 5.0))
    disp = (base[None] + rs.randint(-48, 49, size=(D, H, W))).astype(np.int16)
    mask = rs.rand(D, H, W) < valid
    P = UO.unproject_stack(UO.height_from_disparity(disp), mask)
    return disp, mask, P


def unproject_dyadic(engine, disp, mask, P):
    n = engine.unproject(disp, mask, disparity_scale=-1.0 / 16.0)
    assert n == P.shape[0]
    return n


def dyadic_centroids(P, k, seed, jitter=3):
    """k data points plus small dyadic offsets (multiples of 2^-5): many points sit near or on a
    boundary between two of them."""
    rs = np.random.RandomState(seed)
    idx = rs.choice(P.shape[0], k, replace=False)
    return P[idx] + rs.randint(-jitter * 32, jitter * 32 + 1, size=(k, 3)) * DYADIC_STEP


# ---------------------------------------------------------------------------------------
# 1. host-only self-tests of the references
# ---------------------------------------------------------------------------------------
def test_dyadic_argmin_exact_ties_and_lowest_index():
    P = np.array([[1.0, 0, 0], [1.0, 1.0, 0], [0.5, 0.5, 0.5], [3.0, 3.0, 3.0]])
    C = np.array([[0.0, 0, 0], [2.0, 0, 0], [0.0, 2.0, 0], [2.0, 2.0, 0], [3.0, 3.0, 3.0]])
    assert dyadic_argmin(P, C).tolist() == [0, 0, 0, 4]
    assert dyadic_argmin(P, C[::-1]).tolist() == [3, 1, 4, 0]
    dup = np.array([[1.0, 1, 0], [5.0, 5, 5], [1.0, 1, 0]])
    assert dyadic_argmin(P, dup).tolist() == [0, 0, 0, 1]
    # a gap far below FP32 resolution at this magnitude is still decided exactly
    big = 4095.0
    P2 = np.array([[big, big, big - DYADIC_STEP]])
    C2 = np.array([[0.0, 0, 0], [big, big, big]])
    assert dyadic_argmin(P2, C2).tolist() == [1]
    C3 = np.array([[big - 2 * DYADIC_STEP, big, big], [big, big, big - 2 * DYADIC_STEP]])
    P3 = np.array([[big - DYADIC_STEP, big, big - DYADIC_STEP]])
    assert dyadic_argmin(P3, C3).tolist() == [0]  # exact tie
    assert dyadic_argmin(P3, C3[::-1]).tolist() == [0]
    with pytest.raises(AssertionError):
        dyadic_argmin(np.array([[0.1, 0, 0]]), C)
    with pytest.raises(AssertionError):
        dyadic_argmin(np.array([[4096.0, 0, 0]]), C)
    disp, mask, P4 = dyadic_raster(2, 9, 13, seed=1)
    assert is_dyadic(P4) and P4.shape[0] == mask.sum()


def test_dyadic_argmin_agrees_with_the_oracle_e_step():
    rs = np.random.RandomState(3)
    P = rs.randint(-2000, 2000, size=(3000, 3)) * 0.25
    C = rs.randint(-2000, 2000, size=(50, 3)) * 0.25
    ref = dyadic_argmin(P, C)
    np.testing.assert_array_equal(ref, f64_argmin(P, C))
    cmp = KO.compare_labels(P, C, KO.e_step(P, C), ref, rel_band=0.0)
    assert cmp["n_hard"] == 0, cmp


def test_frame_quantum_restates_compute_frame():
    origin, e = frame_quantum(np.array([[0.0, -1.0, 5.0], [100.0, 1.0, 5.0]]))
    assert origin.tolist() == [50.0, 0.0, 5.0]
    assert e.tolist() == [math.floor(math.log2((2 ** 22 - 2) / (50 * (1 + 1e-6)))),
                          math.floor(math.log2((2 ** 22 - 2) / (1 + 1e-6))), 100]
    # narrower than a unit and away from an integer: a power-of-two step, not the integer 1
    o, e = frame_quantum(np.array([[0.5, 0.0, 0.0], [0.5009765625, 0.0, 0.0]]))
    assert o[0] == 0.5 + 2.0 ** -11 and e[0] == math.floor(math.log2((2 ** 22 - 2) / (2.0 ** -11 * (1 + 1e-6))))
    o, e = frame_quantum(np.array([[-0.2, 0.0, 0.0], [0.3, 0.0, 0.0]]))  # straddles 0: unchanged rule
    assert o[0] == 0.0
    rs = np.random.RandomState(5)
    for scale, off in ((1.0, 0.0), (1e-3, 0.5), (1e3, 4.2e6), (1e6, 0.0), (3.0, -7e4)):
        P = (rs.rand(500, 3) * scale + off).astype(np.float32).astype(np.float64)
        o, e = frame_quantum(P)
        for d in range(3):
            q = np.rint((P[:, d] - o[d]) * 2.0 ** e[d])
            assert np.abs(q).max() < 2 ** 22  # fits the grid ...
            if e[d] < 100:
                assert np.abs((P[:, d] - o[d]) * 2.0 ** (e[d] + 1)).max() * (1 + 1e-6) > 2 ** 22 - 2 - 1  # ... tightly


def test_check_sums_accepts_the_grid_and_rejects_more():
    rs = np.random.RandomState(7)
    P = (rs.rand(400, 3) * 10.0).astype(np.float32).astype(np.float64)
    lab = rs.randint(0, 5, size=400).astype(np.int32)
    counts = np.bincount(lab, minlength=5).astype(np.int64)
    o, e = frame_quantum(P)
    q = np.rint((P - o) * 2.0 ** e)
    sums = np.stack([np.bincount(lab, weights=q[:, d], minlength=5) / 2.0 ** e[d] + counts * o[d] for d in range(3)], 1)
    check_sums(P, lab, sums, counts, 5)  # the rounded-to-grid sums are within the bound
    bad = sums.copy()
    bad[2, 1] += counts[2] * 2.0 ** -(e[1] + 1) * 1.5
    with pytest.raises(AssertionError):
        check_sums(P, lab, bad, counts, 5)
    Pg = np.rint(P * 32) / 32  # on the grid: equality is required
    og, eg = frame_quantum(Pg)
    sg = np.stack([np.bincount(lab, weights=Pg[:, d], minlength=5) for d in range(3)], 1)
    check_sums(Pg, lab, sg, counts, 5)
    sg[0, 0] = np.nextafter(sg[0, 0], np.inf)
    with pytest.raises(AssertionError):
        check_sums(Pg, lab, sg, counts, 5)


# ---------------------------------------------------------------------------------------
# 2. k sweep across every variant boundary
# ---------------------------------------------------------------------------------------
K_SWEEP = [1, 2, 16, 17, 32, 33, 64, 65, 128, 129, 255, 256, 257, 1024, 1025, 2047, 2048]
_CLOUDS = {}


def sweep_cloud(name):
    """'raster16': W % 16 == 0; 'raster': W % 16 != 0 (and groups straddle rows); 'points': a
    set_points cloud in random order.  All dyadic, all with more than 2048 points."""
    if name not in _CLOUDS:
        if name == "raster16":
            _CLOUDS[name] = dyadic_raster(2, 40, 64, seed=16)
        elif name == "raster":
            _CLOUDS[name] = dyadic_raster(1, 45, 101, seed=17, valid=0.8)
        else:
            rs = np.random.RandomState(18)
            ctr = rs.randint(-600, 600, size=(40, 3)) * 0.5
            P = ctr[rs.randint(0, 40, size=6000)] + rs.randint(-640, 641, size=(6000, 3)) * DYADIC_STEP
            _CLOUDS[name] = (None, None, P[rs.permutation(6000)])
    return _CLOUDS[name]


def load_cloud(engine, name):
    disp, mask, P = sweep_cloud(name)
    if disp is None:
        engine.set_points(P.astype(np.float32))
    else:
        unproject_dyadic(engine, disp, mask, P)
    return mask, P


@gpu
@pytest.mark.parametrize("cloud", ["raster16", "raster", "points"])
@pytest.mark.parametrize("k", K_SWEEP)
def test_k_sweep_step_predict_fit_map(engine, k, cloud):
    mask, P = load_cloud(engine, cloud)
    C = dyadic_centroids(P, k, seed=k)
    ref = check_step_predict(engine, P, C)
    if mask is not None:  # the cluster map of the final pass, uint8 / uint16 by k
        cmap = np.zeros(mask.size, dtype=np.uint8 if k <= 255 else np.uint16)
        lab, _ = engine.predict(C, cluster_map_out=cmap)
        np.testing.assert_array_equal(lab, ref)
        assert cmap.tobytes() == ref_map(mask, ref, k).tobytes()
    check_fit(engine, P, C, iters=3, near_ok=True)


@gpu
@pytest.mark.parametrize("k", [17, 129, 257, 2048])
def test_k_sweep_settle_and_two_level_bitwise(engine, k):
    """Settling off, two-level classification forced on and off: the same fit, bit for bit."""
    _, P = load_cloud(engine, "raster")
    C = dyadic_centroids(P, k, seed=k + 1)
    base = engine.fit(C, max_iter=4, tol=0.0)
    step = engine.lloyd_step(C)
    runs = []
    try:
        engine.settle_groups(False)
        runs.append((engine.fit(C, max_iter=4, tol=0.0), engine.lloyd_step(C)))
        engine.settle_groups(True)
        for mode in (0, 1):
            engine.set_option(cabi.OPT_TWO_LEVEL, mode)
            runs.append((engine.fit(C, max_iter=4, tol=0.0), engine.lloyd_step(C)))
    finally:
        engine.settle_groups(True)
        engine.set_option(cabi.OPT_TWO_LEVEL, -1)
    for r, s in runs:
        assert r["centers"].tobytes() == base["centers"].tobytes()
        assert np.array_equal(r["labels"], base["labels"])
        assert r["inertia"] == base["inertia"] and r["n_iter"] == base["n_iter"]
        assert np.array_equal(s[0], step[0]) and s[1].tobytes() == step[1].tobytes()
        assert np.array_equal(s[2], step[2])


@gpu
def test_k_above_the_largest_is_rejected(engine):
    _, P = load_cloud(engine, "points")
    C = dyadic_centroids(P, 2049, seed=3)
    for call in (lambda: engine.lloyd_step(C), lambda: engine.predict(C), lambda: engine.fit(C, max_iter=2)):
        with pytest.raises(cabi.MdkmError) as ei:
            call()
        assert ei.value.code == ERR_INVALID
    assert engine.predict(C[:2048])[0].shape == (P.shape[0],)  # the handle still works


# ---------------------------------------------------------------------------------------
# 3. exact ties under the bucket index
# ---------------------------------------------------------------------------------------
TIE_LATTICES = {(8, 2): (2, 2), (40, 1): (8, 5), (40, 2): (5, 4), (300, 1): (20, 15), (300, 2): (15, 10),
                (2048, 2): (32, 32)}


def tie_case(k, nz, seed, duplicates):
    """A dyadic raster at z = 1 and centroids on a lattice of spacing 2 px (at z = 1, or at
    z = 0.5 and 1.5): pixels between lattice nodes are exactly equidistant from 2, 4 or 8
    centroids.  Indices are shuffled; with ``duplicates`` some centroids are copies of others
    with far-apart indices."""
    nx, ny = TIE_LATTICES[(k, nz)]
    D, H, W = 2, 2 * ny + 1, 2 * nx + 1
    rs = np.random.RandomState(seed)
    disp = np.full((D, H, W), -16, dtype=np.int16)  # z = 1
    mask = rs.rand(D, H, W) < 0.95
    P = UO.unproject_stack(UO.height_from_disparity(disp), mask)
    gy, gx = np.mgrid[0:ny, 0:nx]
    zs = [1.0] if nz == 1 else [0.5, 1.5]
    C = np.concatenate([np.stack([2.0 * gx.ravel() + 1, 2.0 * gy.ravel() + 1, np.full(nx * ny, z)], 1) for z in zs])
    C = C[rs.permutation(k)]
    if duplicates:
        for a in range(0, k // 2, max(1, k // 16)):
            C[k - 1 - a] = C[a]  # the same point at both ends of the index range
    assert C.shape == (k, 3)
    return disp, mask, P, C


@gpu
@pytest.mark.parametrize("duplicates", [False, True])
@pytest.mark.parametrize("k,nz", sorted(TIE_LATTICES))
def test_exact_ties_under_buckets_lowest_index(engine, k, nz, duplicates):
    disp, mask, P, C = tie_case(k, nz, seed=k + nz, duplicates=duplicates)
    unproject_dyadic(engine, disp, mask, P)
    ref = dyadic_argmin(P, C)
    d = ((P - C[ref]) ** 2).sum(1)
    n_equidistant = np.zeros(P.shape[0], dtype=np.int64)
    for c in C:
        n_equidistant += ((P - c) ** 2).sum(1) == d
    assert (n_equidistant > 1).sum() > P.shape[0] // 2  # most pixels really are ties
    for _ in range(2):  # the order inside a bucket comes from shared-memory atomics: twice
        labels, sums, counts, n_ref = engine.lloyd_step(C)
        np.testing.assert_array_equal(labels, ref)
        check_sums(P, labels, sums, counts, k)
        cmap = np.zeros(mask.size, dtype=np.uint8 if k <= 255 else np.uint16)
        plab, inertia = engine.predict(C, cluster_map_out=cmap)
        np.testing.assert_array_equal(plab, ref)
        assert cmap.tobytes() == ref_map(mask, ref, k).tobytes()
        assert inertia == KO.inertia(P, C, ref)  # dyadic: exact


# ---------------------------------------------------------------------------------------
# 4. candidate overflow: more than kCandCap centroids within reach of every group
# ---------------------------------------------------------------------------------------
def squeezed_points(n, seed):
    """x and y in [0, 1) (32 values each), z over [-60, 60]: every x-y tile of the mirror spans
    all the clusters (bench.py's brute-force construction, on the dyadic grid)."""
    rs = np.random.RandomState(seed)
    P = np.stack([rs.randint(0, 32, n) * DYADIC_STEP, rs.randint(0, 32, n) * DYADIC_STEP,
                  rs.randint(-960, 961, n) / 16.0], 1)
    return P


def stacked_raster(k, n_xy, seed):
    """A dyadic raster with z noise over [-40, 40] and k centroids stacked in z above n_xy
    (x, y) positions.  -> (disp, mask, P, C)."""
    rs = np.random.RandomState(seed)
    D, H, W = 2, 40, 100
    disp = rs.randint(-640, 641, size=(D, H, W)).astype(np.int16)
    mask = rs.rand(D, H, W) < 0.9
    P = UO.unproject_stack(UO.height_from_disparity(disp), mask)
    xy = np.stack([rs.randint(0, W, n_xy), rs.randint(0, H, n_xy)], 1).astype(np.float64)
    per = k // n_xy
    C = np.concatenate([np.column_stack([np.repeat(xy[i:i + 1], per, 0),
                                         -40.0 + (np.arange(per) + 0.5) * (80.0 / per)]) for i in range(n_xy)])
    C = np.round(C * 32) / 32
    return disp, mask, P, C[rs.permutation(k)]


@gpu
@pytest.mark.parametrize("k", [300, 2048])
def test_candidate_overflow_squeezed_cloud(engine, k):
    P = squeezed_points(12000, seed=k)
    engine.set_points(P.astype(np.float32))
    C = dyadic_centroids(P, k, seed=k, jitter=1)
    C[:, :2] = np.clip(C[:, :2], 0, 31 * DYADIC_STEP)
    check_step_predict(engine, P, C)
    check_fit(engine, P, C, iters=2, near_ok=True)


@gpu
@pytest.mark.parametrize("k,n_xy", [(300, 4), (2048, 8)])
def test_candidate_overflow_stacked_raster(engine, k, n_xy):
    disp, mask, P, C = stacked_raster(k, n_xy, seed=k)
    unproject_dyadic(engine, disp, mask, P)
    ref = check_step_predict(engine, P, C)
    cmap = np.zeros(mask.size, dtype=np.uint8 if k <= 255 else np.uint16)
    engine.predict(C, cluster_map_out=cmap)  # split-row groups of the final pass (W = 100)
    assert cmap.tobytes() == ref_map(mask, ref, k).tobytes()
    check_fit(engine, P, C, iters=2, near_ok=True)


# ---------------------------------------------------------------------------------------
# 5. frames
# ---------------------------------------------------------------------------------------
def check_cloud_case(engine, P, C, iters=4, near_ok=False, fit_near_ok=True):
    engine.set_points(P.astype(np.float32))
    P = P.astype(np.float32).astype(np.float64)
    check_step_predict(engine, P, C, near_ok=near_ok)
    return check_fit(engine, P, C, iters, near_ok=fit_near_ok)


@gpu
def test_frame_zero_extent_z_raster(engine):
    rs = np.random.RandomState(1)
    disp = np.full((2, 30, 70), -40, dtype=np.int16)  # z = 2.5 everywhere
    mask = rs.rand(*disp.shape) < 0.9
    P = UO.unproject_stack(UO.height_from_disparity(disp), mask)
    unproject_dyadic(engine, disp, mask, P)
    for k in (5, 40):
        C = dyadic_centroids(P, k, seed=k)
        check_step_predict(engine, P, C)
        check_fit(engine, P, C, 4)


@gpu
def test_frame_zero_extent_x_points(engine):
    rs = np.random.RandomState(2)
    P = np.column_stack([np.full(3000, 7.0), rs.randint(-800, 800, 3000) / 8.0, rs.randint(-800, 800, 3000) / 16.0])
    for k in (6, 48):
        check_cloud_case(engine, P, dyadic_centroids(P, k, seed=k))


@gpu
@pytest.mark.parametrize("k", [1, 3])
def test_frame_all_points_identical(engine, k):
    P = np.tile([[3.25, -1.5, 0.75]], (500, 1))
    engine.set_points(P.astype(np.float32))
    C = np.tile(P[:1], (k, 1))  # k = 3: duplicated centroids, the first copy takes everything
    labels, sums, counts, _ = engine.lloyd_step(C)
    assert labels.tolist() == [0] * 500 and counts.tolist() == [500] + [0] * (k - 1)
    check_sums(P, labels, sums, counts, k)
    plab, inertia = engine.predict(C)
    assert plab.tolist() == [0] * 500 and inertia == 0.0
    r = engine.fit(C, max_iter=5, tol=0.0)
    ref = KO.kmeans_fit(P, C, max_iter=5, tol=0.0)
    assert r["n_iter"] == ref["n_iter"] and r["labels"].tolist() == [0] * 500
    np.testing.assert_array_equal(r["centers"], ref["centers"])
    assert r["inertia"] == 0.0


@gpu
def test_frame_utm_like_coordinates(engine):
    """x ~ 5e5, y ~ 4.2e6 (metres), a 1 km extent, centimetre detail (as float32 keeps it)."""
    rs = np.random.RandomState(3)
    ctr = np.column_stack([5.0e5 + rs.rand(12) * 1000, 4.2e6 + rs.rand(12) * 1000, 100 + rs.rand(12) * 50])
    P = ctr[rs.randint(0, 12, 8000)] + np.round(rs.normal(0, 30.0, (8000, 3)), 2)
    C = P[rs.choice(8000, 40, replace=False)].astype(np.float32).astype(np.float64) + np.round(rs.normal(0, 5, (40, 3)), 2)
    check_cloud_case(engine, P, C)
    check_cloud_case(engine, P, C[:9])


@gpu
@pytest.mark.parametrize("k", [40, 300])
def test_frame_wide_extent_fp32_undecided(engine, k):
    """Dyadic points over +-4000 and centroids in pairs 2^-5 apart: ||c'||^2 needs about 36
    bits, and the two distances of a pair differ by less than their FP32 rounding for most
    points near the pair, so only the FP64 re-decision (and a pruning margin that covers that
    rounding) tells them apart."""
    rs = np.random.RandomState(k)
    P = rs.randint(-4000 * 32, 4000 * 32, size=(20000, 3)) * DYADIC_STEP
    P[:, 2] *= 0.01
    P = np.round(P * 32) / 32
    base = dyadic_centroids(P, k // 2, seed=k, jitter=1)
    C = np.concatenate([base, base + [DYADIC_STEP, 0, 0]])[rs.permutation(k)]
    engine.set_points(P.astype(np.float32))
    labels, sums, counts, n_ref = engine.lloyd_step(C)
    ref = check_labels_f64(P, C, labels)
    check_sums(P, labels, sums, counts, k)
    assert n_ref > 0  # some points really were re-decided in FP64
    np.testing.assert_array_equal(engine.predict(C)[0], ref)


@gpu
def test_frame_tiny_extent(engine):
    rs = np.random.RandomState(4)
    P = 0.5 + rs.rand(4000, 3) * 1e-3
    P32 = P.astype(np.float32).astype(np.float64)
    # the origin is not the nearest integer (1), which would leave a half-range of 0.5: the grid
    # is finer than the float32 spacing of the points, so the sums are exact
    assert frame_quantum(P32)[1].min() >= 32 and on_grid(P32)
    for k in (7, 60):
        C = P32[rs.choice(4000, k, replace=False)] + rs.normal(0, 1e-5, (k, 3))
        check_cloud_case(engine, P, C)


@gpu
def test_frame_far_outlier_coarse_quantum(engine):
    rs = np.random.RandomState(5)
    P = np.concatenate([rs.normal(c, 0.3, (1500, 3)) for c in ([0, 0, 0], [2, 1, 0], [1, 3, 1])] + [[[1e6, -1e6, 1e6]]])
    P32 = P.astype(np.float32).astype(np.float64)
    _, e = frame_quantum(P32)
    assert e.max() <= 3  # the grid is coarser than the clusters' detail
    C = P32[rs.choice(4500, 36, replace=False)] + rs.normal(0, 0.05, (36, 3))
    check_cloud_case(engine, P, C, iters=3, near_ok=True)
    check_cloud_case(engine, P, np.vstack([C[:4], P32[-1:]]), iters=3, near_ok=True)


@gpu
def test_frame_centroids_outside_on_every_side(engine):
    rs = np.random.RandomState(6)
    P = np.column_stack([rs.randint(0, 3200, 6000) / 32.0, rs.randint(0, 3200, 6000) / 32.0, rs.randint(0, 320, 6000) / 32.0])
    inside = dyadic_centroids(P, 36, seed=6)
    out = []
    for d, (lo, hi) in enumerate(((0, 100), (0, 100), (0, 10))):
        for v in (lo - 3.5, lo - 1500.0, hi + 2.25, hi + 2000.0):
            c = P[rs.randint(6000)].copy()
            c[d] = v
            out.append(c)
    C = np.vstack([inside[:18], out, inside[18:]])
    C = C[rs.permutation(C.shape[0])]
    assert C.shape[0] >= 33 and is_dyadic(C)
    check_cloud_case(engine, P, C)


@gpu
@pytest.mark.parametrize("k", [6, 40])
def test_frame_centroids_beyond_fp32(engine, k):
    """Centroids at +-1e20: their FP32 ||c'||^2 overflows to inf.  They own no point; the rest
    must be decided as usual, and the fit relocates them as scikit-learn does."""
    rs = np.random.RandomState(k)
    P = np.concatenate([rs.normal(c, 0.5, (1000, 3)) for c in ([0, 0, 0], [3, 0, 1], [0, 4, 2])])
    P32 = P.astype(np.float32).astype(np.float64)
    C = P32[rs.choice(3000, k, replace=False)] + rs.normal(0, 0.1, (k, 3))
    C[1] = [1e20, 1e20, 1e20]
    C[k // 2] = [-1e20, 0.0, 1e20]
    C[-1] = [0.0, -1e20, 0.0]
    engine.set_points(P32.astype(np.float32))
    ref = check_step_predict(engine, P32, C)
    assert not np.isin(ref, [1, k // 2, k - 1]).any()
    r = engine.fit(C, max_iter=4, tol=0.0)
    fr = KO.kmeans_fit(P32, C, max_iter=4, tol=0.0)
    assert r["n_relocations"] >= 3 and r["n_iter"] == fr["n_iter"]
    assert classify(P32, fr["centers"], fr["labels"], r["labels"])[2] == 0
    np.testing.assert_allclose(r["centers"], fr["centers"], rtol=0, atol=1e-6)


# ---------------------------------------------------------------------------------------
# 6. group tails
# ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 1023, 1024, 1025, 8193])
def test_group_tails_points(engine, n):
    rs = np.random.RandomState(n)
    P = rs.randint(-3000, 3000, size=(n, 3)) / 16.0
    engine.set_points(P.astype(np.float32))
    for k in sorted({1, min(n, 3), min(n, 40), min(n, 300), min(n, 2048)}):
        C = P[rs.permutation(n)[:k]] if k == n else dyadic_centroids(P, k, seed=k)
        check_step_predict(engine, P, C)
        if k <= 300 or n <= 2048:
            check_fit(engine, P, C, 3, near_ok=True)


@gpu
def test_group_tail_padding_far_from_origin(engine):
    """The zero padding of the last block sits at the frame origin, far from the last points of
    a cloud whose blobs lie away from its centre: the last group's box grows to include it."""
    rs = np.random.RandomState(8)
    n = 128 * 37 + 3
    ctr = np.array([[3.0e4, -2.0e4, 500.0], [3.0e4 + 800, -2.0e4 + 800, 600.0], [3.0e4, -2.0e4 + 800, 520.0]])
    P = ctr[rs.randint(0, 3, n)] + rs.randint(-320, 321, (n, 3)) / 32.0
    P = P[rs.permutation(n)]
    for k in (4, 37):
        check_cloud_case(engine, P, dyadic_centroids(P, k, seed=k), iters=3)


@gpu
def test_group_tails_one_pixel_per_day(engine):
    rs = np.random.RandomState(9)
    disp = rs.randint(-400, 400, size=(6, 20, 30)).astype(np.int16)
    mask = np.zeros(disp.shape, dtype=bool)
    for d in range(6):
        mask[d, rs.randint(20), rs.randint(30)] = True
    P = UO.unproject_stack(UO.height_from_disparity(disp), mask)
    unproject_dyadic(engine, disp, mask, P)
    for k in (1, 3, 6):
        C = P[:k] + 0.5 if k < 6 else P[::-1].copy()
        ref = check_step_predict(engine, P, C)
        cmap = np.zeros(mask.size, dtype=np.uint8)
        r = engine.fit(C, max_iter=3, tol=0.0, cluster_map_out=cmap)
        fr = KO.kmeans_fit(P, C, max_iter=3, tol=0.0)
        assert r["n_iter"] == fr["n_iter"] and np.array_equal(r["labels"], fr["labels"])
        assert cmap.tobytes() == ref_map(mask, r["labels"], k).tobytes()
        assert ref.shape == (6,)


@gpu
@pytest.mark.parametrize("shape", [(1, 5, 70), (3, 7, 45)])
def test_group_tails_last_group_straddles_a_row(engine, shape):
    disp, mask, P = dyadic_raster(*shape, seed=shape[2], valid=1.0)
    n = unproject_dyadic(engine, disp, mask, P)
    last = (n // 128) * 128
    rows = {int(r) for r in P[last:, 1]}
    assert n % 128 and len(rows) == 2  # the last, partial group runs over a row end
    for k in (5, 40):
        C = dyadic_centroids(P, k, seed=k)
        ref = check_step_predict(engine, P, C)
        cmap = np.zeros(mask.size, dtype=np.uint8)
        engine.predict(C, cluster_map_out=cmap)
        assert cmap.tobytes() == ref_map(mask, ref, k).tobytes()
        check_fit(engine, P, C, 3, near_ok=True)


# ---------------------------------------------------------------------------------------
# 7. many days: more segments than the mirror keeps apart (kMirrorMaxSeg = 1024)
# ---------------------------------------------------------------------------------------
@gpu
def test_many_days(engine):
    D, H, W, k = 1100, 8, 40, 24
    rs = np.random.RandomState(11)
    hm = (rs.randint(-1200, 1200, size=(D, H, W)) / 16.0 + (np.arange(D) % 7)[:, None, None]).astype(np.float32)
    mask = rs.rand(D, H, W) < 0.9
    mask[[3, 500, 1024, 1099]] = False  # empty days: the cluster map's day cursor skips them
    P = UO.unproject_stack(hm, mask)
    assert engine.unproject(hm, mask) == P.shape[0]
    assert len(engine.segment_offsets) == D + 1
    C = dyadic_centroids(P, k, seed=k)
    ref = check_step_predict(engine, P, C)
    res = {}
    for on in (True, False):
        engine.raster_mirror(on)
        try:
            engine.drop_caches()
            cmap = np.zeros((D, H, W), dtype=np.uint8)
            res[on] = (engine.fit(C, max_iter=5, tol=0.0, cluster_map_out=cmap), cmap, engine.lloyd_step(C))
        finally:
            engine.raster_mirror(True)
    a, b = res[True], res[False]
    assert a[0]["centers"].tobytes() == b[0]["centers"].tobytes() and np.array_equal(a[0]["labels"], b[0]["labels"])
    assert a[0]["inertia"] == b[0]["inertia"] and a[0]["n_iter"] == b[0]["n_iter"]
    assert a[1].tobytes() == b[1].tobytes() == ref_map(mask, a[0]["labels"], k).tobytes()
    assert np.array_equal(a[2][0], ref) and np.array_equal(b[2][0], ref) and a[2][1].tobytes() == b[2][1].tobytes()
    fr = KO.kmeans_fit(P, C, max_iter=5, tol=0.0)
    assert a[0]["n_iter"] == fr["n_iter"]
    assert classify(P, fr["centers"], fr["labels"], a[0]["labels"])[2] == 0
    np.testing.assert_allclose(a[0]["centers"], fr["centers"], rtol=0, atol=1e-9)
    # ground levelling per day (last: it rewrites the resident z)
    Pt, hn_ref, lo_ref, hi_ref, off_ref = UO.reference_tail_stack(hm, mask, detrend=False)
    np.testing.assert_array_equal(engine.segment_offsets, off_ref)
    lo, hi, hn = engine.ground_level(True)
    np.testing.assert_array_equal(lo, lo_ref)
    np.testing.assert_array_equal(hi, hi_ref)
    np.testing.assert_array_equal(hn, hn_ref.astype(np.float32))
    np.testing.assert_array_equal(engine.get_cloud(False)[:, 2], Pt[:, 2].astype(np.float32))


# ---------------------------------------------------------------------------------------
# 8. non-finite centroids are rejected
# ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_non_finite_centroids_rejected(pkg, engine, bad):
    disp, mask, P = dyadic_raster(1, 20, 30, seed=12)
    hm = UO.height_from_disparity(disp).astype(np.float32)
    hm[~mask] = np.nan
    unproject_dyadic(engine, disp, mask, P)
    for k, row, col in ((3, 0, 0), (40, 39, 2), (300, 150, 1)):
        C = dyadic_centroids(P, k, seed=k)
        C[row, col] = bad
        calls = (lambda: engine.fit(C, max_iter=3), lambda: engine.predict(C), lambda: engine.lloyd_step(C),
                 lambda: pkg.fuse_multiday_kmeans(hm, n_clusters=k, init=C, max_iter=3, engine=engine))
        for call in calls:
            with pytest.raises(cabi.MdkmError) as ei:
                call()
            assert ei.value.code == ERR_INVALID and "non-finite" in str(ei.value)
    unproject_dyadic(engine, disp, mask, P)
    C = dyadic_centroids(P, 3, seed=3)
    np.testing.assert_array_equal(engine.predict(C)[0], dyadic_argmin(P, C))  # the handle still works
