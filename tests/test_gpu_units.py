"""Detection in any unit.  Scaling the coordinates and both radii by 2^k leaves every result bit-identical
(tests/test_oracle_units.py pins that on the oracle), so a scaled bundled view has the committed goldens and the
unit-scale GPU run on its other side -- and the scale alone decides which variant of the feature kernel runs: the FAST
one needs r2 <= 2^40 and adim >= 2^-20 (features.cu: launch_features), every other radius runs the exact variants, whose
scalar vote loop no unit-scale test reaches.  stats()["fast_math"] proves which variant ran.

Also here: both range limits of the FAST path at A = 4, B = 8 (power-of-two divisors, so only the range guards decide),
the exact variants under slab sharding and on organized frames, and the band where FP32 goes subnormal, against the
oracle at the same scale."""
import hashlib

import numpy as np
import pytest

from conftest import forest_path

pytestmark = pytest.mark.gpu

R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85
F32 = np.float32
VIEWS = ("cheff000", "cheff001", "cheff002")
FORESTS = [forest_path(f) for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]
# (k of the 2^k scale, the feature kernel variant expected: 1 FAST, 0 exact).  At A = 5: adim = 2^(k+2), r2 = 400 * 4^k
SCALE_MATRIX = [(-50, 0), (-23, 0),     # adim < 2^-20
                (-22, 1),               # adim = 2^-20
                (0, 1), (15, 1),        # r2 <= 2^40
                (16, 0), (20, 0), (45, 0)]  # r2 > 2^40
SCALES = [k for k, _ in SCALE_MATRIX if k != 0]
FAST = dict(SCALE_MATRIX)


def same_bits(a, b):
    """bit-identical float arrays; NaNs compare equal whatever their payload (the device writes 0x7FFFFFFF, x86 0/0 gives
    0xFFC00000), so NaN positions must agree"""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def scaled(xyz, k):
    return np.ascontiguousarray(xyz * F32(2.0 ** k))


def detector(kpl, k, forests=FORESTS[:1], A=5, B=10, r_feat=R_FEAT, r_nms=R_NMS, th=TH, fragile=False):
    """TestDetector's configuration with both radii scaled by 2^k (exactly: r_feat and r_nms are floats)"""
    s = F32(2.0 ** k)
    d = kpl.KeypointLearningDetector()
    d.setNAnnulus(A); d.setNBins(B); d.setNonMaxima(True); d.setNonMaximaDrawsRemove(False)
    d.setRadiusSearch(float(F32(r_feat) * s)); d.setNonMaxRadius(float(F32(r_nms) * s))
    d.setPredictionThreshold(float(F32(th))); d.setNormalsMode(1, k=10); d.setReportFragile(fragile)
    assert d.loadForest(forests[0])
    for i, f in enumerate(forests[1:]):
        assert d.addForest(f) == i + 1
    return d


# ---------------------------------------------------------------------------------------------
# the scale matrix: every entry point at every scale, bit-identical to the unit-scale run and to the goldens
# ---------------------------------------------------------------------------------------------
def run_compute(kpl, views, k, fragile=False):
    xyz = scaled(views["cheff001"], k)
    n = len(xyz)
    d = detector(kpl, k, fragile=fragile)
    d.keepIntermediates(True)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    out = dict(normals=d.fetch("normals", n, 4), features=d.fetch("features", n, 50), scores=d.getResponse().copy(),
               keypoints=idx, stats=d.stats())
    if fragile:
        out["fragile"] = d.fetchFragile(n)
    d.close()
    return out


def run_forests(kpl, views, k, fragile=False):
    xyz = scaled(views["cheff001"], k)
    d = detector(kpl, k, forests=FORESTS, fragile=fragile)
    d.setInputCloud(xyz)
    res = d.computeForests()
    out = dict(scores=d.getResponses().copy(), keypoints=[r[1] for r in res], stats=d.stats())
    if fragile:
        out["fragile"] = d.fetchFragile(len(FORESTS) * len(xyz))
    d.close()
    return out


def subset(n, stride):
    """a scattered index list: the golden rows (every `stride`-th point) and 1500 others, shuffled; and where the golden
    rows went"""
    rng = np.random.default_rng(17)
    g = np.arange(0, n, stride)
    idx = np.concatenate([g, rng.choice(np.setdiff1d(np.arange(n), g), 1500, replace=False)]).astype(np.int32)
    perm = rng.permutation(len(idx))
    return idx[perm], np.argsort(perm)[:len(g)]


def run_subset(kpl, views, golden, k):
    xyz = scaled(views["cheff001"], k)
    sub, _ = subset(len(xyz), int(golden["cheff001"]["stride"]))
    d = detector(kpl, k)
    d.setInputCloud(xyz); d.setNormals(None)                    # the normals are estimated on the device (kNN-10)
    rows = d.computePointsForTrainingFeatures(sub)
    out = dict(features=rows, stats=d.stats())
    d.close()
    return out


def run_batch(kpl, views, k):
    d = detector(kpl, k)
    sc, kp = d.computeBatch([scaled(views[v], k) for v in VIEWS])
    out = dict(scores=[s.copy() for s in sc], keypoints=kp, stats=d.stats())
    d.close()
    return out


def run_batch_forests(kpl, views, k):
    d = detector(kpl, k, forests=FORESTS)
    res = d.computeBatchForests([scaled(views[v], k) for v in VIEWS])
    out = dict(scores=[[s.copy() for s, _ in r] for r in res], keypoints=[[i for _, i in r] for r in res], stats=d.stats())
    d.close()
    return out


@pytest.fixture(scope="module")
def unit_runs(kpl, views, golden):
    """the unit-scale runs of every entry point (k = 0), computed once"""
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = {"compute": lambda: run_compute(kpl, views, 0), "fragile": lambda: run_compute(kpl, views, 0, True),
                           "forests": lambda: run_forests(kpl, views, 0), "forests_fragile": lambda: run_forests(kpl, views, 0, True),
                           "subset": lambda: run_subset(kpl, views, golden, 0), "batch": lambda: run_batch(kpl, views, 0),
                           "batch_forests": lambda: run_batch_forests(kpl, views, 0)}[name]()
            assert cache[name]["stats"]["fast_math"] == FAST[0], name
        return cache[name]
    return get


def assert_counters(st, ref, k):
    assert st["fast_math"] == FAST[k], (k, st["fast_math"])
    assert st["feature_pairs"] == ref["feature_pairs"] and st["candidate_pairs"] == ref["candidate_pairs"]


def assert_golden_single(r, g):
    assert sha(r["normals"]) == str(g["normals_sha"])
    assert sha(r["features"]) == str(g["features_sha"])
    assert np.array_equal(r["scores"].view(np.uint32), g["scores"].view(np.uint32))
    assert np.array_equal(r["keypoints"], g["keypoints"])


@pytest.mark.parametrize("fragile", [False, True], ids=["plain", "fragile"])
@pytest.mark.parametrize("k", SCALES)
def test_compute_any_unit(kpl, views, golden, unit_runs, k, fragile):
    """compute(): the single-forest kernel, and with setReportFragile the FRAGILE one (mask unchanged too)"""
    r = run_compute(kpl, views, k, fragile)
    u = unit_runs("fragile" if fragile else "compute")
    assert_counters(r["stats"], u["stats"], k)
    for key in ("normals", "features", "scores"):
        assert same_bits(r[key], u[key]), key
    assert np.array_equal(r["keypoints"], u["keypoints"])
    assert_golden_single(r, golden["cheff001"])
    if fragile:
        assert np.array_equal(r["fragile"], u["fragile"])
        assert r["stats"]["n_fragile_points"] == u["stats"]["n_fragile_points"] == int(r["fragile"].sum()) > 0


@pytest.mark.parametrize("fragile", [False, True], ids=["plain", "fragile"])
@pytest.mark.parametrize("k", SCALES)
def test_compute_forests_any_unit(kpl, views, golden, unit_runs, k, fragile):
    """computeForests() with three forests: the forest-set kernel, with and without the fragile report"""
    r = run_forests(kpl, views, k, fragile)
    u = unit_runs("forests_fragile" if fragile else "forests")
    assert_counters(r["stats"], u["stats"], k)
    assert same_bits(r["scores"], u["scores"])
    for f in range(len(FORESTS)):
        assert np.array_equal(r["keypoints"][f], u["keypoints"][f]), f
    assert np.array_equal(r["scores"][0].view(np.uint32), golden["cheff001"]["scores"].view(np.uint32))
    assert np.array_equal(r["keypoints"][0], golden["cheff001"]["keypoints"])
    if fragile:
        assert np.array_equal(r["fragile"], u["fragile"]) and r["fragile"].sum() > 0


@pytest.mark.parametrize("k", SCALES)
def test_feature_subset_any_unit(kpl, views, golden, unit_runs, k):
    """computePointsForTrainingFeatures on a scattered index subset: the query-list path of the kernel"""
    r = run_subset(kpl, views, golden, k)
    u = unit_runs("subset")
    assert_counters(r["stats"], u["stats"], k)
    assert same_bits(r["features"], u["features"])
    g = golden["cheff001"]
    _, at = subset(len(views["cheff001"]), int(g["stride"]))
    assert np.array_equal(r["features"][at].view(np.uint32), g["features_rows"].view(np.uint32))


@pytest.mark.parametrize("k", SCALES)
def test_batch_any_unit(kpl, views, golden, unit_runs, k):
    """computeBatch() over the three bundled views"""
    r = run_batch(kpl, views, k)
    u = unit_runs("batch")
    assert_counters(r["stats"], u["stats"], k)
    for v, name in enumerate(VIEWS):
        assert np.array_equal(r["scores"][v].view(np.uint32), golden[name]["scores"].view(np.uint32)), name
        assert np.array_equal(r["keypoints"][v], golden[name]["keypoints"]), name


@pytest.mark.parametrize("k", SCALES)
def test_batch_forests_any_unit(kpl, views, golden, unit_runs, k):
    """computeBatchForests() with three forests over the three bundled views"""
    r = run_batch_forests(kpl, views, k)
    u = unit_runs("batch_forests")
    assert_counters(r["stats"], u["stats"], k)
    for f in range(len(FORESTS)):
        for v, name in enumerate(VIEWS):
            assert same_bits(r["scores"][f][v], u["scores"][f][v]), (f, name)
            assert np.array_equal(r["keypoints"][f][v], u["keypoints"][f][v]), (f, name)
    for v, name in enumerate(VIEWS):
        assert np.array_equal(r["scores"][0][v].view(np.uint32), golden[name]["scores"].view(np.uint32)), name
        assert np.array_equal(r["keypoints"][0][v], golden[name]["keypoints"]), name


# ---------------------------------------------------------------------------------------------
# the range limits of the FAST path, at A = 4, B = 8 (every divisor a power of two: only the range guards decide)
# ---------------------------------------------------------------------------------------------
BOUNDARIES = {
    # name: (cloud scale k, radius, unscaled radius with the same result, variant expected at scale)
    "r2_eq_2^40": (16, F32(2.0 ** 20), F32(16.0), 1),                      # neighbours fill [2^39, 2^40)
    "r2_above_2^40": (16, np.nextafter(F32(2.0 ** 20), F32(np.inf)), F32(16.0 * (1 + 2.0 ** -23)), 0),
    "adim_eq_2^-20": (-22, F32(2.0 ** -18), F32(16.0), 1),
    "adim_below_2^-20": (-22, np.nextafter(F32(2.0 ** -18), F32(0)), F32(16.0 * (1 - 2.0 ** -24)), 0),
}


def flann_d2(p, c):
    """the radius-membership expression of the kernel and the oracle, in float32: ((dx*dx) + dy*dy) + dz*dz"""
    d = (p.astype(np.float32) - c.astype(np.float32)).astype(np.float32)
    return ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]).astype(np.float32) + d[..., 2] * d[..., 2]).astype(np.float32)


def test_neighbours_fill_the_top_binade(views):
    """the r2 = 2^40 case really feeds the fast square root the top binade of its range"""
    from scipy.spatial import cKDTree
    xyz = scaled(views["cheff001"], 16)
    q = np.random.default_rng(5).choice(len(xyz), 300, replace=False)
    nb = cKDTree(xyz.astype(np.float64)).query_ball_point(xyz[q].astype(np.float64), 2.0 ** 20 * 1.001)
    d2 = np.concatenate([flann_d2(xyz[i], xyz[np.asarray(j)]) for i, j in zip(q, nb)])
    top = np.count_nonzero((d2 >= F32(2.0 ** 39)) & (d2 < F32(2.0 ** 40)))
    assert top > 0.4 * np.count_nonzero(d2 < F32(2.0 ** 40))


@pytest.mark.parametrize("case", list(BOUNDARIES))
def test_fast_path_boundaries(kpl, views, oracle, case):
    k, r, r_unit, fast = BOUNDARIES[case]
    assert F32(r) == F32(r_unit * F32(2.0 ** k))
    forest = forest_path("synthetic-A4xB8-T20-D8")
    runs = []
    for kk, rr in ((k, r_unit), (0, r_unit)):
        xyz = scaled(views["cheff001"], kk)
        n = len(xyz)
        d = detector(kpl, kk, forests=[forest], A=4, B=8, r_feat=rr, th=0.5)
        d.keepIntermediates(True)
        d.setInputCloud(xyz)
        _, idx = d.compute()
        runs.append(dict(normals=d.fetch("normals", n, 4), features=d.fetch("features", n, 32), scores=d.getResponse().copy(),
                         keypoints=idx, stats=d.stats()))
        d.close()
    got, unit = runs
    assert got["stats"]["fast_math"] == fast          # (the unscaled run's variant is the self-test's verdict on its divisor)
    assert got["stats"]["feature_pairs"] == unit["stats"]["feature_pairs"]
    s = F32(2.0 ** k)
    ref = oracle.detect(scaled(views["cheff001"], k), oracle.load_forest_yaml(forest), float(r), float(F32(R_NMS) * s), 0.5, 4, 8,
                        normals_mode=1, k=10, order=1)
    for key in ("normals", "features", "scores"):
        assert same_bits(got[key], unit[key]), key
        assert same_bits(got[key], ref[key]), key
    assert np.array_equal(got["keypoints"], unit["keypoints"]) and np.array_equal(got["keypoints"], ref["keypoints"])
    assert len(got["keypoints"]) > 1000


# ---------------------------------------------------------------------------------------------
# other paths that run the exact variants
# ---------------------------------------------------------------------------------------------
def test_slab_results_equal_unsharded_exact_variant(kpl, views):
    """in-process slab sharding, world 2, at 2^16 (r2 > 2^40): every slab's scores bit-identical to the unsharded run,
    the keypoints their union -- as test_gpu_parity.py::test_slab_results_equal_unsharded at unit scale"""
    from keypoint_learning_b200 import shard
    from test_gpu_parity import _role_slab
    k, world = 16, 2
    s = F32(2.0 ** k)
    xyz = np.ascontiguousarray(views["cheff001"][:, [1, 0, 2]])      # the longest axis (y) onto x, the slab axis
    full = []
    for kk in (0, k):
        d = detector(kpl, kk)
        d.setInputCloud(scaled(xyz, kk))
        _, idx = d.compute()
        full.append((d.getResponse().copy(), idx, d.stats()["fast_math"]))
        d.close()
    assert full[1][2] == 0
    assert same_bits(full[0][0], full[1][0]) and np.array_equal(full[0][1], full[1][1])
    sc_full, idx_full, _ = full[1]
    xyz_s = scaled(xyz, k)
    plan = shard.plan_slabs(xyz_s, float(F32(R_FEAT) * s), float(F32(R_NMS) * s), 4, world)
    d = detector(kpl, k)
    kps, seen = [], np.zeros(len(xyz), bool)
    for rank in range(world):
        sl = _role_slab(xyz_s, plan, rank)
        d.setForcedGrid(plan.origin, sl["local_dims"], sl["offset"])
        d.setInputCloud(sl["xyz4"])
        _, idx = d.compute(role=sl["role"])
        sc = d.getResponse()
        assert d.stats()["fast_math"] == 0
        owned = sl["role"] == 3
        scored = (sl["role"] & 1) == 1
        assert np.all(np.isnan(sc[~scored]))
        assert not seen[sl["gidx"][owned]].any()
        seen[sl["gidx"][owned]] = True
        assert np.array_equal(sc[scored].view(np.uint32), sc_full[sl["gidx"][scored]].view(np.uint32))
        assert np.all(owned[idx])
        kps.append(sl["gidx"][idx])
    assert seen.all()
    assert np.array_equal(np.sort(np.concatenate(kps)), idx_full)
    d.close()


def organized_frames(k):
    """three 160 x 120 range images (holes in frames 0 and 2) scaled by 2^k.  Not a unit-free check: the depth-change
    test of the integral-image normals has an absolute term, so these frames are compared with the oracle as they are"""
    from keypoint_learning_b200 import synth
    fr = np.stack([synth.organized_range_image(160, 120, seed=11 + f, holes=f % 2 == 0)[0] for f in range(3)])
    return np.ascontiguousarray(fr * F32(2.0 ** k))


def test_organized_batches_exact_variant(kpl, oracle):
    """computeOrganizedBatch and computeOrganizedBatchForests with radius_features = 20 * 2^16 > 2^20 (r2 > 2^40) against
    the oracle on the same frames"""
    k = 16
    s = F32(2.0 ** k)
    r_feat, r_nms, th = float(F32(R_FEAT) * s), float(F32(R_NMS) * s), 0.5
    fr = organized_frames(k)
    d = detector(kpl, k, th=th)
    sc_b, kp_b = d.computeOrganizedBatch(fr)
    assert d.stats()["fast_math"] == 0
    d.close()
    d = detector(kpl, k, forests=FORESTS, th=th)
    res = d.computeOrganizedBatchForests(fr)
    assert d.stats()["fast_math"] == 0
    d.close()
    forests = [oracle.load_forest_yaml(f) for f in FORESTS]
    nkp = 0
    for f in range(len(fr)):
        flat = fr[f].reshape(-1, 3)
        nrm = oracle.normals_integral_image(fr[f], 5.0, (0.0, 0.0, 0.0))
        keep = np.nonzero(np.isfinite(flat).all(axis=1))[0]
        pts = np.ascontiguousarray(flat[keep])
        feat = oracle.features(pts, nrm[keep], r_feat, 5, 10, order=1)
        for j, forest in enumerate(forests):
            sc = oracle.scores(forest, feat, nrm[keep])
            kp = keep[oracle.nms(pts, sc, r_nms, th)]
            got = [(res[j][f][0], res[j][f][1])] + ([(sc_b[f], kp_b[f])] if j == 0 else [])
            for sc_g, kp_g in got:
                assert same_bits(sc_g[keep], sc), (f, j)
                assert np.all(np.isnan(np.delete(sc_g, keep))), (f, j)
                assert np.array_equal(kp_g, kp), (f, j)
            nkp += len(kp)
    assert nkp > 0


# ---------------------------------------------------------------------------------------------
# the subnormal band: squared distances, covariances and moments below FLT_MIN
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [-56, -60, -62, -64])
def test_subnormal_band_against_oracle(kpl, views, oracle, main_forest, k):
    xyz = scaled(views["cheff001"], k)
    n = len(xyz)
    s = F32(2.0 ** k)
    d = detector(kpl, k)
    d.keepIntermediates(True)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    st = d.stats()
    ref = oracle.detect(xyz, main_forest, float(F32(R_FEAT) * s), float(F32(R_NMS) * s), TH, 5, 10, normals_mode=1, k=10, order=1)
    assert st["fast_math"] == 0
    assert same_bits(d.fetch("normals", n, 4), ref["normals"])
    assert same_bits(d.fetch("features", n, 50), ref["features"])
    assert same_bits(d.getResponse(), ref["scores"])
    assert np.array_equal(idx, ref["keypoints"])
    assert st["n_unscored"] == int(np.isnan(ref["scores"]).sum())
    d.close()
    # stand-alone normals: the k-NN grid is sized from the data, not from radius_features
    d = kpl.KeypointLearningDetector()
    d.setNormalsMode(1, k=10)
    assert same_bits(d.computeNormals(xyz), oracle.normals_knn(xyz, 10))
    d.close()
