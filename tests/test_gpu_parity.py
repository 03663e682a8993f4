"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on
the same inputs and against the committed golden vectors.

Bars (BASELINE.json north_star): neighbour index sets and NMS keypoint indices bit-exact;
feature histograms and forest scores within 1e-5 absolute.  Because the oracle (order=1) and the
kernels share one arithmetic contract (FP32 RN, no FMA, canonical accumulation order), the tests
demand MORE than the bar: bit-identical normals, features and scores.  The 1e-5 tolerance is then
checked between the GPU result and the grid-free oracle (order=0: ascending-index accumulation),
whose score differences are the "fragile decisions" the north star asks to report separately.
"""
import hashlib
import os

import numpy as np
import pytest

from conftest import forest_path

pytestmark = pytest.mark.gpu

R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85
TOL = 1e-5   # absolute tolerance of north_star for features and scores


def same_bits(a, b):
    """Bit-identical float arrays; NaNs compare equal whatever their payload (the device writes 0x7FFFFFFF, x86 0/0
    gives 0xFFC00000: both mean "no value")."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def make_detector(kpl, forest=None, **kw):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(kw.get("A", 5)); det.setNBins(kw.get("B", 10))
    det.setNonMaxima(True); det.setNonMaxRadius(kw.get("r_nms", R_NMS)); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(kw.get("th", TH)))); det.setRadiusSearch(kw.get("r_feat", R_FEAT))
    det.setCellsPerRadius(kw.get("cpr", 4))
    assert det.loadForest(forest or forest_path())
    return det


@pytest.fixture(scope="module")
def det(kpl):
    d = make_detector(kpl)
    yield d
    d.close()


# ---------------------------------------------------------------------------------------------
# radius search: neighbour index sets, bit-exact
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("view", ["cheff000", "cheff001", "cheff002"])
def test_neighbor_counts_match_golden(det, views, golden, view):
    xyz = views[view]
    c20, _ = det.radiusStats(xyz, R_FEAT)
    assert np.array_equal(c20, golden[view]["counts_r20"])
    assert int(c20.sum()) == int(golden[view]["pairs_r20"])
    c4, _ = det.radiusStats(xyz, R_NMS)
    assert np.array_equal(c4, golden[view]["counts_r4"])


def test_neighbor_sets_bit_exact(det, views, oracle):
    xyz = views["cheff001"]
    rng = np.random.default_rng(3)
    q = np.sort(rng.choice(len(xyz), 400, replace=False)).astype(np.int32)
    for r in (R_NMS, R_FEAT, 7.3):
        off_o, idx_o = oracle.radius_neighbors(xyz, r, q)
        off_g, idx_g = det.radiusNeighbors(xyz, r, q)
        assert np.array_equal(off_o, off_g)
        assert np.array_equal(idx_o, idx_g)
    # hash of the full neighbour sets of every point vs the oracle lists
    _, h = det.radiusStats(xyz, R_NMS)
    off, idx = oracle.radius_neighbors(xyz, R_NMS)
    mul = np.uint64(0x9E3779B97F4A7C15)
    contrib = (idx.astype(np.uint64) + np.uint64(1)) * mul
    ref = np.add.reduceat(contrib, off[:-1].astype(np.int64)) if len(idx) else np.zeros(len(xyz), np.uint64)
    assert np.array_equal(h, ref)


def test_neighbor_counts_brute_force_crop(det, views, oracle):
    xyz = np.ascontiguousarray(views["cheff002"][:12000])
    for r in (2.0, 20.0):
        c, _ = det.radiusStats(xyz, r)
        assert np.array_equal(c, oracle.radius_counts(xyz, r, brute=True))


# ---------------------------------------------------------------------------------------------
# normals
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("view", ["cheff000", "cheff001", "cheff002"])
def test_knn_normals_bit_exact(det, views, golden, oracle, view):
    xyz = views[view]
    det.setNormalsMode(1, k=10)
    n_gpu = det.computeNormals(xyz)
    n_cpu = oracle.normals_knn(xyz, 10)
    assert np.array_equal(n_gpu.view(np.uint32), n_cpu.view(np.uint32))
    assert sha(n_gpu) == str(golden[view]["normals_sha"])


def test_knn_normals_other_k_and_viewpoint(det, views, oracle):
    xyz = np.ascontiguousarray(views["cheff001"][::3])
    for k, vp, flip in ((5, (0.0, 0.0, 1000.0), False), (16, (10.0, -20.0, 30.0), True), (23, (0.0, 0.0, 0.0), False)):
        det.setNormalsMode(1, k=k, viewpoint=vp, flip=flip)
        n_gpu = det.computeNormals(xyz)
        n_cpu = oracle.normals_knn(xyz, k, vp)
        if flip:
            n_cpu[:, :3] *= -1
        assert np.array_equal(n_gpu.view(np.uint32), n_cpu.view(np.uint32))
    det.setNormalsMode(1, k=10)


def test_radius_normals_bit_exact_and_pipeline(kpl, views, oracle, main_forest):
    """F2' (hpp:130-137): PCA normals over the r_feat ball when setNormals() was not called.  The device
    adds the moments in canonical (cell, index) order = oracle order 1; the whole pipeline on top of those
    normals must then reproduce the oracle's scores and keypoints exactly."""
    xyz = np.ascontiguousarray(views["cheff001"][:30000])
    d = make_detector(kpl)
    for r, vp, flip in ((20.0, (0.0, 0.0, 0.0), False), (7.5, (5.0, -3.0, 400.0), True)):
        d.setRadiusSearch(r)
        d.setNormalsMode(2, viewpoint=vp, flip=flip)
        n_gpu = d.computeNormals(xyz)
        n_cpu = oracle.normals_radius(xyz, r, vp, order=1)
        if flip:
            n_cpu[:, :3] *= -1
        same = (n_gpu.view(np.uint32) == n_cpu.view(np.uint32)) | (np.isnan(n_gpu) & np.isnan(n_cpu))
        assert same.all(), np.argwhere(~same)[:5]
    d.setRadiusSearch(R_FEAT)
    d.setNormalsMode(2)
    d.setInputCloud(xyz); d.setNormals(None)
    _, idx = d.compute()
    ref = oracle.detect(xyz, main_forest, R_FEAT, R_NMS, TH, 5, 10, normals_mode=2, order=1)
    assert np.array_equal(d.getResponse().view(np.uint32), ref["scores"].view(np.uint32))
    assert np.array_equal(idx, ref["keypoints"])
    d.close()


# ---------------------------------------------------------------------------------------------
# features
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("view", ["cheff000", "cheff001", "cheff002"])
def test_features_bit_exact_and_within_tolerance(det, views, golden, oracle, view):
    xyz = views[view]
    nrm = oracle.normals_knn(xyz, 10)
    det.setInputCloud(xyz); det.setNormals(nrm)
    f_gpu = det.computePointsForTrainingFeatures()
    g = golden[view]
    assert sha(f_gpu) == str(g["features_sha"])
    assert np.array_equal(f_gpu[::int(g["stride"])], g["features_rows"])
    # north-star tolerance against the grid-free accumulation order
    sub = np.arange(0, len(xyz), 41, dtype=np.int32)
    f0 = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=0, qidx=sub)
    assert np.abs(f_gpu[sub] - f0).max() <= TOL


def test_features_subset_and_shapes(kpl, views, oracle):
    xyz = views["cheff001"]
    nrm = oracle.normals_knn(xyz, 10)
    sub = np.random.default_rng(5).choice(len(xyz), 300, replace=False).astype(np.int32)
    for A, B, r in ((5, 10, 20.0), (10, 5, 20.0), (4, 8, 10.0), (8, 16, 40.0), (1, 1, 5.0), (3, 7, 12.5)):
        d = kpl.KeypointLearningDetector()
        d.setNAnnulus(A); d.setNBins(B); d.setRadiusSearch(r)
        d.setInputCloud(xyz); d.setNormals(nrm)
        f_gpu = d.computePointsForTrainingFeatures(sub)
        f_cpu = oracle.features(xyz, nrm, r, A, B, order=1, qidx=sub)
        assert f_gpu.shape == (len(sub), A * B)
        assert np.array_equal(f_gpu.view(np.uint32), f_cpu.view(np.uint32)), (A, B, r)
        d.close()


@pytest.mark.parametrize("cpr", [2, 3, 6, 8])
def test_features_other_grid_resolutions(kpl, views, oracle, cpr):
    xyz = np.ascontiguousarray(views["cheff000"][::2])
    nrm = oracle.normals_knn(xyz, 10)
    sub = np.arange(0, len(xyz), 53, dtype=np.int32)
    d = kpl.KeypointLearningDetector()
    d.setRadiusSearch(R_FEAT); d.setCellsPerRadius(cpr)
    d.setInputCloud(xyz); d.setNormals(nrm)
    f_gpu = d.computePointsForTrainingFeatures(sub)
    f_cpu = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1, cpr=cpr, qidx=sub)
    assert np.array_equal(f_gpu.view(np.uint32), f_cpu.view(np.uint32))
    d.close()


def test_nan_neighbor_normals_are_skipped(kpl, views, oracle):
    xyz = np.ascontiguousarray(views["cheff001"][:20000])
    nrm = oracle.normals_knn(xyz, 10)
    bad = np.arange(7, len(xyz), 13)
    nrm[bad, :3] = np.nan
    sub = np.setdiff1d(np.arange(0, len(xyz), 29), bad).astype(np.int32)
    d = kpl.KeypointLearningDetector()
    d.setRadiusSearch(R_FEAT); d.setInputCloud(xyz); d.setNormals(nrm)
    f_gpu = d.computePointsForTrainingFeatures(sub)
    f_cpu = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1, qidx=sub)
    assert np.array_equal(f_gpu.view(np.uint32), f_cpu.view(np.uint32))
    d.close()


# ---------------------------------------------------------------------------------------------
# forest + scores + NMS: the full TestDetector path
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("view", ["cheff000", "cheff001", "cheff002"])
def test_full_pipeline_matches_golden(det, views, golden, view):
    """config 1: bundled view, TestDetector defaults, normals estimated on the GPU (kNN-10)."""
    xyz = views[view]
    g = golden[view]
    det.setNormalsMode(1, k=10)
    det.setInputCloud(xyz); det.setNormals(None)
    kp, idx = det.compute()
    sc = det.getResponse()
    assert np.array_equal(sc.view(np.uint32), g["scores"].view(np.uint32))       # bit-exact, hence <= 1e-5
    assert np.array_equal(idx, g["keypoints"])                                   # NMS indices bit-exact
    assert np.array_equal(kp[:, :3], xyz[idx]) and np.array_equal(kp[:, 3], sc[idx])
    st = det.stats()
    assert st["n_above_threshold"] == int(g["n_above"])
    assert st["feature_pairs"] == int(g["pairs_r20"]) - len(xyz)                 # self excluded
    assert st["n_keypoints"] == len(idx)
    # tolerance report against the grid-free order: scores that differ are fragile tree decisions
    assert len(np.setxor1d(idx, g["keypoints_order0"])) <= 2 * int(g["scores_order0_ndiff"])


def test_pipeline_with_given_normals_pcl_layout(det, views, golden, oracle):
    """setNormals() path with pcl::PointXYZ (16 B) / pcl::Normal (32 B) strides."""
    xyz = views["cheff001"]
    nrm = oracle.normals_knn(xyz, 10)
    xyz4 = np.ones((len(xyz), 4), np.float32); xyz4[:, :3] = xyz
    nrm8 = np.zeros((len(xyz), 8), np.float32); nrm8[:, :3] = nrm[:, :3]; nrm8[:, 4] = nrm[:, 3]
    det.setInputCloud(xyz4); det.setNormals(nrm8)
    _, idx = det.compute()
    assert np.array_equal(idx, golden["cheff001"]["keypoints"])
    assert np.array_equal(det.getResponse().view(np.uint32), golden["cheff001"]["scores"].view(np.uint32))
    det.setNormals(None)


@pytest.mark.parametrize("name,A,B", [("synthetic-SHOT-like-T50-D10", 5, 10), ("synthetic-FPFH-like-T30-D25", 5, 10),
                                      ("synthetic-A10xB5-T20-D8", 10, 5), ("synthetic-A4xB8-T20-D8", 4, 8),
                                      ("synthetic-A8xB16-T20-D8", 8, 16)])
def test_forest_sweep_config2(kpl, views, oracle, name, A, B):
    """config 2: other forests / (annuli, bins) shapes / radii, against the oracle."""
    xyz = views["cheff001"]
    nrm = oracle.normals_knn(xyz, 10)
    F = oracle.load_forest_yaml(forest_path(name))
    for r_feat, r_nms, th in ((20.0, 4.0, 0.85), (10.0, 3.0, 0.7)):
        d = make_detector(kpl, forest_path(name), A=A, B=B, r_feat=r_feat, r_nms=r_nms, th=th)
        d.setInputCloud(xyz); d.setNormals(nrm)
        _, idx = d.compute()
        feat = oracle.features(xyz, nrm, r_feat, A, B, order=1)
        sc = oracle.scores_from_sums(oracle.forest_sum(F, feat), F["ntrees"])
        assert np.array_equal(d.getResponse().view(np.uint32), sc.view(np.uint32))
        assert np.array_equal(idx, oracle.nms(xyz, sc, r_nms, th))
        d.close()


def test_forest_against_opencv(kpl, views, oracle):
    """The forest stage against the real OpenCV implementation (cv2.ml.RTrees, PREDICT_SUM)."""
    cv2 = pytest.importorskip("cv2")
    xyz = views["cheff002"]
    nrm = oracle.normals_knn(xyz, 10)
    rt = cv2.ml.RTrees_load(forest_path())
    d = make_detector(kpl)
    d.setInputCloud(xyz); d.setNormals(nrm)
    d.compute()
    sc_fused = d.getResponse().copy()
    with pytest.raises(kpl.KplError):                 # rows are not materialised by the fused default path
        d.fetch("features", len(xyz), 50)
    d.keepIntermediates(True)
    d.compute()
    assert np.array_equal(sc_fused.view(np.uint32), d.getResponse().view(np.uint32))
    feat = d.fetch("features", len(xyz), 50)
    _, res = rt.predict(feat, flags=cv2.ml.DTREES_PREDICT_SUM)
    ntrees = d.forestInfo()["ntrees"]
    sc_cv = (np.float32(1) - res.ravel().astype(np.float32) / np.float32(ntrees)).astype(np.float32)
    assert np.array_equal(d.getResponse().view(np.uint32), sc_cv.view(np.uint32))
    d.close()


def test_nms_semantics(kpl, oracle):
    """Threshold + local-maximum NMS (hpp:203-256) against the oracle on the golden scores for several radii and
    thresholds: plateaus survive, strictly greater neighbours suppress, d2 == r^2 does not count (hpp:219)."""
    xyz = np.load(os.path.join(os.path.dirname(__file__), "golden", "views", "cheff000.npz"))["xyz"]
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_cheff000.npz"))
    nrm = oracle.normals_knn(xyz, 10)
    for r_nms, th in ((4.0, 0.85), (1.0, 0.5), (8.0, 0.9), (0.0, 0.85), (4.0, 0.0), (4.0, 1.01)):
        d = make_detector(kpl, r_nms=r_nms, th=th)
        d.setInputCloud(xyz); d.setNormals(nrm)
        _, idx = d.compute()
        assert np.array_equal(idx, oracle.nms(xyz, g["scores"], r_nms, th)), (r_nms, th)
        # decisions within 1e-5 of the threshold are reported separately (north star): with T = 100 trees the
        # score k/100 sits exactly on 0.85 / 0.5 / 0.9 for many points
        thd = float(np.float32(th))
        near = int(np.sum(np.abs(g["scores"].astype(np.float64) - thd) <= 1e-5))
        assert d.stats()["n_near_threshold"] == near, (th, d.stats()["n_near_threshold"], near)
        d.close()


def test_nms_draws_remove_branch(kpl, views, oracle):
    """hpp:233-250 (setNonMaximaDrawsRemove(true), the class default): sequential skip-list semantics of the
    reference, resolved on the device in dependency rounds.  Scores are k/ntrees, so ties are everywhere."""
    xyz = views["cheff002"]
    nrm = oracle.normals_knn(xyz, 10)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_cheff002.npz"))
    total = 0
    for r_nms, th, dthr in ((4.0, 0.85, 2.0), (4.0, 0.5, 1.0), (8.0, 0.3, 8.0), (2.0, 0.0, 0.7), (4.0, 0.85, 0.0)):
        d = make_detector(kpl, r_nms=r_nms, th=th)
        d.setNonMaximaDrawsRemove(True); d.setNonMaximaDrawsThreshold(dthr)
        d.setInputCloud(xyz); d.setNormals(nrm)
        _, idx = d.compute()
        assert np.array_equal(d.getResponse().view(np.uint32), g["scores"].view(np.uint32))
        ref = oracle.nms(xyz, g["scores"], r_nms, th, draws_remove=True, draws_thr=dthr)
        assert np.array_equal(idx, ref), (r_nms, th, dthr, len(idx), len(ref))
        plain = oracle.nms(xyz, g["scores"], r_nms, th)
        assert set(idx.tolist()) <= set(plain.tolist())        # the branch only ever removes keypoints
        total += len(plain) - len(idx)
        d.close()
    assert total > 0                                            # the cases really exercise the branch


def test_uniform_sampling_matches_restatement(kpl, views, oracle):
    """--subSampling (main_test_detector.cpp:145-157): one survivor per voxel, closest to the centre."""
    d = kpl.KeypointLearningDetector()
    for view, leaf in (("cheff001", 2.0), ("cheff001", 0.5), ("cheff002", 7.5), ("cheff000", 500.0)):
        xyz = views[view]
        keep = d.uniformSample(xyz, leaf)
        ref = oracle.uniform_sample(xyz, leaf)
        assert np.array_equal(keep, ref), (view, leaf, len(keep), len(ref))
        keep_c = d.uniformSample(xyz, leaf, centre=True)                       # the voxel-centre variant
        assert np.array_equal(keep_c, oracle.uniform_sample(xyz, leaf, centre=True))
        assert len(keep_c) == len(keep) and (leaf > 100 or not np.array_equal(keep_c, keep))
        d.uniformSample(xyz, leaf)                                              # back to PCL 1.8.0's rule
        vox = np.floor(xyz[keep] * (np.float32(1.0) / np.float32(leaf)))
        assert len(np.unique(vox, axis=0)) == len(keep)                  # one survivor per voxel
    assert len(d.uniformSample(views["cheff000"], 500.0)) <= 8
    assert len(d.uniformSample(np.zeros((0, 3), np.float32), 1.0)) == 0
    with pytest.raises(kpl.KplError):
        d.uniformSample(views["cheff000"], 0.0)
    d.close()


def test_cuda_path_against_the_reference_templates(kpl, views, oracle, reference):
    """The CUDA path against oracle/_ref DIRECTLY: the reference's own computePointFeatures / runForest /
    detectKeypoints templates (or their recorded results where oracle/_ref is not built), fed with the canonical
    neighbour order the device uses."""
    xyz = np.ascontiguousarray(views["cheff002"][:3000])
    nrm = oracle.normals_knn(xyz, 10)
    forest = oracle.load_forest_yaml(forest_path("synthetic-SHOT-like-T50-D10"))
    lf = oracle.ref_neighbour_lists(xyz, R_FEAT, 1)
    ln = oracle.ref_neighbour_lists(xyz, R_NMS, 0)
    d = make_detector(kpl, forest=forest_path("synthetic-SHOT-like-T50-D10"), th=0.5)
    d.keepIntermediates(True)
    d.setInputCloud(xyz); d.setNormals(nrm)
    _, idx = d.compute()
    reference.check("cheff002_3k/features", d.fetch("features", len(xyz), 50), lambda: oracle.ref_features(xyz, nrm, R_FEAT, 5, 10, lf))
    reference.check("cheff002_3k/scores", d.getResponse(),
                    lambda: oracle.ref_detect(xyz, nrm, forest, R_FEAT, R_NMS, 0.5, 5, 10, lf, None, non_maxima=False)[1])
    reference.check("cheff002_3k/keypoints", idx, lambda: oracle.ref_detect(xyz, nrm, forest, R_FEAT, R_NMS, 0.5, 5, 10, lf, ln)[0])
    d.setNonMaximaDrawsRemove(True); d.setNonMaximaDrawsThreshold(1.5)
    _, idx_d = d.compute()
    reference.check("cheff002_3k/keypoints_draws", idx_d,
                    lambda: oracle.ref_detect(xyz, nrm, forest, R_FEAT, R_NMS, 0.5, 5, 10, lf, ln, draws_remove=True, draws_thr=1.5)[0])
    d.close()


def test_nearest_point_snap(kpl, views):
    """TrainDetector's 1-NN snap (main_train_detector.cpp:419-436) against brute force in the same FP32 expression."""
    xyz = np.ascontiguousarray(views["cheff000"][:20000])
    rng = np.random.default_rng(3)
    q = np.concatenate([xyz[rng.choice(len(xyz), 300, replace=False)] + rng.normal(0, 0.4, (300, 3)).astype(np.float32),
                        xyz[:50],                                                    # exact cloud points
                        np.float32([[1e4, 0, 0], [-500, -500, -500], [0, 0, 900]])]).astype(np.float32)   # far outside the bounding box
    d = make_detector(kpl)
    idx, d2 = d.nearest(xyz, q)
    for t in range(len(q)):
        e = q[t] - xyz
        dd = ((e[:, 0] * e[:, 0]) + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]
        j = int(np.argmin(dd))                                                       # first minimum = lowest index
        assert idx[t] == j and d2[t].view(np.uint32) == dd[j].view(np.uint32), t
    assert np.array_equal(idx[300:350], np.arange(50))
    d.close()


def test_non_maxima_off_returns_every_point(kpl, views, oracle):
    xyz = np.ascontiguousarray(views["cheff001"][:5000])
    d = make_detector(kpl)
    d.setNonMaxima(False)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    assert np.array_equal(idx, np.arange(len(xyz)))
    d.close()


# ---------------------------------------------------------------------------------------------
# error behaviour of the boundary
# ---------------------------------------------------------------------------------------------
def test_error_codes(kpl, views):
    xyz = np.ascontiguousarray(views["cheff001"][:3000])
    d = kpl.KeypointLearningDetector()
    d.setRadiusSearch(R_FEAT); d.setNonMaxRadius(R_NMS); d.setNonMaximaDrawsRemove(False)
    d.setInputCloud(xyz)
    with pytest.raises(kpl.KplError) as e:
        d.compute()
    assert e.value.code == 2                      # no forest
    assert not d.loadForest("/nonexistent/forest.yaml.gz")
    assert d.loadForest(forest_path("synthetic-A4xB8-T20-D8"))
    with pytest.raises(kpl.KplError) as e:
        d.compute()
    assert e.value.code == 5                      # var_count mismatch (5x10 vs 4x8)
    assert d.loadForest(forest_path())
    with pytest.raises(kpl.KplError) as e:
        d.setNormals(np.zeros((10, 4), np.float32)); d.compute()
    assert e.value.code == 3                      # normals size mismatch
    d.setNormals(None)
    bad = xyz.copy(); bad[17, 1] = np.nan
    with pytest.raises(kpl.KplError) as e:
        d.radiusStats(bad, R_NMS)
    assert e.value.code == 4                      # the C ABI refuses non-finite points ...
    d.setInputCloud(bad)
    _, idx = d.compute()                          # ... the detector facade skips them like the reference (hpp:277)
    assert 17 not in idx and np.isnan(d.getResponse()[17])
    d.setInputCloud(xyz)
    _, idx = d.compute()                          # context still usable after errors
    assert len(idx) >= 0
    d.close()


def test_empty_and_tiny_clouds(kpl, oracle):
    d = make_detector(kpl)
    d.setInputCloud(np.zeros((0, 3), np.float32))
    kp, idx = d.compute()
    assert len(idx) == 0 and kp.shape == (0, 4)
    # fewer than 3 points: kNN normals are NaN -> the points get no score (hpp:277) and no keypoint
    d.setInputCloud(np.array([[0, 0, 0], [1, 0, 0]], np.float32))
    kp, idx = d.compute()
    assert len(idx) == 0 and np.all(np.isnan(d.getResponse())) and d.stats()["n_unscored"] == 2
    # 5 points, k = 10 > n: all points are neighbours
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.1], [0.5, 0.5, 0.3]], np.float32)
    d.setInputCloud(pts)
    _, idx = d.compute()
    nrm = oracle.normals_knn(pts, 10)
    assert np.array_equal(d.fetch("normals", 5, 4).view(np.uint32), nrm.view(np.uint32))
    d.close()


def test_duplicate_points(kpl, oracle, main_forest):
    """exact duplicates: d2 == 0 neighbours that are not the query itself must vote."""
    base = np.load(os.path.join(os.path.dirname(__file__), "golden", "views", "cheff002.npz"))["xyz"][:8000]
    xyz = np.ascontiguousarray(np.concatenate([base, base[100:200], base[100:150]]))
    d = make_detector(kpl)
    d.keepIntermediates(True)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    nrm = oracle.normals_knn(xyz, 10)
    assert np.array_equal(d.fetch("normals", len(xyz), 4).view(np.uint32), nrm.view(np.uint32))
    feat = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1)
    assert np.array_equal(d.fetch("features", len(xyz), 50).view(np.uint32), feat.view(np.uint32))
    sc = oracle.scores_from_sums(oracle.forest_sum(main_forest, feat), main_forest["ntrees"])
    assert np.array_equal(idx, oracle.nms(xyz, sc, R_NMS, TH))
    d.close()


def test_scattered_clusters_and_isolated_points(kpl, oracle, main_forest):
    """The feature kernel's query list (Hilbert order, cut where the curve jumps; grid.cu: build_lists) on a cloud that is
    nothing but jumps: small clusters far apart, isolated points (warps of one query), and a cluster whose points are
    2e-21 apart (d2 in the denormal range: the branch-free square root must give what the IEEE one gives, features.cu)."""
    rng = np.random.default_rng(99)
    base = np.load(os.path.join(os.path.dirname(__file__), "golden", "views", "cheff000.npz"))["xyz"]
    parts = []
    for c in range(40):                                                    # 40 patches of 5..120 points, 300 apart
        m = int(rng.integers(5, 121))
        s = int(rng.integers(0, len(base) - 4000))
        blob = base[s:s + 4000]
        blob = blob[np.argsort(np.linalg.norm(blob - blob[0], axis=1))[:m]]
        parts.append(blob - blob[0] + np.array([300.0 * (c % 7), 300.0 * ((c // 7) % 3), 300.0 * (c // 21)], np.float32))
    parts.append(rng.uniform(-1000, 1000, (200, 3)).astype(np.float32))    # isolated points
    tiny = np.zeros((12, 3), np.float32)
    tiny[:, 0] = np.arange(12, dtype=np.float32) * np.float32(2e-21)       # d2 = 4e-42 .. : denormal squared distances
    tiny[:, 1] = (np.arange(12) % 3).astype(np.float32) * np.float32(1e-21)
    parts.append(tiny)                                                     # at the origin, inside the first patch
    xyz = np.ascontiguousarray(np.concatenate(parts).astype(np.float32))
    xyz = np.ascontiguousarray(xyz[rng.permutation(len(xyz))])
    nrm = oracle.normals_knn(xyz, 10)
    d = make_detector(kpl)
    d.keepIntermediates(True)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    assert same_bits(d.fetch("normals", len(xyz), 4), nrm)                 # (coincident points: NaN curvature on both sides)
    feat = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1)
    assert same_bits(d.fetch("features", len(xyz), 50), feat)
    sc = oracle.scores_from_sums(oracle.forest_sum(main_forest, feat), main_forest["ntrees"])
    sc = np.where(np.isfinite(nrm[:, :3]).all(1), sc, np.nan).astype(np.float32)      # no finite normal: unscored (hpp:277)
    assert same_bits(d.getResponse(), sc)
    assert np.array_equal(idx, oracle.nms(xyz, sc, R_NMS, TH))
    # an index subset that straddles the clusters (its own query list: 32 consecutive entries per warp, several groups)
    sub = rng.choice(len(xyz), 700, replace=False).astype(np.int32)
    d.setNormals(nrm)
    assert same_bits(d.computePointsForTrainingFeatures(sub), feat[sub])
    d.close()


# ---------------------------------------------------------------------------------------------
# full-size synthetic configuration: size-independent properties
# ---------------------------------------------------------------------------------------------
def test_synthetic_view_properties(kpl, oracle, main_forest):
    """config 3 generator at reduced size vs the oracle, then 1 M points through invariants."""
    from keypoint_learning_b200 import synth
    xyz, vp = synth.view_25d(300, 200, seed=9)
    d = make_detector(kpl)
    d.keepIntermediates(True)
    d.setNormalsMode(1, k=10, viewpoint=vp)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    nrm = oracle.normals_knn(xyz, 10, vp)
    feat = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1)
    sc = oracle.scores_from_sums(oracle.forest_sum(main_forest, feat), main_forest["ntrees"])
    assert np.array_equal(d.getResponse().view(np.uint32), sc.view(np.uint32))
    assert np.array_equal(idx, oracle.nms(xyz, sc, R_NMS, TH))

    xyz, vp = synth.view_25d(1250, 800, seed=1234)        # BASELINE.json configs[2]: 1 M points
    d.setInputCloud(xyz)
    _, idx = d.compute()
    sc = d.getResponse()
    st = d.stats()
    assert st["n_points"] == 1_000_000 and len(idx) == st["n_keypoints"]
    assert np.all(np.diff(idx) > 0)                                        # ascending, unique
    assert np.all(sc[idx].astype(np.float64) >= float(np.float32(TH)))     # thresholded
    q = np.round((1.0 - sc.astype(np.float64)) * main_forest["ntrees"])    # scores are k/ntrees quantised
    assert np.all(np.abs((1.0 - sc) * main_forest["ntrees"] - q) < 1e-3) and q.min() >= 0 and q.max() <= main_forest["ntrees"]
    # permutation invariance: shuffling the input permutes scores and keypoints, nothing else
    perm = np.random.default_rng(0).permutation(len(xyz))
    d.setInputCloud(np.ascontiguousarray(xyz[perm]))
    _, idx_p = d.compute()
    feat_rows = d.fetch("features", len(xyz), 50)
    # features are sums in canonical (cell, index) order: a permutation changes the order inside a
    # cell, so scores may differ only through FP32 re-association -> compare within tolerance
    assert np.abs(feat_rows - 0).max() <= 1.0 + 1e-6
    sc_p = d.getResponse()
    frac_diff = np.mean(sc_p != sc[perm])
    assert frac_diff < 5e-3, frac_diff
    # exact oracle check of a sample of the full-size result
    sub = np.random.default_rng(1).choice(len(xyz), 256, replace=False).astype(np.int32)
    d.setInputCloud(xyz)
    d.compute()
    nrm_g = d.fetch("normals", len(xyz), 4)
    f_cpu = oracle.features(xyz, nrm_g, R_FEAT, 5, 10, order=1, qidx=sub)
    f_gpu = d.fetch("features", len(xyz), 50)[sub]
    assert np.array_equal(f_gpu.view(np.uint32), f_cpu.view(np.uint32))
    d.close()


def test_query_without_finite_normal_is_unscored(kpl, views, oracle, main_forest):
    """hpp:277: a point whose normal is NaN gets no score, is no keypoint and suppresses nobody."""
    xyz = np.ascontiguousarray(views["cheff000"][:25000])
    nrm = oracle.normals_knn(xyz, 10)
    bad = np.arange(3, len(xyz), 17)
    nrm[bad, 1] = np.nan
    d = make_detector(kpl)
    d.keepIntermediates(True)
    d.setInputCloud(xyz); d.setNormals(nrm)
    _, idx = d.compute()
    sc_gpu = d.getResponse()
    feat = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1)
    sc = oracle.scores(main_forest, feat, nrm)
    assert np.all(np.isnan(sc_gpu[bad])) and d.stats()["n_unscored"] == len(bad)
    ok = ~np.isnan(sc)
    assert np.array_equal(np.isnan(sc_gpu), ~ok)                      # NaN payloads differ between C and CUDA
    assert np.array_equal(sc_gpu[ok].view(np.uint32), sc[ok].view(np.uint32))
    assert np.array_equal(d.fetch("features", len(xyz), 50).view(np.uint32), feat.view(np.uint32))
    assert np.array_equal(idx, oracle.nms(xyz, sc, R_NMS, TH))
    d.close()


# ---------------------------------------------------------------------------------------------
# per-point roles + forced grid through plain kpl_detect: a slab of a larger cloud, self-contained (the band
# within reach(r_nms) of the owned range is scored locally with role SCORE, no exchange) -- the role semantics of
# include/kpl.h.  The multi-rank schedule of kpl_shard_* is covered by tests/test_gpu_multi.py.
# ---------------------------------------------------------------------------------------------
def _role_slab(xyz, plan, rank, support=2):
    from keypoint_learning_b200 import shard
    world = plan.world
    cx = shard.cell_coords(xyz, plan.origin, plan.cell, 0)
    c0, c1 = int(plan.cuts[rank]), int(plan.cuts[rank + 1])
    halo = plan.reach_nms + plan.reach_feat + support
    lo = c0 - halo if rank > 0 else 0
    hi = c1 + halo if rank < world - 1 else int(plan.dims[0])
    lo, hi = max(lo, 0), min(hi, int(plan.dims[0]))
    gidx = np.nonzero((cx >= lo) & (cx < hi))[0]
    c = cx[gidx]
    role = np.zeros(len(gidx), np.uint8)
    role[(c >= c0 - plan.reach_nms) & (c < c1 + plan.reach_nms)] = 1
    role[(c >= c0) & (c < c1)] = 3
    xyz4 = np.ones((len(gidx), 4), np.float32)
    xyz4[:, :3] = xyz[gidx]
    return dict(xyz4=xyz4, role=role, gidx=gidx, local_dims=np.array([hi - lo, plan.dims[1], plan.dims[2]], np.int32),
                offset=np.array([lo, 0, 0], np.int32), interior=(rank > 0, rank < world - 1))


@pytest.mark.parametrize("world", [2, 3])
def test_slab_results_equal_unsharded(kpl, views, golden, world):
    from keypoint_learning_b200 import shard
    xyz = views["cheff001"]
    # shard along the longest axis of this view (y): rotate it onto x, the slab axis
    xyz_r = np.ascontiguousarray(xyz[:, [1, 0, 2]])
    d = make_detector(kpl)
    d.setNormalsMode(1, k=10)
    d.setInputCloud(xyz_r)
    _, idx_full = d.compute()
    sc_full = d.getResponse().copy()
    plan = shard.plan_slabs(xyz_r, R_FEAT, R_NMS, 4, world)
    kps, seen = [], np.zeros(len(xyz), bool)
    for rank in range(world):
        s = _role_slab(xyz_r, plan, rank)
        d.setForcedGrid(plan.origin, s["local_dims"], s["offset"])
        d.setInputCloud(s["xyz4"])
        _, idx = d.compute(role=s["role"])
        sc = d.getResponse()
        owned = s["role"] == 3
        scored = (s["role"] & 1) == 1
        assert d.stats()["n_scored"] == int(scored.sum())
        assert np.all(np.isnan(sc[~scored]))
        assert not seen[s["gidx"][owned]].any()
        seen[s["gidx"][owned]] = True
        assert np.array_equal(sc[scored].view(np.uint32), sc_full[s["gidx"][scored]].view(np.uint32))   # bit-identical scores
        assert np.all(owned[idx])                                                                      # only owned points are output
        kps.append(s["gidx"][idx])
    assert seen.all()
    assert np.array_equal(np.sort(np.concatenate(kps)), idx_full)
    # the same slab with the clipped-support check armed and no support columns: refused, not silently different
    s = _role_slab(xyz_r, plan, 0, support=0)
    d.setForcedGrid(plan.origin, s["local_dims"], s["offset"], interior=s["interior"], guard_cells=0)
    d.setInputCloud(s["xyz4"])
    with pytest.raises(kpl.KplError) as e:
        d.compute(role=s["role"])
    assert e.value.code == 12
    d.setForcedGrid(None)
    d.close()


# ---------------------------------------------------------------------------------------------
# the headline workload: closed 3-D surfaces at |coords| up to 1000 mm (BASELINE.json configs[3])
# ---------------------------------------------------------------------------------------------
def scene_crop(n_scene, m):
    from keypoint_learning_b200 import synth
    xyz, vp = synth.scene_closed_surfaces(n_scene, seed=4321)
    return synth.cube_crop(xyz, m), vp


def test_scene_closed_surfaces_vs_oracle(kpl, oracle, main_forest):
    """configs[3] geometry (multi-layer z cells, runs crossing a cell row several times, the computeRoots2 fallback of the
    un-centred covariance far from the origin): normals, features, scores and keypoints uint32-exact against the oracle
    (semantics: impl/KeypointLearning.hpp:179-376)."""
    xyz, vp = scene_crop(1_250_000, 300_000)
    assert np.abs(xyz).max() > 300.0
    d = make_detector(kpl)
    d.setNormalsMode(1, k=10, viewpoint=vp)
    d.keepIntermediates(True)
    d.setInputCloud(xyz)
    _, idx = d.compute()
    st = d.stats()
    assert st["grid_dims"][2] > 3                                   # really a 3-D grid
    ref = oracle.detect(xyz, main_forest, R_FEAT, R_NMS, TH, 5, 10, normals_mode=1, k=10, viewpoint=vp, order=1)
    assert same_bits(d.fetch("normals", len(xyz), 4), ref["normals"])
    assert same_bits(d.fetch("features", len(xyz), 50), ref["features"])
    assert same_bits(d.getResponse(), ref["scores"])
    assert np.array_equal(idx, ref["keypoints"])
    assert len(idx) > 0
    assert st["n_unscored"] == int(np.isnan(ref["scores"]).sum())
    # exact pair counter = the oracle's neighbour counts (self excluded) minus the pairs that never vote: a query
    # without a finite normal is not scored (hpp:277) and a neighbour without one is skipped (hpp:338)
    counts = oracle.radius_counts(xyz, R_FEAT)
    bad = np.nonzero(np.isnan(ref["normals"][:, :3]).any(axis=1))[0].astype(np.int32)
    off, nb = oracle.radius_neighbors(xyz, R_FEAT, bad)
    removed = 0
    for k, b in enumerate(bad):
        mine = nb[off[k]:off[k + 1]]
        removed += (len(mine) - 1) + int(np.sum(~np.isin(mine, bad)))
    assert st["feature_pairs"] == int(counts.sum()) - len(xyz) - removed
    d.close()


def test_scene_crop_against_the_reference_templates(kpl, oracle, reference):
    """A 3 k-point crop of the closed-surface scene through oracle/_ref (the reference's own templates)."""
    xyz, vp = scene_crop(1_250_000, 3000)
    nrm = oracle.normals_knn(xyz, 10, vp)
    fname = "synthetic-SHOT-like-T50-D10"
    forest = oracle.load_forest_yaml(forest_path(fname))
    lf = oracle.ref_neighbour_lists(xyz, R_FEAT, 1)
    ln = oracle.ref_neighbour_lists(xyz, R_NMS, 0)
    d = make_detector(kpl, forest=forest_path(fname), th=0.5)
    d.keepIntermediates(True)
    d.setInputCloud(xyz); d.setNormals(nrm)
    _, idx = d.compute()
    reference.check("scene_crop_3k/features", d.fetch("features", len(xyz), 50), lambda: oracle.ref_features(xyz, nrm, R_FEAT, 5, 10, lf))
    reference.check("scene_crop_3k/scores", d.getResponse(),
                    lambda: oracle.ref_detect(xyz, nrm, forest, R_FEAT, R_NMS, 0.5, 5, 10, lf, None, non_maxima=False)[1])
    reference.check("scene_crop_3k/keypoints", idx, lambda: oracle.ref_detect(xyz, nrm, forest, R_FEAT, R_NMS, 0.5, 5, 10, lf, ln)[0])
    d.close()


# ---------------------------------------------------------------------------------------------
# fragile splits (BASELINE.md s5): decisions of forest_->predict (hpp:281) within 1e-5 of the threshold
# ---------------------------------------------------------------------------------------------
def test_fragile_split_report(kpl, views, golden, oracle, main_forest):
    xyz = views["cheff001"]
    nrm = oracle.normals_knn(xyz, 10)
    d = make_detector(kpl)
    d.keepIntermediates(True)
    d.setInputCloud(xyz); d.setNormals(nrm)
    d.compute()
    assert d.stats()["n_fragile_points"] == 0            # off by default
    with pytest.raises(kpl.KplError):
        d.fetchFragile(len(xyz))
    d.setReportFragile(True)
    d.compute()
    assert np.array_equal(d.getResponse().view(np.uint32), golden["cheff001"]["scores"].view(np.uint32))
    feat = d.fetch("features", len(xyz), 50)
    ref = oracle.forest_fragile(main_forest, feat)
    got = d.fetchFragile(len(xyz))
    assert np.array_equal(got, ref)
    assert d.stats()["n_fragile_points"] == int(ref.sum())
    assert 0 < int(ref.sum()) < len(xyz)
    # a score that differs between two accumulation orders implies a fragile decision: the grid-free oracle
    # (ascending-index accumulation) must not disagree on any point that is not flagged
    f0 = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=0)
    s0 = oracle.scores_from_sums(oracle.forest_sum(main_forest, f0), main_forest["ntrees"])
    differs = s0 != d.getResponse()
    assert not np.any(differs & (got == 0))
    d.close()


# ---------------------------------------------------------------------------------------------
# batch of independent views in one pass (BASELINE.json configs[4])
# ---------------------------------------------------------------------------------------------
def test_batch_equals_per_view_calls(kpl, views, golden):
    """kpl_detect_batch: every view bit-identical to its stand-alone kpl_detect run (own grid, own order)."""
    from keypoint_learning_b200 import synth
    clouds = [views["cheff000"], views["cheff002"][:20000], synth.view_25d(200, 150, seed=5)[0], views["cheff001"],
              np.ascontiguousarray(views["cheff001"][:7] + np.float32(300.0))]       # a tiny view: fewer points than k
    d = make_detector(kpl)
    d.setNormalsMode(1, k=10)
    sc_b, kp_b = d.computeBatch(clouds)
    st = d.stats()
    assert st["n_views"] == len(clouds) and st["n_points"] == sum(len(c) for c in clouds)
    pairs = 0
    for c, sc, kp in zip(clouds, sc_b, kp_b):
        d.setInputCloud(c); d.setNormals(None)
        _, idx = d.compute()
        assert np.array_equal(d.getResponse().view(np.uint32), sc.view(np.uint32))
        assert np.array_equal(idx, kp)
        pairs += d.stats()["feature_pairs"]
    assert st["feature_pairs"] == pairs
    assert np.array_equal(sc_b[0].view(np.uint32), golden["cheff000"]["scores"].view(np.uint32))
    assert np.array_equal(kp_b[3], golden["cheff001"]["keypoints"])
    # given normals + one single view behave like kpl_detect
    sc1, kp1 = d.computeBatch([views["cheff001"]])
    assert np.array_equal(kp1[0], golden["cheff001"]["keypoints"])
    with pytest.raises(kpl.KplError):
        d.computeBatchConcat(np.zeros((4, 4), np.float32), np.array([0, 2, 2, 4], np.int64))      # an empty view
    d.close()


# ---------------------------------------------------------------------------------------------
# computePointsForTrainingFeatures on a small index subset of a large cloud (main_train_detector.cpp:419-439)
# ---------------------------------------------------------------------------------------------
def test_feature_subset_is_compact(kpl, oracle):
    import torch
    from keypoint_learning_b200 import synth
    xyz, vp = synth.scene_closed_surfaces(10_000_000, seed=4321)
    rng = np.random.default_rng(11)
    q = rng.choice(len(xyz), 5000, replace=False).astype(np.int32)
    q[10] = q[3]                                                     # duplicates are allowed
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    d = make_detector(kpl)
    d.setNormalsMode(1, k=10, viewpoint=vp)
    d.setInputCloud(xyz)
    rows = d.computePointsForTrainingFeatures(q)
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 < 1.5e9, "kpl_features on 5 k indices of a 10 M-point cloud used %.2f GB" % ((free0 - free1) / 1e9)
    assert rows.shape == (5000, 50)
    # check 40 of the rows against the oracle evaluated on the query's own neighbourhood (canonical order needs the
    # grid of the WHOLE cloud: pass it explicitly)
    org, cell, dims = oracle.canon_grid(xyz, R_FEAT, 4)
    nrm_all = d.fetch("normals", len(xyz), 4)
    for k in range(0, 5000, 125):
        c = xyz[q[k]]
        near = np.nonzero(np.abs(xyz - c).max(axis=1) < R_FEAT + 1.0)[0]
        loc = int(np.searchsorted(near, q[k]))
        f = oracle.features(xyz[near], nrm_all[near], R_FEAT, 5, 10, order=1, qidx=np.array([loc], np.int32),
                            canon=(org, cell, dims))
        assert np.array_equal(f[0].view(np.uint32), rows[k].view(np.uint32)), k
    d.close()


def test_feature_subset_matches_full_rows(kpl, views, oracle):
    xyz = views["cheff002"]
    nrm = oracle.normals_knn(xyz, 10)
    d = make_detector(kpl)
    d.setInputCloud(xyz); d.setNormals(nrm)
    full = d.computePointsForTrainingFeatures()
    rng = np.random.default_rng(2)
    for m in (1, 31, 32, 33, 1000, 20000):
        q = rng.choice(len(xyz), m, replace=(m > 5000)).astype(np.int32)
        rows = d.computePointsForTrainingFeatures(q)
        assert np.array_equal(rows.view(np.uint32), full[q].view(np.uint32)), m
    d.close()


# ---------------------------------------------------------------------------------------------
# stand-alone normal estimation sizes its k-NN grid from the data, whatever the unit of the cloud
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", [1e-3, 1.0, 250.0])
def test_knn_normals_any_unit(kpl, views, oracle, scale):
    import time
    xyz = np.ascontiguousarray(views["cheff001"] * np.float32(scale))
    d = kpl.KeypointLearningDetector()
    d.setNormalsMode(1, k=10)                          # radiusFeatures stays at its default of 20, as in TestDetector's `ne`
    t0 = time.perf_counter()
    got = d.computeNormals(xyz)
    dt = time.perf_counter() - t0
    ref = oracle.normals_knn(xyz, 10)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    cells = d.stats()["grid_cells"]
    assert 1000 < cells < 5e7, cells                   # neither one cell (brute force) nor an exploding grid
    assert dt < 5.0
    d.close()


def test_forest_guards(kpl, views, tmp_path):
    """A forest that splits on a variable >= annuli*bins, or holds a non-numeric threshold, is refused instead of
    reading beyond the feature row."""
    import gzip
    xyz = np.ascontiguousarray(views["cheff001"][:2000])
    d = kpl.KeypointLearningDetector()
    d.setRadiusSearch(R_FEAT); d.setNonMaxRadius(R_NMS); d.setNonMaximaDrawsRemove(False)
    d.setInputCloud(xyz)
    # var_count 0 (unknown) but a split on variable 50 with 5 x 10 = 50 features
    d.setForestArrays(dict(ntrees=1, roots=[0], var=[50, -1, -1], thr=[0.1, 0, 0], left=[1, -1, -1], right=[2, -1, -1], value=[0, 0, 1], var_count=0))
    with pytest.raises(kpl.KplError) as e:
        d.compute()
    assert e.value.code == 5
    d.setForestArrays(dict(ntrees=1, roots=[0], var=[49, -1, -1], thr=[0.1, 0, 0], left=[1, -1, -1], right=[2, -1, -1], value=[0, 0, 1], var_count=0))
    d.compute()
    txt = gzip.open(forest_path("synthetic-A4xB8-T20-D8"), "rt").read()
    import re
    bad = re.sub(r"le:\s*[-+0-9.eE]+", "le:.Inf", txt, count=1)
    assert bad != txt
    p = tmp_path / "inf.yaml"
    p.write_text(bad)
    assert not d.loadForest(str(p))
    d.close()


# ---------------------------------------------------------------------------------------------
# organized clouds: initCompute's IntegralImageNormalEstimation branch (impl/KeypointLearning.hpp:138-145)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(320, 240), (97, 61), (640, 13), (7, 300), (12, 11), (1, 1)])
def test_integral_image_normals_bit_exact(kpl, oracle, shape):
    from keypoint_learning_b200 import synth
    w, h = shape
    xyz, vp = synth.organized_range_image(w, h, seed=w + h)
    d = kpl.KeypointLearningDetector()
    d.setNormalsMode(1, k=10, viewpoint=vp)
    for smoothing in (5.0, 3.0, 10.0):
        got = d.computeNormalsOrganized(xyz, smoothing)
        ref = oracle.normals_integral_image(xyz, smoothing, vp)
        assert same_bits(got, ref), (shape, smoothing)
    d.close()


def test_organized_cloud_detection(kpl, oracle, main_forest):
    """The whole organized path through the Python facade: integral-image normals, NaN points compacted, detection over the
    finite points with those normals == the oracle fed with the same normals."""
    from keypoint_learning_b200 import synth
    xyz, vp = synth.organized_range_image(320, 240, seed=11)
    d = make_detector(kpl, th=0.5)
    d.setNormalsMode(1, k=10, viewpoint=vp)
    kp, idx = d.computeOrganized(xyz, 5.0)
    sc = d.getResponse()
    flat = xyz.reshape(-1, 3)
    nrm = oracle.normals_integral_image(xyz, 5.0, vp)
    keep = np.nonzero(np.isfinite(flat).all(axis=1))[0]
    ref = oracle.detect(np.ascontiguousarray(flat[keep]), main_forest, R_FEAT, R_NMS, 0.5, 5, 10, normals4=nrm[keep], order=1)
    assert same_bits(sc[keep], ref["scores"])
    assert np.all(np.isnan(sc[np.setdiff1d(np.arange(len(flat)), keep)]))
    assert np.array_equal(idx, keep[ref["keypoints"]])
    assert len(idx) > 0
    d.close()


def test_eigen32_normalize_variant(kpl, views, oracle, main_forest):
    """kpl_params.eigen32_normalize: the per-annulus normalisation as Eigen 3.2.x evaluates it, bit-identical to the oracle
    in the same mode; the default (division, Eigen >= 3.3) is untouched."""
    xyz = views["cheff002"]
    nrm = oracle.normals_knn(xyz, 10)
    d = make_detector(kpl)
    d.keepIntermediates(True)
    d.setInputCloud(xyz); d.setNormals(nrm)
    d.setEigen32Normalize(True)
    _, idx = d.compute()
    try:
        oracle.set_normalize_mode(True)
        ref = oracle.detect(xyz, main_forest, R_FEAT, R_NMS, TH, 5, 10, normals4=nrm, order=1)
    finally:
        oracle.set_normalize_mode(False)
    assert np.array_equal(d.fetch("features", len(xyz), 50).view(np.uint32), ref["features"].view(np.uint32))
    assert same_bits(d.getResponse(), ref["scores"])
    assert np.array_equal(idx, ref["keypoints"])
    sc1 = d.getResponse().copy()
    d.setEigen32Normalize(False)
    d.setReportFragile(True)
    d.compute()
    differs = sc1 != d.getResponse()
    assert not np.any(differs & (d.fetchFragile(len(xyz)) == 0))      # only fragile decisions can tell the two Eigen versions apart
    d.close()
