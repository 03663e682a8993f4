"""Every forest of the set over a batch of views (kpl_detect_batch_forests / _device) and over a batch of organized frames
(kpl_detect_batch_organized_forests / _device), from one feature pass.  For forest k and view (or frame) v the scores, as
bits, and the keypoints must be those of kpl_detect_batch / kpl_detect_batch_organized with only forest k loaded and
threshold k."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]
FOREST_A4xB8 = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-A4xB8-T20-D8.yaml.gz")
R_FEAT, R_NMS = 20.0, 4.0
TH = float(np.float32(0.5))
TH3 = [TH, 2.0, float(np.float32(0.3))]          # forest 1 finds no keypoint at 2.0
KPL_E_INVALID, KPL_E_FOREST, KPL_E_NONFINITE, KPL_E_VARCOUNT = 1, 2, 4, 5


def _same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _detector(kpl, forests, draws=False, non_maxima=True, normals_mode=1, th=TH, fragile=False):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(non_maxima); det.setNonMaxRadius(R_NMS)
    det.setNonMaximaDrawsRemove(draws); det.setNonMaximaDrawsThreshold(1.0 if draws else 0.0)
    det.setPredictionThreshold(th); det.setRadiusSearch(R_FEAT); det.setNormalsMode(normals_mode, k=10)
    det.setReportFragile(fragile)
    if forests:
        assert det.loadForest(forests[0])
        for k, f in enumerate(forests[1:]):
            assert det.addForest(f) == k + 1
    return det


_VIEWS = []


def _views():
    """cheff000/001/002 and a crop of the scene: views of different sizes."""
    if not _VIEWS:
        from keypoint_learning_b200 import synth
        for v in ("cheff000", "cheff001", "cheff002"):
            _VIEWS.append(np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", "views", v + ".npz"))["xyz"], np.float32))
        xyz, _ = synth.scene_closed_surfaces(1_250_000, seed=4321)
        _VIEWS.append(np.ascontiguousarray(synth.cube_crop(xyz, 30_000), np.float32))
    return list(_VIEWS)


def _single_batches(kpl, views, thresholds, normals=None, **kw):
    """[k] -> (computeBatch results, stats, fragile mask) with forest k alone at threshold k."""
    out = []
    for k, f in enumerate(FORESTS):
        d = _detector(kpl, [f], th=thresholds[k], **kw)
        sc, kp = d.computeBatch(views, normals)
        frag = d.fetchFragile(sum(len(v) for v in views)) if kw.get("fragile") else None
        out.append(([s.copy() for s in sc], kp, d.stats(), frag))
        d.close()
    return out


def _check_sums(st, ref):
    for key in ("feature_pairs", "candidate_pairs", "n_scored", "n_points", "n_views"):
        assert st[key] == ref[0][1][key], key
    for key in ("n_above_threshold", "n_near_threshold", "n_keypoints", "n_fragile_points", "nms_rounds"):
        assert st[key] == sum(r[1][key] for r in ref), key


VARIANTS = ["plain", "draws", "no_nms", "thresholds", "given", "radius"]


@pytest.mark.parametrize("variant", VARIANTS)
def test_views_equal_single_forest_batches(kpl, variant):
    views = _views()
    kw = dict(draws=variant == "draws", non_maxima=variant != "no_nms", normals_mode=2 if variant == "radius" else 1)
    th = TH3 if variant == "thresholds" else [TH] * 3
    det = _detector(kpl, FORESTS, **kw)
    normals = [det.computeNormals(v) for v in views] if variant == "given" else None
    res = det.computeBatchForests(views, normals, th if variant == "thresholds" else None)
    st = det.stats()
    det.close()
    ref = _single_batches(kpl, views, th, normals, **kw)
    assert len(res) == 3 and all(len(r) == len(views) for r in res)
    for k in range(3):
        for v in range(len(views)):
            assert _same(res[k][v][0], ref[k][0][v]), (k, v)
            assert np.array_equal(res[k][v][1], ref[k][1][v]), (k, v)
    _check_sums(st, [(r[0], r[2]) for r in ref])
    if variant == "thresholds":
        assert all(len(res[1][v][1]) == 0 for v in range(len(views)))
        assert all(len(res[k][v][1]) > 0 for k in (0, 2) for v in range(len(views)))
    if variant == "draws":
        assert st["nms_rounds"] > 0
    assert sum(len(res[k][v][1]) for k in range(3) for v in range(len(views))) > 0


def test_view_against_forests_on_one_cloud(kpl):
    """One (k, v) of the batch is what kpl_detect_forests returns for view v alone."""
    views = _views()
    det = _detector(kpl, FORESTS)
    res = det.computeBatchForests(views, thresholds=TH3)
    det.setInputCloud(views[3])
    one = det.computeForests(TH3)
    resp = det.getResponses()
    det.close()
    for k in range(3):
        assert _same(res[k][3][0], resp[k]) and np.array_equal(res[k][3][1], one[k][1]), k


def test_fragile_masks_and_non_finite_views(kpl):
    views = _views()[:2]
    det = _detector(kpl, FORESTS, fragile=True)
    det.computeBatchForests(views)
    n = sum(len(v) for v in views)
    masks = det.fetchFragile(3 * n)
    st = det.stats()
    ref = _single_batches(kpl, views, [TH] * 3, fragile=True)
    for k in range(3):
        assert np.array_equal(masks[k * n:(k + 1) * n], ref[k][3]), k
    assert st["n_fragile_points"] == sum(r[2]["n_fragile_points"] for r in ref)
    # non-finite points are refused, as by kpl_detect_batch
    bad = [views[0].copy(), views[1]]
    bad[0][7, 2] = np.nan
    with pytest.raises(kpl.KplError) as e:
        det.computeBatchForests(bad)
    assert e.value.code == KPL_E_NONFINITE
    det.close()


def _frames(w, h, count, seed0=0, all_nan=None):
    from keypoint_learning_b200 import synth
    fr = np.stack([synth.organized_range_image(w, h, seed=seed0 + f, holes=f % 2 == 0)[0] for f in range(count)])
    if all_nan is not None:
        fr[all_nan] = np.nan
    return np.ascontiguousarray(fr)


SHAPES = [((320, 240), 4), ((97, 61), 3), ((7, 300), 2), ((12, 11), 2), ((1, 1), 2)]


def _single_organized(kpl, fr, thresholds, draws=False, **kw):
    out = []
    for k, f in enumerate(FORESTS):
        d = _detector(kpl, [f], th=thresholds[k], draws=draws)
        sc, kp = d.computeOrganizedBatch(fr, **kw)
        out.append(([s.copy() for s in sc], kp, d.stats()))
        d.close()
    return out


@pytest.mark.parametrize("draws", [False, True])
def test_frames_equal_single_forest_batches(kpl, draws):
    det = _detector(kpl, FORESTS, draws=draws)
    total = 0
    for (w, h), count in SHAPES:
        fr = _frames(w, h, count, seed0=w + h, all_nan=count - 1 if w == 320 else None)
        res = det.computeOrganizedBatchForests(fr, thresholds=TH3)
        st = det.stats()
        ref = _single_organized(kpl, fr, TH3, draws)
        for k in range(3):
            for f in range(count):
                assert _same(res[k][f][0], ref[k][0][f]), ((w, h), k, f)       # NaN positions and payloads included
                assert np.array_equal(res[k][f][1], ref[k][1][f]), ((w, h), k, f)
                total += len(res[k][f][1])
            if w == 320:
                assert np.all(np.isnan(res[k][-1][0])) and len(res[k][-1][1]) == 0
        _check_sums(st, [(r[0], r[2]) for r in ref])
    assert total > 0
    # no finite point in the whole batch: K*F + 1 zero offsets, all-NaN scores in every slice
    res = det.computeOrganizedBatchForests(np.full((3, 5, 4, 3), np.nan, np.float32))
    assert len(res) == 3 and all(np.all(np.isnan(s)) and len(kp) == 0 for r in res for s, kp in r)
    assert det.stats()["n_keypoints"] == 0 and det.stats()["n_views"] == 3
    det.close()


def test_frames_caller_normals_and_viewpoints(kpl):
    fr = _frames(97, 61, 4, seed0=3)
    vps = np.array([[0, 0, 0], [0, 0, 2000], [400, -300, 700], [-50, 20, 9000]], np.float32)
    rng = np.random.default_rng(5)
    nrm = rng.normal(size=fr.shape[:3] + (4,)).astype(np.float32)
    nrm[..., :3] /= np.linalg.norm(nrm[..., :3], axis=-1, keepdims=True)
    nrm[rng.random(fr.shape[:3]) < 0.05] = np.nan
    det = _detector(kpl, FORESTS)
    for kw in (dict(viewpoints=vps), dict(normals=nrm)):
        res = det.computeOrganizedBatchForests(fr, **kw)
        ref = _single_organized(kpl, fr, [TH] * 3, **kw)
        for k in range(3):
            for f in range(len(fr)):
                assert _same(res[k][f][0], ref[k][0][f]) and np.array_equal(res[k][f][1], ref[k][1][f]), (kw.keys(), k, f)
        assert sum(len(res[k][f][1]) for k in range(3) for f in range(len(fr))) > 0
    # the viewpoints change the result (they flip normals)
    plain = det.computeOrganizedBatchForests(fr)
    flipped = det.computeOrganizedBatchForests(fr, viewpoints=vps)
    assert any(not _same(plain[k][f][0], flipped[k][f][0]) for k in range(3) for f in range(len(fr)))
    det.close()


def test_frames_fragile_masks(kpl):
    fr = _frames(97, 61, 3, seed0=8)
    det = _detector(kpl, FORESTS, fragile=True)
    det.computeOrganizedBatchForests(fr)
    m = det.stats()["n_points"]
    masks = det.fetchFragile(3 * m)
    for k, f in enumerate(FORESTS):
        d = _detector(kpl, [f], fragile=True)
        d.computeOrganizedBatch(fr)
        assert d.stats()["n_points"] == m
        assert np.array_equal(masks[k * m:(k + 1) * m], d.fetchFragile(m)), k
        d.close()
    det.close()


def _device_views(det, views, K, thresholds=None, forests=True):
    import torch
    cat = np.concatenate(views)
    n, nv = len(cat), len(views)
    off = np.zeros(nv + 1, np.int64); off[1:] = np.cumsum([len(v) for v in views])
    x4 = np.ones((n, 4), np.float32); x4[:, :3] = cat
    d_xyz = torch.from_numpy(x4).cuda()
    d_sc = torch.empty(K * n, dtype=torch.float32, device="cuda")
    d_kp = torch.empty(K * n, dtype=torch.int32, device="cuda")
    d_kpo = torch.empty(K * nv + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    if forests:
        nk = det.detectBatchForestsDevice(d_xyz.data_ptr(), off, d_sc.data_ptr(), d_kp.data_ptr(), d_kpo.data_ptr(), thresholds=thresholds)
    else:
        nk = det.detectBatchDevice(d_xyz.data_ptr(), off, d_sc.data_ptr(), d_kp.data_ptr(), d_kpo.data_ptr())
    st = det.stats()
    kpo, kp, sc = d_kpo.cpu().numpy(), d_kp.cpu().numpy(), d_sc.cpu().numpy()
    return nk, st, [[(sc[k * n + off[v]:k * n + off[v + 1]], kp[kpo[k * nv + v]:kpo[k * nv + v + 1]]) for v in range(nv)] for k in range(K)]


def _device_frames(det, fr, K, thresholds=None, forests=True):
    import torch
    nf, h, w, _ = fr.shape
    n = nf * h * w
    x4 = np.ones((nf, h, w, 4), np.float32); x4[..., :3] = fr
    d_xyz = torch.from_numpy(x4).cuda()
    d_sc = torch.empty(K * n, dtype=torch.float32, device="cuda")
    d_kp = torch.empty(K * n, dtype=torch.int32, device="cuda")
    d_kpo = torch.empty(K * nf + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    args = dict(d_scores=d_sc.data_ptr(), d_kp_idx=d_kp.data_ptr(), d_kp_offsets=d_kpo.data_ptr())
    if forests:
        nk = det.detectOrganizedBatchForestsDevice(d_xyz.data_ptr(), w, h, nf, thresholds=thresholds, **args)
    else:
        nk = det.detectOrganizedBatchDevice(d_xyz.data_ptr(), w, h, nf, **args)
    st = det.stats()
    kpo, kp, sc = d_kpo.cpu().numpy(), d_kp.cpu().numpy(), d_sc.cpu().numpy()
    p = h * w
    return nk, st, [[(sc[k * n + f * p:k * n + (f + 1) * p], kp[kpo[k * nf + f]:kpo[k * nf + f + 1]]) for f in range(nf)] for k in range(K)]


def _assert_same_results(a, b):
    assert len(a) == len(b)
    for k in range(len(a)):
        for v in range(len(a[k])):
            assert _same(a[k][v][0], b[k][v][0]) and np.array_equal(a[k][v][1], b[k][v][1]), (k, v)


def test_device_entry_points_and_budget(kpl):
    """The device entry points return what the host ones do.  They synchronise with the host as often as the single-forest
    batch device calls, for every K, and launch K - 1 more kernels (one NMS per further forest).  K = 1 is the single-forest
    call: the same results, launches and syncs."""
    views = _views()
    fr = _frames(160, 120, 8, seed0=40, all_nan=5)
    th = [TH, float(np.float32(0.3)), float(np.float32(0.6))]
    for K in (1, 2, 3):
        det = _detector(kpl, FORESTS[:K])
        host_v = det.computeBatchForests(views, thresholds=th[:K])
        nk, st, dev_v = _device_views(det, views, K, th[:K])
        _assert_same_results(dev_v, host_v)
        assert nk == st["n_keypoints"] == sum(len(kp) for r in host_v for _, kp in r) > 0
        host_f = det.computeOrganizedBatchForests(fr, thresholds=th[:K])
        nk_f, st_f, dev_f = _device_frames(det, fr, K, th[:K])
        _assert_same_results(dev_f, host_f)
        assert nk_f == sum(len(kp) for r in host_f for _, kp in r) > 0
        # the single-forest batch calls with forest 0 on the same inputs
        det.setPredictionThreshold(th[0])
        nk1, st1, one_v = _device_views(det, views, 1, forests=False)
        _, st1_f, one_f = _device_frames(det, fr, 1, forests=False)
        _assert_same_results(one_v, dev_v[:1])
        _assert_same_results(one_f, dev_f[:1])
        assert st["host_syncs"] == st1["host_syncs"] and st_f["host_syncs"] == st1_f["host_syncs"], K
        assert st["kernel_launches"] == st1["kernel_launches"] + K - 1, K
        assert st_f["kernel_launches"] == st1_f["kernel_launches"] + K - 1, K
        if K == 1:
            assert nk == nk1
        det.close()


def test_draws_remove_budget(kpl):
    """With draws-remove each forest runs its own resolution rounds."""
    views = _views()[:2]
    det = _detector(kpl, FORESTS, draws=True)
    _, st, _ = _device_views(det, views, 3)
    _, st1, _ = _device_views(det, views, 1, forests=False)
    assert st["nms_rounds"] >= st1["nms_rounds"] > 0 and st["host_syncs"] >= st1["host_syncs"]
    det.close()


def test_refusals(kpl):
    from keypoint_learning_b200 import capi
    import torch
    L = capi.load_library()
    views = [v[:3000] for v in _views()[:2]]
    xyz = np.ascontiguousarray(np.concatenate(views))
    n = len(xyz)
    off = np.array([0, 3000, n], np.int64)
    det = _detector(kpl, FORESTS)
    det._push()
    f32, i32, i64 = ctypes.c_float, ctypes.c_int32, ctypes.c_int64
    P = capi._ptr
    sc = np.empty(16 * n, np.float32); kp = np.empty(16 * n, np.int32); kpo = np.empty(64, np.int64)

    def call(x=xyz, o=off, nv=2, kp_out=kp, kpo_out=kpo):
        return L.kpl_detect_batch_forests(det._h, P(x, f32), 12, None, 0, P(o, i64), nv, None, P(sc, f32), P(kp_out, i32), P(kpo_out, i64))

    assert call() == 0 and kpo[6] == det.stats()["n_keypoints"]
    assert call(kp_out=None) == KPL_E_INVALID and call(kpo_out=None) == KPL_E_INVALID
    for o in (np.array([1, 3000, n], np.int64), np.array([0, 3000, 3000], np.int64), np.array([0, 4000, 3000], np.int64)):
        assert call(o=o) == KPL_E_INVALID, o
    assert call(nv=0) == KPL_E_INVALID
    # K*n over the limit: refused before the (far too small) input is read
    big = np.array([0, 800_000_000], np.int64)
    assert call(o=big, nv=1) == KPL_E_INVALID and b"forest count x point count" in L.kpl_last_error(det._h)
    frames = _frames(12, 11, 2)
    fsc = np.empty(3 * frames.size, np.float32); fkp = np.empty(3 * frames.size, np.int32); fkpo = np.empty(7, np.int64)

    def fcall(w=12, h=11, nf=2, kp_out=fkp):
        return L.kpl_detect_batch_organized_forests(det._h, P(frames, f32), 12, None, 0, w, h, nf, 5.0, None, None, P(fsc, f32),
                                                    P(kp_out, i32), P(fkpo, i64))

    assert fcall() == 0
    assert fcall(kp_out=None) == KPL_E_INVALID and fcall(w=0) == KPL_E_INVALID
    assert fcall(w=40000, h=10000, nf=2) == KPL_E_INVALID and b"forest count x point count" in L.kpl_last_error(det._h)
    # device entry points: NULL outputs, and K*n over the limit
    d = torch.zeros(n * 4, dtype=torch.float32, device="cuda")
    dk = torch.empty(3 * n, dtype=torch.int32, device="cuda"); dko = torch.empty(64, dtype=torch.int64, device="cuda")
    nkp = i64(0)

    def dcall(x=d.data_ptr(), k=dk.data_ptr(), ko=dko.data_ptr(), o=off, nv=2):
        return L.kpl_detect_batch_forests_device(det._h, ctypes.c_void_p(x), None, P(o, i64), nv, None, None, ctypes.c_void_p(k),
                                                 ctypes.c_void_p(ko), ctypes.byref(nkp))

    def odcall(k=dk.data_ptr(), ko=dko.data_ptr(), w=12, h=11, nf=2):
        return L.kpl_detect_batch_organized_forests_device(det._h, ctypes.c_void_p(d.data_ptr()), None, w, h, nf, 5.0, None, None, None,
                                                           ctypes.c_void_p(k), ctypes.c_void_p(ko), ctypes.byref(nkp))

    assert odcall() == 0
    for kw in (dict(x=None), dict(k=None), dict(ko=None), dict(o=big, nv=1)):
        assert dcall(**kw) == KPL_E_INVALID, kw
    for kw in (dict(k=None), dict(ko=None), dict(w=40000, h=10000, nf=2)):
        assert odcall(**kw) == KPL_E_INVALID, kw
    # a forced grid
    det.setForcedGrid((0.0, 0.0, 0.0), (4, 4, 4))
    det._push()
    assert call() == KPL_E_INVALID and fcall() == KPL_E_INVALID
    det.setForcedGrid(None)
    # a forest of another annuli x bins, named by its index
    assert det.addForest(FOREST_A4xB8) == 3
    det._push()
    assert call() == KPL_E_VARCOUNT and b"forest 3" in L.kpl_last_error(det._h)
    assert fcall() == KPL_E_VARCOUNT and b"forest 3" in L.kpl_last_error(det._h)
    # the single-forest batches keep scoring with forest 0 only
    assert L.kpl_detect_batch(det._h, P(xyz, f32), 12, None, 0, P(off, i64), 2, None, P(kp, i32), P(kpo, i64)) == 0
    # wrong threshold shapes
    for th in ([TH], [TH] * 5, [[TH] * 4]):
        with pytest.raises(ValueError):
            det.computeBatchForests(views, thresholds=th)
        with pytest.raises(ValueError):
            det.computeOrganizedBatchForests(frames, thresholds=th)
    det.close()
    nof = _detector(kpl, [])
    nof._push()
    assert L.kpl_detect_batch_forests(nof._h, P(xyz, f32), 12, None, 0, P(off, i64), 2, None, None, P(kp, i32), P(kpo, i64)) == KPL_E_FOREST
    with pytest.raises(kpl.KplError) as e:
        nof.computeOrganizedBatchForests(frames)
    assert e.value.code == KPL_E_FOREST
    nof.close()


CPP = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include "KeypointLearning.h"

// argv: three forests, binary file (int32 frames, width, height; frames x height x width x 3 float xyz; frames x 3 float origins)
int main(int argc, char** argv)
{
    if (argc < 5) return 2;
    std::ifstream f(argv[4], std::ios::binary);
    int32_t hd[3];
    f.read(reinterpret_cast<char*>(hd), sizeof hd);
    const int F = hd[0], W = hd[1], H = hd[2];
    std::vector<float> xyz((size_t)F * W * H * 3), vp((size_t)F * 3);
    f.read(reinterpret_cast<char*>(xyz.data()), xyz.size() * 4);
    f.read(reinterpret_cast<char*>(vp.data()), vp.size() * 4);
    typedef pcl::PointCloud<pcl::PointXYZ> Cloud;
    std::vector<Cloud::ConstPtr> frames;
    for (int k = 0; k < F; ++k) {
        Cloud::Ptr c(new Cloud);
        for (size_t i = 0; i < (size_t)W * H; ++i) {
            const float* p = xyz.data() + ((size_t)k * W * H + i) * 3;
            c->points.push_back(pcl::PointXYZ(p[0], p[1], p[2]));
        }
        c->width = W; c->height = H; c->is_dense = false;
        for (int a = 0; a < 3; ++a) c->sensor_origin_[a] = vp[(size_t)k * 3 + a];
        frames.push_back(c);
    }
    const std::vector<double> th = {0.5, 0.5, 0.3};
    pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> det(0.5, true, false, 4.0);
    det.setRadiusSearch(20.0);
    if (!det.loadForest(argv[1]) || !det.addForest(argv[2]) || !det.addForest(argv[3])) return 3;
    std::vector<std::vector<pcl::PointCloud<pcl::PointXYZI>>> outs;
    std::vector<std::vector<pcl::PointIndices>> idx;
    if (!det.computeOrganizedBatchForests(frames, outs, &idx, &th)) return 4;
    bool same = outs.size() == 3 && idx.size() == 3;
    size_t total = 0;
    for (int k = 0; same && k < 3; ++k) {
        pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> one(th[k], true, false, 4.0);
        one.setRadiusSearch(20.0);
        if (!one.loadForest(argv[1 + k])) return 5;
        std::vector<pcl::PointCloud<pcl::PointXYZI>> o1;
        std::vector<pcl::PointIndices> i1;
        if (!one.computeOrganizedBatch(frames, o1, &i1)) return 6;
        same = outs[k].size() == (size_t)F && idx[k].size() == (size_t)F;
        for (int f = 0; same && f < F; ++f) {
            same = i1[f].indices == idx[k][f].indices && o1[f].size() == outs[k][f].size() && outs[k][f].width == outs[k][f].size();
            for (size_t j = 0; same && j < o1[f].size(); ++j)
                same = std::memcmp(&o1[f].points[j].x, &outs[k][f].points[j].x, 12) == 0 &&
                       std::memcmp(&o1[f].points[j].intensity, &outs[k][f].points[j].intensity, 4) == 0;
            total += i1[f].indices.size();
        }
    }
    // one threshold per forest
    const std::vector<double> two = {0.5, 0.5};
    const bool refused = !det.computeOrganizedBatchForests(frames, outs, &idx, &two);
    std::printf("keypoints %zu refused %d same %d\n", total, (int)refused, (int)same);
    return 0;
}
"""


def test_cpp_compute_organized_batch_forests(kpl, tmp_path):
    """KeypointLearningDetector::computeOrganizedBatchForests equals computeOrganizedBatch with each forest alone."""
    from keypoint_learning_b200 import build as B
    B.build_host()
    src, exe, data = str(tmp_path / "batch_forests.cpp"), str(tmp_path / "batch_forests"), str(tmp_path / "frames.bin")
    with open(src, "w") as f:
        f.write(CPP)
    common = [os.path.join(B.HOST, f) for f in sorted(os.listdir(B.HOST)) if f.endswith(".cpp") and not f.startswith("main_")]
    subprocess.check_call([B._host_cxx(), "-O2", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", B.HOST, src,
                           *common, "-o", exe, "-L", B.HERE, "-lkpl_b200", "-lpthread", "-Wl,-rpath," + B.HERE])
    fr = _frames(160, 120, 3, seed0=90)
    vps = np.array([[0, 0, 0], [0, 0, 3000], [200, 100, -100]], np.float32)
    with open(data, "wb") as f:
        f.write(np.array([3, 160, 120], np.int32).tobytes()); f.write(fr.tobytes()); f.write(vps.tobytes())
    r = subprocess.run([exe, *FORESTS, data], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "2 thresholds for 3 forests" in r.stderr
    words = r.stdout.split("\n")[-2].split()
    got = dict(zip(words[0::2], words[1::2]))
    assert int(got["keypoints"]) > 0 and got["refused"] == "1" and got["same"] == "1"
