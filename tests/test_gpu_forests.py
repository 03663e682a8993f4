"""Several forests scored from one feature pass (kpl_detect_forests / _device, computeForests).  Forest k's scores and
keypoints must be bit-identical to a kpl_detect call on the same cloud with only forest k loaded and threshold k."""
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
KPL_E_INVALID, KPL_E_FOREST, KPL_E_NONFINITE, KPL_E_VARCOUNT = 1, 2, 4, 5


def _same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _detector(kpl, forests, draws=False, non_maxima=True, normals_mode=1, th=TH, fragile=False):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(non_maxima); det.setNonMaxRadius(R_NMS)
    det.setNonMaximaDrawsRemove(draws); det.setNonMaximaDrawsThreshold(1.0 if draws else 0.0)
    det.setPredictionThreshold(th); det.setRadiusSearch(R_FEAT); det.setNormalsMode(normals_mode, k=10)
    det.setReportFragile(fragile)
    assert det.loadForest(forests[0])
    for k, f in enumerate(forests[1:]):
        assert det.addForest(f) == k + 1
    assert det.forestCount() == len(forests)
    return det


_CLOUDS = {}


def _cloud(name):
    if name not in _CLOUDS:
        if name == "cheff001":
            _CLOUDS[name] = np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff001.npz"))["xyz"], np.float32)
        else:
            from keypoint_learning_b200 import synth
            xyz, _ = synth.scene_closed_surfaces(1_250_000, seed=4321)
            _CLOUDS[name] = np.ascontiguousarray(synth.cube_crop(xyz, 200_000 if name == "scene" else 20_000), np.float32)
    return _CLOUDS[name]


def _singles(kpl, xyz, thresholds, normals=None, **kw):
    """(scores, keypoints, stats) of kpl_detect with forest k alone, for every k."""
    out = []
    for k, f in enumerate(FORESTS):
        d = _detector(kpl, [f], th=thresholds[k], **kw)
        d.setInputCloud(xyz)
        if normals is not None:
            d.setNormals(normals)
        _, idx = d.compute()
        frag = d.fetchFragile(len(xyz)) if kw.get("fragile") else None
        out.append((d.getResponse().copy(), idx.copy(), d.stats(), frag))
        d.close()
    return out


VARIANTS = ["plain", "draws", "no_nms", "thresholds", "given", "radius"]


@pytest.mark.parametrize("cloud", ["cheff001", "scene"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_forests_equal_single_forest_calls(kpl, cloud, variant):
    xyz = _cloud(cloud)
    kw = dict(draws=variant == "draws", non_maxima=variant != "no_nms", normals_mode=2 if variant == "radius" else 1)
    th = [TH, 2.0, float(np.float32(0.3))] if variant == "thresholds" else [TH] * 3
    normals = None
    det = _detector(kpl, FORESTS, **kw)
    if variant == "given":
        normals = det.computeNormals(xyz)
        det.setNormals(normals)
    det.setInputCloud(xyz)
    res = det.computeForests(th if variant == "thresholds" else None)
    st = det.stats()
    resp = det.getResponses()
    assert resp.shape == (3, len(xyz))
    ref = _singles(kpl, xyz, th, normals, **kw)
    for k in range(3):
        sc1, idx1, _, _ = ref[k]
        assert _same(resp[k], sc1), k
        assert np.array_equal(res[k][1], idx1), k
        assert _same(res[k][0][:, 3], sc1[idx1]) and np.array_equal(res[k][0][:, :3], xyz[idx1, :3]), k
    if variant == "thresholds":
        assert len(res[1][1]) == 0 and len(res[0][1]) > 0 and len(res[2][1]) > 0
    # the histograms are counted once, the per-forest decisions summed
    for key in ("feature_pairs", "candidate_pairs", "n_scored"):
        assert st[key] == ref[0][2][key], key
    for key in ("n_above_threshold", "n_near_threshold", "n_keypoints", "nms_rounds"):
        assert st[key] == sum(r[2][key] for r in ref), key
    if variant == "draws":
        assert st["nms_rounds"] > 0
    assert sum(len(r[1]) for r in res) > 0
    det.close()


def test_one_forest_and_a_forest_twice(kpl):
    xyz = _cloud("cheff001")
    det = _detector(kpl, FORESTS[:1])
    det.setInputCloud(xyz)
    _, idx = det.compute()
    sc = det.getResponse().copy()
    res = det.computeForests()
    assert _same(det.getResponses()[0], sc) and np.array_equal(res[0][1], idx) and len(idx) > 0
    assert det.addForest(FORESTS[0]) == 1
    res = det.computeForests()
    r = det.getResponses()
    assert _same(r[0], r[1]) and _same(r[0], sc)
    assert np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[1][1], idx)
    det.close()


def test_each_forest_against_oracle(kpl, oracle):
    xyz = _cloud("scene_small")
    det = _detector(kpl, FORESTS)
    det.setInputCloud(xyz)
    res = det.computeForests()
    resp = det.getResponses()
    det.close()
    for k, f in enumerate(FORESTS):
        ref = oracle.detect(xyz, oracle.load_forest_yaml(f), R_FEAT, R_NMS, TH, 5, 10, normals_mode=1, k=10, order=1)
        assert _same(resp[k], ref["scores"]), k
        assert np.array_equal(res[k][1], ref["keypoints"]), k


def test_non_dense_cloud(kpl):
    xyz = _cloud("scene_small").copy()
    xyz[::97] = np.nan
    det = _detector(kpl, FORESTS)
    det.setInputCloud(xyz)
    res = det.computeForests([TH, TH, float(np.float32(0.3))])
    resp = det.getResponses()
    ref = _singles(kpl, xyz, [TH, TH, float(np.float32(0.3))])
    for k in range(3):
        assert _same(resp[k], ref[k][0]) and np.array_equal(res[k][1], ref[k][1]), k
    assert np.all(np.isnan(resp[:, ::97]))
    det.close()


def test_fragile_masks(kpl):
    xyz = _cloud("cheff001")
    det = _detector(kpl, FORESTS, fragile=True)
    det.setInputCloud(xyz)
    det.computeForests()
    n = len(xyz)
    masks = det.fetchFragile(3 * n)
    st = det.stats()
    ref = _singles(kpl, xyz, [TH] * 3, fragile=True)
    for k in range(3):
        assert np.array_equal(masks[k * n:(k + 1) * n], ref[k][3]), k
    assert st["n_fragile_points"] == sum(r[2]["n_fragile_points"] for r in ref)
    det.close()


def _device_forests(det, xyz, K, thresholds=None):
    import torch
    n = len(xyz)
    x4 = np.ones((n, 4), np.float32); x4[:, :3] = xyz
    d_xyz = torch.from_numpy(x4).cuda()
    d_sc = torch.empty(K * n, dtype=torch.float32, device="cuda")
    d_kp = torch.empty(K * n, dtype=torch.int32, device="cuda")
    d_kpo = torch.empty(K + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    nk = det.detectForestsDevice(d_xyz.data_ptr(), n, thresholds=thresholds, d_scores=d_sc.data_ptr(), d_kp_idx=d_kp.data_ptr(),
                                 d_kp_offsets=d_kpo.data_ptr())
    st = det.stats()
    kpo = d_kpo.cpu().numpy()
    return nk, st, d_sc.cpu().numpy().reshape(K, n), [d_kp.cpu().numpy()[kpo[k]:kpo[k + 1]] for k in range(K)], d_xyz


@pytest.mark.parametrize("draws", [False, True])
def test_device_entry_point_and_budget(kpl, draws):
    """The device entry point returns what the host one does.  Without draws-remove it synchronises with the host exactly as
    often as kpl_detect_device on the same cloud, whatever K is, and launches K + 1 more kernels: K - 1 more NMS launches and
    the two of launch_view_ranges."""
    import torch
    xyz = _cloud("scene")
    th = [TH, float(np.float32(0.3)), float(np.float32(0.6))]
    for K in (1, 2, 3):
        det = _detector(kpl, FORESTS[:K], draws=draws)
        det.setInputCloud(xyz)
        res = det.computeForests(th[:K])
        resp = det.getResponses().copy()
        nk, st, sc, kp, d_xyz = _device_forests(det, xyz, K, th[:K])
        assert nk == sum(len(r[1]) for r in res) == st["n_keypoints"] > 0
        for k in range(K):
            assert _same(sc[k], resp[k]) and np.array_equal(kp[k], res[k][1]), (K, k)
        # kpl_detect_device with forest 0 alone on the same cloud (the forest set does not change it)
        d_kp = torch.empty(len(xyz), dtype=torch.int32, device="cuda")
        det.setPredictionThreshold(th[0])
        det.detectDevice(d_xyz.data_ptr(), len(xyz), d_kp_idx=d_kp.data_ptr())
        st1 = det.stats()
        if not draws:
            assert st["host_syncs"] == st1["host_syncs"], K
            assert st["kernel_launches"] == st1["kernel_launches"] + K + 1, K
        else:
            assert st["host_syncs"] >= st1["host_syncs"] and st["nms_rounds"] >= st1["nms_rounds"]
        det.close()


def test_extra_forests_leave_other_entry_points_alone(kpl):
    xyz = _cloud("cheff001")
    views = [xyz[:40000], xyz[40000:]]
    det = _detector(kpl, FORESTS[:1])

    def run():
        det.setInputCloud(xyz)
        _, idx = det.compute()
        out = [det.getResponse().copy(), idx.copy()]
        s = det.stats()
        out.append((s["kernel_launches"], s["host_syncs"]))
        sc_b, kp_b = det.computeBatch(views)
        out += [np.concatenate(sc_b).copy(), np.concatenate(kp_b).copy()]
        s = det.stats()
        out.append((s["kernel_launches"], s["host_syncs"]))
        out.append(det.computePointsForTrainingFeatures(np.arange(0, len(xyz), 7, dtype=np.int32)))
        return out

    before = run()
    det.addForest(FORESTS[1]); det.addForest(FORESTS[2])
    after = run()
    for a, b in zip(before, after):
        if isinstance(a, tuple):
            assert a == b
        else:
            assert _same(a, b) if a.dtype == np.float32 else np.array_equal(a, b)
    assert det.forestCount() == 3
    assert det.loadForest(FORESTS[1])
    assert det.forestCount() == 1 and det.forestInfo()["ntrees"] == 50
    det.close()


def test_refusals(kpl):
    from keypoint_learning_b200 import capi
    L = capi.load_library()
    xyz = np.ascontiguousarray(_cloud("scene_small")[:3000])
    n = len(xyz)
    det = _detector(kpl, FORESTS)
    det._push()
    f32, i32, i64, f64 = ctypes.c_float, ctypes.c_int32, ctypes.c_int64, ctypes.c_double
    P = capi._ptr
    sc = np.empty(16 * n, np.float32); kp = np.empty(16 * n, np.int32); kpo = np.empty(17, np.int64)

    def call(x=xyz, kp_out=kp, kpo_out=kpo):
        return L.kpl_detect_forests(det._h, P(x, f32), 12, None, 0, len(x), None, P(sc, f32), P(kp_out, i32), P(kpo_out, i64))

    assert call() == 0
    assert call(kp_out=None) == KPL_E_INVALID and call(kpo_out=None) == KPL_E_INVALID
    bad = xyz.copy(); bad[5, 1] = np.inf
    assert call(bad) == KPL_E_NONFINITE
    # a failed add leaves the set as it was
    with pytest.raises(kpl.KplError):
        det.addForest(os.path.join(ROOT, "no-such-forest.yaml.gz"))
    assert det.forestCount() == 3
    broken = dict(ntrees=1, var=[0, -1, -1], thr=[0.5, 0, 0], left=[1, 0, 0], right=[2, 0, 0], value=[0, 1, 0], roots=[5])   # root out of range
    with pytest.raises(kpl.KplError):
        det.addForestArrays(broken)
    assert det.forestCount() == 3 and call() == 0
    # a forest of another annuli x bins, named by its index
    assert det.addForest(FOREST_A4xB8) == 3
    assert call() == KPL_E_VARCOUNT and b"forest 3" in L.kpl_last_error(det._h)
    # kpl_detect keeps scoring with forest 0 only
    assert L.kpl_detect(det._h, P(xyz, f32), 12, None, 0, None, n, None, P(kp, i32), ctypes.byref(i64())) == 0
    # the cap
    assert det.loadForest(FORESTS[0])
    for k in range(1, 16):
        assert det.addForest(FORESTS[k % 3]) == k
    with pytest.raises(kpl.KplError) as e:
        det.addForest(FORESTS[0])
    assert e.value.code == KPL_E_INVALID and det.forestCount() == 16
    assert call() == 0 and kpo[16] == kpo[16 - 3] + (kpo[3] - kpo[0])
    # device entry point
    import torch
    d = torch.zeros(n * 4, dtype=torch.float32, device="cuda")
    dk = torch.empty(16 * n, dtype=torch.int32, device="cuda"); dko = torch.empty(17, dtype=torch.int64, device="cuda")
    nkp = i64(0)
    assert L.kpl_detect_forests_device(det._h, ctypes.c_void_p(d.data_ptr()), None, n, None, None, None, ctypes.c_void_p(dko.data_ptr()),
                                       ctypes.byref(nkp)) == KPL_E_INVALID
    assert L.kpl_detect_forests_device(det._h, ctypes.c_void_p(d.data_ptr()), None, n, None, None, ctypes.c_void_p(dk.data_ptr()), None,
                                       ctypes.byref(nkp)) == KPL_E_INVALID
    det.close()
    # no forest at all; adding needs forest 0 first
    nof = kpl.KeypointLearningDetector()
    nof.setRadiusSearch(R_FEAT)
    nof._push()
    assert L.kpl_detect_forests(nof._h, P(xyz, f32), 12, None, 0, n, None, None, P(kp, i32), P(kpo, i64)) == KPL_E_FOREST
    assert L.kpl_add_forest(nof._h, FORESTS[0].encode(), None) == KPL_E_FOREST and nof.forestCount() == 0
    nof.close()


def test_failed_install_leaves_the_set_alone(kpl):
    """A malformed kpl_set_forest and a kpl_load_forest of a missing file change nothing: neither the three loaded forests
    nor what kpl_detect and kpl_detect_forests return."""
    xyz = _cloud("cheff001")
    det = _detector(kpl, FORESTS)
    det.setInputCloud(xyz)

    def results():
        _, idx = det.compute()
        out = [det.getResponse().copy(), idx.copy()]
        res = det.computeForests()
        return out + [det.getResponses().copy()] + [r[1].copy() for r in res]

    info, before = det.forestInfo(), results()
    assert len(before[1]) > 0
    broken = dict(ntrees=1, var=[0, -1, -1], thr=[0.5, 0, 0], left=[1, 0, 0], right=[2, 0, 0], value=[0, 1, 0], roots=[5])   # root out of range
    with pytest.raises(kpl.KplError) as e:
        det.setForestArrays(broken)
    assert e.value.code == KPL_E_FOREST
    assert not det.loadForest(os.path.join(ROOT, "no-such-forest.yaml.gz"))
    assert det.forestCount() == 3 and det.forestInfo() == info
    after = results()
    for a, b in zip(before, after):
        assert _same(a, b) if a.dtype == np.float32 else np.array_equal(a, b)
    det.close()


CPP = r"""
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include "KeypointLearning.h"

// argv: three forests, binary file (int32 n; n x 3 float xyz)
int main(int argc, char** argv)
{
    if (argc < 5) return 2;
    std::ifstream f(argv[4], std::ios::binary);
    int32_t n = 0;
    f.read(reinterpret_cast<char*>(&n), 4);
    std::vector<float> xyz((size_t)n * 3);
    f.read(reinterpret_cast<char*>(xyz.data()), xyz.size() * 4);
    typedef pcl::PointCloud<pcl::PointXYZ> Cloud;
    size_t total = 0;
    bool same = true;
    for (int dense = 1; dense >= 0; --dense) {
        Cloud::Ptr c(new Cloud);
        for (int32_t i = 0; i < n; ++i) c->points.push_back(pcl::PointXYZ(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        if (!dense)
            for (int32_t i = 0; i < n; i += 53) c->points[(size_t)i].x = std::nanf("");
        c->width = (uint32_t)n; c->height = 1; c->is_dense = dense != 0;
        const std::vector<double> th = {0.5, 0.5, 0.3};
        pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> det(0.5, true, false, 4.0);
        det.setRadiusSearch(20.0);
        if (!det.loadForest(argv[1]) || !det.addForest(argv[2]) || !det.addForest(argv[3])) return 3;
        det.setInputCloud(c);
        std::vector<pcl::PointCloud<pcl::PointXYZI>> outs;
        std::vector<pcl::PointIndices> idx;
        if (!det.computeForests(outs, &idx, &th)) return 4;
        same = same && outs.size() == 3 && idx.size() == 3;
        for (int k = 0; same && k < 3; ++k) {
            pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> one(th[k], true, false, 4.0);
            one.setRadiusSearch(20.0);
            if (!one.loadForest(argv[1 + k])) return 5;
            one.setInputCloud(c);
            pcl::PointCloud<pcl::PointXYZI> out;
            one.compute(out);
            const auto& i1 = one.getKeypointsIndices()->indices;
            same = i1 == idx[k].indices && out.size() == outs[k].size() && outs[k].width == outs[k].size() && out.is_dense == outs[k].is_dense;
            for (size_t j = 0; same && j < out.size(); ++j)
                same = std::memcmp(&out.points[j].x, &outs[k].points[j].x, 12) == 0 &&
                       std::memcmp(&out.points[j].intensity, &outs[k].points[j].intensity, 4) == 0;
            total += i1.size();
        }
        // one threshold per forest
        const std::vector<double> two = {0.5, 0.5};
        same = same && !det.computeForests(outs, &idx, &two);
    }
    std::printf("keypoints %zu same %d\n", total, (int)same);
    return 0;
}
"""


def test_cpp_compute_forests(kpl, tmp_path):
    """KeypointLearningDetector::computeForests equals compute() with each forest alone, on a dense and a non-dense cloud."""
    from keypoint_learning_b200 import build as B
    B.build_host()
    src, exe, data = str(tmp_path / "forests.cpp"), str(tmp_path / "forests"), str(tmp_path / "cloud.bin")
    with open(src, "w") as f:
        f.write(CPP)
    common = [os.path.join(B.HOST, f) for f in sorted(os.listdir(B.HOST)) if f.endswith(".cpp") and not f.startswith("main_")]
    subprocess.check_call([B._host_cxx(), "-O2", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", B.HOST, src,
                           *common, "-o", exe, "-L", B.HERE, "-lkpl_b200", "-lpthread", "-Wl,-rpath," + B.HERE])
    xyz = np.ascontiguousarray(_cloud("scene_small")[:, :3], np.float32)
    with open(data, "wb") as f:
        f.write(np.array([len(xyz)], np.int32).tobytes()); f.write(xyz.tobytes())
    r = subprocess.run([exe, *FORESTS, data], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    words = r.stdout.split("\n")[-2].split()
    got = dict(zip(words[0::2], words[1::2]))
    assert int(got["keypoints"]) > 0 and got["same"] == "1"
