"""Batched detection of organized frames (kpl_detect_batch_organized / _device): integral-image normals of every frame,
the finite pixels compacted on the device, one stacked-grid batch over them.  Every frame's result must be bit-identical
to the single-frame organized path (computeOrganized, KeypointLearningDetector::compute) on that frame alone."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz")
R_FEAT, R_NMS = 20.0, 4.0
KPL_E_INVALID, KPL_E_FOREST = 1, 2
# integral-image scratch of one launch (organized.cu: II_CHUNK_BYTES)
CHUNK_BYTES = 256 << 20


def _detector(kpl, draws=False, th=0.5, forest=True):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS)
    det.setNonMaximaDrawsRemove(draws); det.setNonMaximaDrawsThreshold(1.0 if draws else 0.0)
    det.setPredictionThreshold(float(np.float32(th))); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10)
    if forest:
        assert det.loadForest(FOREST)
    return det


def _frames(w, h, count, seed0=0, all_nan=None):
    """`count` range images of one size, holes on and off in turn; frame `all_nan` holds no measurement at all."""
    from keypoint_learning_b200 import synth
    fr = np.stack([synth.organized_range_image(w, h, seed=seed0 + f, holes=f % 2 == 0)[0] for f in range(count)])
    if all_nan is not None:
        fr[all_nan] = np.nan
    return np.ascontiguousarray(fr)


def _single(det, frame, smoothing=5.0):
    _, idx = det.computeOrganized(frame, smoothing)
    return det.getResponse().copy(), idx


def _same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


SHAPES = [((320, 240), 6), ((97, 61), 3), ((7, 300), 2), ((12, 11), 2), ((1, 1), 2)]


@pytest.mark.parametrize("draws", [False, True])
def test_batch_equals_single_frames(kpl, draws):
    det = _detector(kpl, draws)
    total_kp = 0
    for (w, h), count in SHAPES:
        fr = _frames(w, h, count, seed0=w + h, all_nan=count - 1 if w == 320 else None)
        sc_b, kp_b = det.computeOrganizedBatch(fr)
        assert det.stats()["n_views"] == count
        for f in range(count):
            sc1, idx1 = _single(det, fr[f])
            assert _same(sc_b[f], sc1), ((w, h), f)          # NaN positions and payloads included
            assert np.array_equal(kp_b[f], idx1), ((w, h), f)
            total_kp += len(idx1)
        if w == 320:
            assert np.all(np.isnan(sc_b[-1])) and len(kp_b[-1]) == 0
    assert total_kp > 0
    # a batch in which no frame holds a finite point
    sc_b, kp_b = det.computeOrganizedBatch(np.full((3, 5, 4, 3), np.nan, np.float32))
    assert all(np.all(np.isnan(s)) for s in sc_b) and all(len(k) == 0 for k in kp_b)
    assert det.stats()["n_keypoints"] == 0 and det.stats()["n_points"] == 0
    det.close()


def test_batch_frame_against_oracle(kpl, oracle):
    fr = _frames(160, 120, 3, seed0=11)
    det = _detector(kpl)
    sc_b, kp_b = det.computeOrganizedBatch(fr)
    det.close()
    main_forest = oracle.load_forest_yaml(FOREST)
    xyz = fr[2]
    flat = xyz.reshape(-1, 3)
    nrm = oracle.normals_integral_image(xyz, 5.0, (0.0, 0.0, 0.0))
    keep = np.nonzero(np.isfinite(flat).all(axis=1))[0]
    assert len(keep) < len(flat)                             # frame 2 has holes
    ref = oracle.detect(np.ascontiguousarray(flat[keep]), main_forest, R_FEAT, R_NMS, float(np.float32(0.5)), 5, 10, normals4=nrm[keep], order=1)
    sc = sc_b[2]
    finite = np.isfinite(sc[keep]) | np.isfinite(ref["scores"])
    assert np.array_equal(sc[keep][finite].view(np.uint32), ref["scores"][finite].view(np.uint32))
    assert np.all(np.isnan(np.delete(sc, keep)))
    assert np.array_equal(kp_b[2], keep[ref["keypoints"]]) and len(kp_b[2]) > 0


def test_batched_normals_per_frame_viewpoints(kpl):
    fr = _frames(97, 61, 4, seed0=3)
    vps = np.array([[0, 0, 0], [0, 0, 2000], [400, -300, 700], [-50, 20, 9000]], np.float32)
    det = _detector(kpl)
    flipped = False
    for smoothing in (5.0, 3.0, 10.0):
        det.setNormalsMode(1, k=10, viewpoint=(0.0, 0.0, 0.0))
        det.computeOrganizedBatch(fr, smoothing, viewpoints=vps)
        m = det.stats()["n_points"]
        got = det.fetch("normals", m, 4)
        ref, plain = [], []
        for f in range(len(fr)):
            keep = np.isfinite(fr[f].reshape(-1, 3)).all(axis=1)
            det.setNormalsMode(1, k=10, viewpoint=tuple(float(v) for v in vps[f]))
            ref.append(det.computeNormalsOrganized(fr[f], smoothing)[keep])
            det.setNormalsMode(1, k=10, viewpoint=(0.0, 0.0, 0.0))
            plain.append(det.computeNormalsOrganized(fr[f], smoothing)[keep])
        ref = np.concatenate(ref)
        assert m == len(ref)
        assert _same(got, ref), smoothing
        flipped |= not _same(ref, np.concatenate(plain))
    assert flipped                                           # the viewpoints turned some normals around
    det.close()


@pytest.mark.parametrize("draws", [False, True])
def test_caller_normals(kpl, draws):
    fr = _frames(97, 61, 3, seed0=21)
    rng = np.random.default_rng(5)
    nrm = rng.normal(size=fr.shape[:3] + (4,)).astype(np.float32)
    nrm[..., :3] /= np.linalg.norm(nrm[..., :3], axis=-1, keepdims=True)
    nrm[rng.random(fr.shape[:3]) < 0.05] = np.nan
    det = _detector(kpl, draws)
    sc_b, kp_b = det.computeOrganizedBatch(fr, normals=nrm, viewpoints=np.full((3, 3), 1e6, np.float32))
    total = 0
    for f in range(len(fr)):
        det.setInputCloud(np.ascontiguousarray(fr[f].reshape(-1, 3))); det.setNormals(np.ascontiguousarray(nrm[f].reshape(-1, 4)))
        _, idx = det.compute()
        assert _same(sc_b[f], det.getResponse()), f
        assert np.array_equal(kp_b[f], idx), f
        total += len(idx)
    assert total > 0
    det.close()


def _device_run(det, fr, vps=None):
    import torch
    nf, h, w, _ = fr.shape
    x4 = np.ones((nf, h, w, 4), np.float32)
    x4[..., :3] = fr
    d_xyz = torch.from_numpy(x4).cuda()
    d_sc = torch.empty(nf * h * w, dtype=torch.float32, device="cuda")
    d_kp = torch.empty(nf * h * w, dtype=torch.int32, device="cuda")
    d_kpo = torch.empty(nf + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    nk = det.detectOrganizedBatchDevice(d_xyz.data_ptr(), w, h, nf, 5.0, viewpoints=vps, d_scores=d_sc.data_ptr(), d_kp_idx=d_kp.data_ptr(),
                                        d_kp_offsets=d_kpo.data_ptr())
    st = det.stats()
    kpo = d_kpo.cpu().numpy()
    kp = d_kp.cpu().numpy()
    sc = d_sc.cpu().numpy()
    n = h * w
    return nk, st, [sc[f * n:(f + 1) * n] for f in range(nf)], [kp[kpo[f]:kpo[f + 1]] for f in range(nf)]


def test_device_entry_point_and_budget(kpl):
    """The device entry point returns what the host one does; it synchronises with the host once more than
    kpl_detect_batch_device on the same compacted views, and the launches it adds do not grow with the number of frames."""
    import torch
    fr = _frames(160, 120, 32, seed0=40)
    vps = np.zeros((32, 3), np.float32); vps[::3, 2] = 5000.0
    det = _detector(kpl)
    counts = {}
    for nf in (4, 32):
        sub = np.ascontiguousarray(fr[:nf])
        sc_h, kp_h = det.computeOrganizedBatch(sub, viewpoints=vps[:nf])
        st_h = det.stats()
        nk, st, sc_d, kp_d = _device_run(det, sub, vps[:nf])
        assert nk == sum(len(k) for k in kp_h) > 0
        for f in range(nf):
            assert _same(sc_d[f], sc_h[f]) and np.array_equal(kp_d[f], kp_h[f]), (nf, f)
        # the same compacted views through kpl_detect_batch_device, with the batch's own normals
        m = st["n_points"]
        nrm = det.fetch("normals", m, 4)
        keep = [np.isfinite(sub[f].reshape(-1, 3)).all(axis=1) for f in range(nf)]
        cat = np.ones((m, 4), np.float32)
        cat[:, :3] = np.concatenate([sub[f].reshape(-1, 3)[keep[f]] for f in range(nf)])
        off = np.zeros(nf + 1, np.int64); off[1:] = np.cumsum([k.sum() for k in keep])
        d_xyz, d_nrm = torch.from_numpy(cat).cuda(), torch.from_numpy(nrm).cuda()
        d_kp = torch.empty(m, dtype=torch.int32, device="cuda"); d_kpo = torch.empty(nf + 1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        assert det.detectBatchDevice(d_xyz.data_ptr(), off, d_kp_idx=d_kp.data_ptr(), d_kp_offsets=d_kpo.data_ptr(), d_normals4=d_nrm.data_ptr()) == nk
        st_b = det.stats()
        # one round trip for the per-frame finite counts on top of the batch's; the host entry point adds the copy-out
        assert st["host_syncs"] == st_b["host_syncs"] + 1
        assert st_h["host_syncs"] == st["host_syncs"] + 1
        assert st["n_views"] == nf and st["n_points"] == m
        # launches on top of the batch's (whose radix-sort passes follow the grid's key bits): the same for 4 and 32 frames
        counts[nf] = st["kernel_launches"] - st_b["kernel_launches"]
        t = det.timings()
        assert t["total_ms"] >= t["normals_ms"] > 0
    assert counts[4] == counts[32]
    det.close()


def test_integral_image_chunks(kpl):
    """Frames whose integral images exceed one launch's scratch run in chunks; each frame's result is the one of a batch of
    its own."""
    w, h = 2048, 1536
    per_chunk = CHUNK_BYTES // ((w + 1) * (h + 1) * 24)
    assert per_chunk == 3
    fr = _frames(w, h, 4, seed0=70)
    det = _detector(kpl)
    det.computeOrganizedBatch(np.ascontiguousarray(fr[:3]))
    one_chunk = det.stats()["kernel_launches"]
    sc_b, kp_b = det.computeOrganizedBatch(fr)
    assert det.stats()["kernel_launches"] == one_chunk + 2     # a second chunk: one more integral image and normal launch
    for f in range(len(fr)):
        sc1, kp1 = det.computeOrganizedBatch(np.ascontiguousarray(fr[f:f + 1]))
        assert _same(sc_b[f], sc1[0]) and np.array_equal(kp_b[f], kp1[0]), f
    assert sum(len(k) for k in kp_b) > 0
    det.close()


def test_refusals(kpl):
    from keypoint_learning_b200 import capi
    L = capi.load_library()
    det = _detector(kpl)
    det._push()
    fr = _frames(12, 11, 2)
    f32, i32, i64 = ctypes.c_float, ctypes.c_int32, ctypes.c_int64
    sc = np.empty(fr.size, np.float32); kp = np.empty(fr.size, np.int32); kpo = np.empty(3, np.int64)
    P = lambda a, t: capi._ptr(a, t)

    def call(xyz=fr, stride=12, w=12, h=11, nf=2, s=5.0, normals=None, ns=0, kp_out=kp, kpo_out=kpo):
        return L.kpl_detect_batch_organized(det._h, P(xyz, f32), stride, P(normals, f32), ns, w, h, nf, s, None, P(sc, f32),
                                            P(kp_out, i32), P(kpo_out, i64))

    assert call() == 0
    bad = [dict(w=0), dict(h=0), dict(nf=0), dict(w=-3), dict(w=65536, h=32768, nf=1), dict(w=46341, h=46341, nf=1),
           dict(s=0.0), dict(s=-1.0), dict(s=float("nan")), dict(s=float("inf")), dict(stride=8), dict(stride=14),
           dict(normals=fr, ns=10), dict(xyz=None), dict(kp_out=None), dict(kpo_out=None)]
    for kw in bad:
        assert call(**kw) == KPL_E_INVALID, kw
    # device entry point
    import torch
    d = torch.zeros(fr.size // 3 * 4, dtype=torch.float32, device="cuda")
    dk = torch.empty(fr.size, dtype=torch.int32, device="cuda"); dko = torch.empty(3, dtype=torch.int64, device="cuda")
    nkp = ctypes.c_int64(0)

    def dcall(x=d.data_ptr(), w=12, h=11, nf=2, s=5.0, k=dk.data_ptr(), ko=dko.data_ptr()):
        return L.kpl_detect_batch_organized_device(det._h, ctypes.c_void_p(x), None, w, h, nf, s, None, None, ctypes.c_void_p(k),
                                                   ctypes.c_void_p(ko), ctypes.byref(nkp))

    assert dcall() == 0
    for kw in (dict(x=None), dict(k=None), dict(ko=None), dict(w=0), dict(nf=0), dict(s=0.0), dict(w=65536, h=32768, nf=1)):
        assert dcall(**kw) == KPL_E_INVALID, kw
    # a forced grid
    det.setForcedGrid((0.0, 0.0, 0.0), (4, 4, 4))
    det._push()
    assert call() == KPL_E_INVALID and dcall() == KPL_E_INVALID
    with pytest.raises(kpl.KplError) as e:
        det.computeOrganizedBatch(fr)
    assert e.value.code == KPL_E_INVALID
    det.close()
    nof = _detector(kpl, forest=False)
    with pytest.raises(kpl.KplError) as e:
        nof.computeOrganizedBatch(fr)
    assert e.value.code == KPL_E_FOREST
    nof.close()


CPP = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include "KeypointLearning.h"

// argv: forest, binary file (int32 frames, width, height; frames x height x width x 3 float xyz; frames x 3 float origins)
int main(int argc, char** argv)
{
    if (argc < 3) return 2;
    std::ifstream f(argv[2], std::ios::binary);
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
    pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> det(0.5, true, true, 4.0);
    det.setRadiusSearch(20.0); det.setNonMaximaDrawsThreshold(1.0f);
    if (!det.loadForest(argv[1])) return 3;
    std::vector<pcl::PointCloud<pcl::PointXYZI>> outs;
    std::vector<pcl::PointIndices> idx;
    if (!det.computeOrganizedBatch(frames, outs, &idx)) return 4;
    bool same = outs.size() == (size_t)F && idx.size() == (size_t)F;
    size_t total = 0;
    for (int k = 0; same && k < F; ++k) {
        pcl::PointCloud<pcl::PointXYZI> one;
        det.setInputCloud(frames[k]);
        det.compute(one);
        const auto& i1 = det.getKeypointsIndices()->indices;
        same = i1 == idx[k].indices && one.size() == outs[k].size() && outs[k].width == outs[k].size();
        for (size_t j = 0; same && j < one.size(); ++j)
            same = std::memcmp(&one.points[j].x, &outs[k].points[j].x, 12) == 0 &&
                   std::memcmp(&one.points[j].intensity, &outs[k].points[j].intensity, 4) == 0;
        total += i1.size();
    }
    // frames of different sizes are refused
    Cloud::Ptr other(new Cloud(*frames[0]));
    other->width = W / 2; other->height = H * 2;
    std::vector<Cloud::ConstPtr> mixed = {frames[0], other};
    const bool refused = !det.computeOrganizedBatch(mixed, outs);
    std::printf("keypoints %zu refused %d same %d\n", total, (int)refused, (int)same);
    return 0;
}
"""


def test_cpp_compute_organized_batch(kpl, tmp_path):
    """KeypointLearningDetector::computeOrganizedBatch on organized clouds with distinct sensor origins equals compute() on
    every frame: keypoint indices, xyz and intensity bits."""
    from keypoint_learning_b200 import build as B
    B.build_host()
    src, exe, data = str(tmp_path / "organized_batch.cpp"), str(tmp_path / "organized_batch"), str(tmp_path / "frames.bin")
    with open(src, "w") as f:
        f.write(CPP)
    common = [os.path.join(B.HOST, f) for f in sorted(os.listdir(B.HOST)) if f.endswith(".cpp") and not f.startswith("main_")]
    subprocess.check_call([B._host_cxx(), "-O2", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", B.HOST, src,
                           *common, "-o", exe, "-L", B.HERE, "-lkpl_b200", "-lpthread", "-Wl,-rpath," + B.HERE])
    fr = _frames(160, 120, 3, seed0=90)
    vps = np.array([[0, 0, 0], [0, 0, 3000], [200, 100, -100]], np.float32)
    with open(data, "wb") as f:
        f.write(np.array([3, 160, 120], np.int32).tobytes()); f.write(fr.tobytes()); f.write(vps.tobytes())
    r = subprocess.run([exe, FOREST, data], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "must be organized clouds of one width x height" in r.stderr
    words = r.stdout.split("\n")[-2].split()
    got = dict(zip(words[0::2], words[1::2]))
    assert int(got["keypoints"]) > 0 and got["refused"] == "1" and got["same"] == "1"
