"""Every forest of the set over a slab-sharded cloud from one feature pass (kpl_shard_detect_forests(_group)): in-process
groups on one GPU, a one-rank NCCL communicator, torchrun over 2 / 4 GPUs and the C++ ShardedKeypointLearningDetector.
For every forest k the owned scores (as bits) and the global keypoints must be those of the single-GPU computeForests,
and so those of kpl_detect with only forest k loaded."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

try:        # torch (the torchrun tests' device count) before the one-rank NCCL test loads a libnccl.so.2 of its own
    import torch
except ImportError:
    torch = None

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]
FOREST_A4xB8 = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-A4xB8-T20-D8.yaml.gz")
R_FEAT, R_NMS = 20.0, 4.0
TH = float(np.float32(0.5))
KPL_E_INVALID, KPL_E_VARCOUNT, KPL_E_HALO = 1, 5, 12
NMS = ("plain", "draws", "off")


def _detector(kpl, nms="plain", forests=FORESTS):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(nms != "off"); det.setNonMaxRadius(R_NMS)
    det.setNonMaximaDrawsRemove(nms == "draws"); det.setNonMaximaDrawsThreshold(1.0 if nms == "draws" else 0.0)
    det.setPredictionThreshold(TH); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10)
    _load(det, forests)
    return det


def _load(det, forests):
    assert det.loadForest(forests[0])
    for f in forests[1:]:
        det.addForest(f)
    assert det.forestCount() == len(forests)


def _cheff(name="cheff002"):
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", name + ".npz"))["xyz"]
    return np.ascontiguousarray(xyz[:, [1, 0, 2]])          # the longest axis (y) onto the slab axis


def _single(kpl, xyz, nms, nrm=None, thresholds=None):
    """single-GPU computeForests: ([K keypoint index arrays], (K, n) responses)"""
    det = _detector(kpl, nms)
    det.setInputCloud(xyz)
    if nrm is not None:
        det.setNormals(nrm)
    out = det.computeForests(thresholds)
    sc = det.getResponses().copy()
    det.close()
    return [idx for _, idx in out], sc


def _jobs(kpl, xyz, plan, nms, nrm=None, forests=FORESTS):
    from keypoint_learning_b200 import shard
    dets = [_detector(kpl, nms, forests) for _ in range(plan.world)]
    return dets, [shard.SlabJob(d, xyz, plan, r, None, normals=nrm) for r, d in enumerate(dets)]


def _close(jobs, dets):
    for j in jobs:
        j.close()
    for d in dets:
        d.close()


def _same(kps, scores, jobs, kp_full, sc_full):
    assert len(kps) == len(kp_full)
    for k, (a, b) in enumerate(zip(kps, kp_full)):
        assert np.array_equal(a, b), (k, len(a), len(b))
    for j, sc in zip(jobs, scores):
        assert sc.shape == (len(kp_full), j.n_owned)
        assert np.array_equal(sc.view(np.uint32), sc_full[:, j.gidx].view(np.uint32))


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("nms", NMS)
@pytest.mark.parametrize("normals", ["estimated", "given"])
def test_in_process_group_forests_equal_single_gpu(kpl, world, nms, normals):
    from keypoint_learning_b200 import shard
    xyz = _cheff()
    nrm = None
    if normals == "given":
        d = _detector(kpl, nms)
        nrm = d.computeNormals(xyz)
        d.close()
    kp_full, sc_full = _single(kpl, xyz, nms, nrm)
    assert all(len(k) for k in kp_full)
    if normals == "given":
        plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, world, normal_support_cells=0)
        dets, jobs = _jobs(kpl, xyz, plan, nms, nrm)
        kps, scores = shard.detect_group_forests(jobs)
    else:
        plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, world)
        dets, jobs = _jobs(kpl, xyz, plan, nms)
        kps, scores = shard.detect_group_forests_widening(jobs, xyz, R_FEAT, R_NMS, 4)
    _same(kps, scores, jobs, kp_full, sc_full)
    stats = [d.stats() for d in dets]
    assert sum(s["n_scored"] for s in stats) == len(xyz)
    assert sum(s["n_keypoints"] for s in stats) == sum(len(k) for k in kp_full)
    pairs = sum(s["feature_pairs"] for s in stats)
    if world > 1:
        info = [j.info() for j in jobs]
        extra = 32 if normals == "given" else 16
        assert all(i["halo_bytes"] == (i["send_left"] + i["send_right"]) * (extra + 4 * 3) for i in info)
    # kpl_shard_detect on the same contexts: forest 0 only, from a feature pass of the same size
    kp0, sc0 = shard.detect_group(jobs)
    assert np.array_equal(kp0, kp_full[0])
    for j, s in zip(jobs, sc0):
        assert np.array_equal(s.view(np.uint32), sc_full[0, j.gidx].view(np.uint32))
    assert sum(d.stats()["feature_pairs"] for d in dets) == pairs
    if world > 1:
        assert all(i["halo_bytes"] == (i["send_left"] + i["send_right"]) * (extra + 4) for i in (j.info() for j in jobs))
    _close(jobs, dets)


def test_per_forest_thresholds_with_an_empty_forest(kpl):
    from keypoint_learning_b200 import shard
    xyz = _cheff()
    th = [TH, 1.0e9, float(np.float32(0.3))]
    kp_full, sc_full = _single(kpl, xyz, "plain", thresholds=th)
    assert len(kp_full[0]) and not len(kp_full[1]) and len(kp_full[2])
    plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, 3)
    dets, jobs = _jobs(kpl, xyz, plan, "plain")
    kps, scores = shard.detect_group_forests_widening(jobs, xyz, R_FEAT, R_NMS, 4, thresholds=th)
    _same(kps, scores, jobs, kp_full, sc_full)
    with pytest.raises(ValueError):
        shard.detect_group_forests(jobs, thresholds=th[:2])
    _close(jobs, dets)


@pytest.mark.parametrize("nms", ["plain", "draws"])
def test_one_forest_is_shard_detect(kpl, nms):
    """K = 1 through the forests entry point: kpl_shard_detect's results, kernel launches and host synchronisations."""
    from keypoint_learning_b200 import shard
    xyz = _cheff()
    plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, 3)
    dets, jobs = _jobs(kpl, xyz, plan, nms, forests=FORESTS[:1])
    kp, sc = shard.detect_group_widening(jobs, xyz, R_FEAT, R_NMS, 4)
    ref = [(s["kernel_launches"], s["host_syncs"]) for s in (d.stats() for d in dets)]
    kps, scores = shard.detect_group_forests(jobs)
    assert len(kps) == 1 and np.array_equal(kps[0], kp)
    for a, b in zip(scores, sc):
        assert np.array_equal(a[0].view(np.uint32), b.view(np.uint32))
    assert [(s["kernel_launches"], s["host_syncs"]) for s in (d.stats() for d in dets)] == ref
    _close(jobs, dets)


def test_refusals_leave_the_contexts_usable(kpl):
    from keypoint_learning_b200 import capi, shard
    L = capi.load_library()
    xyz = _cheff()
    kp_full, sc_full = _single(kpl, xyz, "plain")
    plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, 2)
    dets, jobs = _jobs(kpl, xyz, plan, "plain")

    def refused(code):
        with pytest.raises(kpl.KplError) as e:
            shard.detect_group_forests(jobs)
        assert e.value.code == code

    def right():
        _same(*shard.detect_group_forests(jobs), jobs, kp_full, sc_full)

    _same(*shard.detect_group_forests_widening(jobs, xyz, R_FEAT, R_NMS, 4), jobs, kp_full, sc_full)
    _load(dets[1], FORESTS[:2])                       # another forest count
    refused(KPL_E_INVALID)
    _load(dets[1], [FORESTS[0], FORESTS[2], FORESTS[1]])   # another forest at slots 1 and 2
    refused(KPL_E_INVALID)
    _load(dets[1], FORESTS)
    right()
    for d in dets:                                    # a forest that does not match annuli x bins
        d.addForest(FOREST_A4xB8)
    refused(KPL_E_VARCOUNT)
    assert "forest 3" in (L.kpl_last_error(dets[0]._h) or b"").decode()
    for d in dets:
        _load(d, FORESTS)
    right()
    hs = (ctypes.c_void_p * 2)(*[j._h for j in jobs])
    kp = np.empty(4, np.int32)
    off = np.zeros(4, np.int64)
    n = ctypes.c_int64(0)
    rc = L.kpl_shard_detect_forests_group(hs, 2, None, None, kp.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), kp.size,
                                          off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), ctypes.byref(n))
    assert rc == KPL_E_INVALID
    right()
    _close(jobs, dets)


def test_sparse_cloud_widens_for_every_forest(kpl):
    """The cloud of test_clipped_knn_support_is_detected scored with three forests: KPL_E_HALO at support 1, the single-GPU
    result for every forest after widening."""
    from keypoint_learning_b200 import shard
    rng = np.random.default_rng(5)
    xyz = np.stack([rng.uniform(-400, 400, 4000), rng.uniform(-100, 100, 4000), rng.uniform(-3, 3, 4000)], axis=1).astype(np.float32)
    kp_full, sc_full = _single(kpl, xyz, "plain")
    plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, 2, normal_support_cells=1)
    dets, jobs = _jobs(kpl, xyz, plan, "plain")
    with pytest.raises(kpl.KplError) as e:
        shard.detect_group_forests(jobs)
    assert e.value.code == KPL_E_HALO
    _same(*shard.detect_group_forests_widening(jobs, xyz, R_FEAT, R_NMS, 4), jobs, kp_full, sc_full)
    assert jobs[0].plan.normal_support_cells > 1
    _close(jobs, dets)


def test_one_rank_nccl_communicator(kpl):
    from keypoint_learning_b200 import shard
    xyz = _cheff("cheff000")
    kp_full, sc_full = _single(kpl, xyz, "plain")
    det = _detector(kpl)
    plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, 1)
    job = shard.SlabJob(det, xyz, plan, 0, shard.nccl_unique_id())
    job.detect()
    syncs = det.stats()["host_syncs"]
    sc = np.empty(3 * job.n_owned, np.float32)
    n, off, kps = job.detect_forests(scores_out=sc)
    assert n == sum(len(k) for k in kp_full) and off[-1] == n
    for a, b in zip(kps, kp_full):
        assert np.array_equal(a, b)
    assert np.array_equal(sc.reshape(3, -1).view(np.uint32), sc_full.view(np.uint32))
    assert det.stats()["host_syncs"] == syncs + 1
    job.close()
    det.close()


def _ngpus():
    return torch.cuda.device_count() if torch is not None else 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("nms", ["plain", "draws"])
def test_sharded_nccl_forests_equal_single_gpu(tmp_path, kpl, world, nms):
    if _ngpus() < world:
        pytest.skip("needs %d GPUs" % world)
    out = str(tmp_path / "kp.npz")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "forests_multi_gpu_worker.py"), out, nms]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    kp_full, sc_full = _single(kpl, _cheff(), nms)
    got = np.load(out)
    off = got["offsets"]
    for k in range(len(FORESTS)):
        assert np.array_equal(got["keypoints"][off[k]:off[k + 1]], kp_full[k])
    for rank in range(world):
        d = np.load(out + ".rank%d.npz" % rank)
        assert np.array_equal(d["scores"].view(np.uint32), sc_full[:, d["gidx"]].view(np.uint32))


CPP = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include "KeypointLearning.h"
#include "KeypointLearningSharded.h"

// argv: three forests, binary file (int64 n, n x 3 float xyz, n x 4 float normals)
int main(int argc, char** argv)
{
    if (argc < 5) return 2;
    std::ifstream f(argv[4], std::ios::binary);
    int64_t n = 0;
    f.read(reinterpret_cast<char*>(&n), sizeof n);
    std::vector<float> xyz((size_t)n * 3), nrm((size_t)n * 4);
    f.read(reinterpret_cast<char*>(xyz.data()), xyz.size() * 4);
    f.read(reinterpret_cast<char*>(nrm.data()), nrm.size() * 4);
    pcl::PointCloud<pcl::PointXYZ>::Ptr cloud(new pcl::PointCloud<pcl::PointXYZ>);
    pcl::PointCloud<pcl::Normal>::Ptr normals(new pcl::PointCloud<pcl::Normal>);
    for (int64_t i = 0; i < n; ++i) {
        cloud->push_back(pcl::PointXYZ(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        pcl::Normal q;
        q.normal_x = nrm[4 * i]; q.normal_y = nrm[4 * i + 1]; q.normal_z = nrm[4 * i + 2]; q.curvature = nrm[4 * i + 3];
        normals->push_back(q);
    }
    pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> single(0.5, true, false, 4.0);
    pcl::keypoints::ShardedKeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> sharded(3);
    single.setRadiusSearch(20.0);
    sharded.setRadiusSearch(20.0); sharded.setNonMaxRadius(4.0); sharded.setPredictionThreshold(0.5); sharded.setNonMaximaDrawsRemove(false);
    if (!single.loadForest(argv[1]) || !sharded.loadForest(argv[1])) return 3;
    for (int k = 2; k < 4; ++k)
        if (!single.addForest(argv[k]) || !sharded.addForest(argv[k])) return 3;
    single.setInputCloud(cloud); single.setNormals(normals);
    sharded.setInputCloud(cloud); sharded.setNormals(normals);
    std::vector<pcl::PointCloud<pcl::PointXYZI>> out1, out3;
    std::vector<pcl::PointIndices> i1, i3;
    const std::vector<double> two = {0.5, 0.5};
    const bool refused = !sharded.computeForests(out3, &i3, &two);
    if (!single.computeForests(out1, &i1) || !sharded.computeForests(out3, &i3)) return 4;
    bool same = out1.size() == 3 && out3.size() == 3 && i1.size() == 3 && i3.size() == 3;
    size_t total = 0;
    for (size_t k = 0; same && k < 3; ++k) {
        same = i1[k].indices == i3[k].indices && out1[k].size() == out3[k].size();
        for (size_t j = 0; same && j < out1[k].size(); ++j)
            same = std::memcmp(&out1[k].points[j], &out3[k].points[j], sizeof(pcl::PointXYZI)) == 0;
        total += i1[k].indices.size();
    }
    // compute() still scores forest 0 only
    pcl::PointCloud<pcl::PointXYZI> c3;
    same = same && sharded.compute(c3) && sharded.getKeypointsIndices()->indices == i1[0].indices;
    std::printf("keypoints %zu slabs %d refused %d same %d\n", total, sharded.plan().world, (int)refused, (int)same);
    return 0;
}
"""


def test_cpp_sharded_detector_compute_forests(kpl, tmp_path):
    """ShardedKeypointLearningDetector::computeForests at 3 ranks on one GPU equals KeypointLearningDetector::computeForests
    point for point; a thresholds vector of the wrong size is refused."""
    from keypoint_learning_b200 import build as B
    B.build_host()
    src, exe, data = str(tmp_path / "sharded_forests.cpp"), str(tmp_path / "sharded_forests"), str(tmp_path / "cloud.bin")
    with open(src, "w") as f:
        f.write(CPP)
    common = [os.path.join(B.HOST, f) for f in sorted(os.listdir(B.HOST)) if f.endswith(".cpp") and not f.startswith("main_")]
    subprocess.check_call([B._host_cxx(), "-O2", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", B.HOST, src,
                           *common, "-o", exe, "-L", B.HERE, "-lkpl_b200", "-lpthread", "-Wl,-rpath," + B.HERE])
    xyz = _cheff("cheff001")
    det = _detector(kpl)
    nrm = det.computeNormals(xyz)           # the same normals for both detectors (the single one estimates radius normals)
    det.close()
    with open(data, "wb") as f:
        f.write(np.int64(len(xyz)).tobytes()); f.write(xyz.astype(np.float32).tobytes()); f.write(nrm.astype(np.float32).tobytes())
    r = subprocess.run([exe, *FORESTS, data], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "2 thresholds for 3 forests" in r.stderr
    words = r.stdout.split()
    got = dict(zip(words[0::2], words[1::2]))
    assert int(got["keypoints"]) > 0 and got["slabs"] == "3"
    assert got["refused"] == "1" and got["same"] == "1"
