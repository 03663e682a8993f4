"""Slab-sharded detection with the caller's normals (kpl_shard_set_slab_normals / kpl_shard_upload_normals): in-process
groups on one GPU, a one-rank NCCL communicator, torchrun over 2 / 4 GPUs and the C++ ShardedKeypointLearningDetector.
Every result must be bit-identical to the single-GPU kpl_detect with the same normals, on a plan without k-NN support."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz")
# (draws-remove, r_nms, threshold, draws threshold): plain NMS as test_gpu_multi.py, draws-remove with CASES[1] of
# test_gpu_draws_scaling.py
MODES = ((False, 4.0, 0.85, 0.0), (True, 4.0, 0.5, 1.0))


def _detector(kpl, draws=False, r_nms=4.0, th=0.85, dthr=0.0):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(r_nms)
    det.setNonMaximaDrawsRemove(draws); det.setNonMaximaDrawsThreshold(dthr)
    det.setPredictionThreshold(float(np.float32(th))); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    assert det.loadForest(FOREST)
    return det


def _ctx_params(det):
    from keypoint_learning_b200 import capi
    p = capi.KplParams()
    assert capi.load_library().kpl_get_params(det._h, ctypes.byref(p)) == 0
    return {f: (list(v) if isinstance(v, ctypes.Array) else v) for f, v in ((f, getattr(p, f)) for f, _ in p._fields_)}


def _single(det, xyz, nrm):
    det.setInputCloud(xyz); det.setNormals(nrm)
    _, idx = det.compute()
    return idx, det.getResponse().copy()


def _cheff(name):
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", name + ".npz"))["xyz"]
    return np.ascontiguousarray(xyz[:, [1, 0, 2]])          # the longest axis (y) onto the slab axis


def _perturbed(nrm, xyz, plan, seed):
    """Normals the device would not estimate: some replaced by random unit vectors, some flipped, some NaN -- among them
    points in the strip columns on both sides of every interior face."""
    from keypoint_learning_b200 import shard
    rng = np.random.default_rng(seed)
    out = np.array(nrm, np.float32, copy=True)
    n = len(xyz)
    kind = rng.integers(0, 3, n)
    pick = rng.random(n) < 0.1
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    out[pick & (kind == 0), :3] = v[pick & (kind == 0)]
    out[pick & (kind == 1), :3] *= -1
    out[pick & (kind == 2), :3] = np.nan
    cx = shard.cell_coords(xyz, plan.origin, plan.cell, 0)
    for c in plan.cuts[1:-1]:
        for side in ((cx >= c - plan.halo) & (cx < c), (cx >= c) & (cx < c + plan.halo)):
            assert all((pick & side & (kind == k)).any() for k in range(3))
    return out


def _group(kpl, xyz, nrm, plan, mode):
    from keypoint_learning_b200 import shard
    dets = [_detector(kpl, *mode) for _ in range(plan.world)]
    jobs = [shard.SlabJob(d, xyz, plan, r, None, normals=nrm) for r, d in enumerate(dets)]
    return dets, jobs


def _close(jobs, dets):
    for j in jobs:
        j.close()
    for d in dets:
        d.close()


def _same(kp, scores, jobs, idx_full, sc_full):
    assert np.array_equal(kp, idx_full), (len(kp), len(idx_full))
    for j, sc in zip(jobs, scores):
        assert np.array_equal(sc.view(np.uint32), sc_full[j.gidx].view(np.uint32))


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("mode", MODES, ids=["plain", "draws"])
def test_in_process_group_given_normals_equals_single_gpu(kpl, world, mode):
    from keypoint_learning_b200 import shard
    xyz = _cheff("cheff002")
    ref = _detector(kpl, *mode)
    nrm = ref.computeNormals(xyz)
    idx_full, sc_full = _single(ref, xyz, nrm)
    pairs_full = ref.stats()["feature_pairs"]
    ref.close()
    plan = shard.plan_slabs(xyz, 20.0, mode[1], 4, world, normal_support_cells=0)
    assert plan.normal_support_cells == 0 and plan.halo == max(plan.reach_feat, plan.reach_nms)
    dets, jobs = _group(kpl, xyz, nrm, plan, mode)
    before = [_ctx_params(d) for d in dets]
    kp, scores = shard.detect_group(jobs)
    _same(kp, scores, jobs, idx_full, sc_full)
    assert sum(d.stats()["n_scored"] for d in dets) == len(xyz)
    assert sum(d.stats()["feature_pairs"] for d in dets) == pairs_full
    assert [_ctx_params(d) for d in dets] == before
    if world > 1:
        info = [j.info() for j in jobs]
        assert all(i["halo_bytes"] == (i["send_left"] + i["send_right"]) * 36 for i in info)
    _close(jobs, dets)


@pytest.mark.parametrize("mode", MODES, ids=["plain", "draws"])
def test_normals_the_device_would_not_estimate(kpl, mode):
    """Random, flipped and NaN normals in every strip: the sharded result is the single-GPU one with those normals, and not
    the one with estimated normals (a path that ignored the caller's normals would give the latter)."""
    from keypoint_learning_b200 import shard
    xyz = _cheff("cheff002")
    world = 3
    ref = _detector(kpl, *mode)
    plan = shard.plan_slabs(xyz, 20.0, mode[1], 4, world, normal_support_cells=0)
    nrm = _perturbed(ref.computeNormals(xyz), xyz, plan, seed=3)
    idx_full, sc_full = _single(ref, xyz, nrm)
    assert np.isnan(sc_full).any()
    ref.close()
    dets, jobs = _group(kpl, xyz, nrm, plan, mode)
    kp, scores = shard.detect_group(jobs)
    _same(kp, scores, jobs, idx_full, sc_full)
    assert sum(d.stats()["n_unscored"] for d in dets) == int(np.isnan(nrm[:, :3]).any(axis=1).sum())
    _close(jobs, dets)
    # the same group with estimated normals
    est_plan = shard.plan_slabs(xyz, 20.0, mode[1], 4, world)
    dets = [_detector(kpl, *mode) for _ in range(world)]
    jobs = [shard.SlabJob(d, xyz, est_plan, r, None) for r, d in enumerate(dets)]
    kp_est, sc_est = shard.detect_group_widening(jobs, xyz, 20.0, mode[1], 4)
    assert not np.array_equal(kp_est, kp)
    assert not all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(sc_est, scores))
    _close(jobs, dets)


def test_streaming_upload_of_points_and_normals(kpl):
    """A second detection after kpl_shard_upload and kpl_shard_upload_normals, both with new values, is the single-GPU run
    on the new input."""
    from keypoint_learning_b200 import shard
    mode = MODES[1]
    xyz = _cheff("cheff002")
    ref = _detector(kpl, *mode)
    plan = shard.plan_slabs(xyz, 20.0, mode[1], 4, 3, normal_support_cells=0)
    nrm = _perturbed(ref.computeNormals(xyz), xyz, plan, seed=5)
    dets, jobs = _group(kpl, xyz, nrm, plan, mode)
    _same(*shard.detect_group(jobs), jobs, *_single(ref, xyz, nrm))
    # new positions in the same cell columns and the same bounding box (x kept, y / z moved, the extreme points kept)
    rng = np.random.default_rng(9)
    lo, hi = xyz.min(axis=0), xyz.max(axis=0)
    extreme = ((xyz == lo) | (xyz == hi)).any(axis=1)
    xyz2 = xyz.copy()
    xyz2[:, 1:] += rng.uniform(-0.7, 0.7, (len(xyz), 2)).astype(np.float32) * ~extreme[:, None]
    xyz2 = np.clip(xyz2, lo, hi)
    nrm2 = _perturbed(ref.computeNormals(xyz2), xyz2, plan, seed=6)
    for j in jobs:
        own = np.ones((j.n_owned, 4), np.float32)
        own[:, :3] = xyz2[j.gidx]
        j.upload(own)
        j.upload_normals(nrm2)
    idx2, sc2 = _single(ref, xyz2, nrm2)
    assert not np.array_equal(sc2.view(np.uint32), _single(ref, xyz, nrm)[1].view(np.uint32))
    _same(*shard.detect_group(jobs), jobs, idx2, sc2)
    ref.close()
    _close(jobs, dets)


def test_sparse_cloud_needs_no_support_with_given_normals(kpl):
    """The cloud of test_clipped_knn_support_is_detected: estimated k-NN normals are clipped at support 1; given normals need
    no support at all."""
    from keypoint_learning_b200 import shard
    rng = np.random.default_rng(5)
    xyz = np.stack([rng.uniform(-400, 400, 4000), rng.uniform(-100, 100, 4000), rng.uniform(-3, 3, 4000)], axis=1).astype(np.float32)
    ref = _detector(kpl)
    nrm = ref.computeNormals(xyz)
    idx_full, sc_full = _single(ref, xyz, nrm)
    ref.close()
    plan1 = shard.plan_slabs(xyz, 20.0, 4.0, 4, 2, normal_support_cells=1)
    dets = [_detector(kpl) for _ in range(2)]
    jobs = [shard.SlabJob(d, xyz, plan1, r, None) for r, d in enumerate(dets)]
    with pytest.raises(kpl.KplError) as e:
        shard.detect_group(jobs)
    assert e.value.code == 12
    plan0 = shard.plan_slabs(xyz, 20.0, 4.0, 4, 2, normal_support_cells=0)
    for j in jobs:
        j.normals = nrm
        j.replan(xyz, plan0)
    _same(*shard.detect_group(jobs), jobs, idx_full, sc_full)
    _close(jobs, dets)


def test_one_rank_nccl_communicator_given_normals(kpl):
    from keypoint_learning_b200 import shard
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff000.npz"))["xyz"]
    ref = _detector(kpl, *MODES[1])
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, 1, normal_support_cells=0)
    nrm = _perturbed(ref.computeNormals(xyz), xyz, plan, seed=8)
    idx_full, sc_full = _single(ref, xyz, nrm)
    before = _ctx_params(ref)
    job = shard.SlabJob(ref, xyz, plan, 0, shard.nccl_unique_id(), normals=nrm)
    sc = np.empty(job.n_owned, np.float32)
    n, kp = job.detect(scores_out=sc)
    assert n == len(idx_full) and np.array_equal(kp, idx_full)
    assert np.array_equal(sc.view(np.uint32), sc_full.view(np.uint32))
    assert _ctx_params(ref) == before
    job.close()
    ref.close()


def test_refusals(kpl):
    """Ranks that disagree on normals, a bad normals stride, and kpl_shard_upload_normals on a slab set without normals
    fail with KPL_E_INVALID; the contexts are left as they were."""
    from keypoint_learning_b200 import capi, shard
    L = capi.load_library()
    xyz = _cheff("cheff002")
    ref = _detector(kpl)
    nrm = ref.computeNormals(xyz)
    idx_full, _ = _single(ref, xyz, nrm)
    ref.close()
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, 2, normal_support_cells=0)
    dets = [_detector(kpl) for _ in range(2)]
    jobs = [shard.SlabJob(dets[0], xyz, plan, 0, None, normals=nrm), shard.SlabJob(dets[1], xyz, plan, 1, None)]
    before = [_ctx_params(d) for d in dets]
    with pytest.raises(kpl.KplError) as e:
        shard.detect_group(jobs)
    assert e.value.code == 1
    assert [_ctx_params(d) for d in dets] == before
    with pytest.raises(kpl.KplError) as e:
        jobs[1].upload_normals(nrm)
    assert e.value.code == 1
    f32p = ctypes.POINTER(ctypes.c_float)
    own = np.ascontiguousarray(jobs[1].host_xyz4)
    own_n = np.ascontiguousarray(nrm[jobs[1].gidx])
    gp = jobs[1].gidx.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    assert L.kpl_shard_set_slab_normals(jobs[1]._h, own.ctypes.data_as(f32p), 16, own_n.ctypes.data_as(f32p), 10, gp, len(own)) == 1
    assert L.kpl_shard_set_slab_normals(jobs[1]._h, own.ctypes.data_as(f32p), 16, None, 16, gp, len(own)) == 1
    # both ranks with normals: the group runs
    jobs[1].normals = nrm
    jobs[1].replan(xyz, plan)
    assert np.array_equal(shard.detect_group(jobs)[0], idx_full)
    # a plain set_slab returns a rank to estimated normals: the ranks disagree again
    jobs[1].normals = None
    jobs[1].replan(xyz, plan)
    with pytest.raises(kpl.KplError) as e:
        shard.detect_group(jobs)
    assert e.value.code == 1
    _close(jobs, dets)


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_nccl_given_normals_equals_single_gpu(tmp_path, kpl, world):
    if _ngpus() < world:
        pytest.skip("needs %d GPUs" % world)
    out = str(tmp_path / "kp.npz")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "normals_multi_gpu_worker.py"), out]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    xyz = _cheff("cheff002")
    nrm = np.load(out)["normals"]
    ref = _detector(kpl, *MODES[1])
    idx_full, sc_full = _single(ref, xyz, nrm)
    ref.close()
    assert np.isnan(sc_full).any()
    assert np.array_equal(np.load(out)["keypoints"], idx_full)
    for rank in range(world):
        d = np.load(out + ".rank%d.npz" % rank)
        assert np.array_equal(d["scores"].view(np.uint32), sc_full[d["gidx"]].view(np.uint32))


CPP = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include "KeypointLearning.h"
#include "KeypointLearningSharded.h"

// argv: forest, binary file (int64 n, n x 3 float xyz, n x 4 float normals)
int main(int argc, char** argv)
{
    if (argc < 3) return 2;
    std::ifstream f(argv[2], std::ios::binary);
    int64_t n = 0;
    f.read(reinterpret_cast<char*>(&n), sizeof n);
    std::vector<float> xyz((size_t)n * 3), nrm((size_t)n * 4);
    f.read(reinterpret_cast<char*>(xyz.data()), xyz.size() * 4);
    f.read(reinterpret_cast<char*>(nrm.data()), nrm.size() * 4);
    pcl::PointCloud<pcl::PointXYZ>::Ptr cloud(new pcl::PointCloud<pcl::PointXYZ>);
    pcl::PointCloud<pcl::Normal>::Ptr normals(new pcl::PointCloud<pcl::Normal>), few(new pcl::PointCloud<pcl::Normal>);
    for (int64_t i = 0; i < n; ++i) {
        cloud->push_back(pcl::PointXYZ(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        pcl::Normal q;
        q.normal_x = nrm[4 * i]; q.normal_y = nrm[4 * i + 1]; q.normal_z = nrm[4 * i + 2]; q.curvature = nrm[4 * i + 3];
        normals->push_back(q);
    }
    few->points.assign(normals->points.begin(), normals->points.begin() + 10);
    pcl::keypoints::KeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> single(0.5, true, true, 4.0);
    pcl::keypoints::ShardedKeypointLearningDetector<pcl::PointXYZ, pcl::PointXYZI> sharded(3);
    single.setRadiusSearch(20.0); single.setNonMaximaDrawsThreshold(1.0f);
    sharded.setRadiusSearch(20.0); sharded.setNonMaxRadius(4.0); sharded.setPredictionThreshold(0.5);
    sharded.setNonMaximaDrawsRemove(true); sharded.setNonMaximaDrawsThreshold(1.0f);
    if (!single.loadForest(argv[1]) || !sharded.loadForest(argv[1])) return 3;
    pcl::PointCloud<pcl::PointXYZI> out1, out3;
    single.setInputCloud(cloud); single.setNormals(normals);
    single.compute(out1);
    sharded.setInputCloud(cloud); sharded.setNormals(few);
    const bool refused = !sharded.compute(out3);
    sharded.setNormals(normals);
    if (!sharded.compute(out3)) return 4;
    const auto& i1 = single.getKeypointsIndices()->indices;
    const auto& i3 = sharded.getKeypointsIndices()->indices;
    const std::vector<float>& r1 = single.getResponse();
    const std::vector<float>& r3 = sharded.getResponse();
    bool same = i1 == i3 && r1.size() == r3.size() && std::memcmp(r1.data(), r3.data(), r1.size() * 4) == 0 && out1.size() == out3.size();
    for (size_t k = 0; same && k < out1.size(); ++k)
        same = std::memcmp(&out1.points[k], &out3.points[k], sizeof(pcl::PointXYZI)) == 0;
    std::printf("keypoints %zu slabs %d support %d refused %d same %d\n", i1.size(), sharded.plan().world,
                sharded.plan().normal_support_cells, (int)refused, (int)same);
    return 0;
}
"""


def test_cpp_sharded_detector_set_normals(kpl, tmp_path):
    """ShardedKeypointLearningDetector::setNormals at 3 ranks on one GPU equals KeypointLearningDetector with the same
    normals (keypoint cloud, indices, responses); a normals cloud of the wrong size is refused as initCompute does."""
    from keypoint_learning_b200 import build as B
    B.build_host()
    src, exe, data = str(tmp_path / "sharded_normals.cpp"), str(tmp_path / "sharded_normals"), str(tmp_path / "cloud.bin")
    with open(src, "w") as f:
        f.write(CPP)
    common = [os.path.join(B.HOST, f) for f in sorted(os.listdir(B.HOST)) if f.endswith(".cpp") and not f.startswith("main_")]
    subprocess.check_call([B._host_cxx(), "-O2", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", B.HOST, src,
                           *common, "-o", exe, "-L", B.HERE, "-lkpl_b200", "-lpthread", "-Wl,-rpath," + B.HERE])
    xyz = _cheff("cheff001")
    det = _detector(kpl)
    nrm = det.computeNormals(xyz)
    det.close()
    from keypoint_learning_b200 import shard
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, 3, normal_support_cells=0)
    nrm = _perturbed(nrm, xyz, plan, seed=11)
    with open(data, "wb") as f:
        f.write(np.int64(len(xyz)).tobytes()); f.write(xyz.astype(np.float32).tobytes()); f.write(nrm.astype(np.float32).tobytes())
    r = subprocess.run([exe, FOREST, data], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "the number of normals does not match the number of input points" in r.stderr
    words = r.stdout.split()
    got = dict(zip(words[0::2], words[1::2]))
    assert int(got["keypoints"]) > 0 and got["slabs"] == "3" and got["support"] == "0"
    assert got["refused"] == "1" and got["same"] == "1"
