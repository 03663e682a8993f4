"""N-GPU result == 1-GPU result, bit for bit (BASELINE.md s5), through the C entry points kpl_shard_* of include/kpl.h.
On a single GPU: the ranks of an in-process group (peer copies instead of NCCL; every kernel and all host logic of the
sharded step) and a one-rank NCCL communicator.  With 2+ GPUs: real NCCL halo / score exchange under torchrun."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
def test_sharded_nccl_equals_golden(tmp_path, golden, kpl, world):
    if _ngpus() < world:
        pytest.skip("needs %d GPUs" % world)
    out = str(tmp_path / "kp.npz")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multi_gpu_worker.py"), out, "cheff001"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    # the single-GPU, unsharded run of the same (axis-permuted) cloud is the reference
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff001.npz"))["xyz"]
    xyz = np.ascontiguousarray(xyz[:, [1, 0, 2]])
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(4.0); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(0.85))); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    assert det.loadForest(os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz"))
    det.setInputCloud(xyz)
    _, idx_full = det.compute()
    sc_full = det.getResponse().copy()
    det.close()
    assert len(idx_full) == len(golden["cheff001"]["keypoints"]) or len(idx_full) > 0
    assert np.array_equal(np.load(out)["keypoints"], idx_full)
    seen = np.zeros(len(sc_full), bool)
    scored = 0
    for rank in range(world):
        d = np.load(out + ".rank%d.npz" % rank)
        assert not seen[d["gidx"]].any()
        seen[d["gidx"]] = True
        assert np.array_equal(d["scores"].view(np.uint32), sc_full[d["gidx"]].view(np.uint32))
        assert int(d["halo_bytes"]) > 0
        assert int(d["syncs"]) <= 3                      # work lists, counters, results: nothing else waits on the host
        scored += int(d["scored"])
    assert seen.all()
    assert scored == len(sc_full)                        # every point scored exactly once across the ranks


def _single_gpu_reference(kpl, xyz, forest="synthetic-T100-D15"):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(4.0); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(0.85))); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    assert det.loadForest(os.path.join(ROOT, "tests", "golden", "forests", forest + ".yaml.gz"))
    return det


def _ctx_params(det):
    """kpl_get_params of the detector's context, field by field (a sharded call must leave it untouched)."""
    from keypoint_learning_b200 import capi
    p = capi.KplParams()
    assert capi.load_library().kpl_get_params(det._h, ctypes.byref(p)) == 0
    return {f: (list(v) if isinstance(v, ctypes.Array) else v) for f, v in ((f, getattr(p, f)) for f, _ in p._fields_)}


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_in_process_group_equals_single_gpu(kpl, world):
    """All ranks of an in-process group on ONE device: same kernels, same host logic, strips moved by device copies."""
    from keypoint_learning_b200 import shard
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff002.npz"))["xyz"]
    xyz = np.ascontiguousarray(xyz[:, [1, 0, 2]])
    ref = _single_gpu_reference(kpl, xyz)
    ref.setInputCloud(xyz)
    _, idx_full = ref.compute()
    sc_full = ref.getResponse().copy()
    pairs_full = ref.stats()["feature_pairs"]
    ref.close()
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, world)
    dets = [_single_gpu_reference(kpl, xyz) for _ in range(world)]
    jobs = [shard.SlabJob(d, xyz, plan, r, None) for r, d in enumerate(dets)]
    for rep in range(2):
        # the view has stray points whose 10th neighbour lies beyond one cell column: the k-NN support is widened until
        # no normal that matters is clipped (KPL_E_HALO -> re-plan)
        kp, scores = shard.detect_group_widening(jobs, xyz, 20.0, 4.0, 4)
        assert np.array_equal(kp, idx_full)
        for j, sc in zip(jobs, scores):
            assert np.array_equal(sc.view(np.uint32), sc_full[j.gidx].view(np.uint32))
    assert sum(d.stats()["n_scored"] for d in dets) == len(xyz)
    assert sum(d.stats()["feature_pairs"] for d in dets) == pairs_full          # no band is scored twice
    if world > 1:
        assert all(j.info()["halo_bytes"] > 0 for j in jobs)
        assert jobs[0].info()["n_left"] == 0 and jobs[0].info()["n_right"] == jobs[1].info()["send_left"]
    for j in jobs:
        j.close()
    for d in dets:
        d.close()


def test_clipped_knn_support_is_detected(kpl):
    """A slab whose halo is too thin for the k-NN support of a normal that matters fails with KPL_E_HALO on a sparse cloud
    instead of returning different normals than the single-GPU run."""
    from keypoint_learning_b200 import shard
    rng = np.random.default_rng(5)
    # ~6 mm spacing: the 10th neighbour lies ~11 mm away, far beyond one 5 mm cell column
    xyz = np.stack([rng.uniform(-400, 400, 4000), rng.uniform(-100, 100, 4000), rng.uniform(-3, 3, 4000)], axis=1).astype(np.float32)
    ref = _single_gpu_reference(kpl, xyz)
    ref.setInputCloud(xyz)
    _, idx_full = ref.compute()
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, 2, normal_support_cells=1)
    dets = [_single_gpu_reference(kpl, xyz) for _ in range(2)]
    jobs = [shard.SlabJob(d, xyz, plan, r, None) for r, d in enumerate(dets)]
    before = [_ctx_params(d) for d in dets]
    with pytest.raises(kpl.KplError) as e:
        shard.detect_group(jobs)
    assert e.value.code == 12
    # the failed call left every context as it was: a plain detection on it is the single-GPU one
    for d, p in zip(dets, before):
        assert _ctx_params(d) == p
        d.setInputCloud(xyz)
        assert np.array_equal(d.compute()[1], idx_full)
    for j in jobs:
        j.close()
    # a wide enough support passes and reproduces the single-GPU result
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, 2, normal_support_cells=40)
    jobs = [shard.SlabJob(d, xyz, plan, r, None) for r, d in enumerate(dets)]
    kp, scores = shard.detect_group(jobs)
    assert np.array_equal(kp, idx_full)
    for j, sc in zip(jobs, scores):
        full = ref.getResponse()[j.gidx]
        assert np.array_equal(sc.view(np.uint32), full.view(np.uint32))
    for j in jobs:
        j.close()
    for d in dets + [ref]:
        d.close()


def test_one_rank_nccl_communicator(kpl):
    """kpl_shard_detect over a real (one-rank) NCCL communicator: ncclCommInitRank, the record all-gather, the gather path."""
    from keypoint_learning_b200 import shard
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff000.npz"))["xyz"]
    ref = _single_gpu_reference(kpl, xyz)
    ref.setInputCloud(xyz)
    _, idx_full = ref.compute()
    sc_full = ref.getResponse().copy()
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, 1)
    before = _ctx_params(ref)
    job = shard.SlabJob(ref, xyz, plan, 0, shard.nccl_unique_id())
    sc = np.empty(job.n_owned, np.float32)
    n, kp = job.detect(scores_out=sc)
    assert n == len(idx_full) and np.array_equal(kp, idx_full)
    assert np.array_equal(sc.view(np.uint32), sc_full.view(np.uint32))
    # the sharded call left the context as it was: a plain detection on it is the single-GPU one
    assert _ctx_params(ref) == before
    assert np.array_equal(ref.compute()[1], idx_full)
    job.close()
    ref.close()
