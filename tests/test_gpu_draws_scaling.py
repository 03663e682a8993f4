"""Draws-remove NMS (hpp:233-250, the detector's default NMS mode) on the two scaling paths: a batch of views in one pass
and slab-sharded detection (an in-process group on one GPU, a one-rank NCCL communicator, torchrun over 2 / 4 GPUs).
Every result must be bit-identical to the single-GPU kpl_detect with draws-remove on."""
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
# (r_nms, threshold, draws threshold) of test_nms_draws_remove_branch, dthr = 0 included
CASES = ((4.0, 0.85, 2.0), (4.0, 0.5, 1.0), (8.0, 0.3, 8.0), (2.0, 0.0, 0.7), (4.0, 0.85, 0.0))
# one constant leaf: every point with a finite normal scores 1 - 0 / 1 = 1 and ties with all its neighbours
PLATEAU_FOREST = dict(ntrees=1, roots=[0], var=[-1], thr=[0.0], left=[-1], right=[-1], value=[0.0], var_count=0)


def _detector(kpl, r_nms, th, dthr, forest=FOREST):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(r_nms)
    det.setNonMaximaDrawsRemove(True); det.setNonMaximaDrawsThreshold(dthr)
    det.setPredictionThreshold(float(np.float32(th))); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    if isinstance(forest, dict):
        det.setForestArrays(forest)
    else:
        assert det.loadForest(forest)
    return det


def _set_case(det, r_nms, th, dthr):
    det.setNonMaxRadius(r_nms); det.setPredictionThreshold(float(np.float32(th))); det.setNonMaximaDrawsThreshold(dthr)


def _ctx_params(det):
    from keypoint_learning_b200 import capi
    p = capi.KplParams()
    assert capi.load_library().kpl_get_params(det._h, ctypes.byref(p)) == 0
    return {f: (list(v) if isinstance(v, ctypes.Array) else v) for f, v in ((f, getattr(p, f)) for f, _ in p._fields_)}


def _single(det, xyz):
    det.setInputCloud(xyz); det.setNormals(None)
    _, idx = det.compute()
    return idx, det.getResponse().copy()


def _cheff002():
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff002.npz"))["xyz"]
    return np.ascontiguousarray(xyz[:, [1, 0, 2]])          # the longest axis (y) onto the slab axis


def test_batch_draws_remove_equals_per_view_calls(kpl, views):
    """The views of a batch are stacked with empty layers between them and keep their own index order, so the rounds over
    the stacked grid decide every view as its stand-alone run does."""
    import torch
    from keypoint_learning_b200 import synth
    clouds = [views["cheff000"], views["cheff002"][:20000], synth.view_25d(200, 150, seed=5)[0], views["cheff001"],
              np.ascontiguousarray(views["cheff001"][:7] + np.float32(300.0))]       # a tiny view: fewer points than k
    removed = 0
    for r_nms, th, dthr in CASES:
        d = _detector(kpl, r_nms, th, dthr)
        sc_b, kp_b = d.computeBatch(clouds)
        rounds = d.stats()["nms_rounds"]
        assert rounds >= 1
        for c, sc, kp in zip(clouds, sc_b, kp_b):
            idx, sc1 = _single(d, c)
            assert np.array_equal(sc1.view(np.uint32), sc.view(np.uint32))
            assert np.array_equal(idx, kp), (r_nms, th, dthr)
            d.setNonMaximaDrawsRemove(False)
            removed += len(_single(d, c)[0]) - len(idx)
            d.setNonMaximaDrawsRemove(True)
        d.close()
    assert removed > 0                                       # draws-remove really removed keypoints
    # device-resident batch, one case
    r_nms, th, dthr = CASES[1]
    d = _detector(kpl, r_nms, th, dthr)
    sc_b, kp_b = d.computeBatch(clouds)
    cat = np.ones((sum(len(c) for c in clouds), 4), np.float32)
    cat[:, :3] = np.concatenate(clouds)[:, :3]
    off = np.zeros(len(clouds) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in clouds])
    d_xyz = torch.from_numpy(cat).cuda()
    d_sc = torch.empty(len(cat), dtype=torch.float32, device="cuda")
    d_kp = torch.empty(len(cat), dtype=torch.int32, device="cuda")
    d_kpo = torch.empty(len(clouds) + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    nk = d.detectBatchDevice(d_xyz.data_ptr(), off, d_scores=d_sc.data_ptr(), d_kp_idx=d_kp.data_ptr(), d_kp_offsets=d_kpo.data_ptr())
    kpo = d_kpo.cpu().numpy()
    kp = d_kp.cpu().numpy()
    assert nk == int(kpo[-1]) == sum(len(k) for k in kp_b)
    assert np.array_equal(d_sc.cpu().numpy().view(np.uint32), np.concatenate(sc_b).view(np.uint32))
    for v in range(len(clouds)):
        assert np.array_equal(kp[kpo[v]:kpo[v + 1]], kp_b[v])
    d.close()


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_in_process_group_draws_remove_equals_single_gpu(kpl, world):
    from keypoint_learning_b200 import shard
    xyz = _cheff002()
    r_plan = max(r for r, _, _ in CASES)                     # one plan whose halo covers every case's r_nms
    plan = shard.plan_slabs(xyz, 20.0, r_plan, 4, world)
    dets = [_detector(kpl, *CASES[0]) for _ in range(world)]
    jobs = [shard.SlabJob(d, xyz, plan, r, None) for r, d in enumerate(dets)]
    ref = _detector(kpl, *CASES[0])
    for case in CASES:
        _set_case(ref, *case)
        idx_full, sc_full = _single(ref, xyz)
        for d in dets:
            _set_case(d, *case)
            d._push()
        before = [_ctx_params(d) for d in dets]
        kp, scores = shard.detect_group_widening(jobs, xyz, 20.0, r_plan, 4)
        assert np.array_equal(kp, idx_full), (world, case, len(kp), len(idx_full))
        for j, sc in zip(jobs, scores):
            assert np.array_equal(sc.view(np.uint32), sc_full[j.gidx].view(np.uint32))
        assert [_ctx_params(d) for d in dets] == before      # the sharded call leaves every context as it was
        assert len({d.stats()["nms_rounds"] for d in dets}) == 1 and dets[0].stats()["nms_rounds"] >= 1
    for j in jobs:
        j.close()
    for d in dets + [ref]:
        d.close()


def _plateau(seed=7):
    """A planar lattice (pitch 1, 200 x 40) in a random index order."""
    gx, gy = np.meshgrid(np.arange(200, dtype=np.float32), np.arange(40, dtype=np.float32), indexing="ij")
    xyz = np.stack([gx.ravel(), gy.ravel(), np.zeros(gx.size, np.float32)], axis=1)
    return np.ascontiguousarray(xyz[np.random.default_rng(seed).permutation(len(xyz))])


@pytest.mark.parametrize("world", [2, 3, 4])
def test_plateau_chains_across_slab_faces(kpl, oracle, world):
    """Every point ties with all its neighbours; with a draws threshold between the pitch and r_nms the close draws form
    one lattice-wide dependency graph in random global order, so chains cross every slab face.  Deciding a halo point
    locally or comparing local indices gives a different set."""
    from keypoint_learning_b200 import shard
    r_nms, th, dthr = 4.0, 0.5, 1.5
    xyz = _plateau()
    ref = _detector(kpl, r_nms, th, dthr, forest=PLATEAU_FOREST)
    idx_full, sc_full = _single(ref, xyz)
    assert np.all(sc_full == 1.0)                            # kNN normals are finite everywhere on the lattice
    assert ref.stats()["nms_rounds"] > 1
    want = oracle.nms(xyz, sc_full, r_nms, th, draws_remove=True, draws_thr=dthr)
    assert np.array_equal(idx_full, want)
    assert 0 < len(want) < len(xyz) // 3
    plan = shard.plan_slabs(xyz, 20.0, r_nms, 4, world)
    # close-draw pairs straddle every cut
    cx = shard.cell_coords(xyz, plan.origin, plan.cell, 0)
    for c in plan.cuts[1:-1]:
        a, b = xyz[cx == c - 1], xyz[cx == c]
        d = np.sqrt(((a[:, None, :] - b[None, :, :]) ** 2).sum(axis=2))
        assert (d < dthr).any()
    dets = [_detector(kpl, r_nms, th, dthr, forest=PLATEAU_FOREST) for _ in range(world)]
    jobs = [shard.SlabJob(d, xyz, plan, r, None) for r, d in enumerate(dets)]
    kp, scores = shard.detect_group_widening(jobs, xyz, 20.0, r_nms, 4)
    assert np.array_equal(kp, want)
    for j, sc in zip(jobs, scores):
        assert np.array_equal(sc.view(np.uint32), sc_full[j.gidx].view(np.uint32))
    rounds = {d.stats()["nms_rounds"] for d in dets}
    assert len(rounds) == 1 and rounds.pop() > 1
    for j in jobs:
        j.close()
    for d in dets + [ref]:
        d.close()


def test_one_rank_nccl_communicator_draws_remove(kpl):
    from keypoint_learning_b200 import shard
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff000.npz"))["xyz"]
    ref = _detector(kpl, *CASES[1])
    idx_full, sc_full = _single(ref, xyz)
    plan = shard.plan_slabs(xyz, 20.0, CASES[1][0], 4, 1)
    before = _ctx_params(ref)
    job = shard.SlabJob(ref, xyz, plan, 0, shard.nccl_unique_id())
    sc = np.empty(job.n_owned, np.float32)
    n, kp = job.detect(scores_out=sc)
    assert n == len(idx_full) and np.array_equal(kp, idx_full)
    assert np.array_equal(sc.view(np.uint32), sc_full.view(np.uint32))
    assert ref.stats()["nms_rounds"] >= 1
    assert _ctx_params(ref) == before
    assert np.array_equal(_single(ref, xyz)[0], idx_full)
    job.close()
    ref.close()


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
def test_sharded_nccl_draws_remove_equals_single_gpu(tmp_path, kpl, world):
    if _ngpus() < world:
        pytest.skip("needs %d GPUs" % world)
    out = str(tmp_path / "kp.npz")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "draws_multi_gpu_worker.py"), out]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    xyz = _cheff002()
    ref = _detector(kpl, *CASES[1])
    idx_full, sc_full = _single(ref, xyz)
    ref.close()
    assert np.array_equal(np.load(out)["keypoints"], idx_full)
    for rank in range(world):
        d = np.load(out + ".rank%d.npz" % rank)
        assert np.array_equal(d["scores"].view(np.uint32), sc_full[d["gidx"]].view(np.uint32))
        assert int(d["rounds"]) >= 1


def test_role_array_still_refuses_draws_remove(kpl, views):
    """A caller that drives a slab through kpl_detect with a role array cannot see its neighbours' decisions."""
    xyz = views["cheff001"]
    d = _detector(kpl, *CASES[0])
    d.setInputCloud(xyz)
    with pytest.raises(kpl.KplError) as e:
        d.compute(role=np.full(len(xyz), 3, np.uint8))
    assert e.value.code == 10
    d.close()
