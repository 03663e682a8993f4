"""Slab sharding with the caller's normals on CPU: the schedule of csrc/shard.cu with kpl_shard_set_slab_normals -- the
normal strips travel beside the position strips, nothing is estimated, the plan has no k-NN support -- run by `gloo`
ranks with the CPU oracle scoring on the given normals.  The union of the ranks' results must be oracle.detect(normals4=...)
of the whole cloud, with plain and with draws-remove NMS.  Also: the re-plan loop of shard._widening leaves support 0."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85
DRAWS = (4.0, 0.5, 1.0)                      # (r_nms, threshold, draws threshold)
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-SHOT-like-T50-D10.yaml.gz")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _cloud():
    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff001.npz"))["xyz"]
    xyz = np.ascontiguousarray(xyz[:, [1, 0, 2]])          # the longest axis onto the slab axis
    return np.ascontiguousarray(xyz[(xyz[:, 0] > -60) & (xyz[:, 0] < 60) & (xyz[:, 1] < 0)])


def _normals(oracle, xyz, plan):
    """k-NN normals with some replaced by random unit vectors, some flipped and some NaN -- among them points of the strip
    columns on both sides of every interior face."""
    rng = np.random.default_rng(17)
    nrm = oracle.normals_knn(xyz, 10).copy()
    n = len(xyz)
    cx = np.floor((xyz[:, 0].astype(np.float64) - plan.origin[0]) / plan.cell).astype(np.int64)
    kind = rng.integers(0, 3, n)
    pick = rng.random(n) < 0.2
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    nrm[pick & (kind == 0), :3] = v[pick & (kind == 0)]
    nrm[pick & (kind == 1), :3] *= -1
    nrm[pick & (kind == 2), :3] = np.nan
    for c in plan.cuts[1:-1]:
        for side in ((cx >= c - plan.halo) & (cx < c), (cx >= c) & (cx < c + plan.halo)):
            assert all((pick & side & (kind == k)).any() for k in range(3))
    return nrm


def _exchange(rank, world, to_left, to_right):
    """1-d strips of any dtype to / from the two neighbours (ncclSend / ncclRecv in csrc/shard.cu)."""
    got = {}
    for peer, payload in ((rank - 1, to_left), (rank + 1, to_right)):
        if 0 <= peer < world:
            t = torch.from_numpy(np.ascontiguousarray(payload))
            n_in = torch.zeros(1, dtype=torch.int64)
            for r in dist.batch_isend_irecv([dist.P2POp(dist.isend, torch.tensor([len(t)]), peer), dist.P2POp(dist.irecv, n_in, peer)]):
                r.wait()
            buf = torch.empty(int(n_in), dtype=t.dtype)
            for r in dist.batch_isend_irecv([dist.P2POp(dist.isend, t, peer), dist.P2POp(dist.irecv, buf, peer)]):
                r.wait()
            got[peer] = buf.numpy()
    return got.get(rank - 1), got.get(rank + 1)


def _rows(a, width):
    return None if a is None else a.reshape(-1, width)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["OMP_NUM_THREADS"] = "2"
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from keypoint_learning_b200 import shard
    from oracle import oracle as O
    O.lib().kplo_set_threads(2)
    xyz = _cloud()
    forest = O.load_forest_yaml(FOREST)
    plan = shard.plan_slabs(xyz, R_FEAT, max(R_NMS, DRAWS[0]), 4, world, normal_support_cells=0)
    hs = shard.HostSlab(xyz, plan, rank)
    # 1. position strips and, beside them, the strips of the caller's normals (nothing is estimated on any rank)
    xl, xr = (_rows(a, 3) for a in _exchange(rank, world, *(a.ravel() for a in hs.position_strips())))
    p, role = hs.assemble(xl, xr)
    nrm = np.zeros((len(p), 4), np.float32)
    nrm[hs.n_l:hs.n_l + len(hs.own)] = _normals(O, xyz, plan)[hs.gidx]
    nl, nr = (_rows(a, 4) for a in _exchange(rank, world, *(a.ravel() for a in hs.score_strips(nrm))))
    nrm = hs.merge_scores(nrm, nl, nr)
    gl, gr = _exchange(rank, world, *hs.gidx_strips())
    hs.set_local_gidx(gl, gr)
    # 2. scores of the owned points on the given normals, 3. score strips
    q = np.nonzero(role == 3)[0].astype(np.int32)
    feat = O.features(p, nrm, R_FEAT, 5, 10, order=1, qidx=q, canon=(plan.origin, plan.cell, plan.dims))
    sc = np.full(len(p), np.nan, np.float32)
    sc[q] = O.scores(forest, feat, nrm[q])
    sc = hs.merge_scores(sc, *_exchange(rank, world, *hs.score_strips(sc)))
    # 4a. plain NMS
    kp = hs.owned_keypoints(O.nms(p, sc, R_NMS, TH))
    # 4b. draws-remove: the state rounds
    r_nms, th, dthr = DRAWS
    off, idx = O.radius_neighbors(p, r_nms)
    state = hs.draws_classify(sc, off, idx, th, dthr)
    state = hs.merge_states(state, *_exchange(rank, world, *hs.state_strips(state)))
    while True:
        state, undecided = hs.draws_round(state)
        state = hs.merge_states(state, *_exchange(rank, world, *hs.state_strips(state)))
        total = torch.tensor([undecided], dtype=torch.int64)
        dist.all_reduce(total)
        if int(total) == 0:
            break
    result = {}
    for key, mine in (("kp", kp), ("kp_draws", hs.draws_keypoints(state))):
        lists = [None] * world if rank == 0 else None
        dist.gather_object(mine, lists, dst=0)
        result[key] = np.sort(np.concatenate(lists)) if rank == 0 else np.zeros(0, np.int64)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), gidx=hs.gidx, scores=sc[q], halo=plan.halo,
             halo_want=max(plan.reach_feat, plan.reach_nms), **result)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_given_normals_equals_unsharded_gloo(tmp_path, world, oracle, kpl):
    from keypoint_learning_b200 import shard
    xyz = _cloud()
    forest = oracle.load_forest_yaml(FOREST)
    plan = shard.plan_slabs(xyz, R_FEAT, max(R_NMS, DRAWS[0]), 4, world, normal_support_cells=0)
    nrm = _normals(oracle, xyz, plan)
    ref = oracle.detect(xyz, forest, R_FEAT, R_NMS, TH, 5, 10, normals4=nrm, order=1)
    assert np.isnan(ref["scores"]).any() and len(ref["keypoints"]) > 5
    r_nms, th, dthr = DRAWS
    ref_draws = oracle.nms(xyz, ref["scores"], r_nms, th, draws_remove=True, draws_thr=dthr)
    assert len(ref_draws) < len(oracle.nms(xyz, ref["scores"], r_nms, th))          # the case exercises the branch
    # the estimated normals give another result: the given ones matter
    est = oracle.detect(xyz, forest, R_FEAT, R_NMS, TH, 5, 10, order=1)
    assert not np.array_equal(est["keypoints"], ref["keypoints"])
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]
    seen = np.zeros(len(xyz), bool)
    for r in range(world):
        assert int(d[r]["halo"]) == int(d[r]["halo_want"])                           # no k-NN support in the halo
        assert not seen[d[r]["gidx"]].any()
        seen[d[r]["gidx"]] = True
        assert np.array_equal(d[r]["scores"].view(np.uint32), ref["scores"][d[r]["gidx"]].view(np.uint32))
    assert seen.all()
    assert np.array_equal(d[0]["kp"], ref["keypoints"])
    assert np.array_equal(d[0]["kp_draws"], ref_draws)


def test_widening_leaves_support_zero(kpl):
    """A support-0 plan that clips (KPL_E_HALO) is re-planned with support 1, not with 2 * 0 forever."""
    from keypoint_learning_b200 import capi, shard
    xyz = _cloud()
    plan0 = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, 2, normal_support_cells=0)

    class Job:
        world = 2

        def __init__(self):
            self.plan, self.supports = plan0, []

        def replan(self, xyz_, plan):
            self.plan = plan
            self.supports.append(plan.normal_support_cells)

    jobs = [Job(), Job()]
    calls = []

    def detect():
        calls.append(jobs[0].plan.normal_support_cells)
        if len(calls) == 1:
            raise capi.KplError(capi.KPL_E_HALO, "clipped")
        return "done"

    assert shard._widening(detect, jobs, xyz, R_FEAT, R_NMS, 4, 64) == "done"
    assert calls == [0, 1]
    assert all(j.supports == [1] for j in jobs)
