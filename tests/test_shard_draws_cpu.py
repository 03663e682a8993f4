"""Draws-remove NMS over slabs on CPU: the schedule of csrc/shard.cu (global indices of the halo points, owned-only
classification, state strips after the classification and after every round, one global undecided count that stops
every rank together) run by `gloo` ranks with the CPU oracle for the scores and HostSlab's numpy state rounds for NMS.
The union of the ranks' keypoints must be oracle.nms(draws_remove=True) of the whole cloud."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R_FEAT, R_NMS = 20.0, 4.0
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-SHOT-like-T50-D10.yaml.gz")
CASES = ((4.0, 0.5, 1.0), (4.0, 0.3, 2.0), (8.0, 0.3, 8.0), (4.0, 0.5, 0.0))      # (r_nms, threshold, draws threshold)


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
    plan = shard.plan_slabs(xyz, R_FEAT, max(r for r, _, _ in CASES), 4, world)
    hs = shard.HostSlab(xyz, plan, rank)
    xl, xr = (None if a is None else a.reshape(-1, 3) for a in _exchange(rank, world, *(a.ravel() for a in hs.position_strips())))
    p, role = hs.assemble(xl, xr)
    gl, gr = _exchange(rank, world, *hs.gidx_strips())
    loc_gidx = hs.set_local_gidx(gl, gr)
    # scores of the owned points (oracle, global canonical grid), then the score strips
    nrm = O.normals_knn(p, 10)
    q = np.nonzero(role == 3)[0].astype(np.int32)
    feat = O.features(p, nrm, R_FEAT, 5, 10, order=1, qidx=q, canon=(plan.origin, plan.cell, plan.dims))
    sc = np.full(len(p), np.nan, np.float32)
    sc[q] = O.scores(forest, feat, nrm[q])
    sc = hs.merge_scores(sc, *_exchange(rank, world, *hs.score_strips(sc)))
    result = {}
    for c, (r_nms, th, dthr) in enumerate(CASES):
        off, idx = O.radius_neighbors(p, r_nms)
        state = hs.draws_classify(sc, off, idx, th, dthr)
        state = hs.merge_states(state, *_exchange(rank, world, *hs.state_strips(state)))
        rounds = 0
        while True:
            state, undecided = hs.draws_round(state)
            rounds += 1
            state = hs.merge_states(state, *_exchange(rank, world, *hs.state_strips(state)))
            total = torch.tensor([undecided], dtype=torch.int64)
            dist.all_reduce(total)                              # every rank stops on the same global count
            if int(total) == 0:
                break
        lists = [None] * world if rank == 0 else None
        dist.gather_object(hs.draws_keypoints(state), lists, dst=0)
        # close draws of an owned point that another rank owns: the chains this schedule exists for
        i, j = hs._close
        cross = int(np.count_nonzero((role[i] == 3) & (role[j] != 3)))
        result["kp%d" % c] = np.sort(np.concatenate(lists)) if rank == 0 else np.zeros(0, np.int64)
        result["rounds%d" % c] = rounds
        result["cross%d" % c] = cross
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), gidx=hs.gidx, loc_gidx=loc_gidx, scores=sc[q], **result)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_draws_remove_equals_unsharded_gloo(tmp_path, world, oracle, kpl):
    xyz = _cloud()
    forest = oracle.load_forest_yaml(FOREST)
    nrm = oracle.normals_knn(xyz, 10)
    sc = oracle.scores(forest, oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1), nrm)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]
    for r in range(world):
        assert np.array_equal(d[r]["scores"].view(np.uint32), sc[d[r]["gidx"]].view(np.uint32))
        assert np.array_equal(np.sort(d[r]["loc_gidx"]), np.unique(d[r]["loc_gidx"]))     # one global index per held point
    removed = cross = 0
    for c, (r_nms, th, dthr) in enumerate(CASES):
        ref = oracle.nms(xyz, sc, r_nms, th, draws_remove=True, draws_thr=dthr)
        assert np.array_equal(d[0]["kp%d" % c], ref), (world, r_nms, th, dthr, len(d[0]["kp%d" % c]), len(ref))
        assert len({int(x["rounds%d" % c]) for x in d}) == 1                                  # the ranks stopped together
        removed += len(oracle.nms(xyz, sc, r_nms, th)) - len(ref)
        cross += sum(int(x["cross%d" % c]) for x in d)
    assert removed > 0                         # the cases exercise the branch
    assert cross > 0                           # and close draws straddle a cut
