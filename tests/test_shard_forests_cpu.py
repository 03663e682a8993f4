"""Several forests over slabs on CPU: the schedule of kpl_shard_detect_forests (one position exchange, one scoring pass of
the owned points by all K forests, ONE exchange of (n, K) score strips, then each forest's NMS -- plain, or draws-remove
with its own state rounds) run by `gloo` ranks with the CPU oracle for the scores.  For every forest the union of the
ranks' keypoints must be oracle.nms of the whole cloud scored by that forest alone."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R_FEAT, R_NMS, TH, DRAWS_THR = 20.0, 4.0, 0.5, 1.0
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]


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
    """strips of any dtype and shape (n, ...) to / from the two neighbours (ncclSend / ncclRecv in csrc/shard.cu)."""
    got = {}
    for peer, payload in ((rank - 1, to_left), (rank + 1, to_right)):
        if 0 <= peer < world:
            a = np.ascontiguousarray(payload)
            t = torch.from_numpy(a.reshape(-1))
            n_in = torch.zeros(1, dtype=torch.int64)
            for r in dist.batch_isend_irecv([dist.P2POp(dist.isend, torch.tensor([len(t)]), peer), dist.P2POp(dist.irecv, n_in, peer)]):
                r.wait()
            buf = torch.empty(int(n_in), dtype=t.dtype)
            for r in dist.batch_isend_irecv([dist.P2POp(dist.isend, t, peer), dist.P2POp(dist.irecv, buf, peer)]):
                r.wait()
            got[peer] = buf.numpy().reshape((-1,) + a.shape[1:])
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
    forests = [O.load_forest_yaml(f) for f in FORESTS]
    K = len(forests)
    plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, 4, world)
    hs = shard.HostSlab(xyz, plan, rank)
    xl, xr = _exchange(rank, world, *hs.position_strips())
    p, role = hs.assemble(xl, xr)
    hs.set_local_gidx(*_exchange(rank, world, *hs.gidx_strips()))
    # one scoring pass of the owned points: the feature rows once, every forest on them
    nrm = O.normals_knn(p, 10)
    q = np.nonzero(role == 3)[0].astype(np.int32)
    feat = O.features(p, nrm, R_FEAT, 5, 10, order=1, qidx=q, canon=(plan.origin, plan.cell, plan.dims))
    sc = np.full((len(p), K), np.nan, np.float32)
    for k, f in enumerate(forests):
        sc[q, k] = O.scores(f, feat, nrm[q])
    # ONE exchange of the (n, K) score strips
    sc = hs.merge_scores(sc, *_exchange(rank, world, *hs.score_strips(sc)))
    off, idx = O.radius_neighbors(p, R_NMS)
    result = {}
    for k in range(K):
        s = np.ascontiguousarray(sc[:, k])
        result["plain%d" % k] = hs.owned_keypoints(O.nms(p, s, R_NMS, TH))
        state = hs.draws_classify(s, off, idx, TH, DRAWS_THR)
        state = hs.merge_states(state, *_exchange(rank, world, *hs.state_strips(state)))
        while True:
            state, undecided = hs.draws_round(state)
            state = hs.merge_states(state, *_exchange(rank, world, *hs.state_strips(state)))
            total = torch.tensor([undecided], dtype=torch.int64)
            dist.all_reduce(total)                              # every rank stops on the same global count
            if int(total) == 0:
                break
        result["draws%d" % k] = hs.draws_keypoints(state)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), gidx=hs.gidx, scores=sc[q], **result)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_forests_equal_unsharded_gloo(tmp_path, world, oracle, kpl):
    xyz = _cloud()
    nrm = oracle.normals_knn(xyz, 10)
    feat = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]
    removed = 0
    for k, path in enumerate(FORESTS):
        sc = oracle.scores(oracle.load_forest_yaml(path), feat, nrm)
        for r in range(world):
            assert np.array_equal(d[r]["scores"][:, k].view(np.uint32), sc[d[r]["gidx"]].view(np.uint32))
        for nms, ref in (("plain", oracle.nms(xyz, sc, R_NMS, TH)),
                         ("draws", oracle.nms(xyz, sc, R_NMS, TH, draws_remove=True, draws_thr=DRAWS_THR))):
            got = np.sort(np.concatenate([x["%s%d" % (nms, k)] for x in d]))
            assert len(ref) and np.array_equal(got, ref), (world, k, nms, len(got), len(ref))
        removed += len(oracle.nms(xyz, sc, R_NMS, TH)) - len(oracle.nms(xyz, sc, R_NMS, TH, draws_remove=True, draws_thr=DRAWS_THR))
    assert removed > 0                         # the draws-remove branch is exercised
