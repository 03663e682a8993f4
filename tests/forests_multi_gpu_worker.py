"""torchrun worker of tests/test_gpu_shard_forests.py: the three golden forests over a slab-sharded cloud on WORLD_SIZE GPUs
through kpl_shard_detect_forests (NCCL strips of positions, K score slices and draws-remove states inside
libkpl_b200.so), with estimated k-NN normals and the widening loop.  argv: output path, "plain" or "draws".  Every rank
writes its K x n_owned scores, rank 0 the keypoints of all forests and their offsets.  torch.distributed only hands the
NCCL id of rank 0 to the other ranks."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]


def main():
    out_path, nms = sys.argv[1], sys.argv[2]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import shard

    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff002.npz"))["xyz"]
    xyz = np.ascontiguousarray(xyz[:, [1, 0, 2]])
    det = K.KeypointLearningDetector(device=local)
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(4.0)
    det.setNonMaximaDrawsRemove(nms == "draws"); det.setNonMaximaDrawsThreshold(1.0 if nms == "draws" else 0.0)
    det.setPredictionThreshold(float(np.float32(0.5))); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    assert det.loadForest(FORESTS[0])
    for f in FORESTS[1:]:
        det.addForest(f)
    ids = [shard.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, world)
    job = shard.SlabJob(det, xyz, plan, rank, ids[0])
    sc = np.empty(len(FORESTS) * job.n_owned, np.float32)
    n1, off, kps = shard.detect_forests_widening(job, xyz, 20.0, 4.0, 4, scores_out=sc)
    n2, off2, kps2 = job.detect_forests()                      # a second step must give the same answer
    assert n1 == n2 and np.array_equal(off, off2) and off[-1] == n1
    np.savez(out_path + ".rank%d.npz" % rank, gidx=job.gidx, scores=sc.reshape(len(FORESTS), -1))
    if rank == 0:
        assert all(np.array_equal(a, b) for a, b in zip(kps, kps2))
        np.savez(out_path, keypoints=np.concatenate(kps), offsets=off)
    dist.barrier()
    job.close()
    det.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
