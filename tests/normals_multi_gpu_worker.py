"""torchrun worker of tests/test_gpu_shard_normals.py: slab-sharded detection with the caller's normals over WORLD_SIZE GPUs
through kpl_shard_set_slab_normals / kpl_shard_detect (NCCL strips of positions and normals, scores and draws-remove
states inside libkpl_b200.so).  The normals are k-NN normals with a seeded share replaced, flipped or NaN.  Every rank
writes its owned scores, rank 0 the global keypoint list and the normals.  torch.distributed only hands the NCCL id of
rank 0 to the other ranks."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    out_path = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import shard

    xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff002.npz"))["xyz"]
    xyz = np.ascontiguousarray(xyz[:, [1, 0, 2]])
    det = K.KeypointLearningDetector(device=local)
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(4.0)
    det.setNonMaximaDrawsRemove(True); det.setNonMaximaDrawsThreshold(1.0)
    det.setPredictionThreshold(float(np.float32(0.5))); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    assert det.loadForest(os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz"))
    nrm = det.computeNormals(xyz)
    rng = np.random.default_rng(21)
    kind = rng.integers(0, 3, len(xyz))
    pick = rng.random(len(xyz)) < 0.1
    v = rng.normal(size=(len(xyz), 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    nrm[pick & (kind == 0), :3] = v[pick & (kind == 0)]
    nrm[pick & (kind == 1), :3] *= -1
    nrm[pick & (kind == 2), :3] = np.nan
    ids = [shard.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    plan = shard.plan_slabs(xyz, 20.0, 4.0, 4, world, normal_support_cells=0)
    job = shard.SlabJob(det, xyz, plan, rank, ids[0], normals=nrm)
    sc = np.empty(job.n_owned, np.float32)
    n1, kp1 = job.detect(scores_out=sc)
    job.upload()
    job.upload_normals(nrm)
    n2, kp2 = job.detect()                                    # a second step must give the same answer
    assert n1 == n2
    np.savez(out_path + ".rank%d.npz" % rank, gidx=job.gidx, scores=sc)
    if rank == 0:
        assert np.array_equal(kp1, kp2)
        np.savez(out_path, keypoints=kp1, normals=nrm)
    dist.barrier()
    job.close()
    det.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
