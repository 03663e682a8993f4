"""What caller-supplied normals (kpl_shard_set_slab_normals) change on the sharded path, against normals estimated on the
devices, on the same cloud: 2- and 4-rank in-process groups (kpl_shard_detect_group, all ranks on one GPU) over the 2 M-point
crop of the 10 M-point synthetic scene that tools/time_draws_nms.py uses, and the NCCL path (kpl_shard_detect, one rank per
GPU, launched here under torch.distributed.run) when the host has 2+ GPUs.  The two variants alternate call by call.
Estimated normals use the plan the re-plan loop settles on (k-NN support widened until no normal that matters is clipped);
given normals a plan without k-NN support.  Per configuration: halo points (received by all ranks), exchange_ms (device
time of the position and score exchanges, the slowest rank), per-rank normals_ms / total_ms (the library's CUDA events) and
wall_ms (a host clock around a call, which ends in a device synchronisation).  The given normals are the device's own k-NN
normals (kpl_normals); each variant is checked against the single-GPU kpl_detect with the same normals.

    python tools/time_shard_normals.py --steps 10 --out profiles/r3_shard_normals.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz")
R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def detector(K, vp, device=0):
    det = K.KeypointLearningDetector(device=device)
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(TH))); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10, viewpoint=vp)
    assert det.loadForest(FOREST)
    return det


def summary(rows):
    out = {}
    for k in rows[0]:
        v = np.array([r[k] for r in rows], np.float64)
        out[k] = {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}
    return out


def sample(dets, jobs, wall):
    tm = [d.timings() for d in dets]
    return {"exchange_ms_max_rank": max(j.info()["exchange_ms"] for j in jobs), "normals_ms_max_rank": max(t["normals_ms"] for t in tm),
            "total_ms_max_rank": max(t["total_ms"] for t in tm), "wall_ms": wall,
            "normals_ms_per_rank": [t["normals_ms"] for t in tm], "total_ms_per_rank": [t["total_ms"] for t in tm]}


def layout(jobs):
    info = [j.info() for j in jobs]
    return {"normal_support_cells": jobs[0].plan.normal_support_cells, "halo_cells": jobs[0].plan.halo,
            "halo_points": int(sum(i["n_left"] + i["n_right"] for i in info)), "halo_bytes_sent": int(sum(i["halo_bytes"] for i in info)),
            "owned_points": [int(i["n_owned"]) for i in info]}


def per_rank_summary(rows):
    flat = [{k: v for k, v in r.items() if not k.endswith("_per_rank")} for r in rows]
    out = summary(flat)
    for k in ("normals_ms_per_rank", "total_ms_per_rank"):
        out[k] = [float(np.median([r[k][i] for r in rows])) for i in range(len(rows[0][k]))]
    return out


def time_group(K, steps, world, crop, vp, nrm, ref_kp):
    """ref_kp: the single-GPU keypoints, {"estimated": ..., "given": ...}"""
    from keypoint_learning_b200 import shard
    groups = {}
    for m in ("estimated", "given"):
        dets = [detector(K, vp) for _ in range(world)]
        plan = shard.plan_slabs(crop, R_FEAT, R_NMS, 4, world, normal_support_cells=0 if m == "given" else 1)
        groups[m] = (dets, [shard.SlabJob(d, crop, plan, r, None, normals=nrm if m == "given" else None) for r, d in enumerate(dets)])
    rows = {m: [] for m in groups}
    kps = {}
    for step in range(steps + 2):                            # two warm-up calls per variant
        for m, (dets, jobs) in groups.items():
            t0 = time.perf_counter()
            kp, _ = shard.detect_group_widening(jobs, crop, R_FEAT, R_NMS, 4, want_scores=False)
            wall = (time.perf_counter() - t0) * 1e3
            kps[m] = kp
            if step >= 2:
                rows[m].append(sample(dets, jobs, wall))
    res = {"workload": "%d-rank in-process group on one GPU over a %d-point cube crop of the 10 M-point synthetic scene" % (world, len(crop))}
    for m, (dets, jobs) in groups.items():
        assert np.array_equal(kps[m], ref_kp[m]), "%d-rank group, %s normals: differs from the single-GPU run" % (world, m)
        res[m] = dict(layout(jobs), keypoints=int(len(kps[m])), **per_rank_summary(rows[m]))
        for j in jobs:
            j.close()
        for d in dets:
            d.close()
    return res


def single_gpu(K, vp, crop, nrm, device=0):
    """single-GPU keypoints with estimated and with the given normals"""
    ref = detector(K, vp, device)
    ref.setInputCloud(crop)
    out = {"estimated": ref.compute()[1]}
    ref.setNormals(nrm)
    out["given"] = ref.compute()[1]
    ref.close()
    return out


def nccl_worker(out, steps, crop_n):
    """One rank of the NCCL measurement (under torch.distributed.run)."""
    import torch
    import torch.distributed as dist
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import shard, synth
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    xyz, vp = synth.scene_closed_surfaces(10_000_000, seed=4321)
    crop = np.ascontiguousarray(synth.cube_crop(xyz, crop_n))
    det = {m: detector(K, vp, local) for m in ("estimated", "given")}
    nrm = det["given"].computeNormals(crop)
    ids = [shard.nccl_unique_id() if rank == 0 else None, shard.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    jobs = {}
    for i, m in enumerate(("estimated", "given")):
        plan = shard.plan_slabs(crop, R_FEAT, R_NMS, 4, world, normal_support_cells=0 if m == "given" else 1)
        jobs[m] = shard.SlabJob(det[m], crop, plan, rank, ids[i], normals=nrm if m == "given" else None)
    rows = {m: [] for m in jobs}
    kps = {}
    for step in range(steps + 2):
        for m, job in jobs.items():
            dist.barrier()
            t0 = time.perf_counter()
            _, kp = shard.detect_widening(job, crop, R_FEAT, R_NMS, 4)
            wall = (time.perf_counter() - t0) * 1e3
            kps[m] = kp
            if step >= 2:
                rows[m].append(sample([det[m]], [job], wall))
    mine = {m: {"rows": rows[m], "layout": layout([jobs[m]])} for m in jobs}
    every = [None] * world
    dist.all_gather_object(every, mine)
    if rank == 0:
        ref_kp = single_gpu(K, vp, crop, nrm, local)
        res = {"workload": "%d ranks over NCCL, one GPU each, over a %d-point cube crop of the 10 M-point synthetic scene" % (world, len(crop))}
        for m in jobs:
            assert np.array_equal(kps[m], ref_kp[m]), "NCCL %d ranks, %s normals: differs from the single-GPU run" % (world, m)
            lay = [e[m]["layout"] for e in every]
            n = len(every[0][m]["rows"])
            merged = [{"exchange_ms_max_rank": max(e[m]["rows"][s]["exchange_ms_max_rank"] for e in every),
                       "normals_ms_max_rank": max(e[m]["rows"][s]["normals_ms_max_rank"] for e in every),
                       "total_ms_max_rank": max(e[m]["rows"][s]["total_ms_max_rank"] for e in every),
                       "wall_ms": max(e[m]["rows"][s]["wall_ms"] for e in every),
                       "normals_ms_per_rank": [e[m]["rows"][s]["normals_ms_per_rank"][0] for e in every],
                       "total_ms_per_rank": [e[m]["rows"][s]["total_ms_per_rank"][0] for e in every]} for s in range(n)]
            res[m] = dict(normal_support_cells=lay[0]["normal_support_cells"], halo_cells=lay[0]["halo_cells"],
                          halo_points=sum(x["halo_points"] for x in lay), halo_bytes_sent=sum(x["halo_bytes_sent"] for x in lay),
                          owned_points=[x["owned_points"][0] for x in lay], keypoints=int(len(kps[m])), **per_rank_summary(merged))
        with open(out, "w") as f:
            json.dump(res, f)
    dist.barrier()
    for j in jobs.values():
        j.close()
    dist.destroy_process_group()


def time_nccl(steps, world, crop_n):
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "nccl.json")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", "29533", os.path.abspath(__file__), "--nccl-worker", out, "--steps", str(steps), "--crop", str(crop_n)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
        if r.returncode != 0:
            raise SystemExit("NCCL measurement failed:\n" + r.stdout[-3000:] + r.stderr[-3000:])
        with open(out) as f:
            return json.load(f)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--crop", type=int, default=2_000_000, help="points of the scene crop")
    ap.add_argument("--out", default=None)
    ap.add_argument("--nccl-worker", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.nccl_worker:
        return nccl_worker(a.nccl_worker, a.steps, a.crop)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_shard_normals.py measures on the GPU: no CUDA device")
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import synth
    xyz, vp = synth.scene_closed_surfaces(10_000_000, seed=4321)
    crop = np.ascontiguousarray(synth.cube_crop(xyz, a.crop))
    ref = detector(K, vp)
    nrm = ref.computeNormals(crop)
    ref.close()
    ref_kp = single_gpu(K, vp, crop, nrm)
    res = {"card": card(), "radiusNMS": R_NMS, "threshold": TH, "draws_remove": False, "forest": os.path.basename(FOREST), "steps": a.steps,
           "same_keypoints_estimated_and_given": bool(np.array_equal(ref_kp["estimated"], ref_kp["given"]))}
    for world in (2, 4):
        res["group%d" % world] = time_group(K, a.steps, world, crop, vp, nrm, ref_kp)
    gpus = torch.cuda.device_count()
    for world in (2, 4, 8):
        res["nccl%d" % world] = time_nccl(a.steps, world, a.crop) if gpus >= world else "not measured: %d GPU(s) on this host" % gpus
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
