"""Three forests over the sharded path from one feature pass (kpl_shard_detect_forests_group) against three single-forest
kpl_shard_detect_group calls, one per forest, on the same slabs: 2- and 4-rank in-process groups (all ranks on one GPU)
over the 2 M-point crop of the 10 M-point synthetic scene that tools/time_shard_normals.py uses.  The two variants
alternate call by call; each is checked against the other (keypoints of every forest, owned scores as bits).  Per
variant: per-rank features_ms / nms_ms (the library's CUDA events, summed over the three calls of the single-forest
variant), exchange_ms (device time of the position and score exchanges, the slowest rank) and wall_ms (a host clock around
the call or the three calls, which end in a device synchronisation).  Medians of --steps calls after two warm-up calls.

    python tools/time_shard_forests.py --steps 10 --out profiles/r5_shard_forests.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]
R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def detector(K, vp, forests):
    det = K.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(TH))); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10, viewpoint=vp)
    assert det.loadForest(forests[0])
    for f in forests[1:]:
        det.addForest(f)
    return det


def med(v):
    return float(np.median(np.asarray(v, np.float64)))


def time_group(K, steps, world, crop, vp):
    from keypoint_learning_b200 import shard
    plan = shard.plan_slabs(crop, R_FEAT, R_NMS, 4, world)
    groups = {"forests": [detector(K, vp, FORESTS) for _ in range(world)]}
    for k, f in enumerate(FORESTS):
        groups["single%d" % k] = [detector(K, vp, [f]) for _ in range(world)]
    jobs = {g: [shard.SlabJob(d, crop, plan, r, None) for r, d in enumerate(dets)] for g, dets in groups.items()}
    for g in jobs:           # every group on the plan the re-plan loop settles on
        shard.detect_group_widening(jobs[g], crop, R_FEAT, R_NMS, 4, want_scores=False)
    plan = jobs["forests"][0].plan
    for g in jobs:
        if jobs[g][0].plan.normal_support_cells != plan.normal_support_cells:
            for j in jobs[g]:
                j.replan(crop, plan)
    rows = {"forests": [], "single": []}
    for step in range(steps + 2):
        t0 = time.perf_counter()
        kps, sc = shard.detect_group_forests(jobs["forests"])
        wall = (time.perf_counter() - t0) * 1e3
        tm = [d.timings() for d in groups["forests"]]
        row_f = {"wall_ms": wall, "exchange_ms_max_rank": max(j.info()["exchange_ms"] for j in jobs["forests"]),
                 "features_ms": [t["features_ms"] for t in tm], "nms_ms": [t["nms_ms"] for t in tm], "total_ms": [t["total_ms"] for t in tm]}
        row_s = {"wall_ms": 0.0, "exchange_ms_max_rank": 0.0, "features_ms": [0.0] * world, "nms_ms": [0.0] * world, "total_ms": [0.0] * world}
        for k in range(len(FORESTS)):
            g = "single%d" % k
            t0 = time.perf_counter()
            kp, s1 = shard.detect_group(jobs[g])
            row_s["wall_ms"] += (time.perf_counter() - t0) * 1e3
            row_s["exchange_ms_max_rank"] += max(j.info()["exchange_ms"] for j in jobs[g])
            for r, t in enumerate(d.timings() for d in groups[g]):
                for key in ("features_ms", "nms_ms", "total_ms"):
                    row_s[key][r] += t[key]
            assert np.array_equal(kp, kps[k]), "forest %d: the forests call differs from kpl_shard_detect" % k
            assert all(np.array_equal(a[k].view(np.uint32), b.view(np.uint32)) for a, b in zip(sc, s1))
        if step >= 2:
            rows["forests"].append(row_f)
            rows["single"].append(row_s)
    info = [j.info() for j in jobs["forests"]]
    res = {"workload": "%d-rank in-process group on one GPU over a %d-point cube crop of the 10 M-point synthetic scene, 3 forests" % (world, len(crop)),
           "normal_support_cells": plan.normal_support_cells, "halo_points": int(sum(i["n_left"] + i["n_right"] for i in info)),
           "keypoints_per_forest": [int(len(k)) for k in kps]}
    for v, rs in rows.items():
        res[v] = {"wall_ms": med([r["wall_ms"] for r in rs]), "exchange_ms_max_rank": med([r["exchange_ms_max_rank"] for r in rs])}
        for key in ("features_ms", "nms_ms", "total_ms"):
            res[v][key + "_per_rank"] = [med([r[key][i] for r in rs]) for i in range(world)]
    res["wall_speedup"] = res["single"]["wall_ms"] / res["forests"]["wall_ms"]
    for g in jobs:
        for j in jobs[g]:
            j.close()
        for d in groups[g]:
            d.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--crop", type=int, default=2_000_000)
    ap.add_argument("--worlds", default="2,4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import synth
    xyz, vp = synth.scene_closed_surfaces(10_000_000, seed=4321)
    crop = np.ascontiguousarray(synth.cube_crop(xyz, a.crop))
    out = {"card": card(), "steps": a.steps, "groups": [time_group(K, a.steps, int(w), crop, vp) for w in a.worlds.split(",")],
           "nccl": "not measured (needs several GPUs)"}
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
