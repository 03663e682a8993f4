"""What draws-remove NMS (the detector's default NMS mode) costs on the two scaling paths, against the plain local-maximum
NMS on the same inputs: the 32-view batch of 560x360 synthetic views (kpl_detect_batch_device) and 2- and 4-rank
in-process groups (kpl_shard_detect_group, all ranks on one GPU) over a crop of the 10 M-point synthetic scene.  The two
modes alternate call by call.  nms_ms is the library's CUDA-event time of the NMS stage (threshold + NMS + compaction;
with draws-remove the classification, every resolution round and, on the sharded path, the state exchanges); wall_ms a
host clock around a call, which ends in a device synchronisation.  Every result is checked against the single-GPU
kpl_detect with the same mode.

    python tools/time_draws_nms.py --steps 10 --out profiles/r3_draws_nms.json
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
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz")
R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def detector(K, vp, draws, dthr):
    det = K.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS)
    det.setNonMaximaDrawsRemove(draws); det.setNonMaximaDrawsThreshold(dthr)
    det.setPredictionThreshold(float(np.float32(TH))); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10, viewpoint=vp)
    assert det.loadForest(FOREST)
    return det


def summary(rows):
    out = {}
    for k in rows[0]:
        v = np.array([r[k] for r in rows], np.float64)
        out[k] = {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}
    return out


def time_batch(K, torch, steps, dthr):
    from keypoint_learning_b200 import synth
    views = []
    for i in range(32):
        xyz, vp = synth.view_25d(560, 360, seed=i)
        views.append(xyz)
    cat = np.ones((sum(len(v) for v in views), 4), np.float32)
    cat[:, :3] = np.concatenate(views)
    off = np.zeros(33, np.int64)
    off[1:] = np.cumsum([len(v) for v in views])
    d_xyz = torch.from_numpy(cat).cuda()
    d_sc = torch.empty(len(cat), dtype=torch.float32, device="cuda")
    d_kp = torch.empty(len(cat), dtype=torch.int32, device="cuda")
    d_kpo = torch.empty(33, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    dets = {m: detector(K, vp, m == "on", dthr) for m in ("off", "on")}
    rows = {m: [] for m in dets}
    nkp = {}
    for step in range(steps + 2):                            # two warm-up calls per mode
        for m, det in dets.items():
            t0 = time.perf_counter()
            nk = det.detectBatchDevice(d_xyz.data_ptr(), off, d_scores=d_sc.data_ptr(), d_kp_idx=d_kp.data_ptr(), d_kp_offsets=d_kpo.data_ptr())
            wall = (time.perf_counter() - t0) * 1e3
            st, tm = det.stats(), det.timings()
            nkp[m] = nk
            if step >= 2:
                rows[m].append({"nms_ms": tm["nms_ms"], "total_ms": tm["total_ms"], "wall_ms": wall, "nms_rounds": st["nms_rounds"],
                                "host_syncs": st["host_syncs"]})
    # parity: every view of the last call equals its stand-alone kpl_detect (two views checked)
    kp, kpo = d_kp.cpu().numpy(), d_kpo.cpu().numpy()
    for v in (0, 31):
        det = dets["on"]
        det.setInputCloud(views[v])
        _, idx = det.compute()
        assert np.array_equal(idx, kp[kpo[v]:kpo[v + 1]]), "view %d differs from its stand-alone run" % v
    for det in dets.values():
        det.close()
    return {"workload": "32 synthetic 2.5D views of 560x360 px (%d points), kpl_detect_batch_device" % len(cat),
            "keypoints": nkp, "off": summary(rows["off"]), "on": summary(rows["on"])}


def time_group(K, torch, steps, dthr, world, crop):
    from keypoint_learning_b200 import shard
    rows = {"off": [], "on": []}
    groups = {}
    for m in rows:
        dets = [detector(K, VP, m == "on", dthr) for _ in range(world)]
        plan = shard.plan_slabs(crop, R_FEAT, R_NMS, 4, world)
        groups[m] = (dets, [shard.SlabJob(d, crop, plan, r, None) for r, d in enumerate(dets)])
    kps = {}
    for step in range(steps + 2):
        for m, (dets, jobs) in groups.items():
            t0 = time.perf_counter()
            kp, _ = shard.detect_group_widening(jobs, crop, R_FEAT, R_NMS, 4, want_scores=False)
            wall = (time.perf_counter() - t0) * 1e3
            kps[m] = kp
            if step >= 2:
                st = [d.stats() for d in dets]
                rows[m].append({"nms_ms_max_rank": max(d.timings()["nms_ms"] for d in dets),
                                "total_ms_max_rank": max(d.timings()["total_ms"] for d in dets), "wall_ms": wall,
                                "nms_rounds": st[0]["nms_rounds"], "host_syncs_rank0": st[0]["host_syncs"]})
    for m, (dets, jobs) in groups.items():
        ref = detector(K, VP, m == "on", dthr)
        ref.setInputCloud(crop)
        _, idx = ref.compute()
        assert np.array_equal(idx, kps[m]), "%d-rank group, draws-remove %s: differs from the single-GPU run" % (world, m)
        ref.close()
        for j in jobs:
            j.close()
        for d in dets:
            d.close()
    return {"workload": "%d-rank in-process group on one GPU over a %d-point cube crop of the 10 M-point synthetic scene" % (world, len(crop)),
            "keypoints": {m: int(len(k)) for m, k in kps.items()}, "off": summary(rows["off"]), "on": summary(rows["on"])}


VP = (0.0, 0.0, 0.0)


def main():
    global VP
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--draws-threshold", type=float, default=2.0, help="setNonMaximaDrawsThreshold (half of radiusNMS by default)")
    ap.add_argument("--crop", type=int, default=2_000_000, help="points of the scene crop the groups run on")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_draws_nms.py measures on the GPU: no CUDA device")
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import synth
    res = {"card": card(), "radiusNMS": R_NMS, "threshold": TH, "draws_threshold": a.draws_threshold, "forest": os.path.basename(FOREST),
           "steps": a.steps, "batch": time_batch(K, torch, a.steps, a.draws_threshold)}
    xyz, VP = synth.scene_closed_surfaces(10_000_000, seed=4321)
    crop = np.ascontiguousarray(synth.cube_crop(xyz, a.crop))
    for world in (2, 4):
        res["group%d" % world] = time_group(K, torch, a.steps, a.draws_threshold, world, crop)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
