"""Organized frames one by one against one batch: F in {1, 8, 32} range images of organized_range_image(640, 480, seed=f),
draws-remove off, run three ways that alternate call by call:
  (a) loop: computeOrganized per frame (kpl_normals_organized + host NaN compaction + kpl_detect_xyzi),
  (b) batch: computeOrganizedBatch (kpl_detect_batch_organized: host frames in, host results out),
  (c) device: kpl_detect_batch_organized_device on frames already resident on the GPU.
Per way the median over --steps calls after two warm-up calls of: wall_ms (a host clock around the call, which ends in a
device synchronisation), the library's stage times (CUDA events; summed over the frames for the loop), host_syncs and
kernel_launches (summed for the loop).  Also kpl_normals_organized alone on one frame (wall clock, upload and copy-out
included).  The script checks that (a), (b) and (c) return identical scores (bits) and keypoints.

    python tools/time_organized_batch.py --steps 10 --out profiles/r3_organized_batch.json
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
W, H = 640, 480
STAGES = ("grid_ms", "normals_ms", "features_ms", "nms_ms", "total_ms")


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def detector(K):
    det = K.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(TH))); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10)
    assert det.loadForest(FOREST)
    return det


def record(det, wall):
    t, s = det.timings(), det.stats()
    return dict({k: t[k] for k in STAGES}, wall_ms=wall, host_syncs=s["host_syncs"], kernel_launches=s["kernel_launches"])


def median(rows):
    return {k: float(np.median([r[k] for r in rows])) for k in rows[0]}


def run_loop(det, frames):
    rows, sc, kp = [], [], []
    for fr in frames:
        t0 = time.perf_counter()
        _, idx = det.computeOrganized(fr)
        wall = (time.perf_counter() - t0) * 1e3
        # computeOrganized = kpl_normals_organized (1 host sync, 5 launches), then compute(): on a frame with NaN points a
        # kpl_detect_xyzi call refused after its bounding-box pass (1 sync, 2 launches) and the detection of the finite
        # points, whose stats are the ones reported
        dense = bool(np.isfinite(fr).all())
        r = record(det, wall)
        r["host_syncs"] += 1 if dense else 2
        r["kernel_launches"] += 5 if dense else 7
        rows.append(r)
        sc.append(det.getResponse().copy()); kp.append(idx)
    tot = {k: float(sum(r[k] for r in rows)) for k in rows[0]}
    return tot, sc, kp


def run_device(det, d, nf):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    det.detectOrganizedBatchDevice(d["xyz"].data_ptr(), W, H, nf, 5.0, d_scores=d["sc"].data_ptr(), d_kp_idx=d["kp"].data_ptr(),
                                   d_kp_offsets=d["kpo"].data_ptr())
    torch.cuda.synchronize()
    return record(det, (time.perf_counter() - t0) * 1e3)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_organized_batch.py measures on the GPU: no CUDA device")
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import synth
    frames = np.stack([synth.organized_range_image(W, H, seed=f)[0] for f in range(32)])
    det = detector(K)
    res = {"card": card(), "frame": [W, H], "radiusFeatures": R_FEAT, "radiusNMS": R_NMS, "threshold": TH, "draws_remove": False,
           "forest": os.path.basename(FOREST), "steps": a.steps}
    # kpl_normals_organized alone, one frame
    rows = []
    for step in range(a.steps + 2):
        t0 = time.perf_counter()
        det.computeNormalsOrganized(frames[0])
        if step >= 2:
            rows.append({"wall_ms": (time.perf_counter() - t0) * 1e3, "kernel_launches": det.stats()["kernel_launches"],
                         "host_syncs": det.stats()["host_syncs"]})
    res["normals_organized_one_frame"] = median(rows)
    for nf in (1, 8, 32):
        fr = np.ascontiguousarray(frames[:nf])
        x4 = np.ones((nf, H, W, 4), np.float32)
        x4[..., :3] = fr
        d = {"xyz": torch.from_numpy(x4).cuda(), "sc": torch.empty(nf * H * W, dtype=torch.float32, device="cuda"),
             "kp": torch.empty(nf * H * W, dtype=torch.int32, device="cuda"), "kpo": torch.empty(nf + 1, dtype=torch.int64, device="cuda")}
        rows = {"loop": [], "batch": [], "device": []}
        for step in range(a.steps + 2):                      # two warm-up calls per way
            r_loop, sc_a, kp_a = run_loop(det, fr)
            t0 = time.perf_counter()
            sc_b, kp_b = det.computeOrganizedBatch(fr)
            r_batch = record(det, (time.perf_counter() - t0) * 1e3)
            r_dev = run_device(det, d, nf)
            if step >= 2:
                rows["loop"].append(r_loop); rows["batch"].append(r_batch); rows["device"].append(r_dev)
        kpo = d["kpo"].cpu().numpy(); kp_c = d["kp"].cpu().numpy(); sc_c = d["sc"].cpu().numpy()
        for f in range(nf):
            assert np.array_equal(sc_a[f].view(np.uint32), sc_b[f].view(np.uint32)), (nf, f)
            assert np.array_equal(kp_a[f], kp_b[f]), (nf, f)
            assert np.array_equal(sc_c[f * H * W:(f + 1) * H * W].view(np.uint32), sc_b[f].view(np.uint32)), (nf, f)
            assert np.array_equal(kp_c[kpo[f]:kpo[f + 1]], kp_b[f]), (nf, f)
        res["frames%d" % nf] = {"keypoints": int(sum(len(k) for k in kp_b)), "finite_points": int(det.stats()["n_points"]),
                                "identical_loop_batch_device": True, **{w: median(r) for w, r in rows.items()}}
    det.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
