"""K forests over a batch from one feature pass against K single-forest batches: 32 synthetic 2.5-D views of 560 x 360
points (synth.view_25d, seeds 0..31; BASELINE.json configs[4]) and 8 and 32 organized range images of 640 x 480 pixels
(synth.organized_range_image, seeds 0..F-1), K in {1, 2, 3} of the golden 50-variable forests (synthetic-T100-D15,
-SHOT-like-T50-D10, -FPFH-like-T30-D25), draws-remove off, threshold (double)0.85f, k-NN normals for the views and
integral-image normals for the frames.  Per K, two variants alternate call by call on inputs already resident on the GPU:
  (a) set: one kpl_detect_batch_forests_device (views) / kpl_detect_batch_organized_forests_device (frames) with the K
      forests loaded,
  (b) separate: K kpl_detect_batch_device / kpl_detect_batch_organized_device calls, one detector per forest.
Medians over --steps calls after --warmup warm-up calls of: wall_ms (host clock around the call(s), which end in a device
synchronisation), features_ms (CUDA events around the feature kernel with its fused forest tail; summed over the K calls
for (b)), nms_ms, total_ms, host_syncs and kernel_launches.  The script asserts that (a) and (b) return identical scores
(bits) and keypoints, and records the card (name, power limit, max SM clock) in the same run.

    python tools/time_batch_forests.py --steps 10 --out profiles/r3_batch_forests.json
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
NAMES = ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz") for f in NAMES]
R_FEAT, R_NMS, TH = 20.0, 4.0, float(np.float32(0.85))
VIEW_W, VIEW_H, N_VIEWS = 560, 360, 32
FRAME_W, FRAME_H = 640, 480


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def detector(K, forests, vp):
    det = K.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(TH); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10, viewpoint=vp)
    assert det.loadForest(forests[0])
    for f in forests[1:]:
        det.addForest(f)
    return det


def median(rows):
    return {k: float(np.median([r[k] for r in rows])) for k in rows[0]}


def workload(name):
    """(flat float4 points, host view offsets or None, frame shape (F, W, H) or None, viewpoint, description)"""
    from keypoint_learning_b200 import synth
    if name == "views32":
        views = [synth.view_25d(VIEW_W, VIEW_H, seed=v) for v in range(N_VIEWS)]
        xyz = np.concatenate([v[0] for v in views])
        off = np.zeros(N_VIEWS + 1, np.int64); off[1:] = np.cumsum([len(v[0]) for v in views])
        x4 = np.ones((len(xyz), 4), np.float32); x4[:, :3] = xyz[:, :3]
        return x4, off, None, tuple(float(c) for c in views[0][1]), "%d views of %dx%d px" % (N_VIEWS, VIEW_W, VIEW_H)
    F = int(name[len("frames"):])
    fr = np.stack([synth.organized_range_image(FRAME_W, FRAME_H, seed=f)[0] for f in range(F)])
    x4 = np.ones(fr.shape[:3] + (4,), np.float32); x4[..., :3] = fr
    return x4.reshape(-1, 4), None, (F, FRAME_W, FRAME_H), (0.0, 0.0, 0.0), "%d organized frames of %dx%d px" % (F, FRAME_W, FRAME_H)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="views32,frames8,frames32")
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    import keypoint_learning_b200 as K
    out = {"card": card(), "steps": a.steps, "warmup": a.warmup, "threshold": TH, "forests": list(NAMES), "workloads": {}}
    for wl in a.workloads.split(","):
        x4, off, shape, vp, desc = workload(wl)
        n = len(x4)
        groups = len(off) - 1 if off is not None else shape[0]
        d_xyz = torch.from_numpy(x4).cuda()
        singles = [detector(K, [f], vp) for f in FORESTS]
        sets = {k: detector(K, FORESTS[:k], vp) for k in (1, 2, 3)}
        d_sc = torch.empty(3 * n, dtype=torch.float32, device="cuda")
        d_kp = torch.empty(3 * n, dtype=torch.int32, device="cuda")
        d_kpo = torch.empty(3 * groups + 1, dtype=torch.int64, device="cuda")
        s_sc = [torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(3)]
        s_kp = [torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(3)]
        s_kpo = [torch.empty(groups + 1, dtype=torch.int64, device="cuda") for _ in range(3)]
        torch.cuda.synchronize()

        def run(det, forests, sc, kp, kpo):
            args = dict(d_scores=sc.data_ptr(), d_kp_idx=kp.data_ptr(), d_kp_offsets=kpo.data_ptr())
            if off is not None:
                f = det.detectBatchForestsDevice if forests else det.detectBatchDevice
                return f(d_xyz.data_ptr(), off, **args)
            f = det.detectOrganizedBatchForestsDevice if forests else det.detectOrganizedBatchDevice
            return f(d_xyz.data_ptr(), shape[1], shape[2], shape[0], **args)

        rows = {k: {"set": [], "separate": []} for k in (1, 2, 3)}
        for step in range(a.warmup + a.steps):
            for k in (1, 2, 3):
                det = sets[k]
                t0 = time.perf_counter()
                nk = run(det, True, d_sc, d_kp, d_kpo)
                wall = (time.perf_counter() - t0) * 1e3
                t, s = det.timings(), det.stats()
                r_set = dict(wall_ms=wall, features_ms=t["features_ms"], nms_ms=t["nms_ms"], total_ms=t["total_ms"],
                             host_syncs=s["host_syncs"], kernel_launches=s["kernel_launches"], n_keypoints=nk)
                r_sep = dict(wall_ms=0.0, features_ms=0.0, nms_ms=0.0, total_ms=0.0, host_syncs=0, kernel_launches=0, n_keypoints=0)
                nks = []
                t0 = time.perf_counter()
                for j in range(k):
                    nks.append(run(singles[j], False, s_sc[j], s_kp[j], s_kpo[j]))
                r_sep["wall_ms"] = (time.perf_counter() - t0) * 1e3
                for j in range(k):                      # each detector keeps the stage times and counters of its last call
                    t, s = singles[j].timings(), singles[j].stats()
                    for key in ("features_ms", "nms_ms", "total_ms"):
                        r_sep[key] += t[key]
                    r_sep["host_syncs"] += s["host_syncs"]; r_sep["kernel_launches"] += s["kernel_launches"]
                    r_sep["n_keypoints"] += nks[j]
                if step == a.warmup + a.steps - 1 or step == 0:
                    # identical results, bit for bit: forest j's scores and every (j, view) keypoint range
                    kpo = d_kpo.cpu().numpy()
                    sc = d_sc[:k * n].cpu().numpy().reshape(k, n)
                    kp = d_kp.cpu().numpy()
                    for j in range(k):
                        assert np.array_equal(sc[j].view(np.uint32), s_sc[j].cpu().numpy().view(np.uint32)), (wl, k, j)
                        okpo, okp = s_kpo[j].cpu().numpy(), s_kp[j].cpu().numpy()
                        for v in range(groups):
                            assert np.array_equal(kp[kpo[j * groups + v]:kpo[j * groups + v + 1]], okp[okpo[v]:okpo[v + 1]]), (wl, k, j, v)
                    assert nk == sum(nks), (wl, k)
                if step >= a.warmup:
                    rows[k]["set"].append(r_set)
                    rows[k]["separate"].append(r_sep)
        res = {"workload": desc, "points": n}
        for k in (1, 2, 3):
            sep = median(rows[k]["separate"])
            st = median(rows[k]["set"])
            res["K%d" % k] = {"set": st, "separate": sep, "wall_speedup": sep["wall_ms"] / st["wall_ms"]}
            print(wl, k, json.dumps(res["K%d" % k]), flush=True)
        out["workloads"][wl] = res
        for d in singles + list(sets.values()):
            d.close()
        del d_xyz, d_sc, d_kp, s_sc, s_kp, s_kpo
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
