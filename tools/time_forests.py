"""K forests from one feature pass against K separate detections: the 10 M-point closed-surface scene and the 1 M-point
2.5-D view (bench.py's scene10m / view1m), K in {1, 2, 3} of the golden 50-variable forests (synthetic-T100-D15,
-SHOT-like-T50-D10, -FPFH-like-T30-D25), draws-remove off, threshold (double)0.85f, k-NN normals.  Per K, two variants
alternate call by call on a cloud already resident on the GPU:
  (a) set: one kpl_detect_forests_device with the K forests loaded,
  (b) separate: K kpl_detect_device calls, one detector per forest.
Medians over --steps calls after two warm-up calls of: wall_ms (host clock around the call(s), which end in a device
synchronisation), features_ms (CUDA events around the feature kernel with its fused forest tail; summed over the K calls
for (b)), nms_ms, host_syncs and kernel_launches.  The script checks that (a) and (b) return identical scores (bits) and
keypoints, and records the packed size of every forest (32-byte blocks, csrc/forest.cu: pack_forest) and the card.
--report-fragile times every call with kpl_params.report_fragile on (the feature kernel variant that also flags near-split
decisions).

    python tools/time_forests.py --steps 10 --out profiles/r3_forests.json
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


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def packed_bytes(path):
    """Bytes of the forest as pack_forest lays it out: one 32-byte block per root, two more per internal child of a block."""
    from oracle.oracle import load_forest_yaml
    f = load_forest_yaml(path)
    var, left, right = np.asarray(f["var"]), np.asarray(f["left"]), np.asarray(f["right"])
    blocks = 0
    for r in f["roots"]:
        blocks += 1
        queue = [int(r)]
        while queue:
            p = queue.pop()
            if var[p] < 0:
                continue
            for c in (int(left[p]), int(right[p])):
                if var[c] >= 0:
                    blocks += 2
                    queue += [int(left[c]), int(right[c])]
    return blocks * 32


def detector(K, forests, vp, fragile):
    det = K.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(TH); det.setRadiusSearch(R_FEAT); det.setNormalsMode(1, k=10, viewpoint=vp)
    det.setReportFragile(fragile)
    assert det.loadForest(forests[0])
    for f in forests[1:]:
        det.addForest(f)
    return det


def median(rows):
    return {k: float(np.median([r[k] for r in rows])) for k in rows[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="scene10m,view1m")
    ap.add_argument("--report-fragile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import synth
    out = {"card": card(), "steps": a.steps, "warmup": a.warmup, "threshold": TH, "report_fragile": a.report_fragile,
           "forests": [{"name": nm, "packed_bytes": packed_bytes(p)} for nm, p in zip(NAMES, FORESTS)], "workloads": {}}
    for wl in a.workloads.split(","):
        if wl == "scene10m":
            xyz, vp = synth.scene_closed_surfaces(10_000_000, seed=4321)
        else:
            xyz, vp = synth.view_25d(1250, 800, seed=1234)
        vp = tuple(float(v) for v in vp)
        n = len(xyz)
        x4 = np.ones((n, 4), np.float32); x4[:, :3] = xyz[:, :3]
        d_xyz = torch.from_numpy(x4).cuda()
        singles = [detector(K, [f], vp, a.report_fragile) for f in FORESTS]
        sets = {k: detector(K, FORESTS[:k], vp, a.report_fragile) for k in (1, 2, 3)}
        d_sc = torch.empty(3 * n, dtype=torch.float32, device="cuda")
        d_kp = torch.empty(3 * n, dtype=torch.int32, device="cuda")
        d_kpo = torch.empty(4, dtype=torch.int64, device="cuda")
        s_sc = [torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(3)]
        s_kp = [torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(3)]
        torch.cuda.synchronize()
        rows = {k: {"set": [], "separate": []} for k in (1, 2, 3)}
        for step in range(a.warmup + a.steps):
            for k in (1, 2, 3):
                det = sets[k]
                t0 = time.perf_counter()
                nk = det.detectForestsDevice(d_xyz.data_ptr(), n, d_scores=d_sc.data_ptr(), d_kp_idx=d_kp.data_ptr(), d_kp_offsets=d_kpo.data_ptr())
                wall = (time.perf_counter() - t0) * 1e3
                t, s = det.timings(), det.stats()
                r_set = dict(wall_ms=wall, features_ms=t["features_ms"], nms_ms=t["nms_ms"], total_ms=t["total_ms"],
                             host_syncs=s["host_syncs"], kernel_launches=s["kernel_launches"], n_keypoints=nk)
                r_sep = dict(wall_ms=0.0, features_ms=0.0, nms_ms=0.0, total_ms=0.0, host_syncs=0, kernel_launches=0, n_keypoints=0)
                nks = []
                t0 = time.perf_counter()
                for j in range(k):
                    nks.append(singles[j].detectDevice(d_xyz.data_ptr(), n, d_scores=s_sc[j].data_ptr(), d_kp_idx=s_kp[j].data_ptr()))
                r_sep["wall_ms"] = (time.perf_counter() - t0) * 1e3
                for j in range(k):                      # each detector keeps the stage times and counters of its last call
                    t, s = singles[j].timings(), singles[j].stats()
                    for key in ("features_ms", "nms_ms", "total_ms"):
                        r_sep[key] += t[key]
                    r_sep["host_syncs"] += s["host_syncs"]; r_sep["kernel_launches"] += s["kernel_launches"]
                    r_sep["n_keypoints"] += nks[j]
                if step == a.warmup + a.steps - 1 or step == 0:
                    # identical results, bit for bit
                    kpo = d_kpo.cpu().numpy()
                    sc = d_sc[:k * n].cpu().numpy().reshape(k, n)
                    kp = d_kp.cpu().numpy()
                    for j in range(k):
                        assert np.array_equal(sc[j].view(np.uint32), s_sc[j].cpu().numpy().view(np.uint32)), (wl, k, j)
                        assert np.array_equal(kp[kpo[j]:kpo[j + 1]], s_kp[j][:nks[j]].cpu().numpy()), (wl, k, j)
                if step >= a.warmup:
                    rows[k]["set"].append(r_set)
                    rows[k]["separate"].append(r_sep)
        res = {"points": n}
        for k in (1, 2, 3):
            sep = median(rows[k]["separate"])
            st = median(rows[k]["set"])
            res["K%d" % k] = {"set": st, "separate": sep, "wall_speedup": sep["wall_ms"] / st["wall_ms"]}
            print(wl, k, json.dumps(res["K%d" % k]), flush=True)
        out["workloads"][wl] = res
        for d in singles + list(sets.values()):
            d.close()
        del d_xyz, d_sc, d_kp, s_sc, s_kp
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
