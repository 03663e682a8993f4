#!/usr/bin/env python
"""bench.py -- points scored / second through the detection hot path (search + normals + features +
forest + NMS) on N B200s of one node.  Contract: see the task statement; one JSON line on rank 0.

  python bench.py --gpus 1 --steps 5 --warmup 3                 # our arm (CUDA through the C ABI)
  python bench.py --impl reference --steps 1 --warmup 0         # the reference's CPU path (oracle port, all host threads)
  torchrun --nproc-per-node N bench.py --gpus N ...             # slab-sharded through kpl_shard_* (NCCL inside the library)

A "step" is one full detection pass over the workload (BASELINE.json configs[3]: the synthetic 10 M-point scene;
--workload view1m = configs[2], --workload views = configs[4], --workload cheff001 = configs[0]).
`value` times steps whose input is already resident in HBM; `e2e` times the host-buffer entry point (kpl_detect /
kpl_detect_batch / kpl_shard_upload + kpl_shard_detect): H2D of the cloud + compute + D2H of scores and keypoints.
The default N=1 line also carries short sub-records for the other single-GPU configurations (`extra`), a parity check
of the CUDA path against the CPU oracle on a crop of the workload, and sha256 digests of the results that every N
must reproduce.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
FOREST = os.path.join(ROOT, "tests", "golden", "forests", "synthetic-T100-D15.yaml.gz")
DIGESTS = os.path.join(ROOT, "tests", "golden", "bench_digests.json")
R_FEAT, R_NMS, TH, A, B, K_NORMALS = 20.0, 4.0, 0.85, 5, 10, 10
VIEW_W, VIEW_H = 560, 360            # BASELINE.json configs[4]: ~200 k-point 2.5D views
METRIC = "points scored/sec (search+normals+features+RF+NMS)"


def measured_traffic(workload):
    """DRAM bytes per feature-kernel launch from the committed `ncu --set full` capture of the same workload
    (profiles/traffic.json, written from profiles/*_ncu.txt); None when no capture exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(workload)
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def canon_scores(sc):
    """scores with every NaN mapped to one bit pattern, so that the digest does not depend on NaN payloads"""
    out = np.ascontiguousarray(sc, np.float32).copy()
    out[np.isnan(out)] = np.float32(np.nan)
    return out


def stored_digest(key):
    if os.path.exists(DIGESTS):
        with open(DIGESTS) as f:
            return json.load(f).get(key)
    return None


DUMP_BYTES = 64_000_000
UNSCORED = -1.0          # dumped score of a point without a finite normal; real scores 1 - votes/ntrees lie in [0, 1]


def dump_scores(sc):
    """scores as dumped: the NaN of an unscored point becomes UNSCORED, so that every dumped value is finite"""
    out = np.ascontiguousarray(sc, np.float32).copy()
    out[np.isnan(out)] = UNSCORED
    return out


def dump_outputs(directory, arrays):
    """Writes each array as <directory>/<name>.npy, floats as float32 and integers (indices) as float64, so that two builds
    can be compared output for output.  At most DUMP_BYTES in all: an array larger than its share of what is left is
    replaced by a fixed, seeded sample of its elements in ascending index order (the same elements on every run).
    Every value must be finite."""
    for name, a in arrays.items():
        if not np.isfinite(a).all():
            raise ValueError("--dump-outputs: %s holds values that are not finite" % name)
    os.makedirs(directory, exist_ok=True)
    items = sorted(((name, np.ascontiguousarray(a).ravel()) for name, a in arrays.items()), key=lambda t: t[1].nbytes)
    left = DUMP_BYTES - 4096 * len(items)                       # .npy headers
    for i, (name, a) in enumerate(items):
        a = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
        share = left // (len(items) - i)
        note = ""
        if a.nbytes > share:
            keep = share // a.itemsize
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
            note = " (seeded sample of %d elements)" % keep
        np.save(os.path.join(directory, name + ".npy"), a)
        left -= a.nbytes
        sys.stderr.write("bench.py: wrote %s.npy, %d x %s%s\n" % (name, a.size, a.dtype, note))


# ---------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------
def make_workload(name, n_points):
    from keypoint_learning_b200 import synth
    if name == "view1m":
        xyz, vp = synth.view_25d(1250, 800, seed=1234)
        return xyz, vp, "synthetic 1M-point 2.5D view (1250x800 range image, pitch 0.64 mm)"
    if name == "cheff001":
        xyz = np.load(os.path.join(ROOT, "tests", "golden", "views", "cheff001.npz"))["xyz"]
        return np.ascontiguousarray(xyz), (0.0, 0.0, 0.0), "bundled 2.5D view data/point_cloud_test/cheff001.pcd (%d points)" % len(xyz)
    xyz, vp = synth.scene_closed_surfaces(n_points, seed=4321)
    return xyz, vp, ("synthetic %d-point scene (32 closed surfaces 100-300 mm in a 2x2x1 m box, area-uniform, ~0.58 mm spacing: "
                     "~3.8 k neighbours per point in radiusFeatures)" % len(xyz))


def make_views(rank, distinct):
    """`distinct` different 560x360 views for this rank (seeds rank*distinct + i), as (n,4) float32."""
    from keypoint_learning_b200 import synth
    out, vp = [], None
    for i in range(distinct):
        xyz, vp = synth.view_25d(VIEW_W, VIEW_H, seed=rank * distinct + i)
        x4 = np.ones((len(xyz), 4), np.float32); x4[:, :3] = xyz
        out.append(x4)
    return out, vp


def make_config(args, world):
    """The workload description both arms print (identical dicts: arm-specific details live elsewhere in the line)."""
    if args.workload == "views":
        pts = VIEW_W * VIEW_H
        wl = ("batch of synthetic 2.5D views (%dx%d px, %d points each): %d views per GPU per step, %d distinct per GPU, independent "
              "units split over the GPUs, no communication (the full config is 4096 views)" % (VIEW_W, VIEW_H, pts, args.views_per_gpu, args.distinct_views))
        par = "views-dp%d" % world
    else:
        wl = {"view1m": "synthetic 1M-point 2.5D view (1250x800 range image, pitch 0.64 mm)",
              "cheff001": "bundled 2.5D view data/point_cloud_test/cheff001.pcd (63653 points)"}.get(
            args.workload, "synthetic %d-point scene (32 closed surfaces 100-300 mm in a 2x2x1 m box, area-uniform, ~0.58 mm spacing: "
                           "~3.8 k neighbours per point in radiusFeatures)" % args.points)
        par = "slab%d+halo" % world if world > 1 else "single"
    return {"workload": wl, "radiusFeatures": R_FEAT, "radiusNMS": R_NMS, "threshold": TH, "annuli": A, "bins": B,
            "forest": os.path.basename(FOREST), "normals": "kNN-%d" % K_NORMALS, "parallelism": par,
            "l2": "inputs and intermediates of a step exceed the 126 MB L2 (>= 60 B per point resident); no flush needed"
                  if args.workload != "cheff001" else "L2 flushed between steps (256 MB write)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/)
# ---------------------------------------------------------------------------------------------------------------
def host_threads():
    """All host cores, whatever the launcher exported: torchrun sets OMP_NUM_THREADS=1 for its workers."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, n)


def cpu_detect(crop, vp, threads, order=2):
    """order 2: neighbours in the search's own traversal order, as the reference consumes them (timing legs);
    order 1: the canonical (cell key, index) order the CUDA path accumulates in (parity check; costs a sort per point)."""
    from oracle import oracle as O
    forest = O.load_forest_yaml(FOREST)
    t0 = time.perf_counter()
    res = O.detect(crop, forest, R_FEAT, R_NMS, TH, A, B, normals_mode=1, k=K_NORMALS, viewpoint=vp, order=order, threads=threads)
    return res, time.perf_counter() - t0, O.num_threads()


def cpu_baseline_run(xyz, vp, sample_points, threads):
    """The oracle port of the reference's CPU path on a bounded spatial crop of the workload (same density and geometry)."""
    from keypoint_learning_b200 import synth
    crop = synth.cube_crop(xyz, sample_points)
    res, dt, cores = cpu_detect(crop, vp, threads)
    return dict(value=len(crop) / dt, seconds=dt, cores=cores, n=len(crop), stage_ms=res["stage_ms"], crop=crop,
                sample="cube crop of %d points around the median point of the workload, full pipeline, one pass" % len(crop))


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference binary cannot be built
    (PCL/FLANN/Eigen/Boost/OpenCV C++ absent), so this is the oracle port with an OpenMP loop over points on all host
    threads -- more generous to the reference than its own single-threaded loops (hpp:273,203).  Every step is one pass
    over a crop of the workload, sized from a calibration pass so that warmup + steps end within ~2.5 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    threads = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(threads)
    if args.workload == "views":
        hv, vp = make_views(0, 1)
        xyz = hv[0][:, :3].copy()
    else:
        xyz, vp, _ = make_workload(args.workload, args.points)
    from keypoint_learning_b200 import synth
    passes = max(1, args.warmup + args.steps)
    calib_n = min(len(xyz), 60_000)
    _, dt, cores = cpu_detect(synth.cube_crop(xyz, calib_n), vp, threads)
    rate = calib_n / dt
    sample = int(min(args.cpu_sample, len(xyz), max(calib_n, rate * 150.0 / passes)))
    vals, last = [], None
    for s in range(args.warmup + args.steps):
        last = cpu_baseline_run(xyz, vp, sample, threads)
        if s >= args.warmup:
            vals.append(last)
    tot_pts = sum(v["n"] for v in vals); tot_s = sum(v["seconds"] for v in vals)
    value = tot_pts / tot_s
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "points/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(1, len(vals)),
            "higher_is_better": True, "scaling": "weak" if args.workload == "views" else "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": make_config(args, world),
            "cpu_baseline": {"value": value, "unit": "points/s", "cores": last["cores"], "kind": "port", "sample": last["sample"],
                             "stage_ms": last["stage_ms"]},
            "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# the CUDA arm
# ---------------------------------------------------------------------------------------------------------------
def make_detector(K, local, vp, cpr):
    det = K.KeypointLearningDetector(device=local)
    det.setNAnnulus(A); det.setNBins(B); det.setNonMaxima(True); det.setNonMaxRadius(R_NMS); det.setNonMaximaDrawsRemove(False)
    det.setPredictionThreshold(float(np.float32(TH))); det.setRadiusSearch(R_FEAT)
    det.setNormalsMode(1, k=K_NORMALS, viewpoint=vp)
    det.setCellsPerRadius(cpr)
    if not det.loadForest(FOREST):
        raise RuntimeError("forest failed to load")
    return det


class Acc:
    """Per-call accounting of the library's own timers / counters over the timed region."""

    def __init__(self):
        self.reset()

    def reset(self):
        self.feat_ms = 0.0; self.pairs = 0; self.scored = 0; self.cand = 0; self.launches = 0; self.syncs = 0; self.calls = 0
        self.stage = None; self.dev_ms = 0.0

    def add(self, det):
        t = det.timings(); st = det.stats()
        self.feat_ms += t["features_ms"]; self.pairs += st["feature_pairs"]; self.scored += st["n_scored"]
        self.cand += st["candidate_pairs"]; self.launches += st["kernel_launches"]; self.syncs += st["host_syncs"]; self.calls += 1
        self.dev_ms += t["total_ms"]
        if self.stage is None:
            self.stage = dict(t)
        else:
            for k in t:
                self.stage[k] += t[k]


def time_steps(torch, dist, dev, stream, world, step_fn, steps, sampler=None):
    """EXACTLY `steps` calls bracketed by barrier + synchronize, CUDA events on the launch stream, max over ranks."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    barrier()
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record(stream)
    out = None
    for _ in range(steps):
        out = step_fn()
    ev1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = max(ev0.elapsed_time(ev1), 0.0)
    clocks = sampler.stop() if sampler else None
    if world > 1:
        tms = torch.tensor([ms, wall_ms], dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms, wall_ms = float(tms[0]), float(tms[1])
    return ms / steps, wall_ms / steps, out, clocks


def roofline_record(acc, per_call_views, peak_gbs, peak_src, workload, world):
    """Roofline of the dominant kernel (feature_kernel), algorithmic bytes per SURVEY.md 8d: 32 B per (query, neighbour)
    pair with the query itself included, over the launches of the timed region of THIS rank."""
    calls = max(1, acc.calls)
    pairs_self = (acc.pairs + acc.scored) / calls
    feat_bytes = 32.0 * pairs_self
    feat_s = max(acc.feat_ms / calls * 1e-3, 1e-9)
    achieved = feat_bytes / feat_s / 1e9
    tr = measured_traffic(workload) or {}
    return {"bound": "hbm", "kernel": "feature_kernel", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
            "traffic": tr.get("dram_bytes_per_launch") if world == 1 else None, "traffic_source": tr.get("source") if world == 1 else None,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": feat_bytes, "kernel_ms": feat_s * 1e3,
            "points_per_launch": acc.scored / calls, "views_per_launch": per_call_views,
            "pairs_per_s": acc.pairs / calls / feat_s, "candidate_tests_per_s": acc.cand / calls / feat_s,
            "acceptance": acc.pairs / max(1, acc.cand),
            "stage_ms": {k: v / calls for k, v in (acc.stage or {}).items()}, "host_syncs_per_call": acc.syncs / calls}


def single_cloud_leg(torch, K, dev, local, stream, xyz, vp, args, steps, warmup, sampler=None, flush=False, dump=False):
    """One cloud on one GPU: device-resident `value`, host-buffer `e2e`, digests.  Returns a dict; with `dump`, its
    "outputs" are the scores and keypoint indices of the last timed step."""
    n = len(xyz)
    det = make_detector(K, local, vp, args.cpr)
    det.setStream(stream.cuda_stream)
    xyz4 = np.ones((n, 4), np.float32); xyz4[:, :3] = xyz
    host_xyz4 = torch.from_numpy(xyz4).pin_memory()
    d_xyz4 = host_xyz4.to(dev, non_blocking=True)
    d_scores = torch.empty(n, dtype=torch.float32, device=dev)
    d_kp = torch.empty(n, dtype=torch.int32, device=dev)
    flush_buf = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev) if flush else None
    torch.cuda.synchronize(dev)
    acc = Acc()

    def step():
        if flush_buf is not None:
            flush_buf.zero_()                                  # 256 MB write: evicts the 126 MB L2 (a small cloud would stay resident)
        nk = det.detectDevice(d_xyz4.data_ptr(), n, d_scores=d_scores.data_ptr(), d_kp_idx=d_kp.data_ptr())
        acc.add(det)
        return nk
    for _ in range(warmup):
        step()
    acc.reset()
    ms, wall_ms, nkp, clocks = time_steps(torch, None, dev, stream, 1, step, steps, sampler)
    outputs = {"scores": dump_scores(d_scores.cpu().numpy()), "keypoints": d_kp[:nkp].cpu().numpy()} if dump else None
    if flush_buf is not None:                                  # the flush is not part of the path: time it alone and take it out
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev); e0.record(stream)
        for _ in range(steps):
            flush_buf.zero_()
        e1.record(stream); torch.cuda.synchronize(dev)
        ms = max(ms - e0.elapsed_time(e1) / steps, acc.dev_ms / max(1, acc.calls))
    snap = acc
    st = det.stats()
    # e2e through the host entry point
    sc_host = torch.empty(n, dtype=torch.float32).pin_memory().numpy()
    kp_host = torch.empty(n, dtype=torch.int32).pin_memory().numpy()
    host_np = host_xyz4.numpy()
    det.setInputCloud(host_np); det.setNormals(None)
    det.compute(scores_out=sc_host, kp_out=kp_host)
    steps_e2e = max(1, min(steps, 3))
    idx_box = [None]

    def e2e_step():
        _, idx_box[0] = det.compute(scores_out=sc_host, kp_out=kp_host)
    e2e_ms, e2e_wall, _, _ = time_steps(torch, None, dev, stream, 1, e2e_step, steps_e2e)
    e2e_ms = max(e2e_ms, e2e_wall)
    idx = idx_box[0]
    scores = sc_host[:n].copy()
    # un-timed diagnostic pass: near-split report (BASELINE.md s5)
    det.setReportFragile(True)
    det.compute(scores_out=sc_host, kp_out=kp_host)
    fragile = det.stats()["n_fragile_points"]
    det.setReportFragile(False)
    det.close()
    del d_xyz4, d_scores, d_kp, flush_buf
    return dict(n=n, ms=ms, wall_ms=wall_ms, nkp=int(nkp), clocks=clocks, acc=snap, stats=st, e2e_ms=e2e_ms, idx=idx, scores=scores,
                fragile=int(fragile), h2d=int(n * 16), d2h=int(n * 4 + len(idx) * 4), outputs=outputs)


def views_leg(torch, dist, K, dev, local, stream, rank, world, args, steps, warmup, views_per_gpu, sampler=None, dump=False):
    """configs[4]: `views_per_gpu` independent views per GPU per step in ONE kpl_detect_batch call.  With `dump`, the
    result's "outputs" are the scores, view-local keypoint indices and keypoint offsets of the last timed step."""
    host_views, vp = make_views(rank, args.distinct_views)
    pts = len(host_views[0])
    det = make_detector(K, local, vp, args.cpr)
    det.setStream(stream.cuda_stream)
    order = [v % len(host_views) for v in range(views_per_gpu)]
    concat = np.concatenate([host_views[v] for v in order])
    offsets = np.arange(views_per_gpu + 1, dtype=np.int64) * pts
    n_local = len(concat)
    host_cat = torch.from_numpy(concat).pin_memory()
    d_cat = host_cat.to(dev, non_blocking=True)
    d_scores = torch.empty(n_local, dtype=torch.float32, device=dev)
    d_kp = torch.empty(n_local, dtype=torch.int32, device=dev)
    d_kpo = torch.empty(views_per_gpu + 1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize(dev)
    acc = Acc()

    def step():
        nk = det.detectBatchDevice(d_cat.data_ptr(), offsets, d_scores=d_scores.data_ptr(), d_kp_idx=d_kp.data_ptr(), d_kp_offsets=d_kpo.data_ptr())
        acc.add(det)
        return nk
    for _ in range(warmup):
        step()
    acc.reset()
    ms, wall_ms, nkp, clocks = time_steps(torch, dist, dev, stream, world, step, steps, sampler)
    outputs = None
    if dump:
        kpo = d_kpo.cpu().numpy()
        outputs = {"scores": dump_scores(d_scores.cpu().numpy()), "keypoints": d_kp[:int(kpo[-1])].cpu().numpy(), "keypoint_offsets": kpo}
    snap = acc
    st = det.stats()
    sc_host = torch.empty(n_local, dtype=torch.float32).pin_memory().numpy()
    kp_host = torch.empty(n_local, dtype=torch.int32).pin_memory().numpy()
    host_np = host_cat.numpy()
    res = det.computeBatchConcat(host_np, offsets, scores_out=sc_host, kp_out=kp_host)
    steps_e2e = max(1, min(steps, 3))
    box = [res]

    def e2e_step():
        box[0] = det.computeBatchConcat(host_np, offsets, scores_out=sc_host, kp_out=kp_host)
    e2e_ms, e2e_wall, _, _ = time_steps(torch, dist, dev, stream, world, e2e_step, steps_e2e)
    e2e_ms = max(e2e_ms, e2e_wall)
    scores_v, kp_v = box[0]
    # parity of the batch against stand-alone calls on its first views (bit-identical by construction: checked here)
    same = True
    for v in range(min(2, views_per_gpu)):
        det.setInputCloud(host_views[order[v]]); det.setNormals(None)
        _, idx1 = det.compute()
        same = same and np.array_equal(idx1, kp_v[v]) and np.array_equal(canon_scores(det.getResponse()).view(np.uint32), canon_scores(scores_v[v]).view(np.uint32))
    nk_total = sum(len(k) for k in kp_v)
    digest = {"keypoints": sha(np.concatenate(kp_v[:len(host_views)])) if views_per_gpu >= len(host_views) else None,
              "scores": sha(canon_scores(np.concatenate(scores_v[:len(host_views)]))) if views_per_gpu >= len(host_views) else None}
    det.close()
    return dict(pts_view=pts, n_local=n_local, ms=ms, wall_ms=wall_ms, nkp=int(nkp), clocks=clocks, acc=snap, stats=st, e2e_ms=e2e_ms,
                batch_equals_single=bool(same), digest=digest, h2d=int(n_local * 16), d2h=int(n_local * 4 + nk_total * 4 + (views_per_gpu + 1) * 8),
                outputs=outputs)


def run_b200(args):
    import torch
    import torch.distributed as dist
    import keypoint_learning_b200 as K

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # torch.distributed is plumbing only here: barriers, max-over-ranks of the timings, the NCCL id of rank 0.
        # The data path (halo / score strips, keypoint gather) is NCCL inside libkpl_b200.so (csrc/shard.cu).
        dist.init_process_group("gloo")
    peak_gbs, peak_src = measured_peaks()
    stream = torch.cuda.current_stream(dev)
    sampler = ClockSampler(local) if rank == 0 else None
    config = make_config(args, world)
    line = None
    rc = 0
    dump = bool(args.dump_outputs)
    outputs = None

    if args.workload == "views":
        r = views_leg(torch, dist, K, dev, local, stream, rank, world, args, args.steps, args.warmup, args.views_per_gpu, sampler, dump=dump)
        outputs = r["outputs"]
        n_total = r["n_local"] * world
        value = n_total / (r["ms"] * 1e-3)
        e2e_ms = r["e2e_ms"]
        if world > 1:
            t = torch.tensor([e2e_ms], dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_ms = float(t[0])
        roof = roofline_record(r["acc"], args.views_per_gpu, peak_gbs, peak_src, "views", world)
        if rank == 0:
            line = {"metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": config, "roofline": roof, "cpu_baseline": None,
                    "e2e": {"value": n_total / (e2e_ms * 1e-3), "unit": "points/s", "h2d_bytes_per_step": r["h2d"] * world,
                            "d2h_bytes_per_step": r["d2h"] * world, "ms_per_step": e2e_ms,
                            "api": "kpl_detect_batch (pinned host xyz of all views of the step; scores + per-view keypoint lists copied back)"},
                    "gpu_launches": r["acc"].launches, "clocks": r["clocks"], "keypoints": r["nkp"], "n_points": n_total,
                    "points_per_rank": r["n_local"], "views_per_gpu_per_step": args.views_per_gpu,
                    "batch_equals_single_view_calls": r["batch_equals_single"], "digest_rank0": r["digest"],
                    "host_overhead_ms_per_step": max(0.0, r["wall_ms"] - r["acc"].dev_ms / max(1, r["acc"].calls))}
            if not r["batch_equals_single"]:
                rc = 3
    elif world > 1:
        from keypoint_learning_b200 import shard
        xyz, vp, _ = make_workload(args.workload, args.points)
        n_total = len(xyz)
        det = make_detector(K, local, vp, args.cpr)
        det.setStream(stream.cuda_stream)
        ids = [shard.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        plan = shard.plan_slabs(xyz, R_FEAT, R_NMS, args.cpr, world, args.normal_support)
        job = shard.SlabJob(det, xyz, plan, rank, ids[0])
        pinned = torch.from_numpy(job.host_xyz4).pin_memory()
        sc_host = torch.empty(job.n_owned, dtype=torch.float32).pin_memory().numpy()
        kp_host = torch.empty(n_total, dtype=torch.int32).pin_memory().numpy() if rank == 0 else None
        # first detection: widens the k-NN support if a normal that matters was clipped (KPL_E_HALO), every rank in lockstep
        shard.detect_widening(job, xyz, R_FEAT, R_NMS, args.cpr)
        if job.plan is not plan:
            pinned = torch.from_numpy(job.host_xyz4).pin_memory()
            sc_host = torch.empty(job.n_owned, dtype=torch.float32).pin_memory().numpy()
        host_np = pinned.numpy()
        acc = Acc()
        exch = []
        last_kp = [None]

        def step():
            nk, last_kp[0] = job.detect()                       # slab resident in HBM; rank 0 receives the global keypoint list
            acc.add(det); exch.append(job.info()["exchange_ms"])
            return nk
        for _ in range(args.warmup):
            step()
        acc.reset(); exch.clear()
        ms, wall_ms, nkp, clocks = time_steps(torch, dist, dev, stream, world, step, args.steps, sampler)
        if dump and rank == 0:
            outputs = {"keypoints": last_kp[0].copy()}
        snap_calls, snap_dev = acc.calls, acc.dev_ms
        st = det.stats()
        box = [None]

        def e2e_step():
            job.upload(host_np)                                  # H2D of the owned slab from pinned host memory
            box[0] = job.detect(scores_out=sc_host, kp_out=kp_host)      # ... scores of the owned points and the global keypoint list back
        e2e_step()
        steps_e2e = max(1, min(args.steps, 3))
        e2e_ms, e2e_wall, _, _ = time_steps(torch, dist, dev, stream, world, e2e_step, steps_e2e)
        e2e_ms = max(e2e_ms, e2e_wall)
        nk_glob, kp_glob = box[0]
        info = job.info()
        # per-rank picture of the last timed steps + global counters (plumbing: gloo)
        mine = [snap_dev / max(1, snap_calls), float(info["n_owned"] + info["n_left"] + info["n_right"]), float(st["feature_pairs"]), float(st["n_scored"]),
                float(st["n_near_threshold"]), float(np.mean(exch)) if exch else 0.0, float(info["halo_bytes"]), wall_ms]
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        gathered = [None] * world if rank == 0 else None
        dist.gather_object((job.gidx, sc_host[:job.n_owned].copy()), gathered, dst=0)
        roof = roofline_record(acc, 1, peak_gbs, peak_src, args.workload, world)
        if rank == 0:
            full = np.empty(n_total, np.float32)
            for gi, sc in gathered:
                full[gi] = sc
            dig = {"keypoints": sha(kp_glob.astype(np.int32)), "scores": sha(canon_scores(full))}
            key = "%s:%d:cpr%d" % (args.workload, n_total, args.cpr)
            ref_d = stored_digest(key)
            dev_ms = [a[0] for a in allr]
            line = {"metric": METRIC, "value": n_total / (ms * 1e-3), "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": config, "roofline": roof, "cpu_baseline": None,
                    "e2e": {"value": n_total / (e2e_ms * 1e-3), "unit": "points/s", "h2d_bytes_per_step": int(n_total * 16),
                            "d2h_bytes_per_step": int(n_total * 4 + nk_glob * 4), "ms_per_step": e2e_ms,
                            "api": "kpl_shard_upload + kpl_shard_detect on every rank: owned slab H2D from pinned host, NCCL halo + score exchange, "
                                   "owned scores D2H on every rank, global keypoint list D2H on rank 0"},
                    "gpu_launches": acc.launches, "clocks": clocks, "keypoints": int(nkp), "n_points": n_total,
                    "near_threshold_points": int(sum(a[4] for a in allr)), "points_scored_all_ranks": int(sum(a[3] for a in allr)),
                    "pairs_all_ranks": int(sum(a[2] for a in allr)),
                    "digest": dig, "digest_expected": ref_d, "digest_match": (dig == ref_d) if ref_d else None,
                    "per_rank": [{"device_ms": round(a[0], 3), "slab_points": int(a[1]), "pairs": int(a[2]), "owned_scored": int(a[3]),
                                  "exchange_ms": round(a[5], 3), "halo_bytes": int(a[6])} for a in allr],
                    "device_ms_spread": (max(dev_ms) - min(dev_ms)) / max(dev_ms),
                    "host_overhead_ms_per_step": max(0.0, ms - max(dev_ms)),
                    "plan": {"cuts": plan.cuts.tolist() if job.plan is plan else job.plan.cuts.tolist(), "halo_cells": job.plan.halo,
                             "normal_support_cells": job.plan.normal_support_cells, "modelled_cost": [round(c / 1e9, 3) for c in job.plan.cost]}}
            if ref_d and dig != ref_d:
                rc = 4
        job.close()
        det.close()
    else:
        xyz, vp, _ = make_workload(args.workload, args.points)
        n_total = len(xyz)
        flush = n_total * 64 < 126e6
        r = single_cloud_leg(torch, K, dev, local, stream, xyz, vp, args, args.steps, args.warmup, sampler, flush=flush, dump=dump)
        outputs = r["outputs"]
        roof = roofline_record(r["acc"], 1, peak_gbs, peak_src, args.workload, 1)
        pts = r["acc"].scored / max(1, r["acc"].calls)
        pipe_bytes = roof["algorithmic_bytes_per_launch"] + 16.0 * K_NORMALS * pts + 200.0 * pts
        roof["pipeline_frac"] = (pipe_bytes / (r["ms"] * 1e-3) / 1e9) / peak_gbs
        roof["fast_math_selftest_passed"] = bool(r["stats"]["fast_math"])
        dig = {"keypoints": sha(r["idx"].astype(np.int32)), "scores": sha(canon_scores(r["scores"]))}
        key = "%s:%d:cpr%d" % (args.workload, n_total, args.cpr)
        ref_d = stored_digest(key)
        line = {"metric": METRIC, "value": n_total / (r["ms"] * 1e-3), "unit": "points/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "roofline": roof, "cpu_baseline": None,
                "e2e": {"value": n_total / (r["e2e_ms"] * 1e-3), "unit": "points/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                        "ms_per_step": r["e2e_ms"],
                        "api": "kpl_detect (host xyz, pinned; normals estimated on device; scores + keypoint indices copied back)"},
                "gpu_launches": r["acc"].launches, "clocks": r["clocks"], "keypoints": r["nkp"], "n_points": n_total,
                "near_threshold_points": int(r["stats"]["n_near_threshold"]), "fragile_split_points": r["fragile"],
                "unscored_points": int(r["stats"]["n_unscored"]),
                "digest": dig, "digest_expected": ref_d, "digest_match": (dig == ref_d) if ref_d else None,
                "host_overhead_ms_per_step": max(0.0, r["wall_ms"] - r["acc"].dev_ms / max(1, r["acc"].calls))}
        if ref_d and dig != ref_d:
            rc = 4
        if not args.no_cpu:
            # CPU baseline on a crop of the workload -- and the same crop through the CUDA path: the parity check of the
            # headline configuration (scores uint32-identical up to NaN payload, keypoint lists identical)
            c = cpu_baseline_run(xyz, vp, args.cpu_sample, host_threads())
            line["cpu_baseline"] = {"value": c["value"], "unit": "points/s", "cores": c["cores"], "kind": "port", "sample": c["sample"],
                                    "stage_ms": c["stage_ms"]}
            from keypoint_learning_b200 import synth
            pcrop = synth.cube_crop(c["crop"], args.parity_sample)
            pres, _, _ = cpu_detect(pcrop, vp, host_threads(), order=1)
            det = make_detector(K, local, vp, args.cpr)
            det.setInputCloud(pcrop)
            _, idx = det.compute()
            g, o = canon_scores(det.getResponse()), canon_scores(pres["scores"])
            ok_s = bool(np.array_equal(g.view(np.uint32), o.view(np.uint32)))
            ok_k = bool(np.array_equal(idx, pres["keypoints"]))
            line["parity_check"] = {"config": "%s crop" % args.workload, "n": int(len(pcrop)), "scores_bit_identical": ok_s, "keypoints_identical": ok_k,
                                    "keypoints": int(len(idx)), "max_abs_score_diff": float(np.nanmax(np.abs(g - o))) if len(g) else 0.0,
                                    "against": "oracle/libkpl_oracle.so (CPU restatement, canonical accumulation order)"}
            det.close()
            if not (ok_s and ok_k):
                rc = 5
        if args.extras and args.workload == "scene10m":
            extra = {}
            del xyz
            for name in ("view1m", "cheff001"):
                x2, vp2, _ = make_workload(name, 0)
                r2 = single_cloud_leg(torch, K, dev, local, stream, x2, vp2, args, args.steps, args.warmup, None, flush=len(x2) * 64 < 126e6)
                roof2 = roofline_record(r2["acc"], 1, peak_gbs, peak_src, name, 1)
                d2 = {"keypoints": sha(r2["idx"].astype(np.int32)), "scores": sha(canon_scores(r2["scores"]))}
                exp = stored_digest("%s:%d:cpr%d" % (name, len(x2), args.cpr))
                extra[name] = {"value": len(x2) / (r2["ms"] * 1e-3), "ms_per_step": r2["ms"], "e2e": len(x2) / (r2["e2e_ms"] * 1e-3),
                               "frac": roof2["frac"], "kernel_ms": roof2["kernel_ms"], "keypoints": r2["nkp"], "digest": d2,
                               "digest_match": (d2 == exp) if exp else None, "n_points": len(x2),
                               "config": make_config(argparse.Namespace(**{**vars(args), "workload": name}), 1)["workload"]}
                if exp and d2 != exp:
                    rc = 4
            rv = views_leg(torch, None, K, dev, local, stream, 0, 1, args, args.steps, args.warmup, args.views_per_gpu, None)
            roofv = roofline_record(rv["acc"], args.views_per_gpu, peak_gbs, peak_src, "views", 1)
            expv = stored_digest("views:%d:%d:cpr%d" % (args.views_per_gpu, args.distinct_views, args.cpr))
            extra["views"] = {"value": rv["n_local"] / (rv["ms"] * 1e-3), "ms_per_step": rv["ms"], "e2e": rv["n_local"] / (rv["e2e_ms"] * 1e-3),
                              "frac": roofv["frac"], "kernel_ms": roofv["kernel_ms"], "keypoints": rv["nkp"], "digest": rv["digest"],
                              "digest_match": (rv["digest"] == expv) if expv else None,
                              "batch_equals_single_view_calls": rv["batch_equals_single"], "views_per_step": args.views_per_gpu,
                              "host_syncs_per_call": roofv["host_syncs_per_call"], "n_points": rv["n_local"],
                              "config": make_config(argparse.Namespace(**{**vars(args), "workload": "views"}), 1)["workload"]}
            if not rv["batch_equals_single"]:
                rc = 3
            line["extra"] = extra

    if rank == 0 and outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0 and line is not None:
        line["impl_details"] = {"cells_per_radius": args.cpr, "library": "keypoint_learning_b200/libkpl_b200.so (C ABI include/kpl.h)",
                                "multi_gpu": "kpl_shard_* : NCCL ncclSend/ncclRecv inside the library; torch.distributed (gloo) only for barriers and the NCCL id"
                                if world > 1 else None}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rc:
        sys.stderr.write("bench.py: result check failed (rc %d: 3 batch != single, 4 digest mismatch, 5 oracle parity)\n" % rc)
        sys.exit(rc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="scene10m", choices=["scene10m", "view1m", "views", "cheff001"])
    ap.add_argument("--views-per-gpu", type=int, default=32, help="views workload: views per GPU per step (one kpl_detect_batch call)")
    ap.add_argument("--distinct-views", type=int, default=8, help="views workload: different views generated per GPU")
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--cpr", type=int, default=4, help="grid cells per radiusFeatures")
    ap.add_argument("--normal-support", type=int, default=1, help="slab sharding: cell columns of k-NN support in the halo (widened on KPL_E_HALO)")
    ap.add_argument("--cpu-sample", type=int, default=1_500_000, help="points of the workload crop the CPU legs run on (~10-20 s of host work)")
    ap.add_argument("--parity-sample", type=int, default=400_000, help="points of the crop on which the CUDA path is compared with the oracle")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", dest="extras", action="store_false", help="skip the sub-records of the other single-GPU configurations")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last timed step as DIR/<name>.npy "
                                                          "(scores, -1 for an unscored point; keypoint indices; at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm runs on a crop sized from its own timing, so its outputs are not reproducible")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
