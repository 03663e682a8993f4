"""Dump what every kpl_detect* entry point returns, one line per call, so that two builds can be compared line for line.

For each of the 13 entry points, with non-maxima off, plain and draws-remove, and with one forest and with three (the
*_forests entry points), a line holds the return code, the keypoint count, digests of the scores (as bits), the
keypoints, the offsets and kpl_detect_xyzi's keypoint cloud, every field of kpl_stats, the kpl_timings fields that were
filled, and digests of kpl_fetch("normals" / "features") and kpl_fetch_u8("fragile") afterwards.  forest_ms spans two
back-to-back events, so whether it reads 0 is left out.  Then the return codes of single-fault refusals, the stats a
refused call leaves after a successful one, and the codes of two-fault inputs.

    python tools/dump_entry_points.py --root <tree with a built libkpl_b200.so> --out dump.txt

Needs a B200; the inputs are the golden views and seeded synthetic frames.
"""
import argparse
import ctypes as C
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
FORESTS = [os.path.join(REPO, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]
FOREST_A4xB8 = os.path.join(REPO, "tests", "golden", "forests", "synthetic-A4xB8-T20-D8.yaml.gz")
TH3 = [float(np.float32(0.5)), float(np.float32(0.3)), float(np.float32(0.6))]


def digest(a):
    return "-" if a is None else hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


class Dumper:
    def __init__(self, K, capi, synth, torch):
        self.K, self.capi, self.torch = K, capi, torch
        self.L = capi.load_library()
        self.lines = []
        views = [np.ascontiguousarray(np.load(os.path.join(REPO, "tests", "golden", "views", v + ".npz"))["xyz"][:m], np.float32)
                 for v, m in (("cheff000", 9000), ("cheff001", 12000))]
        self.cloud = views[1]
        self.views = np.ascontiguousarray(np.concatenate(views))
        self.off = np.array([0, len(views[0]), len(self.views)], np.int64)
        fr = np.stack([synth.organized_range_image(48, 40, seed=60 + f, holes=f % 2 == 0)[0] for f in range(3)])
        fr[1] = np.nan
        self.frames = np.ascontiguousarray(fr, np.float32)

    def detector(self, nforests, nms="plain", fragile=False, forest0=None):
        d = self.K.KeypointLearningDetector()
        d.setNAnnulus(5); d.setNBins(10); d.setNonMaxima(nms != "off"); d.setNonMaxRadius(4.0)
        d.setNonMaximaDrawsRemove(nms == "draws"); d.setNonMaximaDrawsThreshold(1.0 if nms == "draws" else 0.0)
        d.setPredictionThreshold(TH3[0]); d.setRadiusSearch(20.0); d.setNormalsMode(1, k=10)
        d.setReportFragile(fragile)
        if nforests:
            assert d.loadForest(forest0 or FORESTS[0])
            for f in FORESTS[1:nforests]:
                d.addForest(f)
        d.keepIntermediates(True)
        d._push()
        return d

    # ---- the 13 entry points: (name, host?, K-aware?, layout) -> call(det, K, th, fault) returning (rc, nkp, outputs)
    def call(self, name, det, K, th, fault=None):
        P, L, torch = self.capi._ptr, self.L, self.torch
        f32, i32, i64 = C.c_float, C.c_int32, C.c_int64
        fault = fault or {}
        forests = "forests" in name
        K = K if forests else 1
        thp = P(np.asarray(th[:K], np.float64), C.c_double) if (forests and th is not None) else None
        if "organized" in name:
            nf, h, w, _ = self.frames.shape
            xyz, n, nv = self.frames.reshape(-1, 3), nf * h * w, nf
            w, h, nf = fault.get("w", w), fault.get("h", h), fault.get("nf", nf)
        elif "batch" in name:
            xyz, n, nv = self.views, len(self.views), 2
        else:
            xyz, n, nv = self.cloud, len(self.cloud), 1
        n_arg = fault.get("n", n)
        off = fault.get("off", self.off)
        nv_arg = fault.get("nv", nv)
        nkp = i64(-1)
        if name.endswith("device"):
            x4 = np.ones((len(xyz), 4), np.float32); x4[:, :3] = xyz
            d_xyz = torch.from_numpy(x4).cuda()
            d_sc = torch.empty(max(K * n, 1), dtype=torch.float32, device="cuda")
            d_kp = torch.empty(max(K * n, 1), dtype=torch.int32, device="cuda")
            d_ko = torch.empty(K * nv + 1, dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            X = None if fault.get("xyz") == "null" else C.c_void_p(d_xyz.data_ptr())
            S, KP = C.c_void_p(d_sc.data_ptr()), (None if fault.get("kp") == "null" else C.c_void_p(d_kp.data_ptr()))
            KO = None if fault.get("ko") == "null" else C.c_void_p(d_ko.data_ptr())
            if name == "kpl_detect_device":
                rc = L.kpl_detect_device(det._h, X, None, None, n_arg, S, KP, C.byref(nkp))
            elif name == "kpl_detect_forests_device":
                rc = L.kpl_detect_forests_device(det._h, X, None, n_arg, thp, S, KP, KO, C.byref(nkp))
            elif name == "kpl_detect_batch_device":
                rc = L.kpl_detect_batch_device(det._h, X, None, P(off, i64), nv_arg, S, KP, KO, C.byref(nkp))
            elif name == "kpl_detect_batch_forests_device":
                rc = L.kpl_detect_batch_forests_device(det._h, X, None, P(off, i64), nv_arg, thp, S, KP, KO, C.byref(nkp))
            elif name == "kpl_detect_batch_organized_device":
                rc = L.kpl_detect_batch_organized_device(det._h, X, None, w, h, nf, fault.get("smooth", 5.0), None, S, KP, KO, C.byref(nkp))
            else:
                rc = L.kpl_detect_batch_organized_forests_device(det._h, X, None, w, h, nf, fault.get("smooth", 5.0), None, thp, S, KP, KO,
                                                                 C.byref(nkp))
            torch.cuda.synchronize()
            out = dict(scores=d_sc.cpu().numpy()[:K * n], kp=d_kp.cpu().numpy()[:max(nkp.value, 0)],
                       off=d_ko.cpu().numpy() if KO is not None and name != "kpl_detect_device" else None)
            return rc, nkp.value, out
        sc = np.full(max(K * n, 1), -1, np.float32)
        kp = np.full(max(K * n, 1), -1, np.int32)
        ko = np.full(K * nv + 1, -1, np.int64)
        kx = np.full((max(n, 1), 4), -1, np.float32)
        X = None if fault.get("xyz") == "null" else P(xyz, f32)
        stride = fault.get("stride", 12)
        KP = None if fault.get("kp") == "null" else P(kp, i32)
        KO = None if fault.get("ko") == "null" else P(ko, i64)
        if name in ("kpl_detect", "kpl_detect_xyzi"):
            if name == "kpl_detect":
                rc = L.kpl_detect(det._h, X, stride, None, 0, None, n_arg, P(sc, f32), KP, C.byref(nkp))
            else:
                rc = L.kpl_detect_xyzi(det._h, X, stride, None, 0, None, n_arg, P(sc, f32), KP, P(kx, f32), C.byref(nkp))
            m = max(nkp.value, 0)
            return rc, nkp.value, dict(scores=sc[:n], kp=kp[:m], xyzi=kx[:m] if name == "kpl_detect_xyzi" else None, off=None)
        if name == "kpl_detect_forests":
            rc = L.kpl_detect_forests(det._h, X, stride, None, 0, n_arg, thp, P(sc, f32), KP, KO)
        elif name == "kpl_detect_batch":
            rc = L.kpl_detect_batch(det._h, X, stride, None, 0, P(off, i64), nv_arg, P(sc, f32), KP, KO)
        elif name == "kpl_detect_batch_forests":
            rc = L.kpl_detect_batch_forests(det._h, X, stride, None, 0, P(off, i64), nv_arg, thp, P(sc, f32), KP, KO)
        elif name == "kpl_detect_batch_organized":
            rc = L.kpl_detect_batch_organized(det._h, X, stride, None, 0, w, h, nf, fault.get("smooth", 5.0), None, P(sc, f32), KP, KO)
        else:
            rc = L.kpl_detect_batch_organized_forests(det._h, X, stride, None, 0, w, h, nf, fault.get("smooth", 5.0), None, thp, P(sc, f32),
                                                      KP, KO)
        m = int(ko[-1]) if rc == 0 else 0
        return rc, m, dict(scores=sc[:K * n], kp=kp[:m], off=ko)

    def fetches(self, det, st, K):
        n = st["n_points"]
        res = []
        for what, width in (("normals", 4), ("features", 50)):
            buf = np.empty(max(n, 1) * width, np.float32)
            rc = self.L.kpl_fetch(det._h, what.encode(), self.capi._ptr(buf, C.c_float), buf.size)
            res.append("%s=%s" % (what, digest(buf[:n * width]) if rc == 0 else "rc%d" % rc))
        buf = np.empty(max(n, 1) * K, np.uint8)
        rc = self.L.kpl_fetch_u8(det._h, b"fragile", self.capi._ptr(buf, C.c_uint8), buf.size)
        res.append("fragile=%s" % (digest(buf[:n * K]) if rc == 0 else "rc%d" % rc))
        return " ".join(res)

    def state(self, det):
        st, t = det.stats(), det.timings()
        stats = ",".join("%s=%s" % (k, st[k]) for k in sorted(st))
        filled = ",".join(k for k in sorted(t) if t[k] != 0.0 and k != "forest_ms")
        return st, "stats[%s] timings_filled[%s]" % (stats, filled)


ENTRY_POINTS = ["kpl_detect", "kpl_detect_xyzi", "kpl_detect_device", "kpl_detect_forests", "kpl_detect_forests_device",
                "kpl_detect_batch", "kpl_detect_batch_forests", "kpl_detect_batch_device", "kpl_detect_batch_forests_device",
                "kpl_detect_batch_organized", "kpl_detect_batch_organized_forests", "kpl_detect_batch_organized_device",
                "kpl_detect_batch_organized_forests_device"]


def run(D):
    out = D.lines
    for nms in ("off", "plain", "draws"):
        for K in (1, 3):
            for th in (None, TH3):
                det = D.detector(K, nms, fragile=nms == "plain")
                for name in ENTRY_POINTS:
                    if "forests" not in name and (K > 1 or th is not None):
                        continue
                    rc, nkp, o = D.call(name, det, K, th)
                    st, s = D.state(det)
                    out.append("%s nms=%s K=%d th=%s rc=%d nkp=%d scores=%s kp=%s off=%s xyzi=%s %s %s" % (
                        name, nms, K, "set" if th else "none", rc, nkp, digest(None if o["scores"] is None else o["scores"].view(np.uint32)),
                        digest(o["kp"]), digest(o["off"]), digest(o.get("xyzi")), s, D.fetches(det, st, K if "forests" in name else 1)))
                det.close()
    # an empty cloud
    det = D.detector(3)
    for name in ("kpl_detect", "kpl_detect_xyzi", "kpl_detect_device", "kpl_detect_forests", "kpl_detect_forests_device"):
        rc, nkp, o = D.call(name, det, 3, None, dict(n=0))
        out.append("%s empty rc=%d nkp=%d off=%s %s" % (name, rc, nkp, digest(o["off"]), D.state(det)[1]))
    det.close()
    # single-fault refusals
    faults = [("null_kp", dict(kp="null")), ("null_xyz", dict(xyz="null"))]
    for name in ENTRY_POINTS:
        fl = list(faults)
        if "forests" in name or "batch" in name:
            fl.append(("null_ko", dict(ko="null")))
        if not name.endswith("device"):
            fl.append(("stride", dict(stride=10)))
        if "batch" in name and "organized" not in name:
            fl += [("off0", dict(off=np.array([1, 3000, 21000], np.int64))), ("off_empty", dict(off=np.array([0, 3000, 3000], np.int64))),
                   ("off_desc", dict(off=np.array([0, 4000, 3000], np.int64))), ("nv0", dict(nv=0))]
            if "forests" in name:
                fl.append(("Kn_limit", dict(off=np.array([0, 800_000_000], np.int64), nv=1)))
        if "organized" in name:
            fl += [("w0", dict(w=0)), ("smooth0", dict(smooth=0.0))]
            if "forests" in name:
                fl.append(("Kn_limit", dict(w=40000, h=10000, nf=2)))
        det = D.detector(3)
        for tag, f in fl:
            out.append("refusal %s %s rc=%d" % (name, tag, D.call(name, det, 3, None, f)[0]))
        det.close()
        for tag, det in (("no_forest", D.detector(0)), ("varcount", D.detector(1, forest0=FOREST_A4xB8))):
            out.append("refusal %s %s rc=%d" % (name, tag, D.call(name, det, 1, None)[0]))
            det.close()
        det = D.detector(3)
        det.setForcedGrid((0.0, 0.0, 0.0), (4, 4, 4)); det._push()
        if "batch" in name:
            out.append("refusal %s forced_grid rc=%d" % (name, D.call(name, det, 3, None)[0]))
        det.close()
    # what a refused call leaves after a successful one (intentional change: the reset comes first)
    for name in ENTRY_POINTS:
        det = D.detector(3)
        D.call(name, det, 3, None)
        rc = D.call(name, det, 3, None, dict(kp="null"))[0]
        st, t = det.stats(), det.timings()
        out.append("after_refusal %s rc=%d n_points=%d n_keypoints=%d kernel_launches=%d total_ms_zero=%s" % (
            name, rc, st["n_points"], st["n_keypoints"], st["kernel_launches"], t["total_ms"] == 0.0))
        det.close()
    # two faults (intentional change: one order for every entry point): a bad stride without a forest
    det = D.detector(0)
    for name in ENTRY_POINTS:
        if not name.endswith("device"):
            out.append("two_faults %s stride+no_forest rc=%d" % (name, D.call(name, det, 1, None, dict(stride=10))[0]))
    det.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--root", default=REPO, help="tree whose keypoint_learning_b200 package (and built library) to load")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import keypoint_learning_b200 as K
    from keypoint_learning_b200 import capi, synth
    import torch
    assert os.path.abspath(K.LIB_PATH).startswith(os.path.abspath(args.root)), K.LIB_PATH
    D = Dumper(K, capi, synth, torch)
    run(D)
    with open(args.out, "w") as f:
        f.write("\n".join(D.lines) + "\n")
    print("%d lines -> %s" % (len(D.lines), args.out))


if __name__ == "__main__":
    main()
