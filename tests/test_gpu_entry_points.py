"""What every kpl_detect* entry point shares: the reset before any refusal, one refusal order whatever K is, and a host
entry point that is its device entry point plus one copy-out synchronisation."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORESTS = [os.path.join(ROOT, "tests", "golden", "forests", f + ".yaml.gz")
           for f in ("synthetic-T100-D15", "synthetic-SHOT-like-T50-D10", "synthetic-FPFH-like-T30-D25")]
KPL_E_INVALID, KPL_E_FOREST = 1, 2
TH = float(np.float32(0.5))

# (family, host entry point, device entry point) for K = 1 and for the forest set
FAMILIES = {
    "cloud": (("kpl_detect", "kpl_detect_device"), ("kpl_detect_forests", "kpl_detect_forests_device")),
    "views": (("kpl_detect_batch", "kpl_detect_batch_device"), ("kpl_detect_batch_forests", "kpl_detect_batch_forests_device")),
    "frames": (("kpl_detect_batch_organized", "kpl_detect_batch_organized_device"),
               ("kpl_detect_batch_organized_forests", "kpl_detect_batch_organized_forests_device")),
}
ENTRY_POINTS = ["kpl_detect_xyzi"] + [e for pairs in FAMILIES.values() for pair in pairs for e in pair]


def _detector(kpl, nforests=3):
    det = kpl.KeypointLearningDetector()
    det.setNAnnulus(5); det.setNBins(10); det.setNonMaxima(True); det.setNonMaxRadius(4.0)
    det.setNonMaximaDrawsRemove(False); det.setPredictionThreshold(TH); det.setRadiusSearch(20.0); det.setNormalsMode(1, k=10)
    for k, f in enumerate(FORESTS[:nforests]):
        assert det.loadForest(f) if k == 0 else det.addForest(f) == k
    det._push()
    return det


class Inputs:
    def __init__(self):
        from keypoint_learning_b200 import synth
        views = [np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", "views", v + ".npz"))["xyz"][:m], np.float32)
                 for v, m in (("cheff000", 6000), ("cheff001", 8000))]
        self.cloud = views[1]
        self.views = np.ascontiguousarray(np.concatenate(views))
        self.off = np.array([0, 6000, 14000], np.int64)
        fr = [synth.organized_range_image(160, 120, seed=40 + f, holes=f % 2 == 0)[0] for f in range(2)]
        self.frames = np.ascontiguousarray(np.stack(fr), np.float32)


def _call(kpl, det, x, name, stride=12, null_kp=False):
    """One call of entry point `name` on the inputs of its family; returns (status, keypoints of all forests)."""
    import torch
    from keypoint_learning_b200 import capi
    L, P = capi.load_library(), capi._ptr
    f32, i32, i64 = C.c_float, C.c_int32, C.c_int64
    K = det.forestCount() if "forests" in name else 1
    w = h = nf = 0
    if "organized" in name:
        nf, h, w, _ = x.frames.shape
        xyz, n, nv = x.frames.reshape(-1, 3), nf * h * w, nf
    elif "batch" in name:
        xyz, n, nv = x.views, len(x.views), 2
    else:
        xyz, n, nv = x.cloud, len(x.cloud), 1
    nkp = i64(0)
    if name.endswith("device"):
        x4 = np.ones((n, 4), np.float32); x4[:, :3] = xyz
        d_xyz = torch.from_numpy(x4).cuda()
        d_kp = torch.empty(K * n, dtype=torch.int32, device="cuda"); d_ko = torch.empty(K * nv + 1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        X, KP, KO = C.c_void_p(d_xyz.data_ptr()), (None if null_kp else C.c_void_p(d_kp.data_ptr())), C.c_void_p(d_ko.data_ptr())
        args = {"kpl_detect_device": (X, None, None, n, None, KP),
                "kpl_detect_forests_device": (X, None, n, None, None, KP, KO),
                "kpl_detect_batch_device": (X, None, P(x.off, i64), nv, None, KP, KO),
                "kpl_detect_batch_forests_device": (X, None, P(x.off, i64), nv, None, None, KP, KO),
                "kpl_detect_batch_organized_device": (X, None, w, h, nf, 5.0, None, None, KP, KO),
                "kpl_detect_batch_organized_forests_device": (X, None, w, h, nf, 5.0, None, None, None, KP, KO)}[name]
        rc = getattr(L, name)(det._h, *args, C.byref(nkp))
        torch.cuda.synchronize()
        return rc, nkp.value
    kp = np.empty(K * n, np.int32); ko = np.zeros(K * nv + 1, np.int64); kx = np.empty((n, 4), np.float32)
    X, KP = P(xyz, f32), (None if null_kp else P(kp, i32))
    args = {"kpl_detect": (X, stride, None, 0, None, n, None, KP, C.byref(nkp)),
            "kpl_detect_xyzi": (X, stride, None, 0, None, n, None, KP, P(kx, f32), C.byref(nkp)),
            "kpl_detect_forests": (X, stride, None, 0, n, None, None, KP, P(ko, i64)),
            "kpl_detect_batch": (X, stride, None, 0, P(x.off, i64), nv, None, KP, P(ko, i64)),
            "kpl_detect_batch_forests": (X, stride, None, 0, P(x.off, i64), nv, None, None, KP, P(ko, i64)),
            "kpl_detect_batch_organized": (X, stride, None, 0, w, h, nf, 5.0, None, None, KP, P(ko, i64)),
            "kpl_detect_batch_organized_forests": (X, stride, None, 0, w, h, nf, 5.0, None, None, None, KP, P(ko, i64))}[name]
    rc = getattr(L, name)(det._h, *args)
    return rc, (nkp.value if name in ("kpl_detect", "kpl_detect_xyzi") else int(ko[-1]))


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_refused_call_leaves_reset_stats(kpl, name):
    """A refused call leaves none of the previous call's stats or timings, whichever check refuses it."""
    x = Inputs()
    det = _detector(kpl)
    rc, nk = _call(kpl, det, x, name)
    assert rc == 0 and nk > 0 and det.stats()["kernel_launches"] > 0
    assert _call(kpl, det, x, name, null_kp=True)[0] == KPL_E_INVALID
    st, t = det.stats(), det.timings()
    assert (st["n_points"], st["n_keypoints"], st["kernel_launches"], t["total_ms"]) == (0, 0, 0, 0.0)
    det.close()


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_two_faults_one_order(kpl, family):
    """A bad stride on a context without a forest: the forest check comes first, for K = 1 and for the forest set alike."""
    x = Inputs()
    det = _detector(kpl, nforests=0)
    (one, _), (many, _) = FAMILIES[family]
    assert _call(kpl, det, x, one, stride=10)[0] == _call(kpl, det, x, many, stride=10)[0] == KPL_E_FOREST
    det.close()


def test_detect_forests_device_checks_threshold_shape(kpl):
    import torch
    det = _detector(kpl)
    d = torch.zeros(4 * 100, dtype=torch.float32, device="cuda")
    for th in ([TH], [TH] * 5, [[TH] * 3]):
        with pytest.raises(ValueError):
            det.detectForestsDevice(d.data_ptr(), 100, thresholds=th, d_kp_idx=d.data_ptr(), d_kp_offsets=d.data_ptr())
    det.close()


@pytest.mark.parametrize("family", sorted(FAMILIES))
@pytest.mark.parametrize("forests", [False, True])
def test_host_is_device_plus_one_sync(kpl, family, forests):
    """The host entry point launches what its device entry point launches and synchronises once more, for the copy-out;
    kpl_detect_xyzi adds the keypoint-cloud gather."""
    x = Inputs()
    det = _detector(kpl)
    host, dev = FAMILIES[family][int(forests)]
    runs = {}
    for name in (host, dev) + (("kpl_detect_xyzi",) if host == "kpl_detect" else ()):
        rc, nk = _call(kpl, det, x, name)
        st = det.stats()
        assert rc == 0 and nk == st["n_keypoints"] > 0, name
        runs[name] = st
    assert runs[host]["kernel_launches"] == runs[dev]["kernel_launches"]
    assert runs[host]["host_syncs"] == runs[dev]["host_syncs"] + 1
    if host == "kpl_detect":
        assert runs["kpl_detect_xyzi"]["kernel_launches"] == runs[dev]["kernel_launches"] + 1
        assert runs["kpl_detect_xyzi"]["host_syncs"] == runs[host]["host_syncs"]
    det.close()
