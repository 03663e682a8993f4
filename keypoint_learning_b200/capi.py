"""ctypes binding of libkpl_b200.so (include/kpl.h) + a thin Python mirror of the reference's
``pcl::keypoints::KeypointLearningDetector`` setters (include/KeypointLearning.h:102-155 of the
reference).  No torch, no numpy compute: numpy arrays are only the host buffers handed to the C ABI.
There is no fallback: if the CUDA library is missing or no sm_100 device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkpl_b200.so")

KPL_OK = 0
STATUS = {0: "KPL_OK", 1: "KPL_E_INVALID", 2: "KPL_E_FOREST", 3: "KPL_E_SIZE_MISMATCH", 4: "KPL_E_NONFINITE",
          5: "KPL_E_VARCOUNT", 6: "KPL_E_CUDA", 7: "KPL_E_GRID", 8: "KPL_E_NOMEM", 9: "KPL_E_IO", 10: "KPL_E_UNSUPPORTED",
          11: "KPL_E_NCCL", 12: "KPL_E_HALO"}
KPL_E_HALO = 12
NORMALS_GIVEN, NORMALS_KNN, NORMALS_RADIUS = 0, 1, 2
ROLE_HALO, ROLE_SCORE, ROLE_OWNED = 0, 1, 3

EXPORTS = ["kpl_create", "kpl_destroy", "kpl_last_error", "kpl_version", "kpl_set_stream", "kpl_params_default",
           "kpl_set_params", "kpl_get_params", "kpl_load_forest", "kpl_set_forest", "kpl_forest_info", "kpl_detect", "kpl_detect_xyzi",
           "kpl_normals", "kpl_features", "kpl_radius_stats", "kpl_radius_neighbors", "kpl_detect_device",
           "kpl_get_timings", "kpl_get_stats", "kpl_fetch", "kpl_set_keep_intermediates", "kpl_uniform_sample", "kpl_nearest",
           "kpl_fetch_u8", "kpl_device_count", "kpl_normals_organized", "kpl_detect_batch", "kpl_detect_batch_device",
           "kpl_slab_plan_make", "kpl_slab_partition", "kpl_nccl_unique_id", "kpl_shard_create", "kpl_shard_destroy", "kpl_shard_set_plan",
           "kpl_shard_set_slab", "kpl_shard_upload", "kpl_shard_detect", "kpl_shard_detect_group", "kpl_shard_get_info",
           "kpl_shard_device_scores", "kpl_shard_set_slab_normals", "kpl_shard_upload_normals", "kpl_detect_batch_organized",
           "kpl_detect_batch_organized_device", "kpl_add_forest", "kpl_add_forest_arrays", "kpl_forest_count", "kpl_detect_forests",
           "kpl_detect_forests_device", "kpl_detect_batch_forests", "kpl_detect_batch_forests_device", "kpl_detect_batch_organized_forests",
           "kpl_detect_batch_organized_forests_device", "kpl_shard_detect_forests", "kpl_shard_detect_forests_group"]
KPL_MAX_RANKS = 64
KPL_MAX_FORESTS = 16


class KplParams(C.Structure):
    _fields_ = [("radius_features", C.c_float), ("radius_nms", C.c_float), ("threshold", C.c_double),
                ("n_annulus", C.c_int32), ("n_bins", C.c_int32), ("non_maxima", C.c_int32), ("draws_remove", C.c_int32),
                ("draws_threshold", C.c_float), ("normals_mode", C.c_int32), ("k_normals", C.c_int32),
                ("viewpoint", C.c_float * 3), ("flip_normals", C.c_int32), ("cells_per_radius", C.c_int32),
                ("grid_forced", C.c_int32), ("grid_origin", C.c_double * 3), ("grid_dims", C.c_int32 * 3),
                ("grid_offset", C.c_int32 * 3), ("slab_interior_lo", C.c_int32), ("slab_interior_hi", C.c_int32),
                ("slab_guard_cells", C.c_int32), ("slab_owned_lo", C.c_int32), ("slab_owned_hi", C.c_int32),
                ("uniform_sampling_centre", C.c_int32), ("eigen32_normalize", C.c_int32), ("report_fragile", C.c_int32)]


class KplTimings(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("grid_ms", "normals_ms", "features_ms", "forest_ms", "nms_ms", "total_ms")]


class KplStats(C.Structure):
    _fields_ = [("n_points", C.c_int64), ("n_scored", C.c_int64), ("feature_pairs", C.c_int64), ("candidate_pairs", C.c_int64),
                ("n_above_threshold", C.c_int64), ("n_keypoints", C.c_int64), ("grid_cells", C.c_int64),
                ("grid_dims", C.c_int32 * 3), ("kernel_launches", C.c_int32), ("grid_origin", C.c_double * 3), ("grid_cell", C.c_double),
                ("fast_math", C.c_int32), ("nms_rounds", C.c_int32), ("n_unscored", C.c_int64),
                ("n_near_threshold", C.c_int64), ("n_fragile_points", C.c_int64), ("host_syncs", C.c_int32), ("n_views", C.c_int32)]


class KplSlabPlan(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("cell", C.c_double), ("dims", C.c_int32 * 3), ("world", C.c_int32),
                ("reach_feat", C.c_int32), ("reach_nms", C.c_int32), ("normal_support_cells", C.c_int32), ("halo", C.c_int32),
                ("cuts", C.c_int32 * (KPL_MAX_RANKS + 1)), ("n_points", C.c_int64), ("cost", C.c_double * KPL_MAX_RANKS)]


class KplShardInfo(C.Structure):
    _fields_ = [("n_owned", C.c_int64), ("n_left", C.c_int64), ("n_right", C.c_int64), ("send_left", C.c_int64), ("send_right", C.c_int64),
                ("halo_bytes", C.c_int64), ("local_dims", C.c_int32 * 3), ("local_offset", C.c_int32 * 3), ("rank", C.c_int32),
                ("world", C.c_int32), ("exchange_ms", C.c_float), ("gather_ms", C.c_float)]


class KplError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (STATUS.get(code, code), msg))
        self.code = code


_lib = None


def load_library():
    """Load libkpl_b200.so.  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libkpl_b200.so is missing: run `python -m keypoint_learning_b200.build` (or __graft_entry__.build())")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    f32p, i32p, i64p, u8p, u64p = (C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_uint8), C.POINTER(C.c_uint64))
    L.kpl_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.kpl_destroy.argtypes = [vp]; L.kpl_destroy.restype = None
    L.kpl_last_error.argtypes = [vp]; L.kpl_last_error.restype = C.c_char_p
    L.kpl_version.restype = C.c_char_p
    L.kpl_set_stream.argtypes = [vp, vp]
    L.kpl_params_default.argtypes = [C.POINTER(KplParams)]
    L.kpl_set_params.argtypes = [vp, C.POINTER(KplParams)]
    L.kpl_get_params.argtypes = [vp, C.POINTER(KplParams)]
    L.kpl_load_forest.argtypes = [vp, C.c_char_p]
    L.kpl_set_forest.argtypes = [vp, C.c_int32, C.c_int32, i32p, i32p, f32p, i32p, i32p, f32p, C.c_int32]
    L.kpl_forest_info.argtypes = [vp, i32p, i32p, i32p, i32p]
    L.kpl_add_forest.argtypes = [vp, C.c_char_p, i32p]
    L.kpl_add_forest_arrays.argtypes = [vp, C.c_int32, C.c_int32, i32p, i32p, f32p, i32p, i32p, f32p, C.c_int32, i32p]
    L.kpl_forest_count.argtypes = [vp, i32p]
    f64p = C.POINTER(C.c_double)
    L.kpl_detect_forests.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, C.c_int64, f64p, f32p, i32p, i64p]
    L.kpl_detect_forests_device.argtypes = [vp, vp, vp, C.c_int64, f64p, vp, vp, vp, i64p]
    L.kpl_detect.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, u8p, C.c_int64, f32p, i32p, i64p]
    L.kpl_detect_xyzi.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, u8p, C.c_int64, f32p, i32p, f32p, i64p]
    L.kpl_normals.argtypes = [vp, f32p, C.c_int32, C.c_int64, f32p]
    L.kpl_features.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, C.c_int64, i32p, C.c_int64, f32p]
    L.kpl_radius_stats.argtypes = [vp, f32p, C.c_int32, C.c_int64, C.c_double, i32p, u64p]
    L.kpl_radius_neighbors.argtypes = [vp, f32p, C.c_int32, C.c_int64, C.c_double, i32p, C.c_int64, i64p, i32p]
    L.kpl_detect_device.argtypes = [vp, vp, vp, vp, C.c_int64, vp, vp, i64p]
    L.kpl_get_timings.argtypes = [vp, C.POINTER(KplTimings)]
    L.kpl_get_stats.argtypes = [vp, C.POINTER(KplStats)]
    L.kpl_fetch.argtypes = [vp, C.c_char_p, f32p, C.c_int64]
    L.kpl_set_keep_intermediates.argtypes = [vp, C.c_int]
    L.kpl_uniform_sample.argtypes = [vp, f32p, C.c_int32, C.c_int64, C.c_float, i32p, i64p]
    L.kpl_nearest.argtypes = [vp, f32p, C.c_int32, C.c_int64, f32p, C.c_int32, C.c_int64, i32p, f32p]
    L.kpl_fetch_u8.argtypes = [vp, C.c_char_p, u8p, C.c_int64]
    L.kpl_normals_organized.argtypes = [vp, f32p, C.c_int32, C.c_int32, C.c_int32, C.c_float, f32p]
    L.kpl_slab_plan_make.argtypes = [f32p, C.c_int32, C.c_int64, C.POINTER(KplParams), C.c_int32, C.c_int32, C.POINTER(KplSlabPlan)]
    L.kpl_slab_partition.argtypes = [C.POINTER(KplSlabPlan), f32p, C.c_int32, C.c_int64, C.c_int32, i32p, i64p]
    L.kpl_nccl_unique_id.argtypes = [vp]
    L.kpl_shard_create.argtypes = [vp, C.POINTER(KplSlabPlan), C.c_int32, vp, C.POINTER(vp)]
    L.kpl_shard_destroy.argtypes = [vp]; L.kpl_shard_destroy.restype = None
    L.kpl_shard_set_plan.argtypes = [vp, C.POINTER(KplSlabPlan)]
    L.kpl_shard_set_slab.argtypes = [vp, f32p, C.c_int32, i32p, C.c_int64]
    L.kpl_shard_upload.argtypes = [vp, f32p, C.c_int32]
    L.kpl_shard_set_slab_normals.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, i32p, C.c_int64]
    L.kpl_shard_upload_normals.argtypes = [vp, f32p, C.c_int32]
    L.kpl_shard_detect.argtypes = [vp, f32p, i32p, C.c_int64, i64p]
    L.kpl_shard_detect_group.argtypes = [C.POINTER(vp), C.c_int32, C.POINTER(f32p), i32p, C.c_int64, i64p]
    L.kpl_shard_detect_forests.argtypes = [vp, f64p, f32p, i32p, C.c_int64, i64p, i64p]
    L.kpl_shard_detect_forests_group.argtypes = [C.POINTER(vp), C.c_int32, f64p, C.POINTER(f32p), i32p, C.c_int64, i64p, i64p]
    L.kpl_shard_get_info.argtypes = [vp, C.POINTER(KplShardInfo)]
    L.kpl_shard_device_scores.argtypes = [vp]; L.kpl_shard_device_scores.restype = vp
    L.kpl_detect_batch.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, i64p, C.c_int32, f32p, i32p, i64p]
    L.kpl_detect_batch_device.argtypes = [vp, vp, vp, i64p, C.c_int32, vp, vp, vp, i64p]
    L.kpl_detect_batch_organized.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, f32p, f32p,
                                             i32p, i64p]
    L.kpl_detect_batch_organized_device.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_float, f32p, vp, vp, vp, i64p]
    L.kpl_detect_batch_forests.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, i64p, C.c_int32, f64p, f32p, i32p, i64p]
    L.kpl_detect_batch_forests_device.argtypes = [vp, vp, vp, i64p, C.c_int32, f64p, vp, vp, vp, i64p]
    L.kpl_detect_batch_organized_forests.argtypes = [vp, f32p, C.c_int32, f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, f32p,
                                                     f64p, f32p, i32p, i64p]
    L.kpl_detect_batch_organized_forests_device.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_float, f32p, f64p, vp, vp, vp,
                                                            i64p]
    _lib = L
    return L


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def _vec3(a, name):
    """Accept (n,3) packed or (n,4)/(n,8) strided float32 host arrays; returns (array, stride_bytes)."""
    a = np.asarray(a)
    if a.dtype != np.float32 or a.ndim != 2 or a.shape[1] < 3 or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("%s must be (n, >=3) float32" % name)
    return a, a.shape[1] * 4


class KeypointLearningDetector:
    """Python mirror of the reference detector: same setter names, `compute()` returns
    (keypoints[n_kp,4] = x,y,z,intensity ; indices[n_kp])."""

    def __init__(self, prediction_th=0.5, non_maxima=True, non_maxima_draws_remove=True, non_max_radius=0.0,
                 n_annulus=5, n_bins=10, device=0):
        L = load_library()
        self._L = L
        self._h = C.c_void_p()
        rc = L.kpl_create(int(device), C.byref(self._h))
        if rc != KPL_OK:
            raise KplError(rc, "kpl_create failed (is an sm_100 GPU visible?)")
        self._p = KplParams()
        L.kpl_params_default(C.byref(self._p))
        # constructor defaults of include/KeypointLearning.h:81-88
        self._p.threshold = float(prediction_th)
        self._p.non_maxima = int(bool(non_maxima))
        self._p.draws_remove = int(bool(non_maxima_draws_remove))
        self._p.radius_nms = float(non_max_radius)
        self._p.n_annulus = int(n_annulus)
        self._p.n_bins = int(n_bins)
        self._cloud = None
        self._normals = None
        self._kp_idx = np.empty(0, np.int32)
        self._scores = None
        self._responses = None
        self._xyzi = None

    # ---- lifetime
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.kpl_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != KPL_OK:
            raise KplError(rc, (self._L.kpl_last_error(self._h) or b"").decode())

    def _push(self):
        self._check(self._L.kpl_set_params(self._h, C.byref(self._p)))

    # ---- reference setters
    def setInputCloud(self, cloud):
        if self._normals is not None and self._cloud is not None and cloud is not self._cloud:
            self._normals = None   # impl/KeypointLearning.hpp:52-55
        self._cloud = cloud

    def setNormals(self, normals): self._normals = normals
    def setNonMaxima(self, v): self._p.non_maxima = int(bool(v))
    def setNonMaximaDrawsRemove(self, v): self._p.draws_remove = int(bool(v))
    def setNonMaximaDrawsThreshold(self, v): self._p.draws_threshold = float(v)
    def setPredictionThreshold(self, th): self._p.threshold = float(th)
    def setNonMaxRadius(self, r): self._p.radius_nms = float(r)
    def setNAnnulus(self, a): self._p.n_annulus = int(a)
    def setNBins(self, b): self._p.n_bins = int(b)
    def setRadiusSearch(self, r): self._p.radius_features = float(r)

    def loadForest(self, path):
        rc = self._L.kpl_load_forest(self._h, os.fsencode(path))
        return rc == KPL_OK

    # ---- extensions of the B200 build
    def setNormalsMode(self, mode, k=10, viewpoint=(0.0, 0.0, 0.0), flip=False):
        self._p.normals_mode = int(mode); self._p.k_normals = int(k)
        for i in range(3):
            self._p.viewpoint[i] = float(viewpoint[i])
        self._p.flip_normals = int(bool(flip))

    def setCellsPerRadius(self, cpr): self._p.cells_per_radius = int(cpr)

    def setEigen32Normalize(self, on=True):
        """row.normalize() as Eigen 3.2.x evaluates it (multiply by 1/norm) instead of the default division (Eigen >= 3.3)."""
        self._p.eigen32_normalize = int(bool(on))

    def setReportFragile(self, on=True):
        """Flag the points whose forest walk decided a split within 1e-5 (stats()["n_fragile_points"], fetchFragile())."""
        self._p.report_fragile = int(bool(on))

    def setForcedGrid(self, origin=None, dims=None, offset=(0, 0, 0), interior=(False, False), guard_cells=0):
        """Slab of a larger cloud: the global grid origin, the local dims and the local cell offset.  interior = which x
        faces of the local grid the cloud continues behind (a clipped k-NN normal search fails with KPL_E_HALO there,
        except in the outermost guard_cells columns)."""
        if origin is None:
            self._p.grid_forced = 0
            return
        self._p.grid_forced = 1
        for i in range(3):
            self._p.grid_origin[i] = float(origin[i]); self._p.grid_dims[i] = int(dims[i]); self._p.grid_offset[i] = int(offset[i])
        self._p.slab_interior_lo = int(bool(interior[0])); self._p.slab_interior_hi = int(bool(interior[1]))
        self._p.slab_guard_cells = int(guard_cells)

    def setStream(self, cuda_stream_ptr):
        """Run on a caller-owned cudaStream_t.  0 is the legacy default stream (what torch.cuda.current_stream()
        reports unless a side stream is active): it is passed as cudaStreamLegacy (1), because a NULL handle
        means "the context's own non-blocking stream" to kpl_set_stream, which would not be ordered after
        work the caller enqueued on the default stream.  None resets to the context stream."""
        ptr = None if cuda_stream_ptr is None else (int(cuda_stream_ptr) or 1)
        self._check(self._L.kpl_set_stream(self._h, C.c_void_p(ptr)))

    @staticmethod
    def _forest_args(f):
        arrays = [np.ascontiguousarray(f["roots"], np.int32), np.ascontiguousarray(f["var"], np.int32), np.ascontiguousarray(f["thr"], np.float32),
                  np.ascontiguousarray(f["left"], np.int32), np.ascontiguousarray(f["right"], np.int32), np.ascontiguousarray(f["value"], np.float32)]
        types = [C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_int32, C.c_float]
        return arrays, [int(f["ntrees"]), len(f["var"])] + [_ptr(a, t) for a, t in zip(arrays, types)] + [int(f.get("var_count", 0))]

    def setForestArrays(self, forest):
        keep, args = self._forest_args(forest)
        self._check(self._L.kpl_set_forest(self._h, *args))

    def addForest(self, path):
        """kpl_add_forest: append the forest at `path` to the forest set (forest 0 is loadForest's); returns its index."""
        idx = C.c_int32(-1)
        self._check(self._L.kpl_add_forest(self._h, os.fsencode(path), C.byref(idx)))
        return idx.value

    def addForestArrays(self, forest):
        """kpl_add_forest_arrays: the same from the arrays setForestArrays takes; returns the new forest's index."""
        keep, args = self._forest_args(forest)
        idx = C.c_int32(-1)
        self._check(self._L.kpl_add_forest_arrays(self._h, *args, C.byref(idx)))
        return idx.value

    def forestCount(self):
        k = C.c_int32(0)
        self._check(self._L.kpl_forest_count(self._h, C.byref(k)))
        return k.value

    def forestInfo(self):
        v = [C.c_int32() for _ in range(4)]
        self._check(self._L.kpl_forest_info(self._h, *[C.byref(x) for x in v]))
        return dict(ntrees=v[0].value, nnodes=v[1].value, var_count=v[2].value, max_depth=v[3].value)

    # ---- the hot path
    def compute(self, role=None, scores_out=None, kp_out=None):
        """detector->compute(*keypoint): returns (keypoints (n_kp,4) float32, indices (n_kp,) int32)."""
        if self._cloud is None:
            raise KplError(1, "no input cloud")
        xyz, xs = _vec3(self._cloud, "cloud")
        n = xyz.shape[0]
        nrm = ns = None
        if self._normals is not None:
            nrm, ns = _vec3(self._normals, "normals")
            if nrm.shape[0] != n:
                raise KplError(3, "normals given, but the number of normals does not match the number of input points")
        self._push()
        # caller-provided result buffers (e.g. pinned host memory) are used as they are
        scores = np.empty(n, np.float32) if scores_out is None else scores_out
        kp = np.empty(max(n, 1), np.int32) if kp_out is None else kp_out
        if scores.dtype != np.float32 or scores.size < n or kp.dtype != np.int32 or kp.size < max(n, 1):
            raise KplError(1, "scores_out / kp_out must be float32[n] / int32[n]")
        nkp = C.c_int64(0)
        r = None if role is None else np.ascontiguousarray(role, np.uint8)
        if self._xyzi is None or self._xyzi.shape[0] < max(n, 1):
            self._xyzi = np.empty((max(n, 1), 4), np.float32)          # virtual memory only: the library writes n_kp rows
        rc = self._L.kpl_detect_xyzi(self._h, _ptr(xyz, C.c_float), xs, _ptr(nrm, C.c_float), ns or 0, _ptr(r, C.c_uint8), n,
                                     _ptr(scores, C.c_float), _ptr(kp, C.c_int32), _ptr(self._xyzi, C.c_float), C.byref(nkp))
        if rc == 4:
            # KPL_E_NONFINITE (found by the device's bounding-box pass, no host scan): a non-dense cloud.  The reference's
            # kd-tree ignores NaN points and runForest skips them (hpp:277): compact the finite points, detect, and map
            # indices / scores back (NaN score, never a keypoint).
            return self._compute_compacted(xyz, nrm, np.isfinite(xyz[:, :3]).all(axis=1), role)
        self._check(rc)
        self._scores = scores
        self._kp_idx = kp[:nkp.value].copy()
        return self._xyzi[:nkp.value].copy(), self._kp_idx          # the keypoint cloud was gathered on the device

    @staticmethod
    def _concat_views(clouds, normals):
        arrs = [_vec3(c, "cloud")[0] for c in clouds]
        width = arrs[0].shape[1]
        if any(a.shape[1] != width for a in arrs):
            raise ValueError("all views must share one point layout")
        xyz = np.ascontiguousarray(np.concatenate(arrs)) if len(arrs) > 1 else arrs[0]
        off = np.zeros(len(arrs) + 1, np.int64)
        off[1:] = np.cumsum([len(a) for a in arrs])
        nrm = ns = None
        if normals is not None:
            nrm = np.ascontiguousarray(np.concatenate([_vec3(x, "normals")[0] for x in normals]))
            ns = nrm.shape[1] * 4
        return xyz, off, nrm, ns

    def _thresholds(self, thresholds):
        """None, or one float64 threshold per forest of the set (the shape computeForests checks)."""
        if thresholds is None:
            return None
        K = self.forestCount()
        th = np.ascontiguousarray(thresholds, np.float64)
        if th.shape != (K,):
            raise ValueError("thresholds must hold one value per forest (%d)" % K)
        return th

    def computeBatch(self, clouds, normals=None):
        """kpl_detect_batch: `clouds` is a list of (n_v, >=3) float32 views.  Returns (scores list, keypoint index list),
        one entry per view, exactly what compute() returns for each view alone."""
        return self.computeBatchConcat(*self._concat_views(clouds, normals))

    def computeBatchForests(self, clouds, normals=None, thresholds=None):
        """kpl_detect_batch_forests: every forest of the set over a batch of views, from one feature pass.  thresholds: None
        (the prediction threshold for every forest) or one per forest.  Returns out[k][v] = (scores, view-local keypoint
        indices): what computeBatch() returns for view v with only forest k loaded and threshold k."""
        th = self._thresholds(thresholds)
        xyz, off, nrm, ns = self._concat_views(clouds, normals)
        K, n, nv = self.forestCount(), xyz.shape[0], len(off) - 1
        self._push()
        scores = np.empty((max(K, 1), n), np.float32)
        kp = np.empty(max(K * n, 1), np.int32)
        kpo = np.empty(K * nv + 1, np.int64)
        self._check(self._L.kpl_detect_batch_forests(self._h, _ptr(xyz, C.c_float), xyz.shape[1] * 4, _ptr(nrm, C.c_float), ns or 0,
                                                     _ptr(off, C.c_int64), nv, _ptr(th, C.c_double), _ptr(scores, C.c_float),
                                                     _ptr(kp, C.c_int32), _ptr(kpo, C.c_int64)))
        return [[(scores[k, off[v]:off[v + 1]], kp[kpo[k * nv + v]:kpo[k * nv + v + 1]].copy()) for v in range(nv)] for k in range(K)]

    def computeBatchConcat(self, xyz, offsets, nrm=None, ns=None, scores_out=None, kp_out=None):
        """kpl_detect_batch on an already concatenated host array (what bench.py times)."""
        n = xyz.shape[0]
        nv = len(offsets) - 1
        self._push()
        scores = np.empty(n, np.float32) if scores_out is None else scores_out
        kp = np.empty(max(n, 1), np.int32) if kp_out is None else kp_out
        kpo = np.empty(nv + 1, np.int64)
        off = np.ascontiguousarray(offsets, np.int64)
        self._check(self._L.kpl_detect_batch(self._h, _ptr(xyz, C.c_float), xyz.shape[1] * 4, _ptr(nrm, C.c_float), ns or 0,
                                             _ptr(off, C.c_int64), nv, _ptr(scores, C.c_float), _ptr(kp, C.c_int32), _ptr(kpo, C.c_int64)))
        return ([scores[off[v]:off[v + 1]] for v in range(nv)], [kp[kpo[v]:kpo[v + 1]].copy() for v in range(nv)])

    def detectBatchDevice(self, d_xyz4, offsets, d_scores=0, d_kp_idx=0, d_kp_offsets=0, d_normals4=0):
        """Device-resident batch: raw device pointers (ints), host offsets.  Returns the total keypoint count."""
        self._push()
        off = np.ascontiguousarray(offsets, np.int64)
        nkp = C.c_int64(0)
        self._check(self._L.kpl_detect_batch_device(self._h, C.c_void_p(d_xyz4), C.c_void_p(d_normals4 or None), _ptr(off, C.c_int64),
                                                    len(off) - 1, C.c_void_p(d_scores or None), C.c_void_p(d_kp_idx), C.c_void_p(d_kp_offsets),
                                                    C.byref(nkp)))
        return nkp.value

    def detectBatchForestsDevice(self, d_xyz4, offsets, d_scores=0, d_kp_idx=0, d_kp_offsets=0, d_normals4=0, thresholds=None):
        """kpl_detect_batch_forests_device: raw device pointers (ints), host offsets; d_scores K*n floats (or 0), d_kp_idx K*n
        int32, d_kp_offsets K*n_views + 1 int64, forest-major then view-major.  Returns the keypoint count of all forests."""
        th = self._thresholds(thresholds)
        self._push()
        off = np.ascontiguousarray(offsets, np.int64)
        nkp = C.c_int64(0)
        self._check(self._L.kpl_detect_batch_forests_device(self._h, C.c_void_p(d_xyz4), C.c_void_p(d_normals4 or None), _ptr(off, C.c_int64),
                                                            len(off) - 1, _ptr(th, C.c_double), C.c_void_p(d_scores or None),
                                                            C.c_void_p(d_kp_idx or None), C.c_void_p(d_kp_offsets or None), C.byref(nkp)))
        return nkp.value

    def fetchFragile(self, n):
        """Per-point mask of the last detection: 1 = a split on the point's forest walk was decided within 1e-5."""
        out = np.empty(n, np.uint8)
        self._check(self._L.kpl_fetch_u8(self._h, b"fragile", _ptr(out, C.c_uint8), n))
        return out

    def _compute_compacted(self, xyz, nrm, finite, role):
        keep = np.nonzero(finite)[0]
        sub = np.ascontiguousarray(xyz[keep])
        saved = (self._cloud, self._normals)
        try:
            self._cloud = sub
            self._normals = None if nrm is None else np.ascontiguousarray(nrm[keep])
            kp, idx = self.compute(role=None if role is None else np.ascontiguousarray(role)[keep])
        finally:
            self._cloud, self._normals = saved
        scores = np.full(xyz.shape[0], np.nan, np.float32)
        scores[keep] = self._scores[:len(keep)]
        self._scores = scores
        self._kp_idx = keep[idx].astype(np.int32)
        return kp, self._kp_idx

    def computeForests(self, thresholds=None):
        """kpl_detect_forests: every forest of the set over the input cloud, from one feature pass.  thresholds: None (the
        prediction threshold for every forest) or one per forest.  Returns a list with one (keypoints (n_kp,4) float32,
        indices (n_kp,) int32) per forest -- what compute() returns with only that forest loaded and that threshold --
        and keeps the (K, n) responses for getResponses().  A non-dense cloud is compacted and mapped back as in compute()."""
        if self._cloud is None:
            raise KplError(1, "no input cloud")
        xyz, xs = _vec3(self._cloud, "cloud")
        nrm = ns = None
        if self._normals is not None:
            nrm, ns = _vec3(self._normals, "normals")
            if nrm.shape[0] != xyz.shape[0]:
                raise KplError(3, "normals given, but the number of normals does not match the number of input points")
        K = self.forestCount()
        th = self._thresholds(thresholds)
        self._push()
        finite = None
        scores, kp, kpo = self._detect_forests(xyz, xs, nrm, ns, th, K)
        if scores is None:                            # KPL_E_NONFINITE: a non-dense cloud
            finite = np.nonzero(np.isfinite(xyz[:, :3]).all(axis=1))[0]
            sub = np.ascontiguousarray(xyz[finite])
            subn = None if nrm is None else np.ascontiguousarray(nrm[finite])
            sc, kp, kpo = self._detect_forests(sub, xs, subn, ns, th, K)
            if sc is None:
                self._check(4)
            scores = np.full((K, xyz.shape[0]), np.nan, np.float32)
            scores[:, finite] = sc
        self._responses = scores
        out = []
        for k in range(K):
            idx = kp[kpo[k]:kpo[k + 1]]
            idx = (idx if finite is None else finite[idx]).astype(np.int32)
            pts = np.empty((len(idx), 4), np.float32)
            pts[:, :3] = xyz[idx, :3]
            pts[:, 3] = scores[k, idx]
            out.append((pts, idx))
        return out

    def _detect_forests(self, xyz, xs, nrm, ns, th, K):
        n = xyz.shape[0]
        scores = np.empty((K, n), np.float32)
        kp = np.empty(max(K * n, 1), np.int32)
        kpo = np.empty(K + 1, np.int64)
        rc = self._L.kpl_detect_forests(self._h, _ptr(xyz, C.c_float), xs, _ptr(nrm, C.c_float), ns or 0, n, _ptr(th, C.c_double),
                                        _ptr(scores, C.c_float), _ptr(kp, C.c_int32), _ptr(kpo, C.c_int64))
        if rc == 4:
            return None, None, None
        self._check(rc)
        return scores, kp, kpo

    def getResponses(self):
        """(K, n) responses of the last computeForests()."""
        return self._responses

    def detectForestsDevice(self, d_xyz4, n, d_normals4=0, thresholds=None, d_scores=0, d_kp_idx=0, d_kp_offsets=0):
        """kpl_detect_forests_device: raw device pointers (ints); d_scores K*n floats (or 0), d_kp_idx K*n int32, d_kp_offsets
        K + 1 int64, forest-major.  thresholds: None or one per forest (host).  Returns the keypoint count of all forests."""
        th = self._thresholds(thresholds)
        self._push()
        nkp = C.c_int64(0)
        self._check(self._L.kpl_detect_forests_device(self._h, C.c_void_p(d_xyz4), C.c_void_p(d_normals4 or None), int(n), _ptr(th, C.c_double),
                                                      C.c_void_p(d_scores or None), C.c_void_p(d_kp_idx or None),
                                                      C.c_void_p(d_kp_offsets or None), C.byref(nkp)))
        return nkp.value

    def getKeypointsIndices(self): return self._kp_idx
    def getResponse(self): return self._scores

    def computeNormals(self, cloud):
        xyz, xs = _vec3(cloud, "cloud")
        self._push()
        out = np.empty((xyz.shape[0], 4), np.float32)
        rc = self._L.kpl_normals(self._h, _ptr(xyz, C.c_float), xs, xyz.shape[0], _ptr(out, C.c_float))
        if rc == 4:                                   # non-dense cloud: NaN normals for the NaN points (as PCL)
            finite = np.isfinite(xyz[:, :3]).all(axis=1)
            out = np.full((xyz.shape[0], 4), np.nan, np.float32)
            out[finite] = self.computeNormals(np.ascontiguousarray(xyz[finite]))
            return out
        self._check(rc)
        return out

    def computeNormalsOrganized(self, cloud_hw, smoothing=5.0):
        """kpl_normals_organized: pcl::IntegralImageNormalEstimation(SIMPLE_3D_GRADIENT, smoothing) on a (height, width, >=3)
        organized cloud (NaN = no measurement).  Returns (height*width, 4)."""
        a = np.ascontiguousarray(cloud_hw, np.float32)
        if a.ndim != 3 or a.shape[2] < 3:
            raise ValueError("organized cloud must be (height, width, >=3) float32")
        h, w = a.shape[:2]
        self._push()
        out = np.empty((h * w, 4), np.float32)
        self._check(self._L.kpl_normals_organized(self._h, _ptr(a, C.c_float), a.shape[2] * 4, w, h, float(smoothing), _ptr(out, C.c_float)))
        return out

    def computeOrganized(self, cloud_hw, smoothing=5.0):
        """compute() for an organized cloud without normals, as initCompute does it (hpp:138-145): integral-image normals,
        then the detection over the finite points (NaN points and points without a normal get no score)."""
        a = np.ascontiguousarray(cloud_hw, np.float32)
        nrm = self.computeNormalsOrganized(a, smoothing)
        flat = np.ascontiguousarray(a.reshape(-1, a.shape[2]))
        saved = (self._cloud, self._normals)
        try:
            self._cloud, self._normals = flat, nrm
            return self.compute()
        finally:
            self._cloud, self._normals = saved

    def computeOrganizedBatch(self, frames, smoothing=5.0, normals=None, viewpoints=None):
        """kpl_detect_batch_organized: `frames` is (F, height, width, >=3) float32 (NaN = no measurement).  normals: None
        (integral-image normals of every frame, flipped towards viewpoints[f] -- an (F, 3) array, default the detector's
        viewpoint) or per-pixel normals of the same (F, height, width, >=3) shape.  Returns (scores list, keypoint pixel index
        list), one entry per frame: what computeOrganized() (normals None) or compute() on the flattened frame with
        setNormals (normals given) returns for that frame alone."""
        a, nrm, vp = self._frames(frames, normals, viewpoints)
        nf, h, w, c = a.shape
        self._push()
        n = nf * h * w
        scores = np.empty(n, np.float32)
        kp = np.empty(max(n, 1), np.int32)
        kpo = np.empty(nf + 1, np.int64)
        self._check(self._L.kpl_detect_batch_organized(self._h, _ptr(a, C.c_float), c * 4, _ptr(nrm, C.c_float),
                                                       0 if nrm is None else nrm.shape[3] * 4, w, h, nf, float(smoothing), _ptr(vp, C.c_float),
                                                       _ptr(scores, C.c_float), _ptr(kp, C.c_int32), _ptr(kpo, C.c_int64)))
        return ([scores[f * h * w:(f + 1) * h * w] for f in range(nf)], [kp[kpo[f]:kpo[f + 1]].copy() for f in range(nf)])

    @staticmethod
    def _frames(frames, normals, viewpoints):
        a = np.asarray(frames)
        if a.ndim != 4 or a.shape[3] < 3:
            raise ValueError("frames must be (n_frames, height, width, >=3) float32")
        a = np.ascontiguousarray(a, np.float32)
        nf, h, w, _ = a.shape
        nrm = None
        if normals is not None:
            nrm = np.ascontiguousarray(normals, np.float32)
            if nrm.shape[:3] != (nf, h, w) or nrm.ndim != 4 or nrm.shape[3] < 3:
                raise ValueError("normals must be (n_frames, height, width, >=3) float32")
        vp = None if viewpoints is None else np.ascontiguousarray(viewpoints, np.float32).reshape(nf, 3)
        return a, nrm, vp

    def computeOrganizedBatchForests(self, frames, smoothing=5.0, normals=None, viewpoints=None, thresholds=None):
        """kpl_detect_batch_organized_forests: every forest of the set over a batch of organized frames (arguments as in
        computeOrganizedBatch), from one feature pass.  thresholds: None or one per forest.  Returns out[k][f] = (pixel-order
        scores, frame-local keypoint pixel indices): what computeOrganizedBatch() returns for frame f with only forest k
        loaded and threshold k."""
        th = self._thresholds(thresholds)
        a, nrm, vp = self._frames(frames, normals, viewpoints)
        nf, h, w, c = a.shape
        K, n = self.forestCount(), nf * h * w
        self._push()
        scores = np.empty((max(K, 1), n), np.float32)
        kp = np.empty(max(K * n, 1), np.int32)
        kpo = np.empty(K * nf + 1, np.int64)
        self._check(self._L.kpl_detect_batch_organized_forests(self._h, _ptr(a, C.c_float), c * 4, _ptr(nrm, C.c_float),
                                                               0 if nrm is None else nrm.shape[3] * 4, w, h, nf, float(smoothing),
                                                               _ptr(vp, C.c_float), _ptr(th, C.c_double), _ptr(scores, C.c_float),
                                                               _ptr(kp, C.c_int32), _ptr(kpo, C.c_int64)))
        return [[(scores[k, f * h * w:(f + 1) * h * w], kp[kpo[k * nf + f]:kpo[k * nf + f + 1]].copy()) for f in range(nf)] for k in range(K)]

    def detectOrganizedBatchForestsDevice(self, d_xyz4, width, height, n_frames, smoothing=5.0, d_normals4=0, viewpoints=None, d_scores=0,
                                          d_kp_idx=0, d_kp_offsets=0, thresholds=None):
        """kpl_detect_batch_organized_forests_device: raw device pointers (ints), host viewpoints and thresholds; d_scores
        K*F*W*H floats (or 0), d_kp_idx K*F*W*H int32, d_kp_offsets K*F + 1 int64.  Returns the keypoint count of all forests."""
        th = self._thresholds(thresholds)
        vp = None if viewpoints is None else np.ascontiguousarray(viewpoints, np.float32).reshape(int(n_frames), 3)
        self._push()
        nkp = C.c_int64(0)
        self._check(self._L.kpl_detect_batch_organized_forests_device(self._h, C.c_void_p(d_xyz4), C.c_void_p(d_normals4 or None), int(width),
                                                                      int(height), int(n_frames), float(smoothing), _ptr(vp, C.c_float),
                                                                      _ptr(th, C.c_double), C.c_void_p(d_scores or None),
                                                                      C.c_void_p(d_kp_idx or None), C.c_void_p(d_kp_offsets or None),
                                                                      C.byref(nkp)))
        return nkp.value

    def detectOrganizedBatchDevice(self, d_xyz4, width, height, n_frames, smoothing=5.0, d_normals4=0, viewpoints=None, d_scores=0,
                                   d_kp_idx=0, d_kp_offsets=0):
        """Device-resident organized frames (float4 per pixel): raw device pointers (ints), host viewpoints ((F, 3) or None).
        Returns the total keypoint count."""
        vp = None if viewpoints is None else np.ascontiguousarray(viewpoints, np.float32).reshape(int(n_frames), 3)
        self._push()
        nkp = C.c_int64(0)
        self._check(self._L.kpl_detect_batch_organized_device(self._h, C.c_void_p(d_xyz4), C.c_void_p(d_normals4 or None), int(width), int(height),
                                                              int(n_frames), float(smoothing), _ptr(vp, C.c_float), C.c_void_p(d_scores or None),
                                                              C.c_void_p(d_kp_idx or None), C.c_void_p(d_kp_offsets or None), C.byref(nkp)))
        return nkp.value

    def computePointsForTrainingFeatures(self, indices=None):
        xyz, xs = _vec3(self._cloud, "cloud")
        n = xyz.shape[0]
        nrm = ns = None
        if self._normals is not None:
            nrm, ns = _vec3(self._normals, "normals")
        idx = None if indices is None else np.ascontiguousarray(indices, np.int32)
        m = n if idx is None else len(idx)
        self._push()
        F = self._p.n_annulus * self._p.n_bins
        out = np.empty((m, F), np.float32)
        self._check(self._L.kpl_features(self._h, _ptr(xyz, C.c_float), xs, _ptr(nrm, C.c_float), ns or 0, n, _ptr(idx, C.c_int32), m, _ptr(out, C.c_float)))
        return out

    def radiusStats(self, cloud, radius):
        xyz, xs = _vec3(cloud, "cloud")
        self._push()
        n = xyz.shape[0]
        counts = np.empty(n, np.int32); h = np.empty(n, np.uint64)
        self._check(self._L.kpl_radius_stats(self._h, _ptr(xyz, C.c_float), xs, n, float(radius), _ptr(counts, C.c_int32), _ptr(h, C.c_uint64)))
        return counts, h

    def radiusNeighbors(self, cloud, radius, queries):
        xyz, xs = _vec3(cloud, "cloud")
        self._push()
        q = np.ascontiguousarray(queries, np.int32)
        off = np.empty(len(q) + 1, np.int64)
        self._check(self._L.kpl_radius_neighbors(self._h, _ptr(xyz, C.c_float), xs, xyz.shape[0], float(radius), _ptr(q, C.c_int32), len(q), _ptr(off, C.c_int64), None))
        idx = np.empty(int(off[-1]), np.int32)
        self._check(self._L.kpl_radius_neighbors(self._h, _ptr(xyz, C.c_float), xs, xyz.shape[0], float(radius), _ptr(q, C.c_int32), len(q), _ptr(off, C.c_int64), _ptr(idx, C.c_int32)))
        return off, idx

    def detectDevice(self, d_xyz4, n, d_normals4=0, d_role=0, d_scores=0, d_kp_idx=0):
        """Device-resident call: raw device pointers (ints).  Returns n_kp."""
        self._push()
        nkp = C.c_int64(0)
        self._check(self._L.kpl_detect_device(self._h, C.c_void_p(d_xyz4), C.c_void_p(d_normals4 or None), C.c_void_p(d_role or None), int(n),
                                              C.c_void_p(d_scores or None), C.c_void_p(d_kp_idx), C.byref(nkp)))
        return nkp.value

    def nearest(self, cloud, queries):
        """Index (and squared distance) of the nearest cloud point of every query point (TrainDetector's 1-NN snap)."""
        xyz, xs = _vec3(cloud, "cloud")
        q, qs = _vec3(queries, "queries")
        self._push()
        idx = np.empty(max(1, q.shape[0]), np.int32); d2 = np.empty(max(1, q.shape[0]), np.float32)
        self._check(self._L.kpl_nearest(self._h, _ptr(xyz, C.c_float), xs, xyz.shape[0], _ptr(q, C.c_float), qs, q.shape[0],
                                        _ptr(idx, C.c_int32), _ptr(d2, C.c_float)))
        return idx[:q.shape[0]].copy(), d2[:q.shape[0]].copy()

    def uniformSample(self, cloud, leaf, centre=False):
        """pcl::UniformSampling(leaf) on the device: ascending indices of the surviving points.  centre=False is PCL 1.8.0's
        literal rule (closest to the voxel index vector), True the voxel centre."""
        xyz, xs = _vec3(cloud, "cloud")
        self._p.uniform_sampling_centre = int(bool(centre))
        self._push()
        idx = np.empty(max(1, xyz.shape[0]), np.int32)
        m = C.c_int64(0)
        self._check(self._L.kpl_uniform_sample(self._h, _ptr(xyz, C.c_float), xs, xyz.shape[0], float(leaf), _ptr(idx, C.c_int32), C.byref(m)))
        return idx[:m.value].copy()

    def keepIntermediates(self, on=True):
        """Materialise the feature rows in compute()/detectDevice() so that fetch("features") works."""
        self._check(self._L.kpl_set_keep_intermediates(self._h, int(bool(on))))

    def fetch(self, what, n, width):
        out = np.empty((n, width), np.float32)
        self._check(self._L.kpl_fetch(self._h, what.encode(), _ptr(out, C.c_float), out.size))
        return out

    def timings(self):
        t = KplTimings()
        self._check(self._L.kpl_get_timings(self._h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in KplTimings._fields_}

    def stats(self):
        s = KplStats()
        self._check(self._L.kpl_get_stats(self._h, C.byref(s)))
        d = {k: getattr(s, k) for k, _ in KplStats._fields_}
        d["grid_dims"] = list(s.grid_dims); d["grid_origin"] = list(s.grid_origin)
        return d
