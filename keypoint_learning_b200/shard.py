"""Slab sharding of ONE large cloud over the GPUs of a node (BASELINE.json configs[3]): thin ctypes caller of the
`kpl_slab_*` / `kpl_shard_*` entry points of include/kpl.h.  Planning, strip packing, the NCCL exchanges, role
handling and the keypoint gather all live in csrc/shard.cu; nothing on the step path runs in Python or torch.

The reference is a single process (src/main_test_detector.cpp:123-187); this is what a multi-GPU driver of that loop
uses.  Schedule per detection (see include/kpl.h):
  1. position strips (halo = reach(radiusFeatures) + normal_support_cells columns) to / from the two neighbours
  2. grid with the GLOBAL origin, normals for everything held (estimated, or the caller's: their strips travel with the
     position strips), scores for the OWNED points only
  3. score strips (4 B / point) to / from the two neighbours
  4. threshold + NMS for the owned points, global keypoint list gathered and sorted on rank 0.

`HostSlab` is the same schedule written with numpy, the transport and the detection stage left to the caller: the CPU
tests run it over a `gloo` process group with the oracle in the middle, which pins the schedule itself (what is sent,
what is scored where, what NMS sees) independently of CUDA and NCCL.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi


@dataclass
class SlabPlan:
    origin: np.ndarray      # 3 doubles, global grid origin
    cell: float
    dims: np.ndarray        # 3 int32, global grid dims
    cuts: np.ndarray        # world+1 cell-x cut positions
    halo: int               # halo width in cells
    reach_nms: int
    reach_feat: int
    normal_support_cells: int
    cost: np.ndarray        # modelled per-rank cost
    c_plan: capi.KplSlabPlan

    @property
    def world(self):
        return len(self.cuts) - 1


def _xyz_arg(xyz):
    a = np.ascontiguousarray(xyz, np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("xyz must be (n, >=3) float32")
    return a, a.shape[1] * 4


def plan_slabs(xyz, r_feat, r_nms, cpr, world, normal_support_cells=1) -> SlabPlan:
    """kpl_slab_plan_make (host only, no GPU): balanced x cuts at cell-column boundaries of the grid of the whole cloud."""
    L = capi.load_library()
    p = capi.KplParams()
    L.kpl_params_default(C.byref(p))
    p.radius_features = float(r_feat); p.radius_nms = float(r_nms); p.cells_per_radius = int(cpr)
    a, stride = _xyz_arg(xyz)
    cp = capi.KplSlabPlan()
    rc = L.kpl_slab_plan_make(a.ctypes.data_as(C.POINTER(C.c_float)), stride, len(a), C.byref(p), int(world), int(normal_support_cells), C.byref(cp))
    if rc == 1:
        raise ValueError("cannot cut this cloud into %d slabs of at least one halo width (kpl_slab_plan_make -> KPL_E_INVALID)" % world)
    if rc != 0:
        raise capi.KplError(rc, "kpl_slab_plan_make failed")
    return SlabPlan(np.array(cp.origin[:], np.float64), float(cp.cell), np.array(cp.dims[:], np.int32), np.array(cp.cuts[:world + 1], np.int64),
                    int(cp.halo), int(cp.reach_nms), int(cp.reach_feat), int(cp.normal_support_cells), np.array(cp.cost[:world], np.float64), cp)


def partition(plan: SlabPlan, xyz, rank) -> np.ndarray:
    """kpl_slab_partition: ascending global indices of the points `rank` owns."""
    L = capi.load_library()
    a, stride = _xyz_arg(xyz)
    idx = np.empty(len(a), np.int32)
    m = C.c_int64(0)
    rc = L.kpl_slab_partition(C.byref(plan.c_plan), a.ctypes.data_as(C.POINTER(C.c_float)), stride, len(a), int(rank),
                              idx.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(m))
    if rc != 0:
        raise capi.KplError(rc, "kpl_slab_partition failed")
    return idx[:m.value].copy()


def cell_coords(xyz, origin, cell, axis=0):
    return np.floor((np.asarray(xyz)[:, axis].astype(np.float64) - origin[axis]) / cell).astype(np.int64)


def nccl_unique_id() -> bytes:
    L = capi.load_library()
    buf = C.create_string_buffer(128)
    rc = L.kpl_nccl_unique_id(buf)
    if rc != 0:
        raise capi.KplError(rc, "kpl_nccl_unique_id failed (is libnccl.so.2 loadable?)")
    return buf.raw


class SlabJob:
    """One rank of a sharded detection job on a GPU.  `det` is this rank's KeypointLearningDetector (forest and parameters
    set); `nccl_id` the 128-byte id shared by all ranks (None: a rank of an in-process group, see detect_group).
    `normals`: None (estimated on the devices) or the caller's (n, >=3) normals of the WHOLE cloud
    (kpl_shard_set_slab_normals; plan with plan_slabs(..., normal_support_cells=0)).  Every rank must choose alike."""

    def __init__(self, det, xyz, plan: SlabPlan, rank: int, nccl_id: bytes | None, normals=None):
        self._L = capi.load_library()
        self.det, self.plan, self.rank, self.world = det, plan, int(rank), plan.world
        self.normals = normals
        det._push()
        self._h = C.c_void_p()
        idbuf = C.create_string_buffer(nccl_id, 128) if nccl_id is not None else None
        self._check(self._L.kpl_shard_create(det._h, C.byref(plan.c_plan), self.rank, idbuf, C.byref(self._h)))
        self._set_slab(xyz)

    def replan(self, xyz, plan: SlabPlan):
        """kpl_shard_set_plan + kpl_shard_set_slab(_normals): a new plan for the same communicator (e.g. a wider k-NN support
        after KPL_E_HALO).  The normals given to the constructor are kept."""
        self.plan = plan
        self._check(self._L.kpl_shard_set_plan(self._h, C.byref(plan.c_plan)))
        self._set_slab(xyz)

    def _set_slab(self, xyz):
        plan, rank = self.plan, self.rank
        self.gidx = partition(plan, xyz, rank)
        a = np.asarray(xyz)
        own = np.ones((len(self.gidx), 4), np.float32)
        own[:, :3] = a[self.gidx, :3]
        self.host_xyz4 = own                       # callers may replace this by a pinned copy (same contents)
        self.n_owned, self.n_total = len(self.gidx), len(a)
        f32p, gp = C.POINTER(C.c_float), self.gidx.ctypes.data_as(C.POINTER(C.c_int32))
        if self.normals is None:
            self._check(self._L.kpl_shard_set_slab(self._h, own.ctypes.data_as(f32p), 16, gp, len(self.gidx)))
            return
        nrm = self._owned_normals(self.normals)
        self._check(self._L.kpl_shard_set_slab_normals(self._h, own.ctypes.data_as(f32p), 16, nrm.ctypes.data_as(f32p), nrm.shape[1] * 4,
                                                       gp, len(self.gidx)))

    def _owned_normals(self, normals):
        a = np.asarray(normals)
        if a.ndim != 2 or a.shape[1] < 3 or len(a) != self.n_total:
            raise ValueError("normals must be (n, >=3) for the whole cloud of %d points" % self.n_total)
        return np.ascontiguousarray(a[self.gidx], np.float32)

    def _check(self, rc):
        if rc != 0:
            raise capi.KplError(rc, (self._L.kpl_last_error(self.det._h) or b"").decode())

    def upload(self, host_xyz4=None):
        a = self.host_xyz4 if host_xyz4 is None else host_xyz4
        self._check(self._L.kpl_shard_upload(self._h, a.ctypes.data_as(C.POINTER(C.c_float)), a.shape[1] * 4))

    def upload_normals(self, normals):
        """kpl_shard_upload_normals: new normals of the WHOLE cloud, (n, >=3), for the same partition; replan keeps them."""
        nrm = self._owned_normals(normals)
        self._check(self._L.kpl_shard_upload_normals(self._h, nrm.ctypes.data_as(C.POINTER(C.c_float)), nrm.shape[1] * 4))
        self.normals = normals

    def detect(self, scores_out=None, kp_out=None):
        """kpl_shard_detect.  Returns (global keypoint count, ascending global keypoint indices on rank 0 / None)."""
        self.det._push()
        n = C.c_int64(0)
        kp = kp_out
        if self.rank == 0 and kp is None:
            kp = np.empty(self.n_total, np.int32)
        self._check(self._L.kpl_shard_detect(self._h, None if scores_out is None else scores_out.ctypes.data_as(C.POINTER(C.c_float)),
                                             None if kp is None else kp.ctypes.data_as(C.POINTER(C.c_int32)),
                                             0 if kp is None else kp.size, C.byref(n)))
        return n.value, (kp[:n.value] if self.rank == 0 else None)

    def info(self):
        i = capi.KplShardInfo()
        self._check(self._L.kpl_shard_get_info(self._h, C.byref(i)))
        d = {k: getattr(i, k) for k, _ in capi.KplShardInfo._fields_}
        d["local_dims"] = list(i.local_dims); d["local_offset"] = list(i.local_offset)
        return d

    def device_scores_ptr(self):
        return self._L.kpl_shard_device_scores(self._h)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.kpl_shard_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _widening(detect, jobs, xyz, r_feat, r_nms, cpr, max_support):
    """detect(); on KPL_E_HALO (a k-NN normal that matters was clipped by a slab face -- every rank reports it) re-plan
    `jobs` with twice the k-NN support (1 after 0: a support that stays 0 would clip on every retry) and try again.  The support is
    thereby derived from the data."""
    while True:
        try:
            return detect()
        except capi.KplError as e:
            ns = max(jobs[0].plan.normal_support_cells * 2, 1)
            if e.code != capi.KPL_E_HALO or ns > max_support:
                raise
            plan = plan_slabs(xyz, r_feat, r_nms, cpr, jobs[0].world, ns)
            for j in jobs:
                j.replan(xyz, plan)


def detect_widening(job, xyz, r_feat, r_nms, cpr, max_support=64, **kw):
    """job.detect() with the widening loop of _widening (every rank of an NCCL job runs it in lockstep)."""
    return _widening(lambda: job.detect(**kw), [job], xyz, r_feat, r_nms, cpr, max_support)


def detect_group_widening(jobs, xyz, r_feat, r_nms, cpr, max_support=64, want_scores=True):
    """detect_group() with the widening loop of _widening for an in-process group."""
    return _widening(lambda: detect_group(jobs, want_scores), jobs, xyz, r_feat, r_nms, cpr, max_support)


def detect_group(jobs, want_scores=True):
    """kpl_shard_detect_group: all ranks of an in-process group (created with nccl_id=None) from this thread.
    Returns (global keypoint indices, [owned scores per rank])."""
    L = capi.load_library()
    world = len(jobs)
    for j in jobs:
        j.det._push()
    hs = (C.c_void_p * world)(*[j._h for j in jobs])
    scores = [np.empty(j.n_owned, np.float32) for j in jobs] if want_scores else None
    f32p = C.POINTER(C.c_float)
    sc_ptrs = (f32p * world)(*[s.ctypes.data_as(f32p) for s in scores]) if want_scores else None
    kp = np.empty(jobs[0].n_total, np.int32)
    n = C.c_int64(0)
    rc = L.kpl_shard_detect_group(hs, world, sc_ptrs, kp.ctypes.data_as(C.POINTER(C.c_int32)), kp.size, C.byref(n))
    if rc != 0:
        raise capi.KplError(rc, (L.kpl_last_error(jobs[0].det._h) or b"").decode())
    return kp[:n.value].copy(), scores


# ---------------------------------------------------------------------------------------------------------------
# The schedule in numpy (transport and detection stage supplied by the caller): CPU tests only
# ---------------------------------------------------------------------------------------------------------------
class HostSlab:
    """What rank `rank` of `plan` sends, holds and decides -- the host mirror of csrc/shard.cu, used by
    tests/test_shard_cpu.py over a gloo process group with the CPU oracle as the detection stage."""

    def __init__(self, xyz, plan: SlabPlan, rank: int):
        self.plan, self.rank, self.world = plan, rank, plan.world
        self.gidx = partition(plan, xyz, rank).astype(np.int64)
        self.own = np.ascontiguousarray(np.asarray(xyz, np.float32)[self.gidx, :3])
        cx = cell_coords(self.own, plan.origin, plan.cell, 0)
        c0, c1, H = int(plan.cuts[rank]), int(plan.cuts[rank + 1]), plan.halo
        self.sel_l = np.nonzero(cx < c0 + H)[0] if rank > 0 else np.zeros(0, np.int64)
        self.sel_r = np.nonzero(cx >= c1 - H)[0] if rank < self.world - 1 else np.zeros(0, np.int64)
        self.x0 = max(c0 - H, 0) if rank > 0 else 0
        self.x1 = min(c1 + H, int(plan.dims[0])) if rank < self.world - 1 else int(plan.dims[0])

    def position_strips(self):
        """(to the left neighbour, to the right neighbour): float32 [m, 3]"""
        return self.own[self.sel_l], self.own[self.sel_r]

    def assemble(self, from_left, from_right):
        """[left halo | owned | right halo] and the roles; from_* are the neighbours' strips (None at the ends)."""
        parts = [p for p in (from_left, self.own, from_right) if p is not None and len(p)]
        self.n_l = 0 if from_left is None else len(from_left)
        self.n_r = 0 if from_right is None else len(from_right)
        self.local = np.ascontiguousarray(np.concatenate(parts))
        self.role = np.zeros(len(self.local), np.uint8)
        self.role[self.n_l:self.n_l + len(self.own)] = capi.ROLE_OWNED
        return self.local, self.role

    def score_strips(self, scores_local):
        """(to the left neighbour, to the right neighbour): the owned values of the strip points of a local array"""
        own = scores_local[self.n_l:self.n_l + len(self.own)]
        return own[self.sel_l], own[self.sel_r]

    def merge_scores(self, scores_local, from_left, from_right):
        """the local array with its halo parts replaced by what the neighbours sent"""
        out = scores_local.copy()
        if self.n_l:
            out[:self.n_l] = from_left
        if self.n_r:
            out[self.n_l + len(self.own):] = from_right
        return out

    # draws-remove NMS: the state rounds of csrc/shard.cu (states 0 not a keypoint, 1 keypoint, 2 undecided, 3 skipped)
    state_strips = score_strips
    merge_states = merge_scores

    def gidx_strips(self):
        """global indices of the strip points (exchanged once per slab)"""
        return self.gidx[self.sel_l], self.gidx[self.sel_r]

    def set_local_gidx(self, from_left, from_right):
        parts = [p for p in (from_left, self.gidx, from_right) if p is not None and len(p)]
        self.local_gidx = np.concatenate(parts).astype(np.int64)
        return self.local_gidx

    def draws_classify(self, scores_local, nb_off, nb_idx, th, draws_thr):
        """States of the owned points (halo points 0, their owners decide them) and the close draws the rounds read.
        nb_off / nb_idx: the r_nms neighbour lists (self included) of every local point, CSR."""
        p = self.local.astype(np.float32)
        sc = np.asarray(scores_local, np.float32)
        n = len(p)
        src = np.repeat(np.arange(n), np.diff(nb_off))
        dst = np.asarray(nb_idx, np.int64)
        owned = np.zeros(n, bool)
        owned[self.n_l:self.n_l + len(self.own)] = True
        above = owned & np.isfinite(sc) & ~(sc.astype(np.float64) < th)
        beaten = np.zeros(n, bool)
        np.logical_or.at(beaten, src, sc[src] < sc[dst])
        draw = (sc[src] == sc[dst]) & (src != dst)
        d = p[src] - p[dst]
        dist = np.sqrt(d[:, 0] * d[:, 0] + (d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]))      # Eigen's norm(): a0 + (a1 + a2)
        close = draw & (dist < np.float32(draws_thr))
        has_draw = np.zeros(n, bool); np.logical_or.at(has_draw, src, draw)
        has_close = np.zeros(n, bool); np.logical_or.at(has_close, src, close)
        state = np.zeros(n, np.uint8)
        is_max = above & ~beaten
        state[is_max & ~has_draw] = 1
        state[is_max & has_draw & has_close] = 2
        self._close = (src[close], dst[close])
        return state

    def draws_round(self, state):
        """One resolution round of the owned undecided candidates on the states held now (halo: the owners' last
        decisions).  Returns (new states, owned candidates still undecided)."""
        i, j = self._close
        lower = self.local_gidx[j] < self.local_gidx[i]
        i, j = i[lower], j[lower]
        n = len(state)
        active = np.zeros(n, bool); np.logical_or.at(active, i, state[j] == 1)
        pending = np.zeros(n, bool); np.logical_or.at(pending, i, state[j] == 2)
        undecided = state == 2
        undecided[:self.n_l] = False
        undecided[self.n_l + len(self.own):] = False
        out = state.copy()
        out[undecided & active] = 3
        out[undecided & ~active & ~pending] = 1
        still = undecided & ~active & pending
        return out, int(still.sum())

    def draws_keypoints(self, state):
        """ascending global indices of the owned keypoints"""
        return self.gidx[np.nonzero(state[self.n_l:self.n_l + len(self.own)] == 1)[0]]

    def owned_keypoints(self, kp_local):
        """local keypoint indices (over the assembled cloud) -> ascending global indices of those this rank owns"""
        kp_local = np.asarray(kp_local, np.int64)
        mine = kp_local[(kp_local >= self.n_l) & (kp_local < self.n_l + len(self.own))]
        return self.gidx[mine - self.n_l]
