"""Issue-slot model of the feature kernel's candidate stream (experiments tool, CPU only).

Takes a dense crop of the bench scene, forms the kernel's warps (32 consecutive queries of the Hilbert order over
sub-cells), and replays the tile loop for a sample of interior warps with four candidate streams:
  cells    : rows culled with whole cells, tiles of 32 consecutive sorted positions (the kernel before the filter)
  rowexact : rows culled with the exact query positions, no per-point filter
  box      : every candidate tested against the group's position box + r, survivors compacted into full tiles
             (features.cu)
  ideal    : a candidate kept iff some lane accepts it (upper bound of any filter)
It prints tiles per warp, acceptance (pairs / candidate tests), lane efficiency of the vote phase and issue slots
relative to `cells`.  Instruction model (warp instructions, from the SASS of the tile loop): 6.75 per candidate in
phase 1 (8 at a time), 140 per bit-walk iteration, 122 per in-order iteration (16 of them in tiles whose largest mask
reaches DENSE_TILE), 45 per tile, 12 per raw batch of 32 for the filter and compaction.

    python tools/sim_candidate_filter.py [crop points] [sampled warps]
"""
import sys

import numpy as np

sys.path.insert(0, ".")
sys.path.insert(0, "tools")
from keypoint_learning_b200 import synth  # noqa: E402
from sim_query_order import hilbert3  # noqa: E402

R = 20.0
CPR = 4
CELL = R * (1 + 2.0 ** -20) / CPR
R2 = np.float32(R * R)
RCULL2 = R * R * (1 + 1e-5)
DENSE_TILE = 29
P1, VOTE, DENSE_IT, TILE, FILT = 6.75, 140.0, 122.0, 45.0, 12.0


def main():
    n_crop = int(sys.argv[1]) if len(sys.argv) > 1 else 600_000
    nsample = int(sys.argv[2]) if len(sys.argv) > 2 else 120
    xyz, _ = synth.scene_closed_surfaces()
    xyz = synth.cube_crop(xyz, n_crop).astype(np.float32)
    n = len(xyz)
    lo = xyz.min(0).astype(np.float64)
    c = np.floor((xyz.astype(np.float64) - lo) / CELL).astype(np.int64)
    dim = c.max(0) + 1
    key = (c[:, 2] * dim[1] + c[:, 1]) * dim[0] + c[:, 0]
    order = np.argsort(key, kind="stable")
    sp, sk, sc = xyz[order], key[order], c[order]
    cell_start = np.searchsorted(sk, np.arange(int(dim.prod()) + 1))
    interior = np.all((sp > xyz.min(0) + 2 * R) & (sp < xyz.max(0) - 2 * R), axis=1)
    f = np.floor((sp.astype(np.float64) - lo) / (CELL / 4)).astype(np.int64)
    perm = np.argsort(hilbert3(f[:, 0], f[:, 1], f[:, 2], int(np.ceil(np.log2(f.max() + 1)))), kind="stable")
    warps = [perm[i:i + 32] for i in range(0, n - 31, 32)]
    ok = [w for w in warps if interior[w].all() and np.all(sc[w].max(0) - sc[w].min(0) <= 3)]   # one group per warp
    pick = np.random.default_rng(0).choice(len(ok), size=min(nsample, len(ok)), replace=False)
    print(f"n={n} dim={dim} sampled warps={len(pick)}")

    def rows_cells(qs):
        cc = sc[qs]
        (x0, y0, z0), (x1, y1, z1) = cc.min(0), cc.max(0)
        out = []
        for zz in range(max(z0 - CPR, 0), min(z1 + CPR, dim[2] - 1) + 1):
            for yy in range(max(y0 - CPR, 0), min(y1 + CPR, dim[1] - 1) + 1):
                gy, gz = max(max(y0 - yy, yy - y1) - 1, 0), max(max(z0 - zz, zz - z1) - 1, 0)
                gap2 = (gy * gy + gz * gz) * CELL * CELL
                if gap2 < RCULL2:
                    rx = min(int(np.sqrt(RCULL2 - gap2) / CELL) + 1, CPR)
                    base = (zz * dim[1] + yy) * dim[0]
                    s, e = cell_start[base + max(x0 - rx, 0)], cell_start[base + min(x1 + rx, dim[0] - 1) + 1]
                    if e > s:
                        out.append((s, e))
        return out

    def rows_exact(qs):
        p = sp[qs].astype(np.float64) - lo
        pmn, pmx = p.min(0), p.max(0)
        cc = sc[qs]
        (x0, y0, z0), (x1, y1, z1) = cc.min(0), cc.max(0)
        out = []
        for zz in range(max(z0 - CPR, 0), min(z1 + CPR, dim[2] - 1) + 1):
            gz = max(0.0, pmn[2] - (zz + 1) * CELL, zz * CELL - pmx[2])
            for yy in range(max(y0 - CPR, 0), min(y1 + CPR, dim[1] - 1) + 1):
                gy = max(0.0, pmn[1] - (yy + 1) * CELL, yy * CELL - pmx[1])
                if gy * gy + gz * gz < RCULL2:
                    rx = np.sqrt(RCULL2 - gy * gy - gz * gz)
                    base = (zz * dim[1] + yy) * dim[0]
                    s = cell_start[base + max(int(np.floor((pmn[0] - rx) / CELL)), 0)]
                    e = cell_start[base + min(int(np.floor((pmx[0] + rx) / CELL)), dim[0] - 1) + 1]
                    if e > s:
                        out.append((s, e))
        return out

    def cost(qs, tiles):
        qp = sp[qs]
        t = np.zeros(5)   # candidates, pairs, vote iterations (bit walk), issue slots, tiles
        for idx in tiles:
            d = qp[:, None, :] - sp[idx][None, :, :]
            m = ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]) < R2
            m &= qs[:, None] != idx[None, :]
            pc = m.sum(1)
            mx = int(pc.max())
            dense = mx >= DENSE_TILE
            it = 16 if dense else (mx + 1) // 2
            t += [len(idx), pc.sum(), it, P1 * 8 * ((len(idx) + 7) // 8) + TILE + (DENSE_IT * 16 if dense else VOTE * it), 1]
        return t

    names = ("cells", "rowexact", "box", "ideal")
    tot = {k: np.zeros(5) for k in names}
    for i in pick:
        qs = np.sort(ok[i])
        rr = rows_cells(qs)
        tot["cells"] += cost(qs, [np.arange(tb, min(tb + 32, e)) for s, e in rr for tb in range(s, e, 32)])
        tot["rowexact"] += cost(qs, [np.arange(tb, min(tb + 32, e)) for s, e in rows_exact(qs) for tb in range(s, e, 32)])
        allc = np.concatenate([np.arange(s, e) for s, e in rr])
        raw_batches = sum((e - s + 31) // 32 for s, e in rr)
        qp = sp[qs].astype(np.float64)
        cpos = sp[allc].astype(np.float64)
        g = np.maximum(np.maximum(qp.min(0) - cpos, cpos - qp.max(0)), 0.0)
        for name, keep in (("box", allc[(g * g).sum(1) < RCULL2]),
                           ("ideal", allc[(((qp[:, None, :] - cpos[None, :, :]) ** 2).sum(2) < R * R).any(0)])):
            t = cost(qs, [keep[j:j + 32] for j in range(0, len(keep), 32)])
            t[3] += FILT * raw_batches
            tot[name] += t
    print("| candidate stream | tiles / warp | acceptance | vote lane eff. | issue slots vs cells |")
    print("|---|---|---|---|---|")
    for k in names:
        cand, pairs, it, slots, tiles = tot[k]
        print(f"| {k} | {tiles / len(pick):.1f} | {pairs / (cand * 32):.3f} | {pairs / (it * 64):.3f} | {slots / tot['cells'][3]:.3f} |")


if __name__ == "__main__":
    main()
