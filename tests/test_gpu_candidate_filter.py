"""The feature kernel stages only the candidates that lie within the radius of its query group's position box and
compacts them into full tiles (features.cu).  These clouds put neighbours at r * (1 +- a few ulp) from the points that
span such boxes, along the axes and the diagonals, so a filter that drops one real neighbour or reorders the survivors
changes a histogram; the histograms must stay bit-identical to the oracle's canonical order."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R = 20.0
A, B = 5, 10


def same_bits(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def flann_d2(p, c):
    """the radius-membership expression of the kernel and the oracle, in float32: ((dx*dx) + dy*dy) + dz*dz"""
    d = (p.astype(np.float32) - c.astype(np.float32)).astype(np.float32)
    return ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]).astype(np.float32) + d[..., 2] * d[..., 2]).astype(np.float32)


def directions():
    d = np.array([(x, y, z) for x in (-1, 0, 1) for y in (-1, 0, 1) for z in (-1, 0, 1) if (x, y, z) != (0, 0, 0)], np.float64)
    return d / np.linalg.norm(d, axis=1, keepdims=True)                   # 6 axes, 12 face and 8 body diagonals


def clusters(rng):
    """compact groups of query points, 200 mm apart: one point, a pair, a group inside one cell, groups spanning 2 and
    3 cells per axis, a 4 x 4 x 2 lattice (one warp), and a patch around a non-trivial offset (larger ulps)"""
    out = []
    out.append(np.zeros((1, 3)))
    out.append(np.array([[0.0, 0.0, 0.0], [1.3, -0.7, 0.4]]))
    out.append(rng.uniform(0.2, 4.5, (6, 3)))
    out.append(rng.uniform(0.0, 9.5, (10, 3)))
    out.append(np.stack([np.linspace(0.0, 13.0, 12)] * 3, axis=1) + rng.uniform(-0.3, 0.3, (12, 3)))
    g = np.stack(np.meshgrid(np.arange(4), np.arange(4), np.arange(2), indexing="ij"), -1).reshape(-1, 3) * 1.5
    out.append(g)
    out.append(rng.uniform(0.0, 7.0, (8, 3)) + 1000.0)
    return [c + np.array([200.0 * i, 37.0 * (i % 3), -55.0 * (i % 2)]) for i, c in enumerate(out)]


def build_cloud(seed=0):
    rng = np.random.default_rng(seed)
    dirs = directions()
    eps = np.array([-3, -2, -1, 0, 1, 2, 3], np.float64) * 2.0 ** -23
    parts, pairs = [], []
    for c in clusters(rng):
        c = c.astype(np.float32).astype(np.float64)
        parts.append(c)
        # probes around every point of the group (the box-spanning ones are the tight cases), at r (1 + k ulp)
        probes = (c[:, None, None, :] + dirs[None, :, None, :] * (R * (1.0 + eps))[None, None, :, None]).reshape(-1, 3)
        parts.append(probes)
        pairs.append((c.astype(np.float32), probes.astype(np.float32)))
    xyz = np.concatenate(parts).astype(np.float32)
    # exact duplicates of group points and of probes: d2 == 0 neighbours other than the query itself
    dup = rng.choice(len(xyz), 400, replace=False)
    xyz = np.ascontiguousarray(np.concatenate([xyz, xyz[dup]]))
    xyz = np.ascontiguousarray(xyz[rng.permutation(len(xyz))])
    nrm = rng.normal(size=(len(xyz), 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    nrm = np.concatenate([nrm, np.zeros((len(xyz), 1))], axis=1).astype(np.float32)
    nrm[rng.choice(len(xyz), len(xyz) // 9, replace=False), :3] = np.nan      # neighbours (and queries) without a normal
    return xyz, nrm, pairs


def test_probes_straddle_the_radius():
    """the construction itself (CPU): FLANN d2 of group points and probes falls on both sides of r2 within a few ulp"""
    _, _, pairs = build_cloud()
    r2 = np.float32(R * R)
    d2 = np.concatenate([flann_d2(c[:, None, :], p[None, :, :]).ravel() for c, p in pairs])
    near = np.abs(d2.astype(np.float64) / float(r2) - 1.0) < 1e-6
    assert np.count_nonzero(near & (d2 < r2)) > 100 and np.count_nonzero(near & (d2 >= r2)) > 100


@pytest.fixture(scope="module")
def cloud():
    return build_cloud()


@pytest.mark.parametrize("cpr", [4, 2, 7])
def test_filtered_candidates_whole_cloud(kpl, oracle, cloud, cpr):
    xyz, nrm, _ = cloud
    d = kpl.KeypointLearningDetector()
    d.setNAnnulus(A); d.setNBins(B); d.setRadiusSearch(R); d.setCellsPerRadius(cpr)
    d.setInputCloud(xyz); d.setNormals(nrm)
    f_gpu = d.computePointsForTrainingFeatures()
    st = d.stats()
    d.close()
    f_cpu = oracle.features(xyz, nrm, R, A, B, order=1, cpr=cpr)
    assert same_bits(f_gpu, f_cpu)
    assert np.count_nonzero(f_cpu) > 0
    # every point is a query, scored iff its normal is finite; a neighbour votes iff its normal is finite: each unordered
    # pair of such points within the radius is found twice
    assert st["feature_pairs"] == 2 * count_pairs(xyz, np.isfinite(nrm[:, :3]).all(1))


def count_pairs(xyz, ok):
    """unordered pairs (i, j), i != j, both `ok`, with the FLANN d2 in float32 below r2"""
    from scipy.spatial import cKDTree
    p = cKDTree(xyz.astype(np.float64)).query_pairs(R * 1.001, output_type="ndarray")
    p = p[ok[p[:, 0]] & ok[p[:, 1]]]
    return int(np.count_nonzero(flann_d2(xyz[p[:, 0]], xyz[p[:, 1]]) < np.float32(R * R)))


def test_filtered_candidates_scattered_subset(kpl, oracle, cloud):
    """an index subset: 32 consecutive list entries per warp, scattered over all the groups (several groups a warp)"""
    xyz, nrm, _ = cloud
    sub = np.sort(np.random.default_rng(3).choice(len(xyz), 1500, replace=False)).astype(np.int32)
    d = kpl.KeypointLearningDetector()
    d.setNAnnulus(A); d.setNBins(B); d.setRadiusSearch(R)
    d.setInputCloud(xyz); d.setNormals(nrm)
    f_gpu = d.computePointsForTrainingFeatures(sub)
    d.close()
    assert same_bits(f_gpu, oracle.features(xyz, nrm, R, A, B, order=1, qidx=sub))


def one_warp_patch(seed=1):
    """A 4 x 4 x 2 lattice of 32 points (1.5 mm pitch): as the whole query list it is exactly one warp and one group, whose
    box is the lattice's.  Probes at r (1 + k 2^-23) leave every box-spanning point outwards, along the axes from the
    extreme faces, along the face and body diagonals from the edges and corners; a dense background fills the reach, so
    that survivors overflow the tile and the raw cursor is rewound."""
    rng = np.random.default_rng(seed)
    lat = np.stack(np.meshgrid(np.arange(4), np.arange(4), np.arange(2), indexing="ij"), -1).reshape(-1, 3) * 1.5 + 31.0
    lat = lat.astype(np.float32).astype(np.float64)
    lo, hi = lat.min(0), lat.max(0)
    eps = np.arange(-4, 5, dtype=np.float64) * 2.0 ** -23
    probes = []
    for p in lat:
        for d in directions():
            if all((d[i] > 0 and p[i] == hi[i]) or (d[i] < 0 and p[i] == lo[i]) or d[i] == 0 for i in range(3)):
                probes.append(p[None, :] + d[None, :] * (R * (1.0 + eps))[:, None])
    probes = np.concatenate(probes)
    background = rng.uniform(lo - 1.1 * R, hi + 1.1 * R, (6000, 3))
    xyz = np.concatenate([lat, probes, background, probes[::7], background[::11]]).astype(np.float32)   # with duplicates
    nrm = rng.normal(size=(len(xyz), 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    nrm = np.concatenate([nrm, np.zeros((len(xyz), 1))], axis=1).astype(np.float32)
    bad = rng.choice(np.arange(32, len(xyz)), len(xyz) // 9, replace=False)
    nrm[bad, :3] = np.nan
    return xyz, nrm, np.arange(32, dtype=np.int32)


def test_one_warp_patch_box_edges(kpl, oracle):
    xyz, nrm, sub = one_warp_patch()
    d = kpl.KeypointLearningDetector()
    d.setNAnnulus(A); d.setNBins(B); d.setRadiusSearch(R)
    d.setInputCloud(xyz); d.setNormals(nrm)
    f_gpu = d.computePointsForTrainingFeatures(sub)
    st = d.stats()
    d.close()
    assert same_bits(f_gpu, oracle.features(xyz, nrm, R, A, B, order=1, qidx=sub))
    # the staged candidates are exactly those of the filter (float32, the kernel's expression) with a finite normal
    lat = xyz[:32]
    lo, hi = lat.min(0), lat.max(0)
    g = np.maximum(np.maximum(lo - xyz, xyz - hi), np.float32(0))
    s2 = (g[:, 0] * g[:, 0] + g[:, 1] * g[:, 1]) + g[:, 2] * g[:, 2]
    finite = np.isfinite(nrm[:, :3]).all(1)
    staged = np.count_nonzero(finite & (s2 < np.float32(R * R * (1.0 + 1e-5))))
    assert staged > 20 * 32                                  # many raw batches: survivors overflow the tile
    assert st["candidate_pairs"] == 32 * staged
    # and the pairs found are exactly the FLANN neighbours of the 32 queries (self excluded)
    d2 = flann_d2(lat[:, None, :], xyz[None, :, :])
    d2[np.arange(32), np.arange(32)] = np.inf
    assert st["feature_pairs"] == np.count_nonzero((d2 < np.float32(R * R)) & finite[None, :])
    # the probes just inside the radius of the box's edge points are real neighbours
    assert np.count_nonzero((d2 < np.float32(R * R)) & (d2 > np.float32(R * R * (1 - 1e-6)))) > 50
