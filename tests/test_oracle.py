"""CPU tests of the oracle itself: the pins that exist for it (SURVEY.md 8c).

The reference ships no tests and cannot be built here, so the oracle is pinned against
  * hand-derived known answers of the binning helpers (src/KeypointLearning.cpp:41-92),
  * scipy cKDTree (float64) for neighbour sets and k-NN, brute force O(n^2) for the FP32 predicate,
  * a float64 centred PCA for the normals,
  * the real OpenCV forest implementation (cv2.ml.RTrees, PREDICT_SUM) for the forest stage,
  * the committed golden vectors (tests/golden/, produced by make_golden.py).
"""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, forest_path

R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---------------------------------------------------------------------------------------------
# binning helpers
# ---------------------------------------------------------------------------------------------
def test_annulus_pair_known_answers(oracle):
    # SURVEY.md Appendix B: findAnnulusPair(n=5, distance, support=20) -> (index, pair, weight)
    kat = {0: (0, 0, 0.5), 1: (0, 0, 0.25), 2: (0, 0, 0.0), 3: (0, 1, 0.25), 4: (1, 0, 0.5), 5: (1, 0, 0.25), 6: (1, 0, 0.0),
           10: (2, 1, 0.0), 18: (4, 3, 0.0), 19: (4, 4, 0.25), 20: (4, 4, 0.5)}
    for d, (i, p, w) in kat.items():
        gi, gp, gw = oracle.find_annulus_pair(5, d, 20.0)
        assert (gi, gp) == (i, p) and gw == np.float32(w), (d, gi, gp, gw)
    gi, gp, gw = oracle.find_annulus_pair(5, np.float32(3.9999998), 20.0)
    assert (gi, gp) == (0, 1) and abs(float(gw) - 0.49999994) < 1e-7
    gi, gp, gw = oracle.find_annulus_pair(5, np.float32(17.9), 20.0)
    assert (gi, gp) == (4, 3) and abs(float(gw) - 0.0250000954) < 1e-8


def test_bin_pair_known_answers(oracle):
    # findBinPair(n=10, cosine): clamps, b == B fix, pair clamps (src/KeypointLearning.cpp:68-92)
    kat = [(-0.25, 0, 0, 0.5), (0.0, 0, 0, 0.5), (0.05, 0, 0, 0.25), (0.1, 0, 0, 0.0), (0.15, 0, 1, 0.25000003), (0.3, 1, 0, 0.0),
           (1.0, 5, 4, 0.500000119), (1.1, 5, 4, 0.0), (1.95, 9, 9, 0.249999762), (2.0, 9, 9, 0.499999523), (2.5, 9, 9, 0.499999523)]
    for c, i, p, w in kat:
        gi, gp, gw = oracle.find_bin_pair(10, c)
        assert (gi, gp) == (i, p), (c, gi, gp)
        assert abs(float(gw) - w) < 2e-7, (c, gw)
    k = np.load(os.path.join(GOLDEN, "kat_bins.npz"))
    for x, ref in zip(k["distance"], k["annulus"]):
        assert tuple(map(float, oracle.find_annulus_pair(5, x, 20.0))) == tuple(ref)
    for x, ref in zip(k["cosine"], k["bins"]):
        assert tuple(map(float, oracle.find_bin_pair(10, x))) == tuple(ref)


def test_abs_is_float_abs(oracle):
    """`abs(weight)` resolves to int abs under g++ with only <cmath> (SURVEY.md 7): any off-centre value must
    keep a non-zero weight."""
    _, _, w = oracle.find_annulus_pair(5, 1.0, 20.0)
    assert w == np.float32(0.25)
    _, _, w = oracle.find_bin_pair(10, 0.07)
    assert 0.1 < float(w) < 0.2


def test_weights_sum_to_one_per_neighbour(oracle):
    rng = np.random.default_rng(0)
    for _ in range(200):
        d, c = np.float32(rng.uniform(0, 20)), np.float32(rng.uniform(-0.1, 2.1))
        a, ap, wa = oracle.find_annulus_pair(5, d, 20.0)
        b, bp, wb = oracle.find_bin_pair(10, c)
        assert 0 <= a < 5 and 0 <= ap < 5 and 0 <= b < 10 and 0 <= bp < 10 and abs(a - ap) <= 1 and abs(b - bp) <= 1
        tot = (1 - wb) * (1 - wa) + wb * (1 - wa) + (1 - wb) * wa + wb * wa
        assert abs(float(tot) - 1.0) < 1e-6


# ---------------------------------------------------------------------------------------------
# libm-independent trig
# ---------------------------------------------------------------------------------------------
def test_trig_within_one_ulp_of_libm(oracle):
    rng = np.random.default_rng(1)
    ys = np.abs(rng.normal(size=4000)).astype(np.float32) * np.float32(10.0) ** rng.integers(-6, 3, 4000).astype(np.float32)
    xs = rng.normal(size=4000).astype(np.float32) * np.float32(10.0) ** rng.integers(-6, 3, 4000).astype(np.float32)
    for y, x in zip(ys, xs):
        got = oracle.atan2f(y, x)
        ref = np.float32(np.arctan2(np.float64(y), np.float64(x)))
        assert abs(float(got) - float(ref)) <= np.spacing(ref), (y, x, got, ref)
    for t in rng.uniform(0, np.pi / 3, 4000).astype(np.float32):
        for f, g in ((oracle.cosf, np.cos), (oracle.sinf, np.sin)):
            ref = np.float32(g(np.float64(t)))
            assert abs(float(f(t)) - float(ref)) <= np.spacing(ref), (t,)
    assert oracle.atan2f(0.0, 1.0) == 0 and oracle.atan2f(0.0, -1.0) == np.float32(np.pi)
    assert oracle.atan2f(0.0, 0.0) == 0 and oracle.atan2f(0.0, -0.0) == np.float32(np.pi)
    assert oracle.atan2f(1.0, 0.0) == np.float32(np.pi / 2)


# ---------------------------------------------------------------------------------------------
# radius search / k-NN
# ---------------------------------------------------------------------------------------------
def test_radius_counts_grid_vs_brute_force(oracle, views):
    xyz = np.ascontiguousarray(views["cheff002"][:6000])
    for r in (2.0, 4.0, 20.0):
        assert np.array_equal(oracle.radius_counts(xyz, r), oracle.radius_counts(xyz, r, brute=True))


def test_radius_neighbours_vs_ckdtree(oracle, views):
    sp = pytest.importorskip("scipy.spatial")
    xyz = views["cheff001"]
    q = np.arange(0, len(xyz), 211, dtype=np.int32)
    tree = sp.cKDTree(xyz.astype(np.float64))
    for r in (R_NMS, R_FEAT):
        off, idx = oracle.radius_neighbors(xyz, r, q)
        for k, qi in enumerate(q):
            mine = set(idx[off[k]:off[k + 1]].tolist())
            d = np.linalg.norm(xyz.astype(np.float64) - xyz[qi].astype(np.float64), axis=1)
            sure_in = set(np.nonzero(d < r - 1e-4)[0].tolist())
            maybe = set(tree.query_ball_point(xyz[qi].astype(np.float64), r + 1e-4))
            assert sure_in <= mine <= maybe
            assert qi in mine                      # the query is its own neighbour (d2 = 0 < r^2)


def test_golden_pair_totals(golden):
    # SURVEY.md 6: 158 212 200 / 145 943 273 / 145 293 891 pairs by float64 cKDTree; FP32 strict predicate differs by a handful
    for v, ref in (("cheff000", 158212200), ("cheff001", 145943273), ("cheff002", 145293891)):
        assert abs(int(golden[v]["pairs_r20"]) - ref) <= 16


def test_knn_vs_ckdtree(oracle, views):
    sp = pytest.importorskip("scipy.spatial")
    xyz = np.ascontiguousarray(views["cheff000"][::2])
    idx, d2 = oracle.knn_indices(xyz, 10)
    assert np.array_equal(idx[:, 0], np.arange(len(xyz)))           # the query itself at rank 0
    assert np.all(np.diff(d2, axis=1) >= 0)
    dd, ii = sp.cKDTree(xyz.astype(np.float64)).query(xyz.astype(np.float64), k=10)
    same = (np.sort(idx, axis=1) == np.sort(ii, axis=1)).all(axis=1)
    assert same.mean() > 0.999                                     # differences only at FP32 distance ties
    assert np.allclose(np.sqrt(d2.astype(np.float64)), dd, rtol=1e-5, atol=1e-5)


def test_knn_more_neighbours_than_points(oracle):
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.1], [0.5, 0.5, 0.3]], np.float32)
    idx, _ = oracle.knn_indices(pts, 10)
    assert np.all(np.sort(idx[:, :5], axis=1) == np.arange(5)) and np.all(idx[:, 5:] == -1)
    assert np.isfinite(oracle.normals_knn(pts, 10)).all()
    assert np.isnan(oracle.normals_knn(pts[:2], 10)).all()          # < 3 neighbours -> NaN (PCL computePointNormal)


# ---------------------------------------------------------------------------------------------
# normals
# ---------------------------------------------------------------------------------------------
def test_normals_vs_float64_pca(oracle, views):
    xyz = views["cheff001"]
    nrm = oracle.normals_knn(xyz, 10)
    assert np.isfinite(nrm).all()
    assert np.allclose(np.linalg.norm(nrm[:, :3], axis=1), 1.0, atol=1e-5)
    # flipped towards the viewpoint (0,0,0): n . (vp - p) >= 0
    assert np.all(np.einsum("ij,ij->i", nrm[:, :3].astype(np.float64), -xyz.astype(np.float64)) >= -1e-3)
    idx, _ = oracle.knn_indices(xyz, 10)
    sub = np.arange(0, len(xyz), 37)
    P = xyz[idx[sub]].astype(np.float64)
    P = P - P.mean(axis=1, keepdims=True)
    w, v = np.linalg.eigh(np.einsum("nki,nkj->nij", P, P))
    n64 = v[:, :, 0]
    cosang = np.abs(np.einsum("ij,ij->i", n64, nrm[sub, :3].astype(np.float64)))
    ang = np.degrees(np.arccos(np.clip(cosang, 0, 1)))
    # PCL 1.8.0's un-centred FP32 covariance is noisy by design (SURVEY.md A.3): median 0.03 deg, long tail
    assert np.median(ang) < 0.2 and np.quantile(ang, 0.99) < 3.0


def test_normals_radius_mode_runs(oracle, views):
    xyz = np.ascontiguousarray(views["cheff001"][:4000])
    nrm = oracle.normals_radius(xyz, 5.0)
    ok = np.isfinite(nrm).all(axis=1)          # points with < 3 neighbours in the ball are NaN (PCL)
    cnt = oracle.radius_counts(xyz, 5.0)
    assert np.array_equal(ok, cnt >= 3) or ok.mean() > 0.99
    assert np.allclose(np.linalg.norm(nrm[ok, :3], axis=1), 1.0, atol=1e-5)


def test_binning_helpers_match_the_reference_build(oracle, reference):
    """oracle/_ref: the reference's OWN src/KeypointLearning.cpp compiled from the mounted tree.  The oracle's
    restatement of findAnnulusPair / findBinPair must agree with it bit for bit on a dense sweep that includes
    every bin boundary +- a few ulps, the clamps and the centre-of-bin cases."""
    rng = np.random.default_rng(5)

    def around(values, span=3):
        out = []
        for v in values:
            x = np.float32(v)
            lo = hi = x
            out.append(x)
            for _ in range(span):
                lo = np.nextafter(lo, np.float32(-np.inf)); hi = np.nextafter(hi, np.float32(np.inf))
                out += [lo, hi]
        return np.asarray(out, np.float32)

    for A, support in ((5, 20.0), (4, 7.5), (8, 40.0), (10, 13.37), (1, 2.0), (16, 20.0)):
        dim = np.float32(support) / np.float32(A)
        edges = around(np.arange(0, 2 * A + 1, dtype=np.float32) * dim / np.float32(2))        # boundaries and centres
        d = np.concatenate([edges[(edges >= 0) & (edges <= np.float32(support))],
                            rng.uniform(0, support, 200_000).astype(np.float32), np.float32([0.0, support])])
        reference.check("annulus_sweep/A=%d,support=%g" % (A, support), oracle.annulus_sweep(A, support, d),
                        lambda: oracle.ref_annulus_sweep(A, support, d))
    for B in (10, 5, 8, 16, 1, 3):
        dim = np.float32(2) / np.float32(B)
        edges = around(np.arange(0, 2 * B + 1, dtype=np.float32) * dim / np.float32(2))
        c = np.concatenate([edges, rng.uniform(-0.5, 2.5, 200_000).astype(np.float32), np.float32([-1.0, 0.0, 2.0, 3.0, -0.0])])
        reference.check("bin_sweep/B=%d" % B, oracle.bin_sweep(B, c), lambda: oracle.ref_bin_sweep(B, c))


def test_binning_helpers_match_the_reference_build_random_shapes(oracle, reference):
    """arbitrary (n_annulus, support) / n_bins, not just the shapes the detector is used with: 60 seeded draws of each,
    and hypothesis on top where oracle/_ref is built."""
    rng = np.random.default_rng(11)
    for k in range(60):
        A, B, seed = int(rng.integers(1, 65)), int(rng.integers(1, 65)), int(rng.integers(0, 2**31 - 1))
        support = float(np.float32(2.0 ** rng.uniform(-6, 12)))
        d = np.minimum(np.random.default_rng(seed).uniform(0, support, 2000).astype(np.float32), np.float32(support))
        reference.check("annulus_random/%d" % k, oracle.annulus_sweep(A, support, d), lambda: oracle.ref_annulus_sweep(A, support, d))
        c = np.random.default_rng(seed).uniform(-1.0, 3.0, 2000).astype(np.float32)
        reference.check("bin_random/%d" % k, oracle.bin_sweep(B, c), lambda: oracle.ref_bin_sweep(B, c))
    if not reference.live:
        return
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 64), st.floats(0.015625, 4096.0, allow_nan=False, width=32), st.integers(0, 2**31 - 1))
    def annulus(A, support, seed):
        d = np.random.default_rng(seed).uniform(0, support, 2000).astype(np.float32)
        d = np.minimum(d, np.float32(support))
        for g, r in zip(oracle.annulus_sweep(A, support, d), oracle.ref_annulus_sweep(A, support, d)):
            assert np.array_equal(g.view(np.uint32), r.view(np.uint32))

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 64), st.integers(0, 2**31 - 1))
    def bins(B, seed):
        c = np.random.default_rng(seed).uniform(-1.0, 3.0, 2000).astype(np.float32)
        for g, r in zip(oracle.bin_sweep(B, c), oracle.ref_bin_sweep(B, c)):
            assert np.array_equal(g.view(np.uint32), r.view(np.uint32))

    annulus()
    bins()


# ---------------------------------------------------------------------------------------------
# oracle/_ref: the reference's OWN detector templates (include/KeypointLearning.h + impl/KeypointLearning.hpp)
# compiled from the mounted tree against the stand-in environment oracle/ref_stubs/kplref_env.h.  Search,
# forest traversal and the Eigen reductions are stand-ins (pinned elsewhere: scipy, cv2); everything else --
# slot-0 skip, NaN-normal skip, the four ordered histogram updates, per-annulus normalisation, feature layout,
# the score line, threshold compare, local-maximum NMS, the draws-remove skip list -- is the reference's code.
# ---------------------------------------------------------------------------------------------
def _ref_case(views, n=2500):
    xyz = np.ascontiguousarray(views["cheff001"][:n])
    return xyz


def test_features_match_the_reference_templates(oracle, views, reference):
    xyz = _ref_case(views)
    nrm = oracle.normals_knn(xyz, 10)
    nrm[7::53, 0] = np.nan                                      # neighbours (and queries) without a finite normal
    q = np.arange(0, len(xyz), 3, dtype=np.int32)
    q = q[np.isfinite(nrm[q, 0])]                               # runForest never asks for such a query (hpp:277)
    for r_feat, A, B in ((20.0, 5, 10), (9.0, 4, 8), (14.0, 10, 5)):
        for order in (0, 1):
            f_orc = oracle.features(xyz, nrm, r_feat, A, B, order=order, qidx=q)
            reference.check("features/r=%g,A=%d,B=%d,order=%d" % (r_feat, A, B, order), f_orc,
                            lambda: oracle.ref_features(xyz, nrm, r_feat, A, B, oracle.ref_neighbour_lists(xyz, r_feat, order), q))
    if not reference.live:
        return
    # the order really matters at the last bit: a sorted-kd-tree order gives different (close) rows
    f_sorted = oracle.ref_features(xyz, nrm, 20.0, 5, 10, oracle.ref_neighbour_lists(xyz, 20.0, 2), q)
    f_canon = oracle.features(xyz, nrm, 20.0, 5, 10, order=1, qidx=q)
    assert np.abs(f_sorted - f_canon).max() < 1e-5 and not np.array_equal(f_sorted, f_canon)


def test_detection_matches_the_reference_templates(oracle, views, reference):
    xyz = _ref_case(views)
    nrm = oracle.normals_knn(xyz, 10)
    assert np.isfinite(nrm[:, :3]).all()                        # the reference mis-aligns its response cloud otherwise (hpp:277 vs :203)
    forest = oracle.load_forest_yaml(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "forests", "synthetic-SHOT-like-T50-D10.yaml.gz"))
    r_feat, A, B = 20.0, 5, 10
    lf = oracle.ref_neighbour_lists(xyz, r_feat, 1)
    feat = oracle.features(xyz, nrm, r_feat, A, B, order=1)
    sc = oracle.scores(forest, feat, nrm)
    # runForest: setNonMaxima(false) hands back the response cloud (hpp:189-196)
    reference.check("detect/all", (np.arange(len(xyz), dtype=np.int32), sc),
                    lambda: oracle.ref_detect(xyz, nrm, forest, r_feat, 4.0, 0.5, A, B, lf, None, non_maxima=False))
    for r_nms, th in ((4.0, 0.85), (2.0, 0.5), (6.0, 0.3), (4.0, 0.0)):
        ln = oracle.ref_neighbour_lists(xyz, r_nms, 0)
        idx = oracle.nms(xyz, sc, r_nms, th)
        reference.check("detect/nms=%g,th=%g" % (r_nms, th), (idx, sc[idx]),
                        lambda: oracle.ref_detect(xyz, nrm, forest, r_feat, r_nms, th, A, B, lf, ln, non_maxima=True, draws_remove=False))
        for dthr in (0.0, 1.0, 3.0):
            reference.check("detect/nms=%g,th=%g,draws=%g" % (r_nms, th, dthr), oracle.nms(xyz, sc, r_nms, th, draws_remove=True, draws_thr=dthr),
                            lambda: oracle.ref_detect(xyz, nrm, forest, r_feat, r_nms, th, A, B, lf, ln, non_maxima=True, draws_remove=True,
                                                      draws_thr=dthr)[0])


def test_normals_radius_order_deviation_is_small(oracle, views):
    """Canonical (cell, index) accumulation order (what the device uses) against PCL's sorted (d2, index)
    order: the same un-centred FP32 moment sums re-associated.  On the model-centred bundled view the two
    normals agree to a small fraction of a degree."""
    xyz = np.ascontiguousarray(views["cheff001"][:6000])
    a = oracle.normals_radius(xyz, 10.0, order=0)
    b = oracle.normals_radius(xyz, 10.0, order=1)
    ok = np.isfinite(a).all(axis=1) & np.isfinite(b).all(axis=1)
    assert np.array_equal(np.isfinite(a).all(axis=1), np.isfinite(b).all(axis=1))
    cosang = np.clip(np.abs(np.sum(a[ok, :3] * b[ok, :3], axis=1)), 0.0, 1.0)
    ang = np.degrees(np.arccos(cosang))
    assert np.median(ang) < 0.05 and np.quantile(ang, 0.99) < 1.0, (np.median(ang), np.quantile(ang, 0.99))


# ---------------------------------------------------------------------------------------------
# features
# ---------------------------------------------------------------------------------------------
def _features_numpy(xyz, nrm, q, r, A, B, O):
    """Independent float32 restatement of hpp:321-376 in numpy for one query, ascending-index order."""
    f32 = np.float32
    H = np.zeros((A, B), f32)
    r2 = f32(np.float64(f32(r)) * np.float64(f32(r)))
    for j in range(len(xyz)):
        d = xyz[q] - xyz[j]
        d2 = f32(f32(f32(d[0] * d[0]) + f32(d[1] * d[1])) + f32(d[2] * d[2]))
        if not d2 < r2 or j == q:
            continue
        dot = f32(f32(nrm[q, 0] * nrm[j, 0]) + f32(f32(nrm[q, 1] * nrm[j, 1]) + f32(nrm[q, 2] * nrm[j, 2])))
        a, ap, wa = O.find_annulus_pair(A, np.sqrt(d2), r)
        b, bp, wb = O.find_bin_pair(B, f32(1) - dot)
        H[a, b] += f32((f32(1) - wb) * (f32(1) - wa)); H[a, bp] += f32(wb * (f32(1) - wa))
        H[ap, b] += f32((f32(1) - wb) * wa); H[ap, bp] += f32(wb * wa)
    for a in range(A):
        ss = f32(0)
        for b in range(B):
            ss = f32(ss + f32(H[a, b] * H[a, b]))
        n = np.sqrt(ss)
        if n > 0:
            H[a] = H[a] / n
    return H.ravel()


def test_features_against_numpy_restatement(oracle, views):
    xyz = np.ascontiguousarray(views["cheff001"][:1500])
    nrm = oracle.normals_knn(xyz, 10)
    q = np.array([0, 17, 400, 1499], np.int32)
    for A, B, r in ((5, 10, 20.0), (3, 4, 6.0)):
        got = oracle.features(xyz, nrm, r, A, B, order=0, qidx=q)
        for k, qi in enumerate(q):
            ref = _features_numpy(xyz, nrm, int(qi), r, A, B, oracle)
            assert np.array_equal(got[k].view(np.uint32), ref.view(np.uint32)), (A, B, qi)


def test_feature_orders_agree_within_tolerance(oracle, views):
    xyz = np.ascontiguousarray(views["cheff002"][::3])
    nrm = oracle.normals_knn(xyz, 10)
    q = np.arange(0, len(xyz), 19, dtype=np.int32)
    f0 = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=0, qidx=q)
    f1 = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1, qidx=q)
    f2 = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=2, qidx=q)
    assert np.abs(f0 - f1).max() <= 1e-5 and np.abs(f0 - f2).max() <= 1e-5     # north-star tolerance
    nr = np.linalg.norm(f1.reshape(len(q), 5, 10), axis=2)
    assert np.all((np.abs(nr - 1) < 1e-5) | (nr == 0))                          # per-annulus L2 normalisation
    # canonical order with a different grid resolution is a different, equally valid order
    f1b = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1, cpr=8, qidx=q)
    assert np.abs(f1 - f1b).max() <= 1e-5


def test_self_is_excluded_and_nan_normals_skipped(oracle):
    xyz = np.array([[0, 0, 0], [1, 0, 0], [0, 3, 0], [100, 0, 0]], np.float32)
    nrm = np.array([[0, 0, 1, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 1, 0]], np.float32)
    f = oracle.features(xyz, nrm, 20.0, 5, 10, order=0).reshape(4, 5, 10)
    # query 0: neighbour 1 (d=1, cos=0) and 2 (d=3, cos=1): all mass in annuli 0/1; self (d=0) did NOT vote
    raw_a0 = np.float32(1.0)   # neighbour 1: a=0,pair=0 (w=.25), b=0,pair=0 (w=.5) -> all four votes land in H(0,0) = 1
    assert f[0, 0, 0] > 0 and f[0, 0, 5] > 0 and f[0, 2:].sum() == 0
    # point 3 has no neighbour within 20: zero row (norm == 0 -> not normalised)
    assert np.all(f[3] == 0)
    nrm2 = nrm.copy(); nrm2[1, 0] = np.nan
    g = oracle.features(xyz, nrm2, 20.0, 5, 10, order=0).reshape(4, 5, 10)
    assert g[0, 0, 0] == 0 and g[0, 0, 5] > 0          # neighbour 1 skipped (hpp:338)
    assert np.all(g[1] == 0)                            # query 1 itself is not scored (hpp:277)
    del raw_a0


# ---------------------------------------------------------------------------------------------
# forest
# ---------------------------------------------------------------------------------------------
def test_forest_yaml_against_opencv(oracle, views):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2)
    for name, F in (("synthetic-T100-D15", 50), ("synthetic-FPFH-like-T30-D25", 50), ("synthetic-A4xB8-T20-D8", 32), ("synthetic-A8xB16-T20-D8", 128)):
        forest = oracle.load_forest_yaml(forest_path(name))
        assert forest["var_count"] == F and forest["ntrees"] == len(forest["roots"])
        rt = cv2.ml.RTrees_load(forest_path(name))
        x = rng.random((3000, F), dtype=np.float32) * np.float32(0.6)
        x /= np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-6)
        _, res = rt.predict(x, flags=cv2.ml.DTREES_PREDICT_SUM)
        assert np.array_equal(oracle.forest_sum(forest, x), res.ravel())


def test_score_rounding_known_answer(oracle):
    # SURVEY.md 8a F7: T=100, sum=15 -> exactly 0.85f, which passes `>= (double)0.85f`
    s = oracle.scores_from_sums(np.array([15, 30, 16], np.float32), 100)
    assert s[0] == np.float32(0.85) and float(s[0]) >= float(np.float32(0.85)) and s[2] < np.float32(0.85)
    assert oracle.scores_from_sums(np.array([30], np.float32), 200)[0] == np.float32(0.85)


# ---------------------------------------------------------------------------------------------
# NMS
# ---------------------------------------------------------------------------------------------
def test_nms_semantics(oracle):
    xyz = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0], [10, 0, 0], [14, 0, 0], [30, 0, 0]], np.float32)
    sc = np.array([0.9, 0.9, 0.95, 0.9, 0.99, 0.5], np.float32)
    # r=4: 0,1 are suppressed by 2 (strictly larger within 4); 3 and 4 are exactly 4 apart: d2 == r^2 does NOT count
    assert oracle.nms(xyz, sc, 4.0, 0.85).tolist() == [2, 3, 4]
    # plateau of equal scores: all survive (only strictly greater suppresses, hpp:219)
    assert oracle.nms(xyz[:2], sc[:2], 4.0, 0.85).tolist() == [0, 1]
    # threshold compare is >= in double against (double)(float)th
    assert oracle.nms(xyz, np.full(6, 0.85, np.float32), 1.0, 0.85).tolist() == [0, 1, 2, 3, 4, 5]
    assert oracle.nms(xyz, sc, 4.0, 0.96).tolist() == [4]
    sc2 = sc.copy(); sc2[2] = np.nan                       # unscored points neither win nor suppress
    assert oracle.nms(xyz, sc2, 4.0, 0.85).tolist() == [0, 1, 3, 4]
    # draws-remove branch (hpp:233-250): of a plateau pair closer than the threshold only the first survives
    assert oracle.nms(xyz[:2], sc[:2], 4.0, 0.85, draws_remove=True, draws_thr=2.0).tolist() == [0]
    assert oracle.nms(xyz[:2], sc[:2], 4.0, 0.85, draws_remove=True, draws_thr=0.5).tolist() == []


# ---------------------------------------------------------------------------------------------
# golden vectors: the oracle today == the oracle that froze them
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("view", ["cheff000", "cheff001", "cheff002"])
def test_oracle_reproduces_golden(oracle, views, golden, main_forest, view):
    xyz, g = views[view], golden[view]
    assert np.array_equal(oracle.radius_counts(xyz, R_NMS), g["counts_r4"])
    nrm = oracle.normals_knn(xyz, 10)
    assert sha(nrm) == str(g["normals_sha"]) and np.array_equal(nrm[::int(g["stride"])], g["normals_rows"])
    feat = oracle.features(xyz, nrm, R_FEAT, 5, 10, order=1)
    assert sha(feat) == str(g["features_sha"])
    sc = oracle.scores(main_forest, feat, nrm)
    assert np.array_equal(sc.view(np.uint32), g["scores"].view(np.uint32))
    assert np.array_equal(oracle.nms(xyz, sc, R_NMS, TH), g["keypoints"])
    assert float(g["features_order0_maxdiff"]) <= 1e-5


def test_detect_one_call_equals_stages(oracle, views, golden, main_forest):
    xyz, g = views["cheff001"], golden["cheff001"]
    res = oracle.detect(xyz, main_forest, order=1)
    assert np.array_equal(res["scores"].view(np.uint32), g["scores"].view(np.uint32))
    assert np.array_equal(res["keypoints"], g["keypoints"])


def test_integral_image_normals_restatement(oracle):
    """pcl::IntegralImageNormalEstimation(SIMPLE_3D_GRADIENT, 5.0) as restated by the oracle (hpp:138-145) against a
    direct float64 evaluation of its definition: gradient_x / gradient_y are differences of column / row sums over the
    smoothing rectangle, the normal their cross product turned towards the viewpoint; undefined on the image border,
    next to depth discontinuities and at NaN points."""
    from keypoint_learning_b200 import synth
    xyz, vp = synth.organized_range_image(200, 150, seed=3)
    h, w = xyz.shape[:2]
    n = oracle.normals_integral_image(xyz, 5.0, vp).reshape(h, w, 4)
    fin = np.isfinite(n[..., 0])
    assert 0.5 < fin.mean() < 0.97
    assert not fin[:5].any() and not fin[-5:].any() and not fin[:, :5].any() and not fin[:, -5:].any()      # BORDER_POLICY_IGNORE
    assert not fin[~np.isfinite(xyz[..., 2])].any()
    assert np.all(np.isnan(n[..., 3]))                                                                    # curvature = bad_point
    assert np.allclose(np.linalg.norm(n[fin][:, :3], axis=1), 1.0, atol=1e-6)
    assert np.all(np.einsum("ij,ij->i", n[fin][:, :3], -xyz[fin].astype(np.float64)) >= -1e-3)           # towards the viewpoint
    step = (2 * w) // 3
    assert not fin[20:-20, step - 2:step + 2].any()                                                      # nothing across the depth step
    # full 5 x 5 rectangle away from every discontinuity: compare with the definition
    P = np.nan_to_num(xyz.astype(np.float64))
    rng = np.random.default_rng(1)
    checked = 0
    for _ in range(4000):
        ri, ci = int(rng.integers(12, h - 12)), int(rng.integers(12, w - 12))
        if not np.isfinite(xyz[ri - 8:ri + 9, ci - 8:ci + 9]).all() or abs(ci - step) < 9 or (ri > h // 2 - 9 and ci < w // 4 + 9):
            continue
        gx = P[ri - 2:ri + 3, ci + 2].sum(0) - P[ri - 2:ri + 3, ci - 2].sum(0)
        gy = P[ri + 2, ci - 2:ci + 3].sum(0) - P[ri - 2, ci - 2:ci + 3].sum(0)
        nv = np.cross(gy, gx)
        nv /= np.linalg.norm(nv)
        if np.dot(-P[ri, ci], nv) < 0:
            nv = -nv
        if not fin[ri, ci]:
            continue                                  # a noise spike tripped the depth-change test nearby
        assert np.abs(n[ri, ci, :3] - nv).max() < 2e-6, (ri, ci)
        checked += 1
    assert checked > 300


def test_eigen_normalize_variants_against_the_reference_templates(oracle, views, reference):
    """`row.normalize()` (hpp:360-365) is Eigen code whose arithmetic changed between versions: >= 3.3 divides by the norm,
    3.2.x multiplies by 1/norm.  The reference pins no Eigen version, so both are restated; the reference's own
    computePointFeatures (oracle/_ref) run over either stub variant must equal the oracle in that mode, and the two
    variants differ by at most one ulp per feature."""
    xyz = np.ascontiguousarray(views["cheff000"][:2500])
    nrm = oracle.normals_knn(xyz, 10)
    lf = oracle.ref_neighbour_lists(xyz, 20.0, 1)
    rows = {}
    try:
        for recip in (False, True):
            oracle.set_normalize_mode(recip)
            f = oracle.features(xyz, nrm, 20.0, 5, 10, order=1)
            reference.check("features_normalize/reciprocal=%d" % recip, f, lambda: oracle.ref_features(xyz, nrm, 20.0, 5, 10, lf))
            rows[recip] = f
    finally:
        oracle.set_normalize_mode(False)
    ulps = np.abs(rows[False].view(np.int32).astype(np.int64) - rows[True].view(np.int32).astype(np.int64))
    assert ulps.max() == 1 and 0.01 < (ulps != 0).mean() < 0.5
