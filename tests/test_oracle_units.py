"""Unit invariance of the whole detection (CPU oracle): scaling the coordinates and both radii by 2^k leaves normals,
features, scores and keypoints bit-identical, because every FP32 rounding commutes with an exact power-of-two scale and
the grid is computed in double.  tests/test_gpu_units.py relies on it: a scaled cloud has the committed goldens (or an
unscaled run) on its other side, and the scale picks the feature kernel's variant (DESIGN.md §3)."""
import os

import numpy as np
import pytest

from conftest import forest_path

R_FEAT, R_NMS, TH = 20.0, 4.0, 0.85
# the scales of the GPU scale matrix (k of 2^k): both exact ranges of the feature kernel and both sides of its fast path
SCALES = [-50, -23, -22, 15, 16, 20, 45]
F32 = np.float32
# the fast path's range limits at A = 4, B = 8: (cloud scale k, radius, unscaled radius with the same result)
BOUNDARIES = [
    (16, F32(2.0 ** 20), F32(16.0)),                                                   # r2 = 2^40 exactly
    (16, np.nextafter(F32(2.0 ** 20), F32(np.inf)), F32(16.0 * (1 + 2.0 ** -23))),     # r2 > 2^40
    (-22, F32(2.0 ** -18), F32(16.0)),                                                 # adim = 2^-20 exactly
    (-22, np.nextafter(F32(2.0 ** -18), F32(0)), F32(16.0 * (1 - 2.0 ** -24))),        # adim < 2^-20
]


def same_bits(a, b):
    """bit-identical float arrays; NaNs compare equal whatever their payload (the NaN positions must agree)"""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def xyz():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "views", "cheff001.npz"))["xyz"]


def detect(oracle, xyz, forest, k, r_feat, r_nms, th, A, B):
    s = F32(2.0 ** k)
    return oracle.detect(np.ascontiguousarray(xyz * s), forest, float(F32(r_feat) * s), float(F32(r_nms) * s), th, A, B,
                         normals_mode=1, k=10, order=1)


def assert_same_result(got, ref):
    assert same_bits(got["normals"], ref["normals"])                 # NaN normals at the same positions
    assert same_bits(got["features"], ref["features"])
    assert same_bits(got["scores"], ref["scores"])
    assert np.array_equal(got["keypoints"], ref["keypoints"])


@pytest.fixture(scope="module")
def unit_run(oracle, xyz, main_forest, golden):
    ref = detect(oracle, xyz, main_forest, 0, R_FEAT, R_NMS, TH, 5, 10)
    # the unit-scale oracle run is the committed golden
    assert np.array_equal(ref["scores"].view(np.uint32), golden["cheff001"]["scores"].view(np.uint32))
    assert np.array_equal(ref["keypoints"], golden["cheff001"]["keypoints"])
    return ref


@pytest.mark.parametrize("k", SCALES)
def test_power_of_two_scale_is_bit_identical(oracle, xyz, main_forest, unit_run, k):
    assert_same_result(detect(oracle, xyz, main_forest, k, R_FEAT, R_NMS, TH, 5, 10), unit_run)


@pytest.mark.parametrize("case", range(len(BOUNDARIES)))
def test_fast_path_boundaries_are_scaled_unit_runs(oracle, xyz, case):
    k, r, r_unit = BOUNDARIES[case]
    assert F32(r) == F32(r_unit * F32(2.0 ** k))                  # the scaled radius is exactly the unscaled one times 2^k
    forest = oracle.load_forest_yaml(forest_path("synthetic-A4xB8-T20-D8"))
    ref = oracle.detect(xyz, forest, float(r_unit), R_NMS, 0.5, 4, 8, normals_mode=1, k=10, order=1)
    assert len(ref["keypoints"]) > 1000
    got = detect(oracle, xyz, forest, k, float(r_unit), R_NMS, 0.5, 4, 8)
    assert_same_result(got, ref)
