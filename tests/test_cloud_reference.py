"""Pins the brute-force references of tests/cloud_ref.py to the CPU oracle, bit for bit, on the adversarial clouds, so
that they can be trusted when they judge the GPU kernels (tests/test_gpu_cloud_search.py).  Runs without a GPU."""
import numpy as np
import pytest

import cloud_ref as R
from oracle import oracle

SOR_CLOUDS = {
    "surface_outliers": lambda: R.surface_with_outliers(6000),
    "surface_offset": lambda: R.surface_with_outliers(6000) + R.OFFSET,
    "surface_mirrored": lambda: R.mirrored(R.surface_with_outliers(6000)),
    "lattice": R.lattice,
    "duplicates": R.with_duplicates,
    "collinear": R.collinear,
    "line_on_faces": R.line_on_faces,
    "coplanar": R.coplanar,
    "identical_40": lambda: R.identical(40),
    "identical_300": lambda: R.identical(300),
    "two_clusters": lambda: R.two_clusters(1000),
    "n1": lambda: R.surface(1),
    "n2": lambda: R.surface(2),
    "n3": lambda: R.surface(3),
}


@pytest.mark.parametrize("name", list(SOR_CLOUDS))
def test_mean_dist_and_kept_indices_equal_the_oracle(name):
    p = SOR_CLOUDS[name]()
    s = R.knn_sorted_d2(p, 200)
    assert (R.knn_mean_dist(p, 20) == R.mean_dist_from_sorted(s, 20)).all()
    for k in (1, 2, 20, 32, 33) + (() if name == "coplanar" else (128, 200)):   # the oracle's plain ring walk is slow on a sparse plane
        ref = R.mean_dist_from_sorted(s, k)
        for ratio in (2.0, 0.3):
            oi, od = oracle.remove_statistical_outlier(p, k, ratio)
            assert (od == ref).all(), f"d-bar differs at k={k}"
            kept = R.sor_select(ref, ratio)
            assert len(kept) == len(oi) and (kept == oi).all(), f"kept set differs at k={k}, ratio={ratio}"


def test_duplicates_are_excluded_from_the_statistics():
    p = R.with_duplicates()
    dbar = R.knn_mean_dist(p, 128)
    dup = (p == R.surface(3000, 2)[1000]).all(axis=1)      # the repeated point and its 140 copies
    assert dup.sum() == 141 and (dbar[dup] == 0).all() and (dbar[~dup] > 0).all()
    kept = R.sor_select(dbar, 2.0)
    assert not dup[kept].any()
    # the zeros count in n but add nothing to the mean or sigma
    pos = dbar[~dup]
    assert R.sor_threshold(dbar, 0.0) == np.add.accumulate(pos)[-1] / len(p)


def test_nn_references_on_small_cases():
    p = np.array([[0.0, 0, 0], [1, 0, 0], [1, 0, 0], [0, 2, 0]])
    q = np.array([[0.5, 0, 0], [0.9, 0, 0], [1, 0, 0], [0, 1.0, 0], [5, 5, 5]])
    assert (R.nn_distance(q, p) == [0.5, np.sqrt((0.9 - 1.0) ** 2), 0.0, 1.0, np.sqrt(59.0)]).all()
    idx, d2 = R.nn_within(q, p, 0.5)
    assert idx.tolist() == [-1, 1, 1, -1, -1]             # d2 == r^2 is outside; the lower of two equal targets wins
    assert d2[0] == -1.0 and d2[2] == 0.0
    idx, d2 = R.nn_within(q, np.zeros((0, 3)), 1.0)
    assert (idx == -1).all() and (d2 == -1.0).all()


VDS_CASES = {
    "offset_colours": (lambda: R.surface(5000, 6) - R.OFFSET, 0.01),
    "mirrored": (lambda: R.mirrored(R.surface(5000, 7)), 0.037),
    "on_faces": (lambda: np.concatenate([np.zeros((1, 3)), R.lattice(9, 900) * 16 + 0.125]), 0.25),
    "one_voxel": (lambda: R.surface(3000, 8) * 1e-3, 10.0),
    "own_voxels": (lambda: R.surface(3000, 9), 1e-6),
}


@pytest.mark.parametrize("name", list(VDS_CASES))
def test_voxel_down_sample_equals_the_oracle(name):
    make, v = VDS_CASES[name]
    p = make()
    c = np.random.default_rng(10).random(p.shape)
    rp, rc, rk, rn = R.voxel_down_sample(p, c, v)
    op, oc, ok, on = oracle.voxel_down_sample(p, c, v)
    assert len(rp) == len(op) and (rk == ok).all() and (rn == on).all()
    assert (rp == op).all() and (rc == oc).all()
