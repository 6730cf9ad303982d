"""The cloud search operators of csrc/knn.cu against plain FP64 brute force (tests/cloud_ref.py), bit for bit, on clouds
built to drive each path of the search: statistical outlier removal (per-point mean distance and kept indices),
nearest-neighbour distance, radius-bounded nearest neighbour and voxel down-sampling.

The k-NN search runs on up to three hashed grids (fine, coarse, top) whose cell sizes depend on the cloud and on the
OTSLAM_KNN_OCC / OTSLAM_KNN_RINGS knobs; its result must not.  The knobs are read once per process, so each setting is
checked in a child process."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import cloud_ref as R
from oracle import oracle

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KS = (1, 2, 31, 32, 33, 64, 127, 128)
SIZES = (1023, 1024, 1025, 2047, 2048, 2049)        # segment CTAs hold 1024 points, radix-sort tiles 2048
RATIO = 2.0


def _L():
    from otslam_b200 import _lib
    return _lib


def _pts(a):
    return np.ascontiguousarray(a, np.float64)


def gpu_sor(p, nb, ratio=RATIO):
    """(status, kept indices, per-point mean distance) of otslam_cloud_remove_statistical_outlier."""
    L, p = _L(), _pts(p)
    idx, dbar, m = np.empty(len(p), np.int64), np.full(len(p), np.nan), C.c_int64(-1)
    st = L.lib.otslam_cloud_remove_statistical_outlier(L.ptr(p), len(p), int(nb), float(ratio), L.ptr(idx), C.byref(m),
                                                       L.ptr(dbar), 0)
    return st, idx[:max(m.value, 0)].copy(), dbar


def gpu_nn_distance(q, p):
    L, q, p = _L(), _pts(q), _pts(p)
    out = np.full(len(q), np.nan)
    L.check(L.lib.otslam_cloud_nn_distance(L.ptr(q), len(q), L.ptr(p), len(p), L.ptr(out), 0))
    return out


def gpu_nn_within(q, p, r):
    L, q, p = _L(), _pts(q), _pts(p)
    idx, d2 = np.full(len(q), -7, np.int32), np.full(len(q), -1.0)
    L.check(L.lib.otslam_cloud_nn_within(L.ptr(q), len(q), L.ptr(p) if len(p) else None, len(p), float(r), L.ptr(idx),
                                         L.ptr(d2), 0))
    return idx, d2


def gpu_vds(p, c, v):
    L, p = _L(), _pts(p)
    n = len(p)
    op, oc = np.full((n, 3), np.nan), np.full((n, 3), np.nan)
    ok, on, m = np.full((n, 3), -7, np.int32), np.full(n, -7, np.int32), C.c_int64(-1)
    st = L.lib.otslam_cloud_voxel_down_sample(L.ptr(p), L.ptr(None if c is None else _pts(c)), n, float(v), L.ptr(op),
                                              L.ptr(oc), L.ptr(ok), L.ptr(on), C.byref(m), 0)
    k = max(m.value, 0)
    return st, m.value, op[:k], oc[:k], ok[:k], on[:k], (op, oc, ok, on)


# ---- the clouds; each drives a path of the search (which one is noted beside it)
SOR_CLOUDS = {
    # fine level (crowding >> 32), restarts fine -> coarse -> top for the isolated points, a top level (coarse dims > 24),
    # rings >= 4 on the top level
    "surface_outliers": (R.surface_with_outliers, KS),
    # cell boundaries far from the origin: the 1e-9 cell reach margin against rounded face positions
    "surface_offset": (lambda: R.surface_with_outliers() + R.OFFSET, KS),
    "surface_mirrored": (lambda: R.mirrored(R.surface_with_outliers()), KS),
    # every point on cell faces (cell == H exactly), distances tie everywhere
    "lattice": (R.lattice, KS),
    # 141 copies of one point: d-bar = 0, excluded from mean, sigma and the kept set
    "duplicates": (R.with_duplicates, KS),
    # degenerate extents: the 1e-9 extent clamp, single-cell axes, cells enlarged to extent / 1024
    "collinear": (R.collinear, KS),
    "line_on_faces": (R.line_on_faces, KS),
    "coplanar": (R.coplanar, KS),
    # one cell, sigma = 0; k = n
    "identical_300": (lambda: R.identical(300), KS),
    "identical_40": (lambda: R.identical(40), (1, 32, 33, 40, 128)),
    # an empty middle: the point halfway walks many rings
    "two_clusters": (R.two_clusters, KS),
    "n1": (lambda: R.surface(1, 30), (1, 2, 128)),
    "n2": (lambda: R.surface(2, 31), (1, 2, 3, 128)),
    "n3": (lambda: R.surface(3, 32), (1, 2, 3, 128)),
    **{f"n{n}": ((lambda n=n: R.surface(n, n)), (1, 20, 33, 128)) for n in SIZES},
}


def _far_sides():
    t = R.surface(3000, 11)
    lo, hi = t.min(0), t.max(0)
    ext, mid = (hi - lo).max(), (lo + hi) / 2
    rng = np.random.default_rng(12)
    far = [mid + s * 1e3 * ext * np.eye(3)[a] + rng.normal(scale=0.1, size=(5, 3)) for a in range(3) for s in (-1, 1)]
    return np.concatenate(far + [R.surface(200, 13)]), t


def _grid_queries(n, lo, hi, seed):
    """n queries at multiples of H / 2 in [lo, hi) H: on cell faces and midway between them."""
    return np.random.default_rng(seed).integers(2 * lo, 2 * hi, (n, 3)) * (R.H / 2)


def _line_queries():
    rng = np.random.default_rng(14)
    q = np.zeros((3000, 3))
    q[:, 0] = rng.integers(-20, 2070, 3000) * (R.H / 2)
    q[:, 1:] = rng.integers(-2, 3, (3000, 2)) * (R.H / 2)
    return q


def _between_clusters():
    t = R.two_clusters()
    d = t[-1]
    return np.concatenate([np.linspace(0, 1, 50)[:, None] * d[None], t[:200]]), t


NN_CASES = {
    "far_sides": _far_sides,                                                          # 10^3 x the extent away, 6 sides
    "lattice_faces": lambda: (_grid_queries(4000, -2, 19, 15), R.lattice()),           # queries on cell faces
    "line_faces": lambda: (_line_queries(), R.line_on_faces()),
    "single_target": lambda: (R.surface(1000, 16), R.surface(1, 17)),
    "identical_target": lambda: (np.concatenate([R.surface(1000, 18), R.identical(10)]), R.identical(500)),
    "collinear_target": lambda: (np.random.default_rng(19).random((2000, 3)) * 3 - 1, R.collinear()),
    "more_queries": lambda: (R.surface(20000, 20) + np.random.default_rng(21).normal(scale=0.01, size=(20000, 3)),
                             R.surface(700, 22)),
    "fewer_queries": lambda: (R.surface(50, 23), R.surface_with_outliers()),
    "offset": lambda: (R.surface(8000, 24) + R.OFFSET, R.surface(8000, 25) + [0.3, -0.2, 0.05] + R.OFFSET),
    "mirrored": lambda: (R.mirrored(R.surface(8000, 24)), R.mirrored(R.surface(8000, 25) + [0.3, -0.2, 0.05])),
    "between_clusters": _between_clusters,                                           # long ring walks through empty cells
    "cluster_to_cluster": lambda: (R.two_clusters()[:2000], R.two_clusters()[2001:]),  # every query outside the grid
}

_cache = {}


def _cached(key, fn):
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def sor_cloud(name):
    return _cached(("cloud", name), SOR_CLOUDS[name][0])


def ref_dbar(name, k):
    s = _cached(("sorted", name), lambda: R.knn_sorted_d2(sor_cloud(name), KS[-1]))
    return R.mean_dist_from_sorted(s, k)


def nn_case(name):
    return _cached(("nn", name), NN_CASES[name])


def ref_nn(name):
    return _cached(("nnref", name), lambda: R.nn_distance(*nn_case(name)))


def run_kernels(out_path):
    """Every outlier-filter and nearest-neighbour-distance case on the GPU, saved to `out_path` (.npz)."""
    res = {}
    for name, (_, ks) in SOR_CLOUDS.items():
        for k in ks:
            st, kept, dbar = gpu_sor(sor_cloud(name), k)
            res[f"sor:{name}:{k}:status"], res[f"sor:{name}:{k}:kept"], res[f"sor:{name}:{k}:dbar"] = np.int64(st), kept, dbar
    for name in NN_CASES:
        res[f"nn:{name}"] = gpu_nn_distance(*nn_case(name))
    np.savez(out_path, **res)


def check_sor(name, k, st, kept, dbar):
    n = len(sor_cloud(name))
    ref = ref_dbar(name, k)
    assert st == 0, f"{name} k={k}: status {st}"
    bad = np.nonzero(dbar != ref)[0]
    assert len(bad) == 0, f"{name} k={k}: d-bar differs at {len(bad)} of {n} points, first {bad[:5]}: {dbar[bad[:5]]} != {ref[bad[:5]]}"
    want = R.sor_select(ref, RATIO)
    assert len(kept) == len(want) and (kept == want).all(), f"{name} k={k}: kept indices differ"


@pytest.mark.parametrize("name", list(SOR_CLOUDS))
def test_outlier_filter_matches_brute_force(name):
    for k in SOR_CLOUDS[name][1]:
        check_sor(name, k, *gpu_sor(sor_cloud(name), k))


def test_outlier_filter_statistics_exclude_zero_mean_distances():
    p = sor_cloud("duplicates")
    _, kept, dbar = gpu_sor(p, 128)
    dup = (p == p[np.argmin(dbar)]).all(axis=1)
    assert dup.sum() == 141 and (dbar[dup] == 0).all() and (dbar[~dup] > 0).all()
    assert len(kept) > 0.8 * len(p) and not dup[kept].any()
    _, kept, dbar = gpu_sor(R.identical(300), 20)
    assert (dbar == 0).all() and len(kept) == 0


def test_outlier_filter_on_a_large_cloud():
    """2^17 + 3 points: d-bar equals the oracle everywhere and brute force on a sample; kept set from the reference rule."""
    p = R.surface(2 ** 17 + 3, 33)
    sample = np.random.default_rng(34).choice(len(p), 1500, replace=False)
    for k in (20, 33):
        st, kept, dbar = gpu_sor(p, k)
        assert st == 0
        assert (dbar[sample] == R.mean_dist_from_sorted(R.knn_sorted_d2(p, k, q=p[sample]), k)).all()
        oi, od = oracle.remove_statistical_outlier(p, k, RATIO)
        assert (dbar == od).all()
        want = R.sor_select(od, RATIO)
        assert (want == oi).all() and len(kept) == len(want) and (kept == want).all()


def test_outlier_filter_neighbour_limits():
    L = _L()
    p = R.surface(200, 35)
    st, _, _ = gpu_sor(p, 129)
    assert st == L.ERR_INVALID                                  # k = 129 > 128 with n >= 129: refused
    st, _, _ = gpu_sor(p[:129], 129)
    assert st == L.ERR_INVALID
    st, kept, dbar = gpu_sor(p[:128], 129)                      # nb_neighbors > n: k = n = 128
    assert st == 0 and (dbar == R.knn_mean_dist(p[:128], 128)).all()
    st, kept, dbar = gpu_sor(p[:100], 200)                      # k = n = 100
    ref = R.knn_mean_dist(p[:100], 100)
    assert st == 0 and (dbar == ref).all() and (kept == R.sor_select(ref, RATIO)).all()


SETTINGS = {
    "default": {},
    "no_fine_level": {"OTSLAM_KNN_RINGS": "0"},
    "fine_everywhere": {"OTSLAM_KNN_OCC": "1", "OTSLAM_KNN_RINGS": "1"},
    "occ2_rings3": {"OTSLAM_KNN_OCC": "2", "OTSLAM_KNN_RINGS": "3"},
}


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_search_is_independent_of_cell_size(setting, tmp_path):
    env = {k: v for k, v in os.environ.items() if not k.startswith("OTSLAM_KNN_")}
    env.update(SETTINGS[setting])
    out = str(tmp_path / "gpu.npz")
    code = f"import sys; sys.path[:0] = [{ROOT!r}, {HERE!r}]; import test_gpu_cloud_search as t; t.run_kernels({out!r})"
    r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = np.load(out)
    for name, (_, ks) in SOR_CLOUDS.items():
        for k in ks:
            check_sor(name, k, int(res[f"sor:{name}:{k}:status"]), res[f"sor:{name}:{k}:kept"], res[f"sor:{name}:{k}:dbar"])
    for name in NN_CASES:
        assert (res[f"nn:{name}"] == ref_nn(name)).all(), name


@pytest.mark.parametrize("name", list(NN_CASES))
def test_nn_distance_matches_brute_force(name):
    q, p = nn_case(name)
    got = gpu_nn_distance(q, p)
    bad = np.nonzero(got != ref_nn(name))[0]
    assert len(bad) == 0, f"{len(bad)} of {len(q)} differ, first {bad[:5]}"


def test_nn_distance_rejects_an_empty_target():
    L = _L()
    q, out = np.zeros((3, 3)), np.empty(3)
    assert L.lib.otslam_cloud_nn_distance(L.ptr(q), 3, None, 0, L.ptr(out), 0) == L.ERR_INVALID


def _exact_radius():
    p = np.array([[0.0, 0, 0], [3, 3, 3], [-3, 1, 2]])
    h = 0.5
    q = np.array([[h, 0, 0], [-h, 0, 0], [0, h, 0], [0, -h, 0], [0, 0, h], [0, 0, -h], [np.nextafter(h, 0), 0, 0],
                  [0.3, 0.4, 0], [0, 0, 0], [3, 3, 3.5], [3, 3, 2.6]])
    return q, p, h


def _duplicates():
    a = R.surface(1000, 40)
    p = np.concatenate([a, a[::-1], a])                        # three copies of each point, in different orders
    q = a + np.random.default_rng(41).normal(scale=0.005, size=a.shape)
    return q, p, 0.02


def _lattice_ties():
    p = R.lattice()                                             # repeats: equal targets at different indices
    return _grid_queries(4000, -1, 18, 42), p, R.H             # midpoints are equidistant from targets in 2-8 cells


def _tiny_radius():
    p = R.surface(5000, 43)                                     # extent 1.5: the cell is enlarged from r to 1.5 / 2^20
    rng = np.random.default_rng(44)
    q = p + rng.choice([-3e-7, 0.0, 3e-7, 5e-7], size=p.shape)
    return np.concatenate([q, rng.random((500, 3))]), p, 4e-7


def _huge_radius():
    return np.random.default_rng(45).random((1000, 3)) * 24 - 12, R.surface(2000, 46), 10.0


def _offset_noisy(sign):
    p = R.surface(20000, 47) + R.OFFSET
    q = p[:5000] + np.random.default_rng(48).normal(scale=0.01, size=(5000, 3))
    return (q, p, 0.012) if sign > 0 else (R.mirrored(q - R.OFFSET), R.mirrored(p - R.OFFSET), 0.012)


WITHIN_CASES = {
    "exact_radius": _exact_radius,
    "duplicates": _duplicates,
    "lattice_ties": _lattice_ties,
    "tiny_radius": _tiny_radius,
    "huge_radius": _huge_radius,
    "offset": lambda: _offset_noisy(1),
    "mirrored": lambda: _offset_noisy(-1),
    "empty_target": lambda: (R.surface(100, 49), np.zeros((0, 3)), 0.1),
}


@pytest.mark.parametrize("name", list(WITHIN_CASES))
def test_nn_within_matches_brute_force(name):
    q, p, r = WITHIN_CASES[name]()
    idx, d2 = gpu_nn_within(q, p, r)
    ridx, rd2 = R.nn_within(q, p, r)
    bad = np.nonzero(idx != ridx)[0]
    assert len(bad) == 0, f"{len(bad)} of {len(q)} differ, first {bad[:5]}: {idx[bad[:5]]} != {ridx[bad[:5]]}"
    if len(p):
        assert (d2 == rd2).all()
    if name == "exact_radius":
        assert (idx[:6] == -1).all() and idx[6] == 0 and idx[8] == 0      # d2 == r^2 is outside the radius
    elif name == "empty_target":
        assert (idx == -1).all()
    else:
        assert (idx >= 0).any()
    if name == "duplicates":
        assert (idx < 1000).all()                                           # the first of three equal targets


# ---- voxel down-sampling against the oracle (an independent hash-map implementation)
def _pass_cloud(bits, seed):
    """Points in [0, 2^b - 2] per axis with a unit voxel: 2^b - 1 voxels per axis, so the key takes b bits per axis."""
    S = np.array([2.0 ** b - 2 if b > 1 else 0.0 for b in bits])
    rng = np.random.default_rng(seed)
    p = rng.random((5000, 3)) * S
    p[1::3] = p[0:-1:3][:len(p[1::3])] + 0.1 * rng.random((len(p[1::3]), 3))   # voxels with several points
    p[0], p[-1] = 0.0, S
    return p


def _key_bits(p, v):
    """make_layout's key width for cloud p: per axis, the bits that hold floor((max - (min - v/2)) / v) + 1 cells."""
    mn, mx = p.min(0), p.max(0)
    bits = 0
    for a in range(3):
        cells, b = np.floor((mx[a] - (mn[a] - v * 0.5)) / v) + 1.0, 1
        while b < 62 and 2.0 ** b < cells:
            b += 1
        bits += b
    return bits


PASS_BITS = [(1, 1, 1), (2, 3, 3), (3, 3, 3), (5, 5, 6), (8, 8, 8), (10, 11, 11), (13, 13, 14), (16, 16, 16), (18, 19, 19),
             (19, 19, 19), (21, 21, 21)]


def _on_faces(sign):
    p = np.concatenate([np.zeros((1, 3)), R.lattice(9, 900) * 16 + 0.125])   # min 0: faces at -0.125 + 0.25 j, points on them
    return sign * p - (R.OFFSET if sign < 0 else 0), 0.25


VDS_CASES = {
    "offset": lambda: (R.surface(20000, 50) - R.OFFSET, 0.01),
    "offset_037": lambda: (R.surface(20000, 50) - R.OFFSET, 0.037),
    "mirrored": lambda: (R.mirrored(R.surface(20000, 51)), 0.037),
    "on_faces": lambda: _on_faces(1),
    "on_faces_negative": lambda: _on_faces(-1),
    "one_voxel": lambda: (R.surface(3000, 52) * 1e-3, 10.0),
    "own_voxels": lambda: (R.surface(3000, 53), 1e-6),
    **{f"n{n}": (lambda n=n: (R.surface(n, 54), 0.02)) for n in SIZES + (2 ** 17 + 3,)},
    **{f"bits{sum(b)}": (lambda b=b: (_pass_cloud(b, sum(b)), 1.0)) for b in PASS_BITS},
}


def test_voxel_cases_cover_every_radix_pass_count():
    passes = {max(1, (_key_bits(*VDS_CASES[f"bits{sum(b)}"]()) + 7) // 8) for b in PASS_BITS}
    assert passes == set(range(1, 9))
    assert [_key_bits(*VDS_CASES[f"bits{sum(b)}"]()) for b in PASS_BITS] == [sum(b) for b in PASS_BITS]


@pytest.mark.parametrize("name", list(VDS_CASES))
def test_voxel_down_sample_equals_the_oracle(name):
    p, v = VDS_CASES[name]()
    c = np.random.default_rng(55).random(p.shape)
    st, m, gp, gc, gk, gn, _ = gpu_vds(p, c, v)
    op, oc, ok, on = oracle.voxel_down_sample(p, c, v)
    assert st == 0 and m == len(op)
    assert (gk == ok).all() and (gn == on).all() and (gp == op).all() and (gc == oc).all()
    if name == "one_voxel":
        assert m == 1
    if name == "own_voxels":
        assert m == len(p)


def test_voxel_down_sample_refuses_keys_wider_than_63_bits():
    L = _L()
    p = _pass_cloud((22, 22, 22), 56)
    assert _key_bits(p, 1.0) == 66
    st, m, *_, bufs = gpu_vds(p, None, 1.0)
    assert st == L.ERR_OVERFLOW and m == 0
    assert np.isnan(bufs[0]).all() and np.isnan(bufs[1]).all() and (bufs[2] == -7).all() and (bufs[3] == -7).all()
