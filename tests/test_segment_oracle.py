"""The CPU model of DBSCAN clustering and RANSAC plane segmentation (tests/models/segment_model.cpp) against independent
restatements: Open3D's DBSCAN loop equals the order-free rule (connected components of the core points, border points to
the smallest neighbouring label) restated with scipy; the RANSAC hypotheses, break bound and selection equal a Python
restatement; closed cases (points on a plane, collinear samples, zero iterations or threshold).  Also: the library checks
its arguments before any CUDA call."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree

import cloud_ref
import segment_ref as ref


# ---------------------------------------------------------------------------------------------------------------------
# DBSCAN
# ---------------------------------------------------------------------------------------------------------------------
def rule_dbscan(p, eps, min_points, with_core=False):
    """The order-free rule: labels by the smallest index of each core component, border points the smallest label."""
    p = np.ascontiguousarray(p, np.float64)
    n = len(p)
    pairs = cKDTree(p).query_pairs(eps * (1.0 + 1e-6), output_type="ndarray").reshape(-1, 2)
    i, j = pairs[:, 0], pairs[:, 1]
    e = p[i] - p[j]
    d2 = (e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]
    keep = d2 < eps * eps
    i, j = i[keep], j[keep]
    deg = 1 + np.bincount(i, minlength=n) + np.bincount(j, minlength=n)
    core = deg >= min_points
    cc = core[i] & core[j]
    g = coo_matrix((np.ones(cc.sum()), (i[cc], j[cc])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    labels = np.full(n, -1, np.int64)
    ci = np.nonzero(core)[0]
    if len(ci):
        first = np.full(comp.max() + 1, n)
        np.minimum.at(first, comp[ci], ci)
        used = np.unique(comp[ci])
        order = used[np.argsort(first[used])]
        lab_of = np.full(comp.max() + 1, -1)
        lab_of[order] = np.arange(len(order))
        labels[ci] = lab_of[comp[ci]]
    big = np.iinfo(np.int64).max
    best = np.full(n, big)
    for a, b in ((i, j), (j, i)):        # a non-core, b core
        m = ~core[a] & core[b]
        np.minimum.at(best, a[m], labels[b[m]])
    border = ~core & (best != big)
    labels[border] = best[border]
    out = labels.astype(np.int32), len(ci) and int(labels.max()) + 1
    return out + (core,) if with_core else out


def chain(n=100_000, eps=0.01, seed=7):
    """n points along a wandering path, consecutive points 0.6-0.9 eps apart: one long component."""
    rng = np.random.default_rng(seed)
    step = rng.normal(size=(n, 3))
    step /= np.linalg.norm(step, axis=1, keepdims=True)
    step[:, 0] = np.abs(step[:, 0]) + 0.5            # keep moving forward so that the path does not fold onto itself
    step /= np.linalg.norm(step, axis=1, keepdims=True)
    return np.cumsum(step * (eps * rng.uniform(0.6, 0.9, n))[:, None], axis=0)


def bridged(eps=0.05):
    """Two dense blobs whose nearest members sit at exactly the same distance from one sparse point between them; the
    blob listed second in the array holds the lower cluster label only through its order."""
    rng = np.random.default_rng(11)
    a = rng.normal(scale=0.01, size=(300, 3)) + [-0.1, 0, 0]
    b = rng.normal(scale=0.01, size=(300, 3)) + [0.1, 0, 0]
    a[0] = [-0.75 * eps, 0.0, 0.0]
    b[0] = [0.75 * eps, 0.0, 0.0]
    bridge = np.array([[0.0, 0.0, 0.0]])
    return np.concatenate([b, bridge, a])


def dbscan_clouds():
    H = cloud_ref.H
    return {
        "lattice_eps_exact": (cloud_ref.lattice(), H, 3),
        "lattice_eps_above": (cloud_ref.lattice(), np.nextafter(H, 1.0), 7),
        "duplicates": (cloud_ref.with_duplicates(), 0.02, 10),
        "identical": (cloud_ref.identical(300), 0.01, 10),
        "two_clusters": (cloud_ref.two_clusters(), 0.05, 5),
        "outliers": (cloud_ref.surface_with_outliers(), 0.02, 8),
        "bridged": (bridged(), 0.05, 4),
        "eps_above_cloud": (cloud_ref.surface(500), 100.0, 10),
    }


@pytest.mark.parametrize("name", sorted(dbscan_clouds()))
def test_dbscan_loop_equals_the_rule(name):
    p, eps, mp = dbscan_clouds()[name]
    lab, nc = ref.cluster_dbscan(p, eps, mp)
    want, wn = rule_dbscan(p, eps, mp)
    assert (lab == want).all() and nc == wn


def test_dbscan_chain_is_one_component():
    p = chain()
    lab, nc = ref.cluster_dbscan(p, 0.01, 2)
    want, _ = rule_dbscan(p, 0.01, 2)
    assert nc == 1 and (lab == 0).all() and (want == 0).all()


def test_dbscan_border_point_takes_the_smallest_label():
    p = bridged()
    lab, nc = ref.cluster_dbscan(p, 0.05, 4)
    assert nc == 2 and lab[300] == 0                 # reached by both clusters, joins the one of the smaller label
    assert (lab[:300] == 0).all() and (lab[301:] == 1).all()


@pytest.mark.parametrize("mp", [0, 1, "n", "n+1"])
def test_dbscan_min_points_edges(mp):
    p = cloud_ref.two_clusters()
    n = len(p)
    m = {"n": n, "n+1": n + 1}.get(mp, mp)
    for eps in (0.05, 100.0):
        lab, nc = ref.cluster_dbscan(p, eps, m)
        want, wn = rule_dbscan(p, eps, m)
        assert (lab == want).all() and nc == wn, (eps, m)
    lab, _ = ref.cluster_dbscan(p, 100.0, n)          # every point sees all n: one cluster
    assert (lab == 0).all()
    lab, nc = ref.cluster_dbscan(p, 100.0, n + 1)      # nobody is core
    assert nc == 0 and (lab == -1).all()


def test_dbscan_permutation_permutes_the_partition():
    p = cloud_ref.surface_with_outliers(6000)
    lab, _ = ref.cluster_dbscan(p, 0.03, 12)
    perm = np.random.default_rng(3).permutation(len(p))
    lp, _ = ref.cluster_dbscan(p[perm], 0.03, 12)
    core = rule_dbscan(p, 0.03, 12, with_core=True)[2][perm]
    a, b = lab[perm], lp
    assert ((a < 0) == (b < 0)).all()
    pairs = {}                 # the core points' partition; a border point may join another of its clusters
    for x, y in zip(a[core], b[core]):
        assert pairs.setdefault(x, y) == y
    assert len(set(pairs.values())) == len(pairs)


# ---------------------------------------------------------------------------------------------------------------------
# RANSAC
# ---------------------------------------------------------------------------------------------------------------------
M64 = 0xFFFFFFFFFFFFFFFF


def splitmix64(x):
    x = (x + 0x9E3779B97F4A7C15) & M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def u01(seed, ctr):
    return float(splitmix64((seed * 0xD1342543DE82EF95 + ctr) & M64) >> 11) * (1.0 / 9007199254740992.0)


def floyd(n, r, seed, h):
    s = []
    for k in range(r):
        j = n - r + k
        t = min(math.floor(u01(seed, h * r + k) * float(j + 1)), j)
        s.append(j if t in s else t)
    return s


def plane_from_moments(c, m):
    xx, xy, xz, yy, yz, zz = m
    det_x, det_y, det_z = yy * zz - yz * yz, xx * zz - xz * xz, xx * yy - xy * xy
    if det_x > det_y and det_x > det_z:
        abc = [det_x, xz * yz - xy * zz, xy * yz - xz * yy]
    elif det_y > det_z:
        abc = [xz * yz - xy * zz, det_y, xy * xz - yz * xx]
    else:
        abc = [xy * yz - xz * yy, xy * xz - yz * xx, det_z]
    norm = math.sqrt((abc[0] * abc[0] + abc[1] * abc[1]) + abc[2] * abc[2])
    if norm == 0.0:
        return [0.0] * 4
    a, b, cc = (v / norm for v in abc)
    return [a, b, cc, -((a * c[0] + b * c[1]) + cc * c[2])]


def py_hypothesis(p, r, seed, h):
    s = floyd(len(p), r, seed, h)
    P = [[float(v) for v in p[i]] for i in s]
    if r == 3:
        e0 = [P[1][k] - P[0][k] for k in range(3)]
        e1 = [P[2][k] - P[0][k] for k in range(3)]
        abc = [e0[1] * e1[2] - e0[2] * e1[1], e0[2] * e1[0] - e0[0] * e1[2], e0[0] * e1[1] - e0[1] * e1[0]]
        norm = math.sqrt((abc[0] * abc[0] + abc[1] * abc[1]) + abc[2] * abc[2])
        if norm == 0.0:
            return [0.0] * 4
        a, b, c = (v / norm for v in abc)
        return [a, b, c, -((a * P[0][0] + b * P[0][1]) + c * P[0][2])]
    c = [0.0, 0.0, 0.0]
    for q in P:
        c = [c[k] + q[k] for k in range(3)]
    c = [v / r for v in c]
    m = [0.0] * 6
    for q in P:
        x, y, z = q[0] - c[0], q[1] - c[1], q[2] - c[2]
        m = [m[0] + x * x, m[1] + x * y, m[2] + x * z, m[3] + y * y, m[4] + y * z, m[5] + z * z]
    return plane_from_moments(c, m)


def py_bound(fitness, r, probability, num_iterations):
    if fitness >= 1.0:
        return 0
    num = math.log(1.0 - probability) if probability < 1.0 else -math.inf
    den = math.log(1.0 - math.pow(fitness, r)) if math.pow(fitness, r) < 1.0 else -math.inf
    with np.errstate(divide="ignore", invalid="ignore"):
        q = float(np.float64(num) / np.float64(den))
    return math.floor(q) if 0.0 <= q < num_iterations else num_iterations


def noisy_plane(n=4000, frac=0.6, seed=5):
    """frac of the points near the plane z = 0.3 x - 0.2 y + 0.1 (noise 2 mm), the rest uniform in a 1 m cube."""
    rng = np.random.default_rng(seed)
    k = int(n * frac)
    xy = rng.uniform(-1, 1, (k, 2))
    z = 0.3 * xy[:, 0] - 0.2 * xy[:, 1] + 0.1 + rng.normal(scale=0.002, size=k)
    p = np.concatenate([np.column_stack([xy, z]), rng.uniform(-1, 1, (n - k, 3))])
    return p[rng.permutation(n)]


@pytest.mark.parametrize("r", [3, 4, 7, 16])
def test_hypothesis_planes_equal_python(r):
    p = noisy_plane(500)
    for seed in (0, 12345, 2 ** 63 + 17):
        got = ref.hypothesis_planes(p, r, seed, 0, 40)
        want = np.array([py_hypothesis(p, r, seed, h) for h in range(40)])
        assert (got.view(np.uint64) == want.view(np.uint64)).all(), (r, seed)
    # Floyd's draw: r distinct indices, also when n = r
    for h in range(50):
        s = floyd(r, r, 99, h)
        assert sorted(s) == list(range(r))


def test_bound_formula():
    cases = [(0.5, 3, 0.99999999, 1000), (0.8, 3, 0.99999999, 1000), (0.1, 3, 0.99999999, 1000), (0.1, 5, 0.99, 1000),
             (1e-6, 3, 0.99999999, 1000),        # 1 - f^3 rounds to 1: q = -inf, B = num_iterations
             (0.3, 3, 1.0, 1000),                # probability 1: q = +inf, B = num_iterations
             (0.999, 3, 1e-18, 1000),             # 1 - p rounds to 1: q = -0, B = 0
             (1.0, 3, 0.9, 1000), (0.5, 3, 0.99999999, 10), (0.9, 4, 0.5, 1000), (0.97, 3, 0.999, 3)]
    for f, r, pr, it in cases:
        assert ref.ransac_bound(f, r, pr, it) == py_bound(f, r, pr, it), (f, r, pr, it)
    assert ref.ransac_bound(1e-6, 3, 0.99999999, 1000) == 1000
    assert ref.ransac_bound(0.3, 3, 1.0, 1000) == 1000
    assert ref.ransac_bound(1.0, 3, 0.5, 1000) == 0


def py_segment_plane(p, thr, r, num_iterations, probability, seed):
    """Open3D's SegmentPlane loop, sequential, over the model's hypothesis planes and evaluations."""
    n = len(p)
    B, best, best_fit, best_rmse, evaluated = math.inf, None, 0.0, 0.0, 0
    for h in range(num_iterations):
        if h > B:
            continue
        evaluated += 1
        pl = ref.hypothesis_planes(p, r, seed, h, 1)[0]
        if not pl.any():
            continue
        cnt, s = ref.evaluate(p, pl, thr)
        fit = cnt / n
        rmse = s / math.sqrt(cnt) if cnt else 0.0
        if fit > best_fit or (fit == best_fit and rmse < best_rmse):
            best, best_fit, best_rmse = pl, fit, rmse
            B = py_bound(fit, r, probability, num_iterations)
    return best, evaluated


@pytest.mark.parametrize("r,probability,iters", [(3, 0.99999999, 300), (3, 1.0, 150), (5, 0.999, 200)])
def test_selection_equals_the_sequential_loop(r, probability, iters):
    p = noisy_plane(3000, 0.4)
    best, evaluated = py_segment_plane(p, 0.01, r, iters, probability, 21)
    got = ref.segment_plane(p, 0.01, r, iters, probability, seed=21)
    assert got["n_evaluated"] == evaluated
    d = np.abs(((best[0] * p[:, 0] + best[1] * p[:, 1]) + best[2] * p[:, 2]) + best[3])
    assert (got["inliers"] == np.nonzero(d < 0.01)[0]).all()
    assert np.abs(got["plane"][:3] - np.array([-0.3, 0.2, 1.0]) / math.sqrt(1.13) * np.sign(got["plane"][2])).max() < 0.01


def test_tree_sum_is_a_sum():
    p = noisy_plane(20000)
    pl = np.array([-0.3, 0.2, 1.0, -0.1]) / math.sqrt(1.13)
    cnt, s = ref.evaluate(p, pl, 0.01)
    d = np.abs(((pl[0] * p[:, 0] + pl[1] * p[:, 1]) + pl[2] * p[:, 2]) + pl[3])
    assert cnt == (d < 0.01).sum() and abs(s - d[d < 0.01].sum()) < 1e-12 * cnt


def test_points_on_a_plane_stop_after_one_hypothesis():
    rng = np.random.default_rng(8)
    p = np.column_stack([rng.uniform(-1, 1, (5000, 2)), np.zeros(5000)])
    r = ref.segment_plane(p, 0.01, 3, 1000, seed=4)
    assert r["n_evaluated"] == 1 and len(r["inliers"]) == 5000
    assert list(r["plane"]) == [0.0, 0.0, 1.0, 0.0]


def test_collinear_samples_are_skipped():
    x = np.random.default_rng(9).uniform(-1, 1, 2000)
    line = np.column_stack([x, np.zeros_like(x), np.zeros_like(x)])
    r = ref.segment_plane(line, 0.01, 3, 200, seed=1)
    assert r["n_evaluated"] == 200 and len(r["inliers"]) == 0 and not r["plane"].any()
    # a few points off the line: the hypotheses on the line are invalid, the others compete
    p = np.concatenate([line, [[0.0, 0.5, 0.0], [0.3, 0.0, 0.5], [0.1, 0.2, 0.3]]])
    best, evaluated = py_segment_plane(p, 0.01, 3, 300, 0.99999999, 5)
    got = ref.segment_plane(p, 0.01, 3, 300, seed=5)
    assert got["n_evaluated"] == evaluated and best is not None and len(got["inliers"]) >= 2000


def test_zero_iterations_and_zero_threshold():
    p = noisy_plane(1000)
    for thr, iters in ((0.01, 0), (0.0, 50)):
        r = ref.segment_plane(p, thr, 3, iters, seed=2)
        assert len(r["inliers"]) == 0 and not r["plane"].any() and r["n_evaluated"] == iters


def test_library_checks_arguments_before_cuda():
    from otslam_b200 import _lib
    L = _lib.lib
    p = np.zeros((10, 3))
    lab = np.empty(10, np.int32)
    for eps, mp, n in ((0.0, 1, 10), (-1.0, 1, 10), (math.inf, 1, 10), (math.nan, 1, 10), (0.1, -1, 10), (0.1, 1, -1), (0.1, 1, 2 ** 31)):
        assert L.otslam_cloud_cluster_dbscan(_lib.ptr(p), n, eps, mp, _lib.ptr(lab), None, 0) == _lib.ERR_INVALID, (eps, mp, n)
    assert L.otslam_cloud_cluster_dbscan(None, 10, 0.1, 1, _lib.ptr(lab), None, 0) == _lib.ERR_INVALID
    assert L.otslam_cloud_cluster_dbscan(_lib.ptr(p), 10, 0.1, 1, None, None, 0) == _lib.ERR_INVALID
    plane = np.empty(4)
    inl = np.empty(10, np.int64)
    m = C.c_int64()

    def seg(n=10, thr=0.01, r=3, it=10, prob=0.9, pts=p, out=inl):
        return L.otslam_cloud_segment_plane(_lib.ptr(pts), n, thr, r, it, prob, C.c_uint64(0), _lib.ptr(plane), _lib.ptr(out), C.byref(m),
                                            None, 0)
    for kw in ({"thr": -0.1}, {"thr": math.inf}, {"thr": math.nan}, {"r": 2}, {"r": 17}, {"it": -1}, {"prob": 0.0}, {"prob": 1.5},
               {"prob": math.nan}, {"n": 2}, {"n": -1}, {"n": 2 ** 31}, {"pts": None}, {"out": None}):
        assert seg(**kw) == _lib.ERR_INVALID, kw
    seg(n=2)
    assert "There must be at least 'ransac_n' points." in _lib.last_error()
