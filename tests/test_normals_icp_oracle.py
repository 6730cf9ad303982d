"""Normal estimation and point-to-plane ICP pinned on the CPU (DESIGN.md §4 "Normals and point-to-plane registration").
The reference is tests/models/normals_icp_model.cpp (tests/normals_icp_ref.py); tests/test_gpu_normals_icp.py compares the
CUDA kernels with it bit for bit.  Here it is pinned against brute force and closed forms: neighbour lists equal a brute
(d2, index) sort on the adversarial clouds, planes give their normal, spheres give radial normals and NumPy's eigh agrees
wherever the eigen gap is large, the fallback and sign rules hold, and point-to-plane ICP recovers a known motion in far
fewer iterations than point-to-point.  The C entry points' argument checks run here too: they fail before any CUDA call."""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial import cKDTree

import cloud_ref
import normals_icp_ref as ref


def brute_lists(p, radius, max_nn):
    k = min(max_nn, len(p))
    r2 = float(radius) * float(radius)
    idx = np.full((len(p), max_nn), -1, np.int32)
    cnt = np.empty(len(p), np.int32)
    for s, d2 in cloud_ref.brute_d2(p, p):
        for r in range(len(d2)):
            j = np.nonzero(d2[r] < r2)[0]
            o = j[np.lexsort((j, d2[r][j]))][:k]
            idx[s + r, :len(o)] = o
            cnt[s + r] = len(o)
    return idx, cnt


ADVERSARIAL = {
    "lattice": lambda: cloud_ref.lattice(m=9, n=1500),
    "duplicates": lambda: cloud_ref.with_duplicates(n=1500, copies=60),
    "identical": lambda: cloud_ref.identical(200),
    "collinear": lambda: cloud_ref.collinear(1500),
    "coplanar": lambda: cloud_ref.coplanar(),
    "mirrored_lattice": lambda: cloud_ref.mirrored(cloud_ref.lattice(m=9, n=1500)),
}


@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
@pytest.mark.parametrize("radius,max_nn", [(np.inf, 1), (np.inf, 30), (np.inf, 33), (np.inf, 128), (3 * cloud_ref.H, 30),
                                           (2 * cloud_ref.H, 128)])
def test_neighbour_lists_equal_brute_force(name, radius, max_nn):
    p = ADVERSARIAL[name]()
    if name == "coplanar" and np.isfinite(radius):
        radius *= 16          # its grid is spaced 16 H
    idx, cnt = ref.neighbours(p, radius, max_nn)
    want_idx, want_cnt = brute_lists(p, radius, max_nn)
    assert (cnt == want_cnt).all()
    assert (idx == want_idx).all()


def tilted_plane(n=4000, seed=0):
    rng = np.random.default_rng(seed)
    nrm = np.array([1.0, 2.0, 2.0]) / 3.0
    e1 = np.array([2.0, -1.0, 0.0]) / np.sqrt(5.0)
    e2 = np.cross(nrm, e1)
    uv = rng.random((n, 2)) - 0.5
    return uv[:, :1] * e1 + uv[:, 1:] * e2, nrm


# centred, with at least 8 neighbours: E[xx^T] - mu mu^T (Open3D's formula) cancels little and no triple is near-collinear
@pytest.mark.parametrize("radius,max_nn", [(np.inf, 8), (np.inf, 30), (np.inf, 128), (0.05, 30)])
def test_planes_give_the_plane_normal(radius, max_nn):
    p, nrm = tilted_plane()
    n = ref.estimate_normals(p, radius, max_nn)
    assert np.abs(np.abs(n @ nrm) - 1.0).max() < 1e-12
    assert (n @ nrm > 0).all()          # largest component (z or y of (1, 2, 2) / 3: the first, y) positive
    flat = ref.estimate_normals(cloud_ref.coplanar(), np.inf, 30)
    assert (flat == np.array([0.0, 0.0, 1.0])).all()


def sphere(n=20000, r=0.5, seed=1):
    v = np.random.default_rng(seed).normal(size=(n, 3))
    return r * v / np.linalg.norm(v, axis=1, keepdims=True)


def test_sphere_normals_are_radial_and_agree_with_eigh():
    p = sphere()
    n = ref.estimate_normals(p, np.inf, 30)
    radial = p / np.linalg.norm(p, axis=1, keepdims=True)
    assert np.abs(np.abs(np.einsum("ij,ij->i", n, radial)) - 1.0).max() < 1e-3
    assert np.abs(np.linalg.norm(n, axis=1) - 1.0).max() < 1e-15 * 4
    idx, cnt = ref.neighbours(p, np.inf, 30)
    nb = p[idx]                                                      # [n, 30, 3]
    mu = nb.mean(axis=1)
    cov = np.einsum("nki,nkj->nij", nb, nb) / 30 - np.einsum("ni,nj->nij", mu, mu)
    w, v = np.linalg.eigh(cov)
    gap = (w[:, 1] - w[:, 0]) / w[:, 2]
    ok = gap > 1e-2
    assert ok.mean() > 0.9
    assert np.abs(np.abs(np.einsum("ij,ij->i", n[ok], v[ok, :, 0])) - 1.0).max() < 1e-9


def test_fallback_and_sign_rules():
    p, nrm = tilted_plane(500)
    # fewer than 3 neighbours: C = I, whose smallest-eigenvalue vector (highest index among equals) is (0, 0, 1)
    for k in (1, 2):
        assert (ref.estimate_normals(p, np.inf, k) == [0.0, 0.0, 1.0]).all()
    prior = np.tile([0.0, 0.0, -1.0], (len(p), 1))
    assert (ref.estimate_normals(p, np.inf, 2, prior) == [0.0, 0.0, -1.0]).all()
    # a radius below the spacing: only the point itself
    assert (ref.estimate_normals(p, 1e-9, 30) == [0.0, 0.0, 1.0]).all()
    # zero covariance (identical points with exact binary coordinates): the zero vector becomes (0, 0, 1) or the prior
    same = cloud_ref.identical(50)
    assert (ref.estimate_normals(same, np.inf, 30) == [0.0, 0.0, 1.0]).all()
    pr = np.tile([0.6, 0.0, -0.8], (50, 1))
    assert (ref.estimate_normals(same, np.inf, 30, pr) == pr).all()
    # priors orient: the opposite prior flips every normal
    n0 = ref.estimate_normals(p, np.inf, 30)
    assert (ref.estimate_normals(p, np.inf, 30, -n0) == -n0).all()
    assert (ref.estimate_normals(p, np.inf, 30, n0) == n0).all()
    # no priors: the largest-magnitude component is positive
    s = ref.estimate_normals(sphere(3000), np.inf, 30)
    big = s[np.arange(len(s)), np.argmax(np.abs(s), axis=1)]
    assert (big > 0).all()


def blob(n=30000, seed=11):
    """An ellipsoid with unequal axes on a floor: no continuous symmetry, so every degree of freedom is constrained."""
    rng = np.random.default_rng(seed)
    v = rng.normal(size=(n // 2, 3))
    v = v / np.linalg.norm(v, axis=1, keepdims=True) * np.array([0.3, 0.2, 0.15]) + np.array([0.0, 0.0, 0.16])
    f = np.zeros((n - n // 2, 3))
    f[:, :2] = rng.random((n - n // 2, 2)) * 0.8 - 0.4
    return np.concatenate([v, f])


def known_motion():
    a = 0.03
    T = np.eye(4)
    T[:3, :3] = [[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]
    T[:3, 3] = [0.01, -0.008, 0.005]
    return T


def moved(p, T):
    return p @ T[:3, :3].T + T[:3, 3]


def point_to_point_iterations(src, tgt, thr, max_iteration=2000):
    """Open3D's RegistrationICP with the point-to-point (Umeyama) estimate, in NumPy: the iteration count from a start."""
    from otslam_b200.o3d_compat.pipelines import TransformationEstimationPointToPoint
    tree = cKDTree(tgt)
    cur, T = src.copy(), np.eye(4)

    def evaluate():
        d, j = tree.query(cur, distance_upper_bound=thr)
        ok = np.isfinite(d)
        return ok, j, (ok.sum() / len(cur)), (np.sqrt((d[ok] ** 2).mean()) if ok.any() else 0.0)

    ok, j, fit, rmse = evaluate()
    for it in range(max_iteration):
        U = TransformationEstimationPointToPoint.compute_transformation(cur[ok], tgt[j[ok]])
        T, cur = U @ T, moved(cur, U)
        f0, r0 = fit, rmse
        ok, j, fit, rmse = evaluate()
        if abs(f0 - fit) < 1e-6 and abs(r0 - rmse) < 1e-6:
            return it + 1, T
    return max_iteration, T


def test_point_to_plane_recovers_a_known_motion():
    tgt = blob()
    tn = ref.estimate_normals(tgt, np.inf, 30)
    T_true = known_motion()
    src = moved(tgt[::2], np.linalg.inv(T_true))
    r = ref.icp_point_to_plane(src, tgt, tn, 0.05, np.eye(4), max_iteration=2000)
    assert np.abs(r["transformation"] - T_true).max() < 1e-4
    assert r["fitness"] > 0.99
    c = r["corr"]
    assert (c >= 0).mean() == r["fitness"]
    it_pp, T_pp = point_to_point_iterations(src, tgt, 0.05)
    assert r["iterations"] * 3 < it_pp, (r["iterations"], it_pp)


def test_single_plane_is_rank_deficient_and_stops_with_the_identity():
    p, nrm = tilted_plane(3000)
    tn = np.tile(nrm, (len(p), 1))
    init = known_motion()
    r = ref.icp_point_to_plane(p[::3], p, tn, 0.2, init, max_iteration=30)
    # a plane leaves three degrees of freedom unconstrained: every solve fails, every update is the identity
    assert (r["transformation"] == init).all()
    assert r["iterations"] == 1


def test_no_correspondences_returns_the_init():
    p, nrm = tilted_plane(1000)
    tn = np.tile(nrm, (len(p), 1))
    init = known_motion()
    r = ref.icp_point_to_plane(p + 10.0, p, tn, 0.05, init, max_iteration=30)
    assert (r["transformation"] == init).all() and r["fitness"] == 0.0 and r["inlier_rmse"] == 0.0
    assert (r["corr"] == -1).all()
    e = ref.icp_point_to_plane(p, np.zeros((0, 3)), np.zeros((0, 3)), 0.05, init, max_iteration=30)
    assert (e["transformation"] == init).all() and e["fitness"] == 0.0


def test_argument_checks_before_any_cuda_call():
    from otslam_b200 import _lib
    L = _lib.lib
    p = np.zeros((4, 3))
    out = np.empty((4, 3))
    ok = dict(points=_lib.ptr(p), n=4, prior=None, radius=float("inf"), max_nn=30, out=_lib.ptr(out))

    def normals(**kw):
        a = dict(ok, **kw)
        return L.otslam_cloud_estimate_normals(a["points"], a["n"], a["prior"], a["radius"], a["max_nn"], a["out"], 0)

    for bad in (dict(max_nn=0), dict(max_nn=129), dict(radius=0.0), dict(radius=-1.0), dict(radius=float("nan")),
                dict(radius=float("-inf")), dict(points=None), dict(out=None), dict(n=-1), dict(n=1 << 31)):
        assert normals(**bad) == _lib.ERR_INVALID, bad
    assert "max_nn" in (normals(max_nn=200) and _lib.last_error())
    T = np.eye(4).reshape(16)
    To = np.empty(16)

    def icp(src=_lib.ptr(p), ns=4, tgt=_lib.ptr(p), tn=_lib.ptr(p), nt=4, d=0.1, init=_lib.ptr(T), rf=1e-6, rr=1e-6, it=30,
            out=_lib.ptr(To)):
        return L.otslam_cloud_icp_point_to_plane(src, ns, tgt, tn, nt, d, init, rf, rr, it, out, None, None, None, None, 0)

    bad_init = np.full(16, np.nan)
    for bad in (dict(src=None), dict(tgt=None), dict(tn=None), dict(init=None), dict(out=None), dict(ns=-1), dict(nt=-1),
                dict(d=0.0), dict(d=float("inf")), dict(d=float("nan")), dict(rf=-1.0), dict(rr=float("nan")), dict(it=-1),
                dict(init=_lib.ptr(bad_init)), dict(ns=1 << 31)):
        assert icp(**bad) == _lib.ERR_INVALID, bad
    # an empty source needs no device: init comes back, 0 iterations
    fit, it = C.c_double(1.0), C.c_int32(5)
    T2 = np.arange(16.0)
    T2[12:] = [0, 0, 0, 1]
    assert L.otslam_cloud_icp_point_to_plane(None, 0, None, None, 0, 0.1, _lib.ptr(T2), 1e-6, 1e-6, 30, _lib.ptr(To), C.byref(fit),
                                             None, C.byref(it), None, 0) == _lib.OK
    assert (To == T2).all() and fit.value == 0.0 and it.value == 0
    assert normals(n=0) == _lib.OK


def test_compat_search_params_and_orientation():
    import otslam_b200.o3d_compat as o3d
    with pytest.raises(RuntimeError, match="128"):
        o3d.geometry.KDTreeSearchParamRadius(0.05)
    assert o3d.geometry.KDTreeSearchParamKNN()._radius_max_nn() == (np.inf, 30)
    assert o3d.geometry.KDTreeSearchParamHybrid(0.02, 30)._radius_max_nn() == (0.02, 30)
    with pytest.raises(RuntimeError):
        o3d.pipelines.registration.TransformationEstimationPointToPlane(kernel=object())
    pc = o3d.geometry.PointCloud(np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0], [0.0, 2.0, 0.0]]))
    with pytest.raises(RuntimeError, match="EstimateNormals"):
        pc.orient_normals_to_align_with_direction()
    pc.normals = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    pc.orient_normals_towards_camera_location((0.0, 0.0, 0.0))
    assert (np.asarray(pc.normals) == [[0.0, 0.0, -1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]]).all()
    pc.orient_normals_to_align_with_direction((0.0, 1.0, 0.0))
    assert (np.asarray(pc.normals) == [[0.0, 0.0, -1.0], [-1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]).all()
    pc.normals = np.zeros((3, 3))
    pc.orient_normals_to_align_with_direction((0.0, 0.0, 2.0))
    assert (np.asarray(pc.normals) == [0.0, 0.0, 2.0]).all()
    tgt = o3d.geometry.PointCloud(np.zeros((4, 3)))
    with pytest.raises(RuntimeError, match="require pre-computed normal vectors for target PointCloud"):
        o3d.pipelines.registration.registration_icp(pc, tgt, 0.05, np.eye(4),
                                                    o3d.pipelines.registration.TransformationEstimationPointToPlane())
