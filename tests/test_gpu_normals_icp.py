"""otslam_cloud_estimate_normals and otslam_cloud_icp_point_to_plane on the GPU equal their CPU model
(tests/models/normals_icp_model.cpp) bit for bit: normals; ICP transform, fitness, RMSE, iterations and correspondence
indices.  Clouds: mesh samples and extract_point_cloud points of config-1 table frames, the cloud_ref adversarial sets;
max_nn 1, 3, 30, 32, 33 and 128 in k-NN and hybrid modes, with and without priors.  Also: device pointers give the
host-pointer results, and the compat registration_icp(..., TransformationEstimationPointToPlane()) recovers a motion."""
import ctypes as C

import numpy as np
import pytest

import cloud_ref
import normals_icp_ref as ref
from oracle import oracle
from test_normals_icp_oracle import blob, known_motion, moved

pytestmark = pytest.mark.gpu


def gpu_normals(p, radius=np.inf, max_nn=30, prior=None):
    from otslam_b200 import _lib
    p = np.ascontiguousarray(p, np.float64)
    pr = None if prior is None else np.ascontiguousarray(prior, np.float64)
    out = np.empty_like(p)
    _lib.check(_lib.lib.otslam_cloud_estimate_normals(_lib.ptr(p), len(p), _lib.ptr(pr), float(radius), int(max_nn), _lib.ptr(out), 0))
    return out


def gpu_icp(src, tgt, tn, dist, init, max_iteration=30, rf=1e-6, rr=1e-6):
    from otslam_b200 import _lib
    s, t, n = (np.ascontiguousarray(a, np.float64) for a in (src, tgt, tn))
    T0 = np.ascontiguousarray(init, np.float64).reshape(16)
    T = np.empty(16)
    fit, rmse, it = C.c_double(), C.c_double(), C.c_int32()
    corr = np.empty(len(s), np.int32)
    _lib.check(_lib.lib.otslam_cloud_icp_point_to_plane(_lib.ptr(s), len(s), _lib.ptr(t), _lib.ptr(n), len(t), float(dist), _lib.ptr(T0),
                                                        rf, rr, max_iteration, _lib.ptr(T), C.byref(fit), C.byref(rmse), C.byref(it),
                                                        _lib.ptr(corr), 0))
    return {"transformation": T.reshape(4, 4), "fitness": fit.value, "inlier_rmse": rmse.value, "iterations": it.value, "corr": corr}


def same_icp(a, b):
    assert (a["transformation"] == b["transformation"]).all()
    assert a["fitness"] == b["fitness"] and a["inlier_rmse"] == b["inlier_rmse"] and a["iterations"] == b["iterations"]
    assert (a["corr"] == b["corr"]).all()


@pytest.fixture(scope="module")
def table_clouds(table_seq):
    """(mesh samples with their normals, extract_point_cloud points with TSDF normals) of three table frames."""
    from otslam_b200.volume import TSDFVolume
    seq, d, c = table_seq
    v = TSDFVolume(0.01, 0.04)
    v.integrate_batch(d[:3], c[:3], seq.fxfycxcy, seq.extrinsic[:3])
    verts, cols, nrm, faces, _ = v.extract_triangle_mesh()
    sp, _, sn, _ = oracle.sample_uniform(verts, cols, nrm, faces, 30000, seed=11)
    p, _, _, pn = v.extract_point_cloud(normals=True)
    v.close()
    return sp, sn, p, pn


CASES = [(np.inf, 1), (np.inf, 3), (np.inf, 30), (np.inf, 32), (np.inf, 33), (np.inf, 128), (0.02, 1), (0.02, 3), (0.02, 30),
         (0.02, 32), (0.02, 33), (0.02, 128)]


@pytest.mark.parametrize("radius,max_nn", CASES)
@pytest.mark.parametrize("which", ["samples", "extracted"])
def test_table_normals_equal_the_model(table_clouds, which, radius, max_nn):
    sp, sn, p, pn = table_clouds
    pts, prior = (sp, sn) if which == "samples" else (p, pn)
    for pr in (None, prior):
        want = ref.estimate_normals(pts, radius, max_nn, pr)
        got = gpu_normals(pts, radius, max_nn, pr)
        assert (got.view(np.uint64) == want.view(np.uint64)).all(), (which, radius, max_nn, pr is None)


ADVERSARIAL = {
    "lattice": lambda: cloud_ref.lattice(),
    "duplicates": lambda: cloud_ref.with_duplicates(),
    "identical": lambda: cloud_ref.identical(300),
    "collinear": lambda: cloud_ref.collinear(),
    "coplanar": lambda: cloud_ref.coplanar(),
    "line_on_faces": lambda: cloud_ref.line_on_faces(),
    "two_clusters": lambda: cloud_ref.two_clusters(),
    "outliers": lambda: cloud_ref.surface_with_outliers(),
    "mirrored_lattice": lambda: cloud_ref.mirrored(cloud_ref.lattice()),
}


@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
@pytest.mark.parametrize("radius,max_nn", [(np.inf, 1), (np.inf, 3), (np.inf, 32), (np.inf, 33), (np.inf, 128),
                                           (3 * cloud_ref.H, 30), (2 * cloud_ref.H, 128)])
def test_adversarial_normals_equal_the_model(name, radius, max_nn):
    p = ADVERSARIAL[name]()
    prior = np.tile([0.0, 0.0, -1.0], (len(p), 1))
    for pr in (None, prior):
        want = ref.estimate_normals(p, radius, max_nn, pr)
        got = gpu_normals(p, radius, max_nn, pr)
        assert (got.view(np.uint64) == want.view(np.uint64)).all(), (name, radius, max_nn, pr is None)


def test_icp_equals_the_model(table_clouds):
    sp, sn, p, pn = table_clouds
    T_true = known_motion()
    tn = ref.estimate_normals(sp, np.inf, 30)
    src = moved(sp[::2], np.linalg.inv(T_true))
    want = ref.icp_point_to_plane(src, sp, tn, 0.05, np.eye(4), max_iteration=2000)
    got = gpu_icp(src, sp, tn, 0.05, np.eye(4), max_iteration=2000)
    same_icp(got, want)
    assert np.abs(got["transformation"] - T_true).max() < 1e-3 and got["fitness"] > 0.99
    # the extracted cloud with its TSDF normals as the target, a few iterations from a perturbed init
    init = known_motion() @ known_motion()
    same_icp(gpu_icp(p[::3], p, pn, 0.03, init, max_iteration=7), ref.icp_point_to_plane(p[::3], p, pn, 0.03, init, max_iteration=7))
    # the blob, a single plane (identity updates) and no correspondences at all
    b = blob()
    bn = ref.estimate_normals(b, np.inf, 30)
    bs = moved(b[::2], np.linalg.inv(T_true))
    same_icp(gpu_icp(bs, b, bn, 0.05, np.eye(4), 100), ref.icp_point_to_plane(bs, b, bn, 0.05, np.eye(4), max_iteration=100))
    plane = cloud_ref.coplanar()
    pln = np.tile([0.0, 0.0, 1.0], (len(plane), 1))
    same_icp(gpu_icp(plane[::2], plane, pln, 0.1, T_true, 30), ref.icp_point_to_plane(plane[::2], plane, pln, 0.1, T_true, max_iteration=30))
    same_icp(gpu_icp(bs + 10.0, b, bn, 0.05, T_true, 30), ref.icp_point_to_plane(bs + 10.0, b, bn, 0.05, T_true, max_iteration=30))
    same_icp(gpu_icp(bs, np.zeros((0, 3)), np.zeros((0, 3)), 0.05, T_true, 5),
             ref.icp_point_to_plane(bs, np.zeros((0, 3)), np.zeros((0, 3)), 0.05, T_true, max_iteration=5))


def test_device_pointers_give_the_host_results(table_clouds):
    import torch
    from otslam_b200 import _lib
    sp, sn, _, _ = table_clouds
    host = gpu_normals(sp, 0.02, 30, sn)
    dp, dn = torch.from_numpy(sp).cuda(), torch.from_numpy(sn).cuda()
    dout = torch.empty_like(dp)
    torch.cuda.synchronize()
    _lib.check(_lib.lib.otslam_cloud_estimate_normals(_lib.ptr(dp), len(sp), _lib.ptr(dn), 0.02, 30, _lib.ptr(dout), 0))
    assert (dout.cpu().numpy().view(np.uint64) == host.view(np.uint64)).all()
    src = moved(sp[::2], np.linalg.inv(known_motion()))
    want = gpu_icp(src, sp, host, 0.05, np.eye(4), 50)
    ds = torch.from_numpy(np.ascontiguousarray(src)).cuda()
    dcorr = torch.empty(len(src), dtype=torch.int32, device="cuda")
    T = np.empty(16)
    fit, rmse, it = C.c_double(), C.c_double(), C.c_int32()
    torch.cuda.synchronize()
    _lib.check(_lib.lib.otslam_cloud_icp_point_to_plane(_lib.ptr(ds), len(src), _lib.ptr(dp), _lib.ptr(dout), len(sp), 0.05,
                                                        _lib.ptr(np.eye(4).reshape(16)), 1e-6, 1e-6, 50, _lib.ptr(T), C.byref(fit),
                                                        C.byref(rmse), C.byref(it), _lib.ptr(dcorr), 0))
    same_icp({"transformation": T.reshape(4, 4), "fitness": fit.value, "inlier_rmse": rmse.value, "iterations": it.value,
              "corr": dcorr.cpu().numpy()}, want)


def test_compat_point_to_plane_recovers_the_motion(table_clouds):
    import otslam_b200.o3d_compat as o3d
    sp, _, _, _ = table_clouds
    T_true = known_motion()
    reg = o3d.pipelines.registration
    tgt = o3d.geometry.PointCloud(sp)
    src = o3d.geometry.PointCloud(sp[::2].copy())
    src.transform(np.linalg.inv(T_true))
    with pytest.raises(RuntimeError, match="require pre-computed normal vectors for target PointCloud"):
        reg.registration_icp(src, tgt, 0.05, np.eye(4), reg.TransformationEstimationPointToPlane())
    tgt.estimate_normals(o3d.geometry.KDTreeSearchParamHybrid(radius=0.05, max_nn=30))
    assert (np.asarray(tgt.normals).view(np.uint64) == ref.estimate_normals(sp, 0.05, 30).view(np.uint64)).all()
    r = reg.registration_icp(src, tgt, 0.05, np.eye(4), reg.TransformationEstimationPointToPlane(),
                             reg.ICPConvergenceCriteria(max_iteration=2000))
    assert r.fitness > 0.99 and np.abs(r.transformation - T_true).max() < 1e-3
    cs = np.asarray(r.correspondence_set)
    assert len(cs) == round(r.fitness * len(src.points)) and cs.shape[1] == 2
    pp = reg.registration_icp(src, tgt, 0.05, np.eye(4), reg.TransformationEstimationPointToPoint(),
                              reg.ICPConvergenceCriteria(max_iteration=2000))
    assert np.abs(pp.transformation - T_true).max() < 2e-3
