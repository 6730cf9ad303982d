"""otslam_cloud_cluster_dbscan and otslam_cloud_segment_plane on the GPU equal their CPU model (tests/models/segment_model.cpp)
bit for bit: labels and cluster counts; plane, inliers and hypotheses evaluated.  Clouds: mesh samples (2e5 and 1e6) of a
chair + table reconstruction, the adversarial DBSCAN clouds of test_segment_oracle and the cloud_ref sets.  Also: device
pointers give the host-pointer results, the DeviceCloud chain gives the compat results, and on the chair + table samples the
plane is the floor and the two largest clusters are the table and the chair."""
import ctypes as C

import numpy as np
import pytest

import cloud_ref
import segment_ref as ref
from oracle import oracle
from test_segment_oracle import chain, dbscan_clouds, noisy_plane

pytestmark = pytest.mark.gpu

TABLE_XY = ((-0.6, 0.6), (-0.4, 0.4))            # synth.table(0, 0) and synth.chair(0, -0.85) footprints
CHAIR_XY = ((-0.225, 0.225), (-1.075, -0.625))


def gpu_dbscan(p, eps, min_points):
    from otslam_b200 import _lib
    p = np.ascontiguousarray(p, np.float64)
    lab = np.empty(len(p), np.int32)
    nc = C.c_int32()
    _lib.check(_lib.lib.otslam_cloud_cluster_dbscan(_lib.ptr(p), len(p), float(eps), int(min_points), _lib.ptr(lab), C.byref(nc), 0))
    return lab, nc.value


def gpu_plane(p, thr, r, iters, probability=0.99999999, seed=0):
    from otslam_b200 import _lib
    p = np.ascontiguousarray(p, np.float64)
    plane = np.empty(4)
    inl = np.empty(len(p), np.int64)
    m, ev = C.c_int64(), C.c_int32()
    _lib.check(_lib.lib.otslam_cloud_segment_plane(_lib.ptr(p), len(p), float(thr), int(r), int(iters), float(probability),
                                                   C.c_uint64(seed), _lib.ptr(plane), _lib.ptr(inl), C.byref(m), C.byref(ev), 0))
    return {"plane": plane, "inliers": inl[:m.value].copy(), "n_evaluated": ev.value}


def same_plane(got, want):
    assert (got["plane"].view(np.uint64) == want["plane"].view(np.uint64)).all(), (got["plane"], want["plane"])
    assert got["n_evaluated"] == want["n_evaluated"]
    assert len(got["inliers"]) == len(want["inliers"]) and (got["inliers"] == want["inliers"]).all()


@pytest.fixture(scope="module")
def chair_table():
    """{n: mesh samples} of the chair + table scene (every 10th of 300 frames, 1 cm voxels), n = 2e5 and 1e6."""
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq = synth.make_sequence("chair_table", 300, subsample=(0, 10))
    d, c = seq.numpy()
    v = TSDFVolume(0.01, 0.04)
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    verts, cols, nrm, faces, _ = v.extract_triangle_mesh()
    v.close()
    return {n: oracle.sample_uniform(verts, cols, nrm, faces, n, seed=3)[0] for n in (200_000, 1_000_000)}


@pytest.mark.parametrize("n", [200_000, 1_000_000])
def test_chair_table_equals_the_model_and_separates_the_objects(chair_table, n):
    p = chair_table[n]
    want = ref.segment_plane(p, 0.01, 3, 1000, seed=7)
    got = gpu_plane(p, 0.01, 3, 1000, seed=7)
    same_plane(got, want)
    a, b, c, d = got["plane"]
    assert abs(c) > 0.99 and abs(d) < 0.01                      # the floor z = 0
    rest = np.delete(p, got["inliers"], axis=0)
    lab, nc = gpu_dbscan(rest, 0.02, 10)
    wl, wn = ref.cluster_dbscan(rest, 0.02, 10)
    assert nc == wn and (lab == wl).all()
    sizes = np.bincount(lab[lab >= 0])
    top = np.argsort(-sizes, kind="stable")[:2]
    boxes = []
    for L in top:
        q = rest[lab == L]
        boxes.append((q[:, 0].min(), q[:, 0].max(), q[:, 1].min(), q[:, 1].max()))

    def inside(box, fp, margin=0.03):
        return (fp[0][0] - margin <= box[0] and box[1] <= fp[0][1] + margin and fp[1][0] - margin <= box[2] and box[3] <= fp[1][1] + margin)
    assert sorted([inside(bx, TABLE_XY) for bx in boxes]) == [False, True]
    assert sorted([inside(bx, CHAIR_XY) for bx in boxes]) == [False, True]
    # the full hypothesis budget and the other parameters
    same_plane(gpu_plane(p, 0.01, 3, 1000, probability=1.0, seed=7), ref.segment_plane(p, 0.01, 3, 1000, probability=1.0, seed=7))
    if n == 200_000:
        same_plane(gpu_plane(p, 0.005, 6, 300, 0.999, seed=9), ref.segment_plane(p, 0.005, 6, 300, 0.999, seed=9))
        lab, nc = gpu_dbscan(p, 0.015, 20)
        wl, wn = ref.cluster_dbscan(p, 0.015, 20)
        assert nc == wn and (lab == wl).all()


ADVERSARIAL = dict(dbscan_clouds())
ADVERSARIAL.update({
    "chain": (chain(), 0.01, 2),
    "lattice_min1": (cloud_ref.lattice(), cloud_ref.H * 1.5, 1),
    "collinear": (cloud_ref.collinear(), 0.01, 5),
    "coplanar": (cloud_ref.coplanar(), 0.02, 6),
    "line_on_faces": (cloud_ref.line_on_faces(), cloud_ref.H * 1.01, 3),
    "mirrored_lattice": (cloud_ref.mirrored(cloud_ref.lattice()), cloud_ref.H * 2, 20),
    "min_points_0": (cloud_ref.two_clusters(), 0.05, 0),
    "min_points_n": (cloud_ref.two_clusters(), 100.0, len(cloud_ref.two_clusters())),
    "min_points_n1": (cloud_ref.two_clusters(), 100.0, len(cloud_ref.two_clusters()) + 1),
})


@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
def test_adversarial_dbscan_equals_the_model(name):
    p, eps, mp = ADVERSARIAL[name]
    lab, nc = gpu_dbscan(p, eps, mp)
    wl, wn = ref.cluster_dbscan(p, eps, mp)
    assert nc == wn and (lab == wl).all()


PLANE_CLOUDS = {
    "noisy_plane": lambda: noisy_plane(20000, 0.5),
    "coplanar": lambda: cloud_ref.coplanar(),
    "collinear": lambda: cloud_ref.collinear(),
    "lattice": lambda: cloud_ref.lattice(),
    "duplicates": lambda: cloud_ref.with_duplicates(),
    "identical": lambda: cloud_ref.identical(300),
    "outliers": lambda: cloud_ref.surface_with_outliers(),
    "two_clusters": lambda: cloud_ref.two_clusters(),
}


@pytest.mark.parametrize("name", sorted(PLANE_CLOUDS))
@pytest.mark.parametrize("thr,r,iters,prob", [(0.01, 3, 1000, 0.99999999), (0.02, 3, 200, 1.0), (0.01, 5, 150, 0.999), (0.0, 3, 50, 0.9),
                                              (0.01, 3, 0, 0.9), (0.01, 16, 70, 0.99)])
def test_adversarial_planes_equal_the_model(name, thr, r, iters, prob):
    p = PLANE_CLOUDS[name]()
    same_plane(gpu_plane(p, thr, r, iters, prob, seed=5), ref.segment_plane(p, thr, r, iters, prob, seed=5))


def test_points_on_a_plane_and_on_a_line():
    rng = np.random.default_rng(8)
    p = np.column_stack([rng.uniform(-1, 1, (5000, 2)), np.zeros(5000)])
    got = gpu_plane(p, 0.01, 3, 1000, seed=4)
    same_plane(got, ref.segment_plane(p, 0.01, 3, 1000, seed=4))
    assert got["n_evaluated"] == 1 and list(got["plane"]) == [0.0, 0.0, 1.0, 0.0]
    line = np.column_stack([rng.uniform(-1, 1, 3000), np.zeros(3000), np.zeros(3000)])
    got = gpu_plane(line, 0.01, 3, 100, seed=1)
    assert got["n_evaluated"] == 100 and len(got["inliers"]) == 0 and not got["plane"].any()


def test_device_pointers_give_the_host_results(chair_table):
    import torch
    from otslam_b200 import _lib
    p = chair_table[200_000]
    want_p = gpu_plane(p, 0.01, 3, 400, seed=3)
    want_l, want_n = gpu_dbscan(p, 0.02, 10)
    dp = torch.from_numpy(p).cuda()
    dlab = torch.empty(len(p), dtype=torch.int32, device="cuda")
    dinl = torch.empty(len(p), dtype=torch.int64, device="cuda")
    nc, m, ev = C.c_int32(), C.c_int64(), C.c_int32()
    plane = np.empty(4)
    torch.cuda.synchronize()
    _lib.check(_lib.lib.otslam_cloud_cluster_dbscan(_lib.ptr(dp), len(p), 0.02, 10, _lib.ptr(dlab), C.byref(nc), 0))
    _lib.check(_lib.lib.otslam_cloud_segment_plane(_lib.ptr(dp), len(p), 0.01, 3, 400, 0.99999999, C.c_uint64(3), _lib.ptr(plane),
                                                   _lib.ptr(dinl), C.byref(m), C.byref(ev), 0))
    assert nc.value == want_n and (dlab.cpu().numpy() == want_l).all()
    same_plane({"plane": plane, "inliers": dinl[:m.value].cpu().numpy(), "n_evaluated": ev.value}, want_p)


def test_device_cloud_chain_equals_compat(chair_table):
    import otslam_b200.o3d_compat as o3d
    from otslam_b200.cloud import DeviceCloud
    p = chair_table[200_000]
    pc = o3d.geometry.PointCloud(p)
    plane, inl = pc.segment_plane(0.01, 3, 1000, seed=7)
    rest = pc.select_by_index(inl, invert=True)
    labels = rest.cluster_dbscan(0.02, 10)
    assert isinstance(labels, np.ndarray) and labels.dtype == np.int32
    big = int(np.argmax(np.bincount(labels[labels >= 0])))
    obj = rest.select_by_index(np.nonzero(labels == big)[0])

    dc = DeviceCloud.from_numpy(p)
    dplane, dinl = dc.segment_plane(0.01, 3, 1000, seed=7)
    drest = dc.select_by_index(dinl, invert=True)
    dlabels = drest.cluster_dbscan(0.02, 10)
    dobj = drest.select_by_index((dlabels == big).nonzero().flatten())
    assert (dplane.view(np.uint64) == plane.view(np.uint64)).all() and dinl.cpu().numpy().tolist() == inl
    assert (dlabels.cpu().numpy() == labels).all()
    assert (dobj.to_numpy()[0] == np.asarray(obj.points)).all()
    # the seed through o3d.utility.random.seed, and errors with the library's message
    from otslam_b200.o3d_compat import geometry
    o3d.utility.random_seed(7)
    used = 7 + geometry._SEED_COUNTER[0]
    a = pc.segment_plane(0.01, 3, 100)
    b = pc.segment_plane(0.01, 3, 100, seed=used)
    assert (a[0] == b[0]).all() and a[1] == b[1]
    with pytest.raises(RuntimeError, match="There must be at least 'ransac_n' points."):
        o3d.geometry.PointCloud(p[:2]).segment_plane(0.01, 3, 100)
    with pytest.raises(RuntimeError, match="eps"):
        pc.cluster_dbscan(0.0, 10)
