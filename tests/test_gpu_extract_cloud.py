"""GPU parity for extraction (K5-K7) and the cloud operators (K1b, K8-K13) vs the oracle.
Integer / index outputs bit-exact; FP64 outputs are produced with the oracle's operation order and
are expected bit-exact too (chamfer <= 0.25 voxel is the contract's outer bound)."""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial import cKDTree

import cloud_ref
from conftest import canon_mesh, lexorder
from oracle import oracle

pytestmark = pytest.mark.gpu


def build_pair(seq, d, c, vl, slab=None):
    from otslam_b200.volume import TSDFVolume
    ov = oracle.Volume(vl, 4 * vl, slab=slab)
    for k in range(len(seq)):
        ov.integrate(oracle.depth_convert(d[k]), c[k], seq.fxfycxcy, seq.extrinsic[k])
    gv = TSDFVolume(vl, 4 * vl, slab=slab)
    gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    return gv, ov


@pytest.mark.parametrize("slab", [None, (0, 2, 2, 0), (0, 2, 2, 1), (1, 1, 3, 2)])
def test_mesh_and_points_parity(table_seq, slab):
    seq, d, c = table_seq
    vl = 0.01
    gv, ov = build_pair(seq, d, c, vl, slab)
    gverts, gcols, gnrm, gfaces, gek = gv.extract_triangle_mesh()
    overts, ocols, ofaces, oek = ov.extract_triangle_mesh()
    assert len(gverts) == len(overts) > 1000 and len(gfaces) == len(ofaces)
    A, B = canon_mesh(overts, ocols, ofaces, oek), canon_mesh(gverts, gcols, gfaces, gek)
    assert (A[3] == B[3]).all()                                  # same lattice edges
    assert (A[0] == B[0]).all()                                  # vertex positions bit-exact (<< 0.25 voxel)
    assert np.abs(A[1] - B[1]).max() <= 1e-9                     # colours (integer sums vs FP64 running mean)
    assert (A[2] == B[2]).all()                                  # same triangles, same winding
    d1 = cKDTree(overts).query(gverts)[0].mean() + cKDTree(gverts).query(overts)[0].mean()
    assert d1 <= 0.25 * vl
    assert (oracle.vertex_normals(gverts, gfaces) == gnrm).all()      # summed in triangle order: bit-exact
    gp, gc, gpe, gpn = gv.extract_point_cloud(normals=True)
    op, oc, ope = ov.extract_point_cloud()
    a, b = lexorder(ope), lexorder(gpe)
    # colours: FP32 interpolation of float-cast voxel colours on both sides (exact sum / count vs FP64 running mean: 1 ulp of float)
    assert len(gp) == len(op) and (ope[a] == gpe[b]).all() and (op[a] == gp[b]).all() and np.abs(oc[a] - gc[b]).max() <= 2e-7
    if slab is None:
        # extract_point_cloud's normals = normalised TSDF gradient (GetNormalAt); same FP64 operation order on both sides
        on = ov.point_normals(gp)
        assert np.abs(on - gpn).max() <= 1e-12
        ln = np.linalg.norm(gpn, axis=1)
        assert (np.abs(ln[ln > 0] - 1) < 1e-12).all() and (ln > 0).mean() > 0.99
    gv.close()


def test_slab_union_equals_full_volume(table_seq):
    from otslam_b200 import slab as slabmod
    seq, d, c = table_seq
    full, _ = build_pair(seq, d, c, 0.01)
    parts = [build_pair(seq, d, c, 0.01, slab=(0, 4, 3, r))[0] for r in range(3)]
    fv = full.extract_triangle_mesh(normals=False)
    merged = slabmod.merge_mesh_parts([(p[0], p[1], p[3], p[4]) for p in (v.extract_triangle_mesh(normals=False) for v in parts)])
    A, B = canon_mesh(fv[0], fv[1], fv[3], fv[4]), canon_mesh(*merged)
    assert (A[3] == B[3]).all() and (A[0] == B[0]).all() and (A[2] == B[2]).all()
    fk = {tuple(k) for k in full.export_blocks(color=False)[0].tolist()}
    pk = set()
    for v in parts:
        pk |= {tuple(k) for k in v.export_blocks(color=False)[0].tolist()}
    assert pk == fk
    for v in parts + [full]:
        v.close()


@pytest.mark.parametrize("n_ranks,thickness,axis", [(2, 1, 0), (3, 2, 0), (3, 1, 3), (4, 2, 3), (8, 1, 3)])
def test_halo_exchange_mode_equals_full_volume(table_seq, n_ranks, thickness, axis):
    """slab.halo = 0: owned blocks only during integration, boundary planes exchanged before extraction
    (ranks emulated as separate volumes on one GPU; the torch.distributed transport is covered by
    tests/test_slab_gloo.py)."""
    from otslam_b200 import slab as slabmod
    seq, d, c = table_seq
    full, _ = build_pair(seq, d, c, 0.01)
    parts = [build_pair(seq, d, c, 0.01, slab=(axis, thickness, n_ranks, r, 0))[0] for r in range(n_ranks)]
    n_owned = [v.num_blocks() for v in parts]
    assert sum(n_owned) == full.num_blocks()                        # a true partition: no replicated integration
    assert sum(v.stats()["weight_sum"] for v in parts) == full.stats()["weight_sum"]
    exports = [v.halo_export() for v in parts]
    for r, v in enumerate(parts):
        for src, (keys, dest, planes) in enumerate(exports):
            sel = dest == r
            assert src != r or not sel.any()
            if sel.any():
                v.halo_import(keys[sel], planes[sel])
    assert all(v.num_blocks() >= n for v, n in zip(parts, n_owned)) and sum(v.num_blocks() for v in parts) > sum(n_owned)
    fv = full.extract_triangle_mesh(normals=False)
    merged = slabmod.merge_mesh_parts([(p[0], p[1], p[3], p[4]) for p in (v.extract_triangle_mesh(normals=False) for v in parts)])
    A, B = canon_mesh(fv[0], fv[1], fv[3], fv[4]), canon_mesh(*merged)
    assert len(A[0]) == len(B[0]) and (A[3] == B[3]).all() and (A[0] == B[0]).all() and (A[2] == B[2]).all()
    assert np.abs(A[1] - B[1]).max() == 0.0
    fp, fc, fe = full.extract_point_cloud()
    pp = [v.extract_point_cloud() for v in parts]
    pe = np.concatenate([p[2] for p in pp])
    a, b = lexorder(fe), lexorder(pe)
    assert len(fe) == len(pe) and (fe[a] == pe[b]).all() and (fp[a] == np.concatenate([p[0] for p in pp])[b]).all()
    for v in parts + [full]:
        v.close()


def test_empty_volume_extraction():
    from otslam_b200.volume import TSDFVolume
    v = TSDFVolume(0.01, 0.04)
    verts, cols, nrm, faces, ek = v.extract_triangle_mesh()
    assert len(verts) == 0 and len(faces) == 0
    assert len(v.extract_point_cloud()[0]) == 0
    v.close()


@pytest.fixture(scope="module")
def mesh(table_seq):
    seq, d, c = table_seq
    ov = oracle.Volume(0.01, 0.04)
    for k in range(3):
        ov.integrate(oracle.depth_convert(d[k]), c[k], seq.fxfycxcy, seq.extrinsic[k])
    v, col, f, ek = ov.extract_triangle_mesh()
    return v, col, f, oracle.vertex_normals(v, f)


def test_backproject_and_depth_convert(table_seq):
    import otslam_b200.o3d_compat as o3d
    seq, d, c = table_seq
    rgbd = o3d.geometry.RGBDImage.create_from_color_and_depth(o3d.geometry.Image(c[0]), o3d.geometry.Image(d[0]), 1000.0, 5.0, False)
    intr = o3d.camera.PinholeCameraIntrinsic(640, 480, *seq.fxfycxcy)
    for ext in (None, seq.extrinsic[0]):
        pc = o3d.geometry.PointCloud.create_from_rgbd_image(rgbd, intr) if ext is None else \
            o3d.geometry.PointCloud.create_from_rgbd_image(rgbd, intr, ext)
        op, oc = oracle.backproject_rgbd(oracle.depth_convert(d[0], 1000.0, 5.0), c[0], seq.fxfycxcy, ext)
        assert len(pc.points) == len(op) and (pc.points == op).all() and (pc.colors == oc).all()


def test_vertex_normals_and_sampling(mesh):
    import otslam_b200.o3d_compat as o3d
    v, col, f, n = mesh
    m = o3d.geometry.TriangleMesh()
    m.vertices, m.vertex_colors, m.triangles = v, col, f
    m.compute_vertex_normals()
    assert (np.asarray(m.vertex_normals) == n).all()
    m.vertex_normals = n
    pc = m.sample_points_uniformly(number_of_points=100000, seed=11)
    op, oc, on, tri = oracle.sample_uniform(v, col, n, f, 100000, seed=11)
    assert (pc.points == op).all() and (pc.colors == oc).all() and (pc.normals == on).all()   # same counter RNG -> point by point
    pc2 = m.sample_points_uniformly(number_of_points=100000, seed=12)
    assert not (pc2.points == op).all()
    d2 = cKDTree(op).query(pc2.points)[0].mean() + cKDTree(pc2.points).query(op)[0].mean()
    assert d2 <= 0.25 * 0.01 * 2 * 4                              # different seeds: same surface
    with pytest.raises(RuntimeError):
        o3d.geometry.TriangleMesh().sample_points_uniformly(10)
    with pytest.raises(RuntimeError):
        m.sample_points_uniformly(0)


def test_zfilter_vds_sor(mesh):
    import otslam_b200.o3d_compat as o3d
    from otslam_b200 import _lib
    v, col, f, n = mesh
    pts, cols, _, _ = oracle.sample_uniform(v, col, None, f, 60000, seed=1)
    zp, zc = oracle.zfilter(pts, cols, 0.03)
    gp, gc, m = np.empty_like(pts), np.empty_like(cols), C.c_int64(0)
    _lib.check(_lib.lib.otslam_cloud_zfilter(_lib.ptr(pts), _lib.ptr(cols), len(pts), 0.03, _lib.ptr(gp), _lib.ptr(gc), C.byref(m), 0))
    assert m.value == len(zp) and (gp[:m.value] == zp).all() and (gc[:m.value] == zc).all()
    pc = o3d.geometry.PointCloud(); pc.points, pc.colors = zp, zc
    for vs in (0.01, 0.037):
        ds = pc.voxel_down_sample(vs)
        op, oc, ok, on = oracle.voxel_down_sample(zp, zc, vs)
        assert len(ds.points) == len(op) and (ds.points == op).all() and (ds.colors == oc).all()
    gk = np.empty((len(zp), 3), np.int32); gn = np.empty(len(zp), np.int32)
    _lib.check(_lib.lib.otslam_cloud_voxel_down_sample(_lib.ptr(zp), None, len(zp), 0.037, _lib.ptr(gp), None, _lib.ptr(gk), _lib.ptr(gn), C.byref(m), 0))
    assert (gk[:m.value] == ok).all() and (gn[:m.value] == on).all()            # voxel keys and counts bit-exact
    rng = np.random.default_rng(0)
    noisy = zp.copy()
    noisy[::61] += rng.normal(0, 0.08, noisy[::61].shape)
    noisy[10] = noisy[11]                                                        # duplicate point
    for k, ratio in ((20, 2.0), (8, 1.0), (100, 2.5)):
        sel, idx = (lambda r: (r[0], np.array(r[1])))(o3d.geometry.PointCloud(noisy).remove_statistical_outlier(k, ratio))
        oi, odb = oracle.remove_statistical_outlier(noisy, k, ratio)
        assert len(idx) == len(oi) and (idx == oi).all()                         # kept indices bit-exact
        assert (sel.points == noisy[oi]).all()
    with pytest.raises(RuntimeError):
        o3d.geometry.PointCloud(noisy).remove_statistical_outlier(0, 1.0)
    with pytest.raises(RuntimeError):
        pc.voxel_down_sample(0.0)
    tiny = o3d.geometry.PointCloud(noisy[:5])
    sel, idx = tiny.remove_statistical_outlier(20, 2.0)                          # fewer points than neighbours
    assert idx == oracle.remove_statistical_outlier(noisy[:5], 20, 2.0)[0].tolist()


def test_point_cloud_distance_vs_ckdtree(mesh):
    """eval metric (accuracy / completeness = mean nearest-neighbour distance both ways)."""
    import otslam_b200.o3d_compat as o3d
    v, col, f, n = mesh
    a, _, _, _ = oracle.sample_uniform(v, None, None, f, 30000, seed=2)
    b, _, _, _ = oracle.sample_uniform(v, None, None, f, 50000, seed=3)
    b = b + np.array([0.3, -0.2, 0.05])                       # partially overlapping: queries outside the target grid too
    pa, pb = o3d.geometry.PointCloud(a), o3d.geometry.PointCloud(b)
    d_ab = pa.compute_point_cloud_distance(pb)
    d_ba = pb.compute_point_cloud_distance(pa)
    # exact FP64 in the (dx^2 + dy^2) + dz^2 order: bit-exact against the reference (brute force on a sample ties it down)
    ref_ab, ref_ba = cloud_ref.nn_distance_large(a, b), cloud_ref.nn_distance_large(b, a)
    assert (ref_ab[:2000] == cloud_ref.nn_distance(a[:2000], b)).all() and (ref_ba[:2000] == cloud_ref.nn_distance(b[:2000], a)).all()
    assert (d_ab == ref_ab).all() and (d_ba == ref_ba).all()
    assert np.allclose(d_ab, cKDTree(b).query(a)[0], rtol=1e-12, atol=1e-15)
    assert np.allclose(d_ba, cKDTree(a).query(b)[0], rtol=1e-12, atol=1e-15)
    assert (pa.compute_point_cloud_distance(pa) == 0).all()
    with pytest.raises(RuntimeError):
        pa.compute_point_cloud_distance(o3d.geometry.PointCloud())


def test_grid_points_and_merge_pack(tmp_path):
    import otslam_b200.o3d_compat as o3d
    from otslam_b200 import _lib, synth
    img = synth.occupancy_map(701, 533, 0.02, 3)
    og = oracle.grid_to_points(img, 0.05, -17.3, -13.1, 100)
    gg, m = np.empty((img.size, 3)), C.c_int64(0)
    _lib.check(_lib.lib.otslam_grid_to_points(_lib.ptr(img), 701, 533, 0.05, -17.3, -13.1, 100, _lib.ptr(gg), C.byref(m), 0))
    assert m.value == len(og) and (gg[:m.value] == og).all()
    rng = np.random.default_rng(4)
    clouds = [og, rng.normal(size=(1000, 3)), rng.normal(size=(777, 3)), np.zeros((0, 3))]
    paint = [[0.2, 0.2, 0.2], [1, 0, 0], [1, 0, 0], [0, 1, 0]]
    rec = o3d.io.pack_cloud_records(clouds, paint=paint)
    ref = np.concatenate([oracle.pack_ply_cloud(c, np.tile(p, (len(c), 1))) for c, p in zip(clouds, paint)])
    assert rec.shape == ref.shape and (rec == ref).all()                         # PLY bytes identical
    cols = [rng.random((len(c), 3)) * 1.2 - 0.1 for c in clouds]                 # includes out-of-range colours (clamped)
    rec2 = o3d.io.pack_cloud_records(clouds, colors_list=cols)
    ref2 = np.concatenate([oracle.pack_ply_cloud(c, k) for c, k in zip(clouds, cols)])
    assert (rec2 == ref2).all()
    pc = o3d.geometry.PointCloud(); pc.points = clouds[1]; pc.colors = np.clip(cols[1], 0, 1)
    p = str(tmp_path / "x.ply")
    o3d.io.write_point_cloud(p, pc)
    back = o3d.io.read_point_cloud(p)
    assert (back.points == pc.points).all() and np.abs(back.colors - pc.colors).max() <= 0.5 / 255 + 1e-12
    assert len(open(p, "rb").read().split(b"end_header\n", 1)[1]) == 27 * 1000


def test_scratch_cache_and_operator_timer():
    """Operators reuse cached device blocks (csrc/scratch.cu) and report the device time of their kernel section."""
    import otslam_b200.o3d_compat as o3d
    from otslam_b200 import _lib
    rng = np.random.default_rng(5)
    pc = o3d.geometry.PointCloud()
    pc.points = rng.random((50000, 3))
    a = pc.voxel_down_sample(0.05)
    assert 0.0 < _lib.last_op_device_ms() < 1000.0
    assert _lib.lib.otslam_trim_scratch() == 0                 # cache back to the driver ...
    b = pc.voxel_down_sample(0.05)                             # ... and the operators still work, same result
    assert (np.asarray(a.points) == np.asarray(b.points)).all()
    want, _, _, _ = oracle.voxel_down_sample(np.asarray(pc.points), None, 0.05)
    assert (np.asarray(b.points) == want).all()


def test_icp_point_to_point_recovers_a_known_motion(mesh):
    """o3d.pipelines.registration.registration_icp as eval_table_chair.py:90-104 calls it (point-to-point, identity init,
    max_iteration=2000): correspondences (otslam_cloud_nn_within) equal a cKDTree radius-bounded nearest-neighbour search,
    and ICP undoes a small known rigid motion of the cloud."""
    import otslam_b200.o3d_compat as o3d
    from otslam_b200 import _lib
    v, col, f, nrm = mesh
    op, _, _, _ = oracle.sample_uniform(v, col, nrm, f, 30000, seed=11)
    rng = np.random.default_rng(5)
    # correspondences: nearest target strictly within the radius, -1 otherwise
    q = op[:5000] + rng.normal(scale=0.01, size=(5000, 3))
    idx = np.empty(len(q), np.int32); d2 = np.empty(len(q))
    _lib.check(_lib.lib.otslam_cloud_nn_within(_lib.ptr(np.ascontiguousarray(q)), len(q), _lib.ptr(op), len(op), 0.012, _lib.ptr(idx),
                                               _lib.ptr(d2), 0))
    dist, nn = cKDTree(op).query(q)
    inside = dist < 0.012
    assert (idx >= 0).sum() == inside.sum() and ((idx >= 0) == inside).all()
    diff = np.linalg.norm(q[inside] - op[idx[inside]], axis=1)
    assert np.abs(diff - dist[inside]).max() <= 1e-12 and np.abs(np.sqrt(d2[inside]) - dist[inside]).max() <= 1e-12
    # ICP: target = the cloud, source = the cloud moved by a small rotation + translation
    a = 0.03
    R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
    T_true = np.eye(4); T_true[:3, :3] = R; T_true[:3, 3] = [0.01, -0.008, 0.005]
    src = o3d.geometry.PointCloud(op[::2].copy())
    src.transform(np.linalg.inv(T_true))
    tgt = o3d.geometry.PointCloud(op)
    reg = o3d.pipelines.registration.registration_icp(
        src, tgt, 0.05, np.eye(4), o3d.pipelines.registration.TransformationEstimationPointToPoint(),
        o3d.pipelines.registration.ICPConvergenceCriteria(max_iteration=2000))
    assert reg.fitness > 0.99 and reg.inlier_rmse < 2e-3
    assert np.abs(reg.transformation - T_true).max() < 2e-3
    before = o3d.pipelines.registration.evaluate_registration(src, tgt, 0.05)
    assert before.inlier_rmse > 3 * reg.inlier_rmse and len(reg.correspondence_set) >= len(before.correspondence_set)
    src.transform(reg.transformation)                                           # eval_table_chair.py:103
    assert src.compute_point_cloud_distance(tgt).mean() < 1e-3
