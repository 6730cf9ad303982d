"""Ray casting on the GPU (otslam_volume_raycast): the CUDA kernel equals the CPU model (tests/models/raycast_model.cpp on
the oracle's volume) bit for bit (colour within one level), renders the synthetic scene at its analytic depth, gives the
same bits however it is called, and leaves the volume exactly as it was."""
import os

import numpy as np
import pytest

from conftest import ROOT, canon_mesh

pytestmark = pytest.mark.gpu

VL = 0.005
ATTRS = ("depth", "vertex", "normal", "color")


def novel(extrinsic, angle_deg=12.0, shift=(0.08, -0.05, 0.12)):
    """a pose near a capture pose: rotated about the camera's y axis and moved"""
    a = np.radians(angle_deg)
    d = np.eye(4)
    d[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
    d[:3, 3] = shift
    return d @ extrinsic


def same_bits(a, b, keys=ATTRS):
    for k in keys:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, k
        assert (np.asarray(a[k]).view(np.uint8) == np.asarray(b[k]).view(np.uint8)).all(), k


def assert_equals_oracle(g, o):
    """hit mask, depth, vertex and normal bit for bit; colour within one level (exact sums vs an FP64 running mean)"""
    gm, om = g["depth"] > 0, o["depth"] > 0
    assert gm.any() and (gm == om).all()
    for k in ("depth", "vertex", "normal"):
        assert (g[k].view(np.uint32) == o[k].view(np.uint32)).all(), k
    assert np.abs(g["color"].astype(np.int16) - o["color"].astype(np.int16)).max() <= 1


def both(depth, rgb, intr, extrinsics, voxel, trunc, views, W, H, **kw):
    """the GPU volume's render and the CPU model's render of the oracle's volume of the same frames"""
    from oracle import oracle
    from otslam_b200.volume import TSDFVolume
    from test_raycast_oracle import raycast
    gv = TSDFVolume(voxel, trunc)
    gv.integrate_batch(depth, rgb, intr, extrinsics)
    ov = oracle.Volume(voxel, trunc)
    for k in range(len(depth)):
        ov.integrate(oracle.depth_convert(depth[k]), rgb[k], intr, extrinsics[k])
    return gv.ray_cast(intr, views, W, H, **kw), raycast(ov, intr, views, W, H, **kw)


@pytest.fixture(scope="module")
def window():
    """64 contiguous frames of configs[1] (frames 468..531 of the 1000-frame chair+table sequence), 5 mm voxels"""
    from otslam_b200 import synth
    seq = synth.make_sequence("chair_table", 1000, poses=synth.trajectory("chair_table", 1000)[468:532], device="cuda")
    d, c = seq.numpy()
    return seq, d, c


@pytest.fixture(scope="module")
def window_volume(window):
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    v = TSDFVolume(VL, 4 * VL)
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    return v


def test_small_sequence_equals_oracle():
    z = np.load(os.path.join(ROOT, "tests", "golden", "small_sequence.npz"))
    intr, (vl, tr) = tuple(z["intr"]), z["voxel"]
    e = z["extrinsic"]
    views = np.concatenate([e, np.stack([novel(x, 20.0, (0.2, 0.0, -0.1)) for x in e])])
    H, W = z["depth"].shape[1:]
    g, o = both(z["depth"], z["rgb"], intr, e, float(vl), float(tr), views, W, H)
    assert_equals_oracle(g, o)


def test_window_equals_oracle(window):
    seq, d, c = window
    e = seq.extrinsic
    views = np.stack([e[0], e[40], novel(e[20]), novel(e[60], -15.0, (-0.1, 0.05, -0.2))])
    g, o = both(d, c, seq.fxfycxcy, e, VL, 4 * VL, views, 640, 480)
    assert_equals_oracle(g, o)


def test_hd_golden_equals_oracle():
    z = np.load(os.path.join(ROOT, "tests", "golden", "hd_sequence.npz"))
    intr, (vl, tr) = tuple(z["intr"]), z["voxel"]
    e = z["extrinsic"]
    views = np.stack([e[3], novel(e[5])])
    g, o = both(z["depth"], z["rgb"], intr, e, float(vl), float(tr), views, 1280, 720)
    assert_equals_oracle(g, o)


def test_depth_against_the_scene(window, window_volume):
    """median |rendered - analytic| <= 0.25 voxel on pixels valid in both and >= 2 px from a depth edge"""
    from scipy.ndimage import binary_dilation
    from otslam_b200 import synth
    seq, _, _ = window
    prims = synth.SCENES["chair_table"]()
    idx = [0, 21, 42, 63]
    out = window_volume.ray_cast(seq.fxfycxcy, seq.extrinsic[idx], 640, 480)
    for j, k in enumerate(idx):
        ref, _ = synth.render(prims, seq.pose_ros[k] @ synth.T_FIX, seq.intr, "cuda", depth_m=True)
        ref = ref.cpu().numpy()
        got = out["depth"][j].astype(np.float64)
        jump = np.zeros(ref.shape, bool)
        jump[:, 1:] |= np.abs(np.diff(ref, axis=1)) > 0.02
        jump[1:, :] |= np.abs(np.diff(ref, axis=0)) > 0.02
        jump |= ref == 0
        m = (got > 0) & (ref > 0) & ~binary_dilation(jump, iterations=2)
        assert m.sum() > 0.2 * m.size
        assert np.median(np.abs(got[m] - ref[m])) <= 0.25 * VL, k


def test_call_equivalences(window, window_volume, tmp_path):
    """n views in one call == n calls; host == CUDA tensors; subsets == the full call; two runs agree; save + load"""
    from otslam_b200.volume import TSDFVolume
    seq, _, _ = window
    v, intr = window_volume, seq.fxfycxcy
    views = np.stack([seq.extrinsic[5], novel(seq.extrinsic[30]), seq.extrinsic[50]])
    full = v.ray_cast(intr, views, 640, 480)
    for i in range(len(views)):
        one = v.ray_cast(intr, views[i], 640, 480)
        assert one["depth"].shape == (480, 640)
        same_bits({k: full[k][i] for k in ATTRS}, one)
    t = v.ray_cast_tensors(intr, views, 640, 480)
    same_bits(full, {k: x.cpu().numpy() for k, x in t.items()})
    for sub in (("depth",), ("normal", "color"), ("vertex",)):
        part = v.ray_cast(intr, views, 640, 480, attributes=sub)
        assert set(part) == set(sub)
        same_bits(full, part, sub)
    same_bits(full, v.ray_cast(intr, views, 640, 480))
    p = tmp_path / "v.otslam"
    v.save(p)
    w = TSDFVolume(VL, 4 * VL)
    w.load(p)
    same_bits(full, w.ray_cast(intr, views, 640, 480))


def test_many_views_chunked_host_and_device(window, window_volume):
    """more views than one staging chunk: host and device outputs agree view for view"""
    seq, _, _ = window
    views = seq.extrinsic[:40]
    h = window_volume.ray_cast(seq.fxfycxcy, views, 640, 480)
    d = window_volume.ray_cast_tensors(seq.fxfycxcy, views, 640, 480)
    same_bits(h, {k: x.cpu().numpy() for k, x in d.items()})
    assert (h["depth"] > 0).mean() > 0.5


def test_state_untouched(window):
    from otslam_b200.o3d_compat import pipelines
    seq, d, c = window
    vol = pipelines.ScalableTSDFVolume(VL, 4 * VL, pipelines.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d[:16], c[:16], _intrinsic(seq), seq.extrinsic[:16])
    stats = vol._vol.stats()
    lazy = vol.extract_triangle_mesh()                 # arrays still in HBM
    before = vol._vol.extract_triangle_mesh(normals=False)
    lazy2 = vol.extract_triangle_mesh()
    r = vol.ray_cast(_intrinsic(seq), seq.extrinsic[3])
    assert (r["depth"] > 0).any()
    assert vol._vol.stats() == stats
    verts, tris = np.asarray(lazy2.vertices), np.asarray(lazy2.triangles)
    after = vol._vol.extract_triangle_mesh(normals=False)
    A, B = canon_mesh(before[0], before[1], before[3], before[4]), canon_mesh(after[0], after[1], after[3], after[4])
    assert all((x == y).all() for x, y in zip(A, B))
    assert (verts == before[0]).all() and (tris == before[3]).all()
    del lazy


def _intrinsic(seq):
    from otslam_b200.o3d_compat import camera
    W, H, fx, fy, cx, cy = seq.intr
    return camera.PinholeCameraIntrinsic(W, H, fx, fy, cx, cy)


def test_slab_volume_refused_and_unchanged(window):
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    v = TSDFVolume(VL, 4 * VL, slab=(0, 8, 2, 0))
    v.integrate_batch(d[:8], c[:8], seq.fxfycxcy, seq.extrinsic[:8])
    stats, keys = v.stats(), v.export_blocks(color=False)
    with pytest.raises(RuntimeError, match="part file"):
        v.ray_cast(seq.fxfycxcy, seq.extrinsic[0], 640, 480)
    assert v.stats() == stats
    after = v.export_blocks(color=False)
    assert (keys[0] == after[0]).all() and (keys[1].view(np.uint32) == after[1].view(np.uint32)).all()


def test_arena_object_equals_own_volume(window):
    from otslam_b200.volume import ArenaView, TSDFVolume
    seq, d, c = window
    intr, e = seq.fxfycxcy, seq.extrinsic
    arena = TSDFVolume(VL, 4 * VL)
    arena.set_objects(2)
    ids = np.array([0] * 32 + [1] * 32, np.int32)
    arena.integrate_batch(d, c, intr, e, object_ids=ids)
    own = TSDFVolume(VL, 4 * VL)
    own.integrate_batch(d[:32], c[:32], intr, e[:32])
    views = np.stack([e[10], novel(e[20])])
    same_bits(own.ray_cast(intr, views, 640, 480), ArenaView(arena, 0).ray_cast(intr, views, 640, 480))
    assert (ArenaView(arena, 1).ray_cast(intr, e[40], 640, 480)["depth"] > 0).any()
    # object 1's blocks sit 2^18 blocks further along x in the shared key space: a camera of object 0 placed there sees nothing
    shift = np.eye(4)
    shift[0, 3] = -(1 << 18) * 16 * VL
    r = ArenaView(arena, 0).ray_cast(intr, e[40] @ shift, 640, 480)
    assert not r["depth"].any()


def test_nocolor_volume_renders_no_colour(window):
    from otslam_b200.volume import TSDFVolume
    seq, d, _ = window
    v = TSDFVolume(VL, 4 * VL, color=False)
    v.integrate_batch(d[:8], None, seq.fxfycxcy, seq.extrinsic[:8])
    r = v.ray_cast(seq.fxfycxcy, seq.extrinsic[4], 640, 480)
    assert (r["depth"] > 0).any() and not r["color"].any()


def test_compat_ray_cast(window, window_volume):
    from otslam_b200.o3d_compat import pipelines
    seq, d, c = window
    vol = pipelines.ScalableTSDFVolume(VL, 4 * VL, pipelines.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d, c, _intrinsic(seq), seq.extrinsic)
    got = vol.ray_cast(_intrinsic(seq), seq.extrinsic[12])
    ref = window_volume.ray_cast(seq.fxfycxcy, seq.extrinsic[12], 640, 480, depth_min=0.1, depth_max=3.0)
    same_bits(ref, got)
