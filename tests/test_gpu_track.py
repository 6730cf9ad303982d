"""Frame-to-model tracking on the GPU (otslam_volume_track): the CUDA kernels equal the CPU model
(tests/models/track_model.cpp on the oracle's volume) bit for bit, recover perturbed poses of the synthetic scene, hold
drift down in a track -> integrate loop, give the same bits however they are called, and leave the volume as it was."""
import os

import numpy as np
import pytest

from conftest import ROOT, canon_mesh
from test_track_oracle import perturb, pose_error, rot

pytestmark = pytest.mark.gpu

VL = 0.005
OUTS = ("extrinsic", "status", "iterations", "fitness", "inlier_rmse")


def same_bits(a, b):
    for k in OUTS:
        x, y = np.atleast_1d(a[k]), np.atleast_1d(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape, k
        assert (x.view(np.uint8) == y.view(np.uint8)).all(), k


def seeded_starts(extrinsics, seed, cm=(1.0, 3.0), deg=(1.0, 2.0)):
    """each extrinsic moved by 1-3 cm and turned by 1-2 degrees, in seeded random directions"""
    rng = np.random.default_rng(seed)
    out = []
    for e in extrinsics:
        d = rng.normal(size=3)
        out.append(perturb(e, rng.normal(size=3), rng.uniform(*deg) * rng.choice([-1, 1]),
                           d / np.linalg.norm(d) * rng.uniform(*cm) / 100))
    return np.stack(out)


def both(depth, rgb, intr, extrinsics, voxel, trunc, frames, inits, **kw):
    """the GPU volume's tracking and the CPU model's tracking on the oracle's volume of the same frames"""
    from oracle import oracle
    from otslam_b200.volume import TSDFVolume
    from test_track_oracle import track
    gv = TSDFVolume(voxel, trunc)
    gv.integrate_batch(depth, rgb, intr, extrinsics)
    ov = oracle.Volume(voxel, trunc)
    for k in range(len(depth)):
        ov.integrate(oracle.depth_convert(depth[k]), rgb[k], intr, extrinsics[k])
    return gv.track(frames, intr, inits, **kw), track(ov, frames, intr, inits, **kw)


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


def test_small_sequence_equals_model():
    z = np.load(os.path.join(ROOT, "tests", "golden", "small_sequence.npz"))
    intr, (vl, tr) = tuple(z["intr"]), z["voxel"]
    e = z["extrinsic"]
    inits = seeded_starts(e, 1)
    g, o = both(z["depth"], z["rgb"], intr, e, float(vl), float(tr), z["depth"], inits)
    same_bits(g, o)
    assert (g["status"] != 3).all()


def test_window_equals_model(window):
    seq, d, c = window
    idx = [3, 17, 31, 45, 59]
    g, o = both(d, c, seq.fxfycxcy, seq.extrinsic, VL, 4 * VL, d[idx], seeded_starts(seq.extrinsic[idx], 2))
    same_bits(g, o)
    assert (g["status"] == 0).all()


def test_recovers_poses(window):
    """integrate the even frames, track the odd ones from seeded 1-3 cm / 1-2 degree errors"""
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    e = seq.extrinsic
    v = TSDFVolume(VL, 4 * VL)
    v.integrate_batch(d[0::2], c[0::2], seq.fxfycxcy, e[0::2])
    r = v.track(d[1::2], seq.fxfycxcy, seeded_starts(e[1::2], 3))
    err = np.array([pose_error(x, t) for x, t in zip(r["extrinsic"], e[1::2])])
    report = np.column_stack([r["status"], r["iterations"], err])
    # Single scale: from these starts a frame can end in a wrong minimum.  It then runs out of iterations (status 1), which
    # the caller sees; one of the 32 does here (DESIGN §4 "Frame-to-model tracking", measured).  Every frame that reports
    # convergence must be within the bounds.
    ok = r["status"] == 0
    assert np.isin(r["status"], (0, 1)).all() and ok.sum() >= 30, report
    assert np.median(err[:, 0]) <= 0.2 * VL, report
    assert err[ok, 0].max() <= 0.5 * VL and err[ok, 1].max() <= 0.2, report


def test_drift_loop(window):
    """16 frames at their true poses, then track -> integrate one frame at a time from the previous tracked pose composed
    with the true relative motion and a seeded drift of about 1 mm and 0.05 degree per frame"""
    from scipy.ndimage import binary_dilation
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    e, intr = seq.extrinsic, seq.fxfycxcy
    rng = np.random.default_rng(4)
    axis, direction = rng.normal(size=3), rng.normal(size=3)
    v = TSDFVolume(VL, 4 * VL)
    v.integrate_batch(d[:16], c[:16], intr, e[:16])
    tracked, loose = e[15], e[15]
    worst, worst_loose = 0.0, 0.0
    for k in range(16, len(e)):
        drift = np.eye(4)
        drift[:3, :3] = rot(axis + 0.3 * rng.normal(size=3), 0.05)
        step = direction + 0.3 * rng.normal(size=3)
        drift[:3, 3] = step / np.linalg.norm(step) * 0.001
        rel = e[k] @ np.linalg.inv(e[k - 1])
        init = drift @ rel @ tracked
        loose = drift @ rel @ loose
        r = v.track(d[k], intr, init)
        assert r["status"] == 0, (k, r)
        tracked = r["extrinsic"]
        v.integrate_batch(d[k:k + 1], c[k:k + 1], intr, tracked[None])
        worst = max(worst, pose_error(tracked, e[k])[0])
        worst_loose = max(worst_loose, pose_error(loose, e[k])[0])
    assert worst <= VL, worst
    assert worst_loose >= 5 * VL, worst_loose
    prims = synth.SCENES["chair_table"]()
    idx = [0, 21, 42, 63]
    out = v.ray_cast(intr, e[idx], 640, 480)
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
    """n frames in one call == n calls; host u16 == CUDA tensor; more frames than one chunk; two runs; save + load"""
    import torch
    from otslam_b200.volume import TSDFVolume
    seq, d, _ = window
    v, intr = window_volume, seq.fxfycxcy
    idx = np.arange(0, 64, 3)[:8]
    inits = seeded_starts(seq.extrinsic[idx], 5)
    full = v.track(d[idx], intr, inits)
    for i in range(len(idx)):
        one = v.track(d[idx[i]], intr, inits[i])
        assert one["extrinsic"].shape == (4, 4)
        same_bits({k: full[k][i] for k in OUTS}, one)
    same_bits(full, v.track(torch.from_numpy(d[idx]).cuda(), intr, inits))
    same_bits(full, v.track(d[idx], intr, inits))
    many = seeded_starts(seq.extrinsic[:40], 6)
    m = v.track(d[:40], intr, many)
    same_bits({k: a[32:] for k, a in m.items()}, v.track(d[32:40], intr, many[32:]))
    p = tmp_path / "v.otslam"
    v.save(p)
    w = TSDFVolume(VL, 4 * VL)
    w.load(p)
    same_bits(full, w.track(d[idx], intr, inits))


def test_state_untouched(window):
    from otslam_b200.o3d_compat import pipelines
    seq, d, c = window
    vol = pipelines.ScalableTSDFVolume(VL, 4 * VL, pipelines.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d[:16], c[:16], _intrinsic(seq), seq.extrinsic[:16])
    stats = vol._vol.stats()
    keys = vol._vol.export_blocks(color=True)
    lazy = vol.extract_triangle_mesh()                 # arrays still in HBM
    before = vol._vol.extract_triangle_mesh(normals=False)
    lazy2 = vol.extract_triangle_mesh()
    r = vol._vol.track(d[3:6], seq.fxfycxcy, seeded_starts(seq.extrinsic[3:6], 7))
    assert (r["status"] == 0).all()
    assert vol._vol.stats() == stats
    after_keys = vol._vol.export_blocks(color=True)
    assert all((x.view(np.uint8) == y.view(np.uint8)).all() for x, y in zip(keys, after_keys))
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
        v.track(d[0], seq.fxfycxcy, seq.extrinsic[0])
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
    idx = [5, 20, 30]
    inits = seeded_starts(e[idx], 8)
    same_bits(own.track(d[idx], intr, inits), ArenaView(arena, 0).track(d[idx], intr, inits))


def test_nocolor_volume_same_poses(window):
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    a, b = TSDFVolume(VL, 4 * VL), TSDFVolume(VL, 4 * VL, color=False)
    a.integrate_batch(d[:16], c[:16], seq.fxfycxcy, seq.extrinsic[:16])
    b.integrate_batch(d[:16], None, seq.fxfycxcy, seq.extrinsic[:16])
    inits = seeded_starts(seq.extrinsic[4:8], 9)
    same_bits(a.track(d[4:8], seq.fxfycxcy, inits), b.track(d[4:8], seq.fxfycxcy, inits))


def test_compat_track_frame_to_model(window, window_volume):
    from otslam_b200.o3d_compat import geometry, pipelines
    seq, d, c = window
    vol = pipelines.ScalableTSDFVolume(VL, 4 * VL, pipelines.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d, c, _intrinsic(seq), seq.extrinsic)
    init = seeded_starts(seq.extrinsic[12:13], 10)[0]
    img = geometry.RGBDImage.create_from_color_and_depth(c[12], d[12], depth_scale=1000.0, convert_rgb_to_intensity=False)
    got = vol.track_frame_to_model(img, _intrinsic(seq), init)
    ref = window_volume.track(d[12], seq.fxfycxcy, init)
    assert (got.transformation.view(np.uint8) == ref["extrinsic"].view(np.uint8)).all()
    assert got.fitness == ref["fitness"] and got.inlier_rmse == ref["inlier_rmse"] and got.converged == (ref["status"] == 0)
