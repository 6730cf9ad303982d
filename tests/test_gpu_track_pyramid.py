"""Coarse-to-fine frame-to-model tracking on the GPU (otslam_volume_track_pyramid): the CUDA kernels equal the CPU model
(tests/models/track_pyramid_model.cpp on the oracle's volume) bit for bit at 2 and 3 levels, one level is TSDFVolume.track,
TRACK_PYRAMID recovers starts that single-scale tracking loses, the result does not depend on how the call is made, and
the volume is left as it was."""
import os

import numpy as np
import pytest

from conftest import ROOT, canon_mesh
from test_gpu_track import OUTS, VL, _intrinsic, same_bits, seeded_starts, window, window_volume  # noqa: F401
from test_track_oracle import pose_error

pytestmark = pytest.mark.gpu

LEVELS = {2: ((0.07, 0.15), (20, 10)), 3: ((0.07, 0.15, 0.3), (20, 10, 10))}


def both(depth, rgb, intr, extrinsics, voxel, trunc, frames, inits, levels):
    """the GPU volume's pyramid tracking and the CPU model's on the oracle's volume of the same frames"""
    from oracle import oracle
    from otslam_b200.volume import TSDFVolume
    from test_track_pyramid_oracle import track_pyramid
    dd, mi = LEVELS[levels]
    gv = TSDFVolume(voxel, trunc)
    gv.integrate_batch(depth, rgb, intr, extrinsics)
    ov = oracle.Volume(voxel, trunc)
    for k in range(len(depth)):
        ov.integrate(oracle.depth_convert(depth[k]), rgb[k], intr, extrinsics[k])
    return gv.track(frames, intr, inits, depth_diff=dd, max_iterations=mi), track_pyramid(ov, frames, intr, inits, dd, mi)


@pytest.mark.parametrize("levels", [2, 3])
def test_small_sequence_equals_model(levels):
    z = np.load(os.path.join(ROOT, "tests", "golden", "small_sequence.npz"))
    intr, (vl, tr) = tuple(z["intr"]), z["voxel"]
    e = z["extrinsic"]
    g, o = both(z["depth"], z["rgb"], intr, e, float(vl), float(tr), z["depth"], seeded_starts(e, 1), levels)
    same_bits(g, o)
    assert (g["status"] != 3).all()


@pytest.mark.parametrize("levels", [2, 3])
def test_window_equals_model(window, levels):
    seq, d, c = window
    idx = [3, 17, 31, 45, 59]
    g, o = both(d, c, seq.fxfycxcy, seq.extrinsic, VL, 4 * VL, d[idx], seeded_starts(seq.extrinsic[idx], 2), levels)
    same_bits(g, o)
    assert (g["status"] == 0).all()


@pytest.mark.parametrize("levels", [2, 3])
def test_hd_golden_equals_model(levels):
    z = np.load(os.path.join(ROOT, "tests", "golden", "hd_sequence.npz"))
    intr, (vl, tr) = tuple(z["intr"]), z["voxel"]
    e = z["extrinsic"]
    idx = [1, 6]
    g, o = both(z["depth"], z["rgb"], intr, e, float(vl), float(tr), z["depth"][idx], seeded_starts(e[idx], 3), levels)
    same_bits(g, o)


def test_cropped_window_equals_model(window):
    """a frame size that 2^(levels - 1) does not divide: 637x477 (the last odd column and row of each level dropped)"""
    seq, d, c = window
    idx = [10, 40]
    crop = np.ascontiguousarray(d[idx, :477, :637])
    g, o = both(d, c, seq.fxfycxcy, seq.extrinsic, VL, 4 * VL, crop, seeded_starts(seq.extrinsic[idx], 4), 3)
    same_bits(g, o)
    assert (g["status"] == 0).all()


def test_one_level_equals_track(window, window_volume):
    seq, d, _ = window
    idx = [2, 22, 42]
    inits = seeded_starts(seq.extrinsic[idx], 5)
    v = window_volume
    same_bits(v.track(d[idx], seq.fxfycxcy, inits), v.track(d[idx], seq.fxfycxcy, inits, depth_diff=[0.07], max_iterations=[20]))
    same_bits(v.track(d[idx], seq.fxfycxcy, inits, depth_diff=0.05, max_iterations=7),
              v.track(d[idx], seq.fxfycxcy, inits, depth_diff=(0.05,), max_iterations=7))
    with pytest.raises(ValueError):
        v.track(d[idx], seq.fxfycxcy, inits, depth_diff=(0.07, 0.15), max_iterations=(20, 10, 10))


def _recover(window, seed, cm, deg):
    from otslam_b200.volume import TRACK_PYRAMID, TSDFVolume
    seq, d, c = window
    e = seq.extrinsic
    v = TSDFVolume(VL, 4 * VL)
    v.integrate_batch(d[0::2], c[0::2], seq.fxfycxcy, e[0::2])
    r = v.track(d[1::2], seq.fxfycxcy, seeded_starts(e[1::2], seed, cm, deg), **TRACK_PYRAMID)
    err = np.array([pose_error(x, t) for x, t in zip(r["extrinsic"], e[1::2])])
    report = np.column_stack([r["status"], r["iterations"], err])
    assert (r["status"] == 0).all(), report
    assert err[:, 0].max() <= 0.5 * VL and err[:, 1].max() <= 0.2, report


def test_recovers_poses(window):
    """integrate the even frames, track the odd ones from the seeded 1-3 cm / 1-2 degree starts of test_gpu_track.py"""
    _recover(window, 3, (1.0, 3.0), (1.0, 2.0))


def test_recovers_larger_starts(window):
    _recover(window, 12, (3.0, 5.0), (2.0, 4.0))


def test_hd_2deg_starts():
    """HD golden volume, 1-3 cm / 2 degree starts: every frame that TRACK_PYRAMID reports converged is within one voxel and
    0.2 degree, and it converges at least as many frames as single-scale tracking from the same starts.  Not every frame
    converges: on the large room some starts end in a wrong minimum at every level (DESIGN §4, measured)."""
    from otslam_b200.volume import TRACK_PYRAMID, TSDFVolume
    z = np.load(os.path.join(ROOT, "tests", "golden", "hd_sequence.npz"))
    intr, (vl, tr) = tuple(z["intr"]), z["voxel"]
    e = z["extrinsic"]
    v = TSDFVolume(float(vl), float(tr))
    v.integrate_batch(z["depth"], z["rgb"], intr, e)
    inits = seeded_starts(e, 13, deg=(2.0, 2.0))
    r = v.track(z["depth"], intr, inits, **TRACK_PYRAMID)
    single = v.track(z["depth"], intr, inits)
    err = np.array([pose_error(x, t) for x, t in zip(r["extrinsic"], e)])
    report = np.column_stack([r["status"], r["iterations"], err, single["status"]])
    ok = r["status"] == 0
    assert ok.sum() >= (single["status"] == 0).sum() and ok.any(), report
    assert err[ok, 0].max() <= float(vl) and err[ok, 1].max() <= 0.2, report


def test_call_equivalences(window, window_volume, tmp_path):
    """n frames in one call == n calls; host u16 == CUDA tensor; more frames than one chunk; two runs; save + load"""
    import torch
    from otslam_b200.volume import TRACK_PYRAMID, TSDFVolume
    seq, d, _ = window
    v, intr = window_volume, seq.fxfycxcy
    idx = np.arange(0, 64, 3)[:8]
    inits = seeded_starts(seq.extrinsic[idx], 5)
    full = v.track(d[idx], intr, inits, **TRACK_PYRAMID)
    for i in range(len(idx)):
        one = v.track(d[idx[i]], intr, inits[i], **TRACK_PYRAMID)
        assert one["extrinsic"].shape == (4, 4)
        same_bits({k: full[k][i] for k in OUTS}, one)
    same_bits(full, v.track(torch.from_numpy(d[idx]).cuda(), intr, inits, **TRACK_PYRAMID))
    same_bits(full, v.track(d[idx], intr, inits, **TRACK_PYRAMID))
    many = seeded_starts(seq.extrinsic[:40], 6)
    m = v.track(d[:40], intr, many, **TRACK_PYRAMID)
    same_bits({k: a[32:] for k, a in m.items()}, v.track(d[32:40], intr, many[32:], **TRACK_PYRAMID))
    p = tmp_path / "v.otslam"
    v.save(p)
    w = TSDFVolume(VL, 4 * VL)
    w.load(p)
    same_bits(full, w.track(d[idx], intr, inits, **TRACK_PYRAMID))


def test_state_untouched(window):
    from otslam_b200.o3d_compat import pipelines
    from otslam_b200.volume import TRACK_PYRAMID
    seq, d, c = window
    vol = pipelines.ScalableTSDFVolume(VL, 4 * VL, pipelines.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d[:16], c[:16], _intrinsic(seq), seq.extrinsic[:16])
    stats = vol._vol.stats()
    keys = vol._vol.export_blocks(color=True)
    lazy = vol.extract_triangle_mesh()                 # arrays still in HBM
    before = vol._vol.extract_triangle_mesh(normals=False)
    lazy2 = vol.extract_triangle_mesh()
    r = vol._vol.track(d[3:6], seq.fxfycxcy, seeded_starts(seq.extrinsic[3:6], 7), **TRACK_PYRAMID)
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


def test_slab_volume_refused_and_unchanged(window):
    from otslam_b200.volume import TRACK_PYRAMID, TSDFVolume
    seq, d, c = window
    v = TSDFVolume(VL, 4 * VL, slab=(0, 8, 2, 0))
    v.integrate_batch(d[:8], c[:8], seq.fxfycxcy, seq.extrinsic[:8])
    stats, keys = v.stats(), v.export_blocks(color=False)
    with pytest.raises(RuntimeError, match="part file"):
        v.track(d[0], seq.fxfycxcy, seq.extrinsic[0], **TRACK_PYRAMID)
    assert v.stats() == stats
    after = v.export_blocks(color=False)
    assert (keys[0] == after[0]).all() and (keys[1].view(np.uint32) == after[1].view(np.uint32)).all()


def test_arena_object_equals_own_volume(window):
    from otslam_b200.volume import TRACK_PYRAMID, ArenaView, TSDFVolume
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
    same_bits(own.track(d[idx], intr, inits, **TRACK_PYRAMID), ArenaView(arena, 0).track(d[idx], intr, inits, **TRACK_PYRAMID))


def test_compat_track_frame_to_model(window, window_volume):
    from otslam_b200.o3d_compat import geometry, pipelines
    from otslam_b200.volume import TRACK_PYRAMID
    seq, d, c = window
    vol = pipelines.ScalableTSDFVolume(VL, 4 * VL, pipelines.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d, c, _intrinsic(seq), seq.extrinsic)
    init = seeded_starts(seq.extrinsic[12:13], 10, (3.0, 5.0), (2.0, 4.0))[0]
    img = geometry.RGBDImage.create_from_color_and_depth(c[12], d[12], depth_scale=1000.0, convert_rgb_to_intensity=False)
    dd, mi = (list(x) for x in (TRACK_PYRAMID["depth_diff"], TRACK_PYRAMID["max_iterations"]))
    got = vol.track_frame_to_model(img, _intrinsic(seq), init, depth_diff=dd, max_iterations=mi)
    ref = window_volume.track(d[12], seq.fxfycxcy, init, depth_diff=dd, max_iterations=mi)
    assert (got.transformation.view(np.uint8) == ref["extrinsic"].view(np.uint8)).all()
    assert got.fitness == ref["fitness"] and got.inlier_rmse == ref["inlier_rmse"] and got.converged == (ref["status"] == 0)
