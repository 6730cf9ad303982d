"""The volume's long-lived device resources on the paths no other test reaches: staging buffers re-sized inside one volume
(new image size, u16 -> f32 depth, host -> device frames), a borrowed stream, and per-kernel profiling.  Each run must
give the volume a fresh one gives."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VL = 0.01
SMALL = (320, 240, 282.80045, 282.80045, 160.25, 120.25)    # the reference camera at half resolution


@pytest.fixture(scope="module")
def frames():
    """The same four poses of the table scene at 640x480 and at 320x240."""
    from otslam_b200 import synth
    large = synth.make_sequence("table", 300, subsample=(0, 75), device="cuda")
    small = synth.make_sequence("table", 300, intr=SMALL, subsample=(0, 75), device="cuda")
    return {"large": large, "small": small}


def integrate(v, seq, kind):
    """u16 / f32: frames from host memory (staged through the volume's raw buffers); device: frames already in HBM"""
    if kind == "u16":
        d, c = seq.numpy()
        v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    elif kind == "f32":
        d, c = seq.numpy()
        for k in range(len(seq)):
            v.integrate_f32(d[k].astype(np.float32) / np.float32(1000.0), c[k], seq.fxfycxcy, seq.extrinsic[k])
    else:
        v.integrate_batch(seq.depth.cuda(), seq.rgb.cuda(), seq.fxfycxcy, seq.extrinsic)


def state(v):
    return v.stats(), [a.tobytes() for a in v.export_blocks()]


@pytest.mark.parametrize("first,second", [("large", "small"), ("small", "large")])
@pytest.mark.parametrize("kinds", [("u16", "u16"), ("u16", "f32"), ("u16", "device")], ids=["u16", "u16-f32", "host-device"])
def test_restaged_after_reset(frames, first, second, kinds):
    """reset() keeps the staging buffers: the second pass runs on buffers re-sized for another image size (the packed
    frames' zero sentinels move), another depth format or another frame source."""
    from otslam_b200.volume import TSDFVolume
    v = TSDFVolume(VL, 4 * VL)
    integrate(v, frames[first], kinds[0])
    assert v.num_blocks() > 0
    v.reset()
    integrate(v, frames[second], kinds[1])
    got = state(v)
    v.close()
    ref = TSDFVolume(VL, 4 * VL)
    integrate(ref, frames[second], kinds[1])
    want = state(ref)
    ref.close()
    assert got[0]["n_blocks"] > 0
    assert got == want


def test_borrowed_stream(frames):
    """Integration on the caller's stream, then back on the volume's own: the same volume, and the caller's stream
    outlives the volume."""
    import torch
    from otslam_b200.volume import TSDFVolume
    seq = frames["large"]
    d, c = seq.numpy()
    s = torch.cuda.Stream()
    v = TSDFVolume(VL, 4 * VL)
    v.set_stream(s.cuda_stream)
    v.integrate_batch(d[:2], c[:2], seq.fxfycxcy, seq.extrinsic[:2])
    half = state(v)
    v.set_stream(None)
    v.integrate_batch(d[2:], c[2:], seq.fxfycxcy, seq.extrinsic[2:])
    got = state(v)
    v.close()
    ev = torch.cuda.Event()
    ev.record(s)
    ev.synchronize()
    s.synchronize()

    ref = TSDFVolume(VL, 4 * VL)
    ref.integrate_batch(d[:2], c[:2], seq.fxfycxcy, seq.extrinsic[:2])
    assert half == state(ref)
    ref.integrate_batch(d[2:], c[2:], seq.fxfycxcy, seq.extrinsic[2:])
    assert got == state(ref)
    ref.close()


def test_profiling(frames):
    """Event pairs around every pack, allocation and integration launch (recycled across calls); results unchanged."""
    from otslam_b200.volume import TSDFVolume
    seq = frames["large"]
    d, c = seq.numpy()
    v = TSDFVolume(VL, 4 * VL)
    v.set_batch(2)
    v.profile(True)
    v.integrate_batch(d[:2], c[:2], seq.fxfycxcy, seq.extrinsic[:2])
    v.integrate_batch(d[2:], c[2:], seq.fxfycxcy, seq.extrinsic[2:])
    prof = v.profile(False)
    for k in ("pack", "alloc", "integrate"):
        assert prof[k][1] > 0, (k, prof)
    got = state(v)
    v.close()
    ref = TSDFVolume(VL, 4 * VL)
    ref.set_batch(2)
    ref.integrate_batch(d[:2], c[:2], seq.fxfycxcy, seq.extrinsic[:2])
    ref.integrate_batch(d[2:], c[2:], seq.fxfycxcy, seq.extrinsic[2:])
    assert got == state(ref)
    ref.close()


def test_failed_extraction_leaves_no_result(frames):
    """An extraction releases the old mesh / points first and keeps a new one only when it completes.  On an arena with no
    object selected it fails after that release: sampling then finds no triangles, the copies copy nothing, and the next
    good extraction gives what a fresh arena gives."""
    from otslam_b200 import _lib
    from otslam_b200.volume import TSDFVolume
    seq = frames["large"]
    d, c = seq.numpy()

    def arena():
        a = TSDFVolume(VL, 4 * VL)
        a.set_objects(2)
        a.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic, object_ids=np.ones(len(seq), np.int32))
        a.select_object(1)
        return a

    def results(a):
        mesh = a.extract_triangle_mesh()
        sample = a.mesh_sample(4096, 11, colors=True, normals=True)
        return [x.tobytes() for x in mesh + sample + a.extract_point_cloud(normals=True)]

    v = arena()
    nv, nf = v.extract_mesh_resident()
    n_pts = len(v.extract_point_cloud()[0])
    assert nv > 0 and nf > 0 and n_pts > 0
    v.select_object(-1)
    with pytest.raises(RuntimeError, match="select_object"):
        v.extract_mesh_resident()
    with pytest.raises(RuntimeError, match="select_object"):
        v.extract_point_cloud()
    with pytest.raises(RuntimeError, match="no triangles"):
        v.mesh_sample(4096, 11)
    mesh = [np.full((nv, 3), 7.0), np.full((nv, 3), 7.0), np.full((nv, 3), 7.0), np.full((nf, 3), 7, np.int32),
            np.full((nv, 4), 7, np.int32)]
    points = [np.full((n_pts, 3), 7.0), np.full((n_pts, 3), 7.0), np.full((n_pts, 4), 7, np.int32)]
    normals = np.full((n_pts, 3), 7.0)
    _lib.check(_lib.lib.otslam_volume_mesh_copy(v._h, *(_lib.ptr(a) for a in mesh)))
    _lib.check(_lib.lib.otslam_volume_points_copy(v._h, *(_lib.ptr(a) for a in points)))
    _lib.check(_lib.lib.otslam_volume_points_normals(v._h, _lib.ptr(normals)))
    for a in mesh + points + [normals]:
        assert (a == 7).all()
    v.select_object(1)
    got = results(v)
    v.close()
    ref = arena()
    want = results(ref)
    ref.close()
    assert got == want
