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
