"""The integration kernel's brick cull changes no result: volumes integrated with the cull (default) and without it
(OTSLAM_K4_CULL=0) are equal bit for bit -- keys, TSDF, weights, colour -- and equal the CPU oracle, on the frames of
cull_ref.scene that stress the test, at every z-split, at two batch sizes, for NoColor volumes, f32 depth, device-resident
frames, a multi-object arena and one rank of a diagonal-slab volume."""
import numpy as np
import pytest

import cull_ref
from oracle import oracle

pytestmark = pytest.mark.gpu
COLOR_TOL = 1.0


def oracle_volume(depth, rgb, intr, ext, vl, trunc, dtr, slab=None):
    ov = oracle.Volume(vl, trunc, slab=slab)
    for k in range(len(depth)):
        ov.integrate(oracle.depth_convert(depth[k], 1000.0, dtr), rgb[k], intr, ext[k])
    return ov.export_blocks()


def gpu_volume(monkeypatch, cull, integrate, vl, trunc, color=True, zsplit=None, batch=None, slab=None):
    from otslam_b200.volume import TSDFVolume
    monkeypatch.setenv("OTSLAM_K4_CULL", "1" if cull else "0")   # read when the volume is created
    gv = TSDFVolume(vl, trunc, color=color, slab=slab)
    if zsplit:
        gv.set_zsplit(zsplit)
    if batch:
        gv.set_batch(batch)
    integrate(gv)
    out = gv.export_blocks()
    gv.close()
    return out


def assert_same(a, b):
    for x, y, what in zip(a, b, ("keys", "TSDF", "weights", "colour")):
        assert x.shape == y.shape and np.array_equal(x, y), f"{what} differ with and without the cull"


def assert_oracle(g, o, color=True):
    gk, gt, gw, gc = g
    ok, ot, ow, oc = o
    assert gk.shape == ok.shape and (gk == ok).all(), "block keys differ from the oracle"
    assert (gw == ow).all(), "weights differ from the oracle"
    assert (gt == ot).all(), "TSDF differs from the oracle"
    seen = ow > 0
    assert seen.any()
    if color:
        assert np.abs(gc - oc)[seen].max() <= COLOR_TOL
    else:
        assert (gc == 0).all()


@pytest.mark.parametrize("zsplit", [1, 2, 4, 8])
@pytest.mark.parametrize("name", cull_ref.SCENES)
def test_cull_on_off_and_oracle(monkeypatch, name, zsplit):
    depth, rgb, ext, intr, vl, trunc, dtr = cull_ref.scene(name)
    run = lambda gv: gv.integrate_batch(depth, rgb, intr, ext, depth_trunc=dtr)
    on = gpu_volume(monkeypatch, True, run, vl, trunc, zsplit=zsplit)
    off = gpu_volume(monkeypatch, False, run, vl, trunc, zsplit=zsplit)
    assert_same(on, off)
    assert_oracle(on, oracle_volume(depth, rgb, intr, ext, vl, trunc, dtr))


@pytest.mark.parametrize("name", ["near_wedge", "holes", "default"])
def test_batch7_nocolor_f32_resident(monkeypatch, name):
    import torch
    depth, rgb, ext, intr, vl, trunc, dtr = cull_ref.scene(name)
    ref = oracle_volume(depth, rgb, intr, ext, vl, trunc, dtr)
    batch7 = lambda gv: gv.integrate_batch(depth, rgb, intr, ext, depth_trunc=dtr)
    assert_same(gpu_volume(monkeypatch, True, batch7, vl, trunc, batch=7), gpu_volume(monkeypatch, False, batch7, vl, trunc, batch=7))
    nocol = lambda gv: gv.integrate_batch(depth, None, intr, ext, depth_trunc=dtr)
    on = gpu_volume(monkeypatch, True, nocol, vl, trunc, color=False)
    assert_same(on, gpu_volume(monkeypatch, False, nocol, vl, trunc, color=False))
    assert_oracle(on, ref, color=False)
    dm = np.stack([oracle.depth_convert(d, 1000.0, dtr) for d in depth])

    def f32(gv):
        for k in range(len(dm)):
            gv.integrate_f32(dm[k], rgb[k], intr, ext[k])
    on = gpu_volume(monkeypatch, True, f32, vl, trunc)
    assert_same(on, gpu_volume(monkeypatch, False, f32, vl, trunc))
    assert_oracle(on, ref)
    dd, rr = torch.from_numpy(depth.view(np.int16)).cuda().view(torch.uint16), torch.from_numpy(rgb).cuda()
    resident = lambda gv: gv.integrate_batch(dd, rr, intr, ext, depth_trunc=dtr)
    on = gpu_volume(monkeypatch, True, resident, vl, trunc)
    assert_same(on, gpu_volume(monkeypatch, False, resident, vl, trunc))
    assert_oracle(on, ref)


def test_arena_objects(monkeypatch):
    from otslam_b200.volume import ArenaView, TSDFVolume
    scenes = [cull_ref.scene(n) for n in ("near_wedge", "border")]
    depth = np.stack([s[0][k] for k in range(6) for s in scenes])
    rgb = np.stack([s[1][k] for k in range(6) for s in scenes])
    ext = np.stack([s[2][k] for k in range(6) for s in scenes])
    ids = np.array([o for _ in range(6) for o in range(2)], np.int32)
    intr, vl, trunc = scenes[0][3], 0.01, 0.04
    views = {}
    for cull in (True, False):
        monkeypatch.setenv("OTSLAM_K4_CULL", "1" if cull else "0")
        arena = TSDFVolume(vl, trunc)
        arena.set_objects(2)
        arena.integrate_batch(depth, rgb, intr, ext, object_ids=ids)
        views[cull] = [ArenaView(arena, o).export_blocks() for o in range(2)]
        arena.close()
    for o in range(2):
        assert_same(views[True][o], views[False][o])
        sel = ids == o
        assert_oracle(views[True][o], oracle_volume(depth[sel], rgb[sel], intr, ext[sel], vl, trunc, 3.0))


def test_slab_rank(monkeypatch):
    depth, rgb, ext, intr, vl, trunc, dtr = cull_ref.scene("default")
    slab = (3, 1, 8, 3, 0)
    run = lambda gv: gv.integrate_batch(depth, rgb, intr, ext, depth_trunc=dtr)
    on = gpu_volume(monkeypatch, True, run, vl, trunc, slab=slab)
    assert_same(on, gpu_volume(monkeypatch, False, run, vl, trunc, slab=slab))
    assert_oracle(on, oracle_volume(depth, rgb, intr, ext, vl, trunc, dtr, slab=slab))
