"""The integration kernel's brick cull (modelled by cull_ref.brick_need) never skips a (brick, frame) pair that holds a voxel
the CPU oracle updates, on frames chosen to stress it, at every z-split."""
import numpy as np
import pytest

import cull_ref
from oracle import oracle


@pytest.mark.parametrize("name", cull_ref.SCENES)
def test_culled_pairs_do_not_update(name):
    depth, rgb, ext, intr, vl, trunc, dtr = cull_ref.scene(name)
    H, W = depth.shape[1:]
    culled = tested = 0
    for k in range(len(depth)):
        d = oracle.depth_convert(depth[k], 1000.0, dtr)
        ov = oracle.Volume(vl, trunc)
        ov.integrate(d, rgb[k], intr, ext[k])
        keys, _, weight, _ = ov.export_blocks(color=False)
        keep = (weight > 0).any(1)
        keys, upd = keys[keep], weight[keep].reshape(-1, 16, 16, 16) > 0
        assert len(keys) > 0
        tiles = cull_ref.tile_max(d)
        for zs in (1, 2, 4, 8):
            need = cull_ref.brick_need(keys, ext[k], vl, trunc, intr, W, H, tiles, zsplit=zs)
            for i in range(len(keys)):
                u = cull_ref.brick_updates(upd[i], zs)
                assert not (u & ~need[i]).any(), f"{name}: frame {k}, block {tuple(keys[i])}, z-split {zs}"
            culled += int((~need).sum())
            tested += need.size
    # blocks with updates are mostly in front of or at the surface, but some of their bricks lie behind it
    assert culled > 0 or name in ("grazing",), f"{name}: nothing culled in {tested} pairs"


def test_tile_max_ragged():
    d = np.arange(7 * 10, dtype=np.float32).reshape(7, 10)
    t = cull_ref.tile_max(d, 4)
    assert t.shape == (2, 3)
    assert t[1, 2] == d[4:7, 8:10].max() and t[0, 0] == d[:4, :4].max()
