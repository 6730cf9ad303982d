"""How many voxel-frame pairs the integration kernel's brick cull skips (CPU, NumPy; the model is tests/cull_ref.py).

The kernel gives each warp a brick of 4 x-rows x 8 y-columns and tests, per gather group of 8 z-slices (z-split 2) and per
frame, whether the brick lies wholly behind the frame's surface: its minimum camera z, lowered by a rounding bound, exceeds
the maximum depth over the 4 px tiles that its projected footprint can reach by at least the truncation distance.  This
script replays the exact test on frames of the benchmark's sequences, reports the share of all visited voxel-frame pairs
the test skips, and asserts that no skipped pair updates (the update sets come from the CPU oracle).

Visited pairs are estimated the way the allocation kernel finds blocks: every 4th pixel back-projected, +-trunc box.
Usage: python tools/study_culling_bricks.py [--hd] [--frames N] [--tile T] [--max-tiles N] [--zsplit Z]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np

import cull_ref
from oracle import oracle
from otslam_b200 import synth


def visited_keys(d, E, intr, unit, trunc):
    fx, fy, cx, cy = intr
    H, W = d.shape
    ii, jj = np.meshgrid(np.arange(0, H, 4), np.arange(0, W, 4), indexing="ij")
    z = d[ii, jj].astype(np.float64)
    m = z > 0
    x = (jj[m] - cx) * z[m] / fx
    y = (ii[m] - cy) * z[m] / fy
    P = np.linalg.inv(E)
    pw = (P[:3, :3] @ np.stack([x, y, z[m]])).T + P[:3, 3]
    keys = set()
    for dx in (-trunc, trunc):
        for dy in (-trunc, trunc):
            for dz in (-trunc, trunc):
                keys |= set(map(tuple, np.floor((pw + [dx, dy, dz]) / unit).astype(int)))
    return np.array(sorted(keys), np.int64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hd", action="store_true", help="room scene, 1280x720, 2 mm voxels, 8 mm truncation")
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--tile", type=int, default=cull_ref.TILE)
    ap.add_argument("--max-tiles", type=int, default=cull_ref.MAX_TILES)
    ap.add_argument("--zsplit", type=int, default=2)
    a = ap.parse_args()
    if a.hd:
        scene, n, intr_full, vl = "room", 2000, synth.HD_INTRINSICS, 0.002
    else:
        scene, n, intr_full, vl = "chair_table", 1000, synth.REF_INTRINSICS, 0.005
    trunc = 4 * vl
    seq = synth.make_sequence(scene, n, intr=intr_full, subsample=(37, n // a.frames))
    depth, rgb = seq.numpy()
    intr = seq.fxfycxcy
    H, W = depth.shape[1:]
    tot = dict(pairs=0, upd=0, skip=0, skip_units=0, units=0)
    for k in range(len(seq)):
        d = oracle.depth_convert(depth[k], 1000.0, 3.0)
        E = seq.extrinsic[k]
        ov = oracle.Volume(vl, trunc)
        ov.integrate(d, rgb[k], intr, E)
        upd = cull_ref.updated_by_frame((np.zeros((0, 3)), None, np.zeros((0, 4096))), ov.export_blocks(color=False))
        keys = visited_keys(d, E, intr, 16 * vl, trunc)
        need = cull_ref.brick_need(keys, E, vl, trunc, intr, W, H, cull_ref.tile_max(d, a.tile), a.zsplit, a.tile, a.max_tiles)
        for i, key in enumerate(map(tuple, keys)):
            if key in upd:
                u = cull_ref.brick_updates(upd[key], a.zsplit)
                assert not (u & ~need[i]).any(), f"culled pair updates: block {key}, frame {k}"
                tot["upd"] += int(upd[key].sum())
        ng = need.shape[2]
        tot["pairs"] += len(keys) * 4096
        tot["skip"] += int((~need).sum()) * 32 * (16 // ng)
        tot["units"] += need.size
        tot["skip_units"] += int((~need).sum())
        missing = set(upd) - set(map(tuple, keys))
        assert not missing or len(missing) < 0.01 * len(upd), "visited-block estimate misses updated blocks"
    p = tot["pairs"]
    print(f"{'hd' if a.hd else 'default'} {W}x{H} voxel {vl * 1000:g} mm trunc {trunc * 1000:g} mm, {len(seq)} frames, "
          f"tile {a.tile} px, max {a.max_tiles} tiles, zsplit {a.zsplit}: updating {tot['upd'] / p:.3f}, "
          f"culled {tot['skip'] / p:.3f} of all visited pairs; no culled pair updates")


if __name__ == "__main__":
    main()
