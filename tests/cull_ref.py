"""NumPy model of the integration kernel's brick cull test (csrc/volume.cu, integrate_kernel's prologue).

A warp of the kernel owns a brick of 4 x-rows x 8 y-columns of a block; the brick's z-range is split into gather groups of
kzg = min(16 / zsplit, 8) slices.  For every (brick, group, frame) the kernel decides from the frame's max-depth tiles
whether any voxel of the group can update.  This module replays that decision with the same operations in the same
precision (FP32; the kernel's fused multiply-adds are evaluated in FP64 and rounded once), so that tests and the study
tool can check the test against the CPU oracle and count how many pairs it skips.
"""
import numpy as np

TILE = 4              # tile edge in pixels (kCullTile)
MAX_TILES = 36       # a footprint covering more tiles than this is not tested (kCullMaxTiles)
Z_FLOOR = np.float32(2.0 ** -9)
COORD_MAX = np.float32(2.0 ** 20)
REL = np.float32(2.0 ** -18)
TINY = np.float32(2.0 ** -100)

f32 = np.float32


def tile_max(depth_f32, tile=TILE):
    """Max converted depth over tile x tile pixel squares (0 where every pixel is invalid), [th, tw] float32."""
    H, W = depth_f32.shape
    th, tw = -(-H // tile), -(-W // tile)
    d = np.zeros((th * tile, tw * tile), np.float32)
    d[:H, :W] = depth_f32
    return d.reshape(th, tile, tw, tile).max(axis=(1, 3))


def _fma(a, b, c):
    return (np.float64(a) * np.float64(b) + np.float64(c)).astype(np.float32)


def column_coords(keys, vl):
    """The kernel's per-column world coordinates px(x), py(y) [n, 16] and pz [n] (FP32, via the same FP64 sums)."""
    vlf = f32(vl)
    half = f32(vlf * f32(0.5))
    unit = float(vl) * 16.0
    idx = np.arange(16, dtype=np.float32)
    off = (half + vlf * idx).astype(np.float32).astype(np.float64)          # RN(half + RN(vl * i))
    k = np.asarray(keys, np.float64)
    px = (off[None, :] + k[:, 0:1] * unit).astype(np.float32)
    py = (off[None, :] + k[:, 1:2] * unit).astype(np.float32)
    pz = (np.float64(half) + k[:, 2] * unit).astype(np.float32)
    return px, py, pz


def frame_consts(extrinsic, vl):
    E = np.asarray(extrinsic, np.float64)[:3, :4].astype(np.float32)
    es = (E[:, 2] * f32(vl)).astype(np.float32)
    return E, es


def brick_need(keys, extrinsic, vl, trunc, intr, W, H, tiles, zsplit=2, tile=TILE, max_tiles=MAX_TILES):
    """need[n, 8, n_groups]: False where the kernel skips (block, warp brick, z-group) for this frame."""
    keys = np.asarray(keys).reshape(-1, 3)
    kzg = min(16 // zsplit, 8)
    ng = 16 // kzg
    px, py, pz = column_coords(keys, vl)
    E, es = frame_consts(extrinsic, vl)
    fx, fy, cx, cy = (f32(c) for c in intr)
    trunc = f32(trunc)
    n = len(keys)
    w = np.arange(8)
    x0 = 4 * (w >> 1)
    y0 = 8 * (w & 1)
    # corner coordinates [n, 8 warps, ng groups] per end: px0/px1, py0/py1, k0/k1
    PX = np.stack([px[:, x0], px[:, x0 + 3]], -1)[:, :, None, :]            # [n, 8, 1, 2]
    PY = np.stack([py[:, y0], py[:, y0 + 7]], -1)[:, :, None, :]
    PZ = pz[:, None, None]
    g = np.arange(ng, dtype=np.float32)
    K = np.stack([g * kzg, g * kzg + (kzg - 1)], -1).astype(np.float32)[None, None, :, :]   # [1, 1, ng, 2]
    corner, S = [], []
    for c in range(3):
        t0 = _fma(E[c, 2], PZ, E[c, 3])                                      # [n, 1, 1]
        a = _fma(E[c, 0], PX, t0[..., None])                                 # [n, 8, 1, 2(x)]
        b = _fma(E[c, 1], PY[..., None, :], a[..., :, None])                 # [n, 8, 1, 2(x), 2(y)]
        v = _fma(K[..., None, None, :], es[c], b[..., None])                 # [n, 8, ng, 2, 2, 2(k)]
        corner.append(v.reshape(n, 8, ng, 8))
        s = (abs(E[c, 0]) * np.abs(PX).max(-1) + abs(E[c, 1]) * np.abs(PY).max(-1)).astype(np.float32)
        s = (s + abs(E[c, 2]) * np.abs(PZ) + abs(E[c, 3]) + f32(16) * abs(es[c])).astype(np.float32)
        S.append(np.broadcast_to(s, (n, 8, ng)))
    X, Y, Z = corner
    dx, dy, dz = (s * REL + TINY for s in S)
    zlo = (Z.min(-1) - dz).astype(np.float32)
    ok = (S[0] < COORD_MAX) & (S[1] < COORD_MAX) & (S[2] < COORD_MAX) & (zlo >= Z_FLOOR)
    with np.errstate(all="ignore"):
        rx = (X / Z).astype(np.float32)
        ry = (Y / Z).astype(np.float32)
        bounds = []
        for r, d, f, c, lim in ((rx, dx, fx, cx, W), (ry, dy, fy, cy, H)):
            R = np.abs(r).max(-1)
            m = ((d + R * dz) / zlo).astype(np.float32)
            M = (abs(f) * m + f32(2.0 ** -18) * (abs(f) * (R + m) + abs(c) + f32(1))).astype(np.float32)
            lo = ((f * r).min(-1) + c + f32(0.5) - M).astype(np.float32)
            hi = ((f * r).max(-1) + c + f32(0.5) + M).astype(np.float32)
            p0 = np.floor(np.maximum(lo, f32(0))).astype(np.float64)
            p1 = np.floor(np.minimum(hi, f32(lim))).astype(np.float64)
            p0 = np.where(ok, p0, 0).astype(np.int64)
            p1 = np.where(ok, np.minimum(p1, lim - 1), -1).astype(np.int64)
            bounds.append((p0, p1))
    (u0, u1), (v0, v1) = bounds
    need = np.ones((n, 8, ng), bool)
    empty = ok & ((u0 > u1) | (v0 > v1))
    need[empty] = False
    tx0, tx1, ty0, ty1 = u0 // tile, u1 // tile, v0 // tile, v1 // tile
    test = ok & ~empty & ((tx1 - tx0 + 1) * (ty1 - ty0 + 1) <= max_tiles)
    for i in zip(*np.nonzero(test)):
        dmax = tiles[ty0[i]:ty1[i] + 1, tx0[i]:tx1[i] + 1].max()
        need[i] = not (f32(zlo[i] - dmax) >= trunc)
    return need


def updated_by_frame(before, after):
    """Voxels whose weight a frame changed: {block key: bool[16(x), 16(y), 16(z)]} from two oracle exports."""
    kb = {tuple(k): w for k, w in zip(before[0], before[2])}
    out = {}
    for k, w in zip(after[0], after[2]):
        prev = kb.get(tuple(k))
        upd = w != (prev if prev is not None else 0)
        if upd.any():
            out[tuple(k)] = upd.reshape(16, 16, 16)
    return out


def brick_updates(upd, zsplit=2):
    """bool[16, 16, 16] (x, y, z) -> any update per [8 warps, n_groups]."""
    kzg = min(16 // zsplit, 8)
    u = upd.reshape(4, 4, 2, 8, 16 // kzg, kzg)                              # [xb, x, yb, y, g, z]
    return u.any(axis=(1, 3, 5)).reshape(8, 16 // kzg)                       # warp = 2 * xb + yb


# ---- frames that stress the test: each returns depth u16 [n, H, W], rgb [n, H, W, 3], extrinsics [n, 4, 4], intrinsics,
#      voxel length, truncation and depth_trunc
def _rot(ax, deg, t=(0.0, 0.0, 0.0)):
    a = np.deg2rad(deg)
    c, s = np.cos(a), np.sin(a)
    i, j = [(1, 2), (0, 2), (0, 1)][ax]
    e = np.eye(4)
    e[i, i], e[i, j], e[j, i], e[j, j] = c, -s, s, c
    e[:3, 3] = t
    return e


def _plane_depth(W, H, intr, n, p0, rng):
    """Depth of the plane n . X = p0 (camera frame) with 2 mm noise; 0 where it lies behind the camera or past 8 m."""
    fx, fy, cx, cy = intr
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float64)
    ray = np.stack([(xs - cx) / fx, (ys - cy) / fy, np.ones_like(xs)], -1)
    den = ray @ np.asarray(n, np.float64)
    with np.errstate(all="ignore"):
        z = np.where(np.abs(den) > 1e-9, p0 / den, 0.0)
    z = np.where((z > 0) & (z < 8.0), z + rng.uniform(0, 0.002, z.shape), 0.0)
    return np.round(z * 1000.0).astype(np.uint16)


def scene(name, seed=0):
    rng = np.random.default_rng(seed)
    W, H, intr = 64, 48, (40.0, 40.0, 31.5, 23.5)
    if name == "near_wedge":     # tests/test_gpu_integrate_paths.py near_scene: blocks straddle the camera plane
        ys, xs = np.mgrid[0:H, 0:W].astype(np.float64)
        n = 6
        depth = np.empty((n, H, W), np.uint16)
        for k in range(n):
            d = 0.010 + 0.59 * (xs / (W - 1)) ** 2 * (0.6 + 0.4 * ys / (H - 1)) + rng.uniform(0, 0.004, (H, W))
            depth[k] = np.round(d * 1000.0).astype(np.uint16)
        ext = np.stack([_rot(0, 8.0 + 3.0 * k, (0.002 * k, -0.001 * k, 0.0)) for k in range(n)])
        vl, trunc, dtr = 0.01, 0.04, 3.0
    elif name == "border":       # a wall seen off-centre, poses shifted so that blocks straddle the image edges
        n = 6
        depth = np.stack([_plane_depth(W, H, intr, (0.0, 0.0, 1.0), 0.8 + 0.1 * k, rng) for k in range(n)])
        ext = np.stack([_rot(1, 15.0 * (k - 2.5), (0.05 * k, -0.03 * k, 0.02 * k)) for k in range(n)])
        vl, trunc, dtr = 0.005, 0.02, 3.0
    elif name == "grazing":      # planes at 80-89 degrees to the optical axis: long, thin footprints
        n = 6
        depth = np.stack([_plane_depth(W, H, intr, (0.0, np.cos(np.deg2rad(a)), np.sin(np.deg2rad(a))), 0.3, rng)
                          for a in (1.0, 3.0, 5.0, 7.0, 9.0, 10.0)])
        ext = np.stack([_rot(0, 2.0 * k, (0.0, 0.01 * k, 0.0)) for k in range(n)])
        vl, trunc, dtr = 0.005, 0.02, 3.0
    elif name == "holes":        # large invalid regions and a depth_trunc cut through the surface
        n = 6
        depth = np.stack([_plane_depth(W, H, intr, (0.3, 0.2, 1.0), 0.8 + 0.03 * k, rng) for k in range(n)])
        for k in range(n):
            y0, x0 = rng.integers(0, H // 2), rng.integers(0, W // 2)
            depth[k, y0:y0 + H // 2, x0:x0 + W // 2] = 0
            depth[k, :, rng.integers(W // 2, W):] = 0
        ext = np.stack([_rot(2, 10.0 * k, (0.01 * k, 0.0, -0.02 * k)) for k in range(n)])
        vl, trunc, dtr = 0.005, 0.02, 1.0
    elif name == "default":      # the benchmark's sequence (640x480, 5 mm voxels), two frames
        from otslam_b200 import synth
        seq = synth.make_sequence("chair_table", 1000, subsample=(37, 500))
        depth, rgb = seq.numpy()
        return depth, rgb, seq.extrinsic, seq.fxfycxcy, 0.005, 0.02, 3.0
    else:
        raise KeyError(name)
    rgb = rng.integers(0, 256, depth.shape + (3,), dtype=np.uint8)
    return depth, rgb, ext, intr, vl, trunc, dtr


SCENES = ("near_wedge", "border", "grazing", "holes", "default")
