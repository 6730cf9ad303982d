"""The integration kernel's less common paths against the CPU oracle, bit for bit: warps whose columns
disagree on the branch-free projection guard, intrinsics that rule the branch-free projection out,
extreme truncation distances, NoColor volumes and more than 256 updates of one voxel (the carry of the
split 16-bit count)."""
import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

W, H = 64, 48
INTR = (40.0, 40.0, 31.5, 23.5)
COLOR_TOL = 1.0


def rot_x(deg, t=(0.0, 0.0, 0.0)):
    a = np.deg2rad(deg)
    e = np.eye(4)
    e[1:3, 1:3] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    e[:3, 3] = t
    return e


def near_scene(n, near=0.010, far=0.60, seed=0):
    """A wedge surface from 1 cm to 60 cm in front of a camera tilted about x: the blocks around its
    near edge straddle the camera plane, so within one warp (two x-rows of 16 y-columns) some columns
    come within 2^-9 m of z = 0 and fail the projection guard while their neighbours pass."""
    rng = np.random.default_rng(seed)
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float64)
    depth = np.empty((n, H, W), np.uint16)
    for k in range(n):
        d = near + (far - near) * (xs / (W - 1)) ** 2 * (0.6 + 0.4 * ys / (H - 1)) + rng.uniform(0, 0.004, (H, W))
        depth[k] = np.round(d * 1000.0).astype(np.uint16)
    rgb = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    ext = np.stack([rot_x(8.0 + 3.0 * k, (0.002 * k, -0.001 * k, 0.0)) for k in range(n)])
    return depth, rgb, ext


def oracle_run(depth, rgb, intr, ext, vl, trunc, depth_trunc=3.0):
    ov = oracle.Volume(vl, trunc)
    nupd = 0
    for k in range(len(depth)):
        nupd += ov.integrate(oracle.depth_convert(depth[k], 1000.0, depth_trunc), rgb[k], intr, ext[k])[1]
    return ov, nupd


def gpu_run(depth, rgb, intr, ext, vl, trunc, color=True, zsplit=None, batch=None):
    from otslam_b200.volume import TSDFVolume
    gv = TSDFVolume(vl, trunc, color=color)
    if zsplit:
        gv.set_zsplit(zsplit)
    if batch:
        gv.set_batch(batch)
    gv.integrate_batch(depth, rgb, intr, ext)
    out = gv.export_blocks()
    st = gv.stats()
    gv.close()
    return out, st


def assert_bits(g, ov, color=True):
    gk, gt, gw, gc = g
    ok, ot, ow, oc = ov.export_blocks()
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
def test_mixed_guard_within_warp(zsplit):
    depth, rgb, ext = near_scene(6)
    assert depth.min() <= 12                                   # surface within ~1 cm of the camera
    ov, nupd = oracle_run(depth, rgb, INTR, ext, 0.01, 0.04)
    g, st = gpu_run(depth, rgb, INTR, ext, 0.01, 0.04, zsplit=zsplit)
    assert_bits(g, ov)
    assert st["weight_sum"] == nupd


@pytest.mark.parametrize("intr", [(40.0, 40.0, 1e-7, 23.5), (0.75, 0.75, 31.5, 23.5)], ids=["tiny_cx", "sub_pixel_focal"])
def test_fast_projection_ruled_out(intr):
    """|cx| in (0, 2^-20) and a focal length below 1 pixel both make the host disable the branch-free
    projection: every column takes the IEEE path."""
    depth, rgb, ext = near_scene(4, near=0.2, seed=1)
    ov, nupd = oracle_run(depth, rgb, intr, ext, 0.01, 0.04)
    g, st = gpu_run(depth, rgb, intr, ext, 0.01, 0.04)
    assert_bits(g, ov)
    assert st["weight_sum"] == nupd


@pytest.mark.parametrize("vl,trunc", [(0.01, 1e-4), (0.02, 0.45)], ids=["tiny_trunc", "huge_trunc"])
def test_extreme_sdf_trunc(vl, trunc):
    depth, rgb, ext = near_scene(4, seed=2)
    ov, nupd = oracle_run(depth, rgb, INTR, ext, vl, trunc)
    g, st = gpu_run(depth, rgb, INTR, ext, vl, trunc)
    assert_bits(g, ov)
    assert st["weight_sum"] == nupd


@pytest.mark.parametrize("with_rgb", [True, False])
def test_no_color(with_rgb):
    """A NoColor volume keeps zero colour sums whether or not colour images are passed."""
    depth, rgb, ext = near_scene(5, seed=3)
    ov, nupd = oracle_run(depth, rgb, INTR, ext, 0.01, 0.04)
    g, st = gpu_run(depth, rgb if with_rgb else None, INTR, ext, 0.01, 0.04, color=False)
    assert_bits(g, ov, color=False)
    assert st["weight_sum"] == nupd


def test_count_carry_past_256_updates():
    """300 frames of one static view: every observed voxel is updated up to 300 times, so the low byte
    of its count (top byte of .y) wraps and carries into .z; colours vary per frame."""
    n = 300
    rng = np.random.default_rng(4)
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float64)
    d = np.round((0.45 + 0.2 * xs / (W - 1) + 0.05 * ys / (H - 1)) * 1000.0).astype(np.uint16)
    depth = np.repeat(d[None], n, axis=0)
    depth[rng.random(depth.shape) < 0.02] = 0                 # a few invalid pixels: counts differ per voxel
    rgb = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    ext = np.repeat(rot_x(5.0)[None], n, axis=0)
    ov, nupd = oracle_run(depth, rgb, INTR, ext, 0.01, 0.04)
    g, st = gpu_run(depth, rgb, INTR, ext, 0.01, 0.04)
    assert_bits(g, ov)
    assert st["weight_sum"] == nupd
    w = g[2]
    assert w.max() == n and ((w > 256) & (w < n)).any()
