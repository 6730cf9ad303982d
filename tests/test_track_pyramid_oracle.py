"""Coarse-to-fine frame-to-model tracking pinned on the CPU (DESIGN.md §4 "Frame-to-model tracking"): the depth pyramid of
tests/models/track_pyramid_model.cpp equals a NumPy restatement bit for bit; each level's intrinsics look along the rays through
the centres of the pixel blocks it averages; on the room corner of test_track_oracle.py the pyramid recovers starts that
single-scale tracking loses; one level is single-scale tracking, bit for bit; and the new argument checks of
otslam_volume_track_pyramid run without a GPU.  The model is tests/models/track_pyramid_model.cpp (which includes the
single-scale model, tests/models/track_model.cpp); tests/test_gpu_track_pyramid.py uses it as the reference for the CUDA
kernels."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_raycast_oracle import INTR, VL, H, W, interior, plane_depth, raycast, volume
from test_track_oracle import CAMS, ROOT, STARTS, corner_depth, perturb, pose_error, track, u16

_p = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731


_MODEL = None


def _lib():
    """track_pyramid_model.cpp + raycast_model.cpp compiled like the oracle (g++ -O2 -fopenmp -ffp-contract=off) into a
    temporary dir"""
    global _MODEL
    if _MODEL is not None:
        return _MODEL
    d = tempfile.mkdtemp(prefix="otslam_track_pyramid_model_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "track_pyramid_model.so")
    m = os.path.join(ROOT, "tests", "models")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-fopenmp", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(m, "track_pyramid_model.cpp"), os.path.join(m, "raycast_model.cpp")])
    lib = C.CDLL(so)
    lib.track_model_pyramid.restype = C.c_int
    lib.track_model_pyramid.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int,
                                        C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                        C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
    lib.track_model_levels.restype = C.c_int64
    lib.track_model_levels.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int,
                                       C.c_void_p]
    lib.track_model_level_intr.restype = None
    lib.track_model_level_intr.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    _MODEL = lib
    return lib


def track_pyramid(vol, depth, intr, init_extrinsics, depth_diff, max_iterations, depth_scale=1000.0, depth_min=0.1,
                  depth_max=3.0):
    """track() over a pyramid of len(depth_diff) levels (index = level, 0 = full resolution) on the CPU model"""
    keys, tsdf, weight, _ = vol.export_blocks(color=False)
    d = np.ascontiguousarray(depth, np.uint16).reshape(-1, *np.shape(depth)[-2:])
    n, h, w = d.shape
    e = np.ascontiguousarray(init_extrinsics, np.float64).reshape(n, 16)
    k = np.ascontiguousarray(intr, np.float64).reshape(4)
    dd = np.ascontiguousarray(depth_diff, np.float64)
    mi = np.ascontiguousarray(max_iterations, np.int32)
    assert len(dd) == len(mi)
    out = {"extrinsic": np.empty((n, 4, 4)), "status": np.empty(n, np.int32), "iterations": np.empty(n, np.int32),
           "fitness": np.empty(n), "inlier_rmse": np.empty(n)}
    r = _lib().track_model_pyramid(len(keys), _p(keys), _p(tsdf), _p(weight), vol.voxel_length, vol.sdf_trunc, n, _p(d), w, h,
                                   _p(k), _p(e), depth_scale, depth_min, depth_max, len(dd), _p(dd), _p(mi),
                                   _p(out["extrinsic"]), _p(out["status"]), _p(out["iterations"]), _p(out["fitness"]),
                                   _p(out["inlier_rmse"]))
    if r < 0:
        raise RuntimeError("bad tracking arguments")
    return out


def model_levels(depth, depth_scale, depth_max, voxel_length, n_levels):
    """levels 1 .. n_levels - 1 of the model's pyramid of one u16 frame"""
    d = np.ascontiguousarray(depth, np.uint16)
    h, w = d.shape
    sizes = [(h >> l, w >> l) for l in range(1, n_levels)]
    out = np.empty(sum(a * b for a, b in sizes), np.float32)
    assert _lib().track_model_levels(1, _p(d), w, h, depth_scale, depth_max, voxel_length, n_levels, _p(out)) == out.size
    levels, at = [], 0
    for a, b in sizes:
        levels.append(out[at:at + a * b].reshape(a, b))
        at += a * b
    return levels


def level_intr(intr, level):
    out = np.empty(4)
    _lib().track_model_level_intr(_p(np.ascontiguousarray(intr, np.float64)), level, _p(out))
    return out


def numpy_levels(depth, depth_scale, depth_max, voxel_length, n_levels):
    """the pyramid restated: level 0 is raw / scale in FP32, valid when > 0 and < depth_max; a coarse pixel keeps the valid
    depths of its 2x2 block within 4 voxels of the block's smallest, sums them in FP64 in raster order, divides by their
    count and rounds to FP32 (0 when none is valid)"""
    d = depth.astype(np.float32) / np.float32(depth_scale)
    valid = (d > 0) & (d.astype(np.float64) < depth_max)
    out = []
    for _ in range(1, n_levels):
        h, w = d.shape[0] >> 1, d.shape[1] >> 1
        quad = [d[dy:2 * h:2, dx:2 * w:2] for dy in (0, 1) for dx in (0, 1)]        # raster order: TL, TR, BL, BR
        ok = [valid[dy:2 * h:2, dx:2 * w:2] for dy in (0, 1) for dx in (0, 1)]
        lo = np.min([np.where(o, q, np.inf) for q, o in zip(quad, ok)], axis=0).astype(np.float64)
        s, n = np.zeros((h, w)), np.zeros((h, w))
        for q, o in zip(quad, ok):
            keep = o & (q.astype(np.float64) - lo <= 4.0 * voxel_length)
            s = np.where(keep, s + q.astype(np.float64), s)
            n += keep
        d = np.where(n > 0, (s / np.maximum(n, 1)).astype(np.float32), np.float32(0))
        valid = d > 0
        out.append(d)
    return out


def test_pyramid_equals_numpy_restatement():
    rng = np.random.default_rng(0)
    for h, w in ((120, 160), (61, 83), (17, 33)):
        # smooth depth with depth edges (jumps beyond the 4-voxel band and within it), holes, all-invalid blocks, and
        # depths at and beyond depth_max
        base = 1500 + 400 * np.sin(np.arange(w) / 7.0)[None, :] + 300 * np.cos(np.arange(h) / 5.0)[:, None]
        raw = base + rng.choice([0, 5, 19, 20, 21, 60, 400], size=(h, w), p=[0.5, 0.1, 0.08, 0.08, 0.08, 0.08, 0.08])
        raw[rng.random((h, w)) < 0.1] = 0
        raw[rng.random((h, w)) < 0.03] = 3000             # exactly depth_max: invalid
        raw[rng.random((h, w)) < 0.03] = 3001
        raw[rng.random((h, w)) < 0.03] = 2999
        raw[:4, :4] = 0                                    # an all-invalid block at every level up to 4x4
        raw[-2:, 4:8] = 3000
        raw = np.clip(raw, 0, 65535).astype(np.uint16)
        for vl in (0.005, 0.01):
            got = model_levels(raw, 1000.0, 3.0, vl, 4)
            ref = numpy_levels(raw, 1000.0, 3.0, vl, 4)
            for l, (g, r) in enumerate(zip(got, ref), 1):
                assert g.shape == (h >> l, w >> l) and r.shape == g.shape, (h, w, l)
                assert (g.view(np.uint32) == r.view(np.uint32)).all(), (h, w, vl, l)
            assert (got[0][:2, :2] == 0).all() and (got[0] > 0).any()
            assert got[0].max() < 3.0


def test_level_intrinsics_look_through_block_centres():
    """a fronto-parallel plane at 1 m: at every level, the model's vertex at coarse pixel (u', v') is the plane's point on
    the level-0 ray through the centre of the block the pixel covers, within the 0.1-voxel bound of the level-0 render
    (a half-pixel error in cx / cy moves that point by 1.8 mm or more at level 1)"""
    E = np.eye(4)
    dep = plane_depth(E, np.array([0.0, 0.0, 1.0]), 1.0)
    v = volume([dep], [E])
    fx, fy, cx, cy = INTR
    inside = interior(dep > 0, 6)
    for level in range(4):
        s = 1 << level
        w, h = W >> level, H >> level
        k = level_intr(INTR, level)
        if level == 0:
            assert tuple(k) == INTR
        out = raycast(v, k, E[None], w, h)
        u, vv = np.meshgrid(s * np.arange(w) + (s - 1) / 2, s * np.arange(h) + (s - 1) / 2)
        ref = np.stack([(u - cx) / fx, (vv - cy) / fy, np.ones_like(u)], -1)          # the plane z = 1 along those rays
        m = inside[::s, ::s][:h, :w] & inside[s - 1::s, s - 1::s][:h, :w]
        assert m.sum() > 0.3 * m.size, level
        got = out["vertex"][0].astype(np.float64)
        assert np.abs(out["depth"][0][m] - 1.0).max() <= 0.1 * VL, level
        assert np.linalg.norm(got[m] - ref[m], axis=-1).max() <= 0.1 * VL, level


# Starts that single-scale tracking with the 7 cm gate cannot recover (the comment above test_track_oracle.STARTS): a turn
# and a shift that move the image the same way add up, and the back wall leaves the gate.
HARD = [((0, 1, 0), 2.0, (0.02, 0.0, 0.0)), ((0, 1, 0), -2.0, (-0.02, 0.0, 0.0)), ((1, 0, 0), -2.0, (0.0, -0.02, 0.0)),
        ((1, 0, 0), 2.0, (0.0, 0.02, 0.0)), ((1, 1, 0), 2.0, (0.0141, -0.0141, 0.0)), ((1, 1, 0), -2.0, (-0.0141, 0.0141, 0.0))]
PYRAMID = ((0.07, 0.15, 0.3), (20, 10, 10))


@pytest.fixture(scope="module")
def corner():
    return volume([corner_depth(e) for e in CAMS], CAMS)


def test_pyramid_recovers_where_single_scale_fails(corner):
    truth = CAMS[0]
    dep = np.stack([u16(corner_depth(truth))] * len(HARD))
    inits = np.stack([perturb(truth, *s) for s in HARD])
    single = track(corner, dep, INTR, inits, depth_scale=10000.0)
    pyr = track_pyramid(corner, dep, INTR, inits, *PYRAMID, depth_scale=10000.0)
    lost = 0
    for i in range(len(HARD)):
        dt, dr = pose_error(pyr["extrinsic"][i], truth)
        assert pyr["status"][i] == 0, (i, pyr["status"][i], pyr["iterations"][i])
        assert dt <= 0.2 * VL and dr <= 0.1, (i, dt, dr)
        assert pyr["fitness"][i] > 0.8 and pyr["inlier_rmse"][i] < 0.1 * VL
        st, (dt1, dr1) = single["status"][i], pose_error(single["extrinsic"][i], truth)
        lost += st != 0 or dt1 > 0.2 * VL or dr1 > 0.1
    assert lost >= 1
    # every level runs at least one iteration, and the sum is reported
    assert (pyr["iterations"] >= 3).all() and (pyr["iterations"] <= sum(PYRAMID[1])).all()


def test_one_level_equals_single_scale(corner):
    truth = CAMS[0]
    inits = np.stack([perturb(truth, *s) for s in STARTS + HARD[:2]])
    dep = np.stack([u16(corner_depth(truth))] * len(inits))
    for diff, it in ((0.07, 20), (0.03, 4)):
        a = track(corner, dep, INTR, inits, depth_scale=10000.0, depth_diff=diff, max_iterations=it)
        b = track_pyramid(corner, dep, INTR, inits, [diff], [it], depth_scale=10000.0)
        for k in a:
            assert (a[k].view(np.uint8) == b[k].view(np.uint8)).all(), k


def test_model_refuses_bad_pyramids(corner):
    dep = u16(corner_depth(CAMS[0]))[None]
    for dd, mi in (([], []), ([0.07] * 5, [10] * 5), ([0.07, 0.0], [10, 10]), ([0.07, 0.1], [10, 0]), ([0.07, 0.1], [10, 101])):
        with pytest.raises(RuntimeError):
            track_pyramid(corner, dep, INTR, CAMS[0][None], dd, mi, depth_scale=10000.0)
    with pytest.raises(RuntimeError):          # 160x120 >> 4 is below one 16x8 tile
        track_pyramid(corner, dep[:, :, :120], INTR, CAMS[0][None], [0.07] * 4, [5] * 4, depth_scale=10000.0)


def test_track_pyramid_argument_checks_without_gpu():
    """every new argument of otslam_volume_track_pyramid is checked before any CUDA call (a null volume last)"""
    from otslam_b200 import _lib
    L = _lib.lib
    k = np.array(INTR, np.float64)
    e = np.eye(4).reshape(1, 16).copy()
    d = np.zeros((1, H, W), np.uint16)
    out = np.zeros((1, 16))

    def call(n=1, w=W, h=H, levels=3, diff=(0.07, 0.15, 0.3), iters=(20, 10, 10), scale=1000.0, ext=e, mem=_lib.MEM_HOST):
        dd = None if diff is None else np.ascontiguousarray(diff, np.float64)
        mi = None if iters is None else np.ascontiguousarray(iters, np.int32)
        st = L.otslam_volume_track_pyramid(None, n, _lib.ptr(d), w, h, _lib.ptr(k), _lib.ptr(ext), scale, 0.1, 3.0, levels,
                                           _lib.ptr(dd), _lib.ptr(mi), _lib.ptr(out), None, None, None, None, mem)
        return st, _lib.last_error()

    cases = {
        "levels 0": call(levels=0), "levels 5": call(levels=5, diff=[0.07] * 5, iters=[10] * 5),
        "null diff": call(diff=None), "null iters": call(iters=None),
        "diff 0 at level 2": call(diff=(0.07, 0.15, 0.0)), "diff < 0 at level 1": call(diff=(0.07, -0.1, 0.3)),
        "diff nan": call(diff=(np.nan, 0.15, 0.3)), "diff inf": call(diff=(0.07, np.inf, 0.3)),
        "iters 0 at level 1": call(iters=(20, 0, 10)), "iters 101 at level 2": call(iters=(20, 10, 101)),
        "coarsest narrower than 16": call(w=63), "coarsest shorter than 8": call(h=31),
        "4 levels of 160x120": call(levels=4, diff=[0.07] * 4, iters=[10] * 4, w=120),
        # otslam_volume_track's own checks still hold
        "n": call(n=-1), "scale": call(scale=0.0), "memory": call(mem=7), "singular": call(ext=np.zeros((1, 16))),
    }
    for name, (st, msg) in cases.items():
        assert st == _lib.ERR_INVALID, name
        assert "null volume" not in msg, name
    for ok in (call(), call(w=64, h=32), call(levels=4, diff=[0.07] * 4, iters=[1] * 4), call(levels=1, diff=[0.07], iters=[1], w=1, h=1)):
        st, msg = ok
        assert st == _lib.ERR_INVALID and "null volume" in msg
