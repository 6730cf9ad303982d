"""Ray casting pinned analytically on the CPU oracle (DESIGN.md §4 "Ray casting"): planes and a sphere integrated from f32
depth (no millimetre quantisation) render back at their analytic depth with the right normals; empty volumes, windows
that exclude the surface, cameras facing away and cameras inside an object see nothing; the block-grid DDA does not step
over a lone allocated block.  Argument checks of otslam_volume_raycast run without a GPU.

The ray caster's CPU restatement is tests/models/raycast_model.cpp; `raycast` below runs it on the voxels of an oracle
volume (oracle.Volume.export_blocks) and on the camera poses of oracle.inverse4.  tests/test_gpu_raycast.py uses it as the
reference for the CUDA kernel."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_MODEL = None


def model():
    """tests/models/raycast_model.cpp compiled like the oracle (g++ -O2 -fopenmp -ffp-contract=off) into a temporary dir"""
    global _MODEL
    if _MODEL is None:
        d = tempfile.mkdtemp(prefix="otslam_raycast_model_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "raycast_model.so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-fopenmp", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-o", so,
                               os.path.join(ROOT, "tests", "models", "raycast_model.cpp")])
        lib = C.CDLL(so)
        lib.raycast_model.restype = C.c_int64
        lib.raycast_model.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int,
                                      C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
        _MODEL = lib
    return _MODEL


def raycast(vol, intr, extrinsics, width, height, depth_min=0.1, depth_max=3.0):
    """Render n views of oracle volume `vol`: dict of depth [n,H,W] f32, vertex / normal [n,H,W,3] f32, color [n,H,W,3] u8
    (0 = no hit) and n_hits.  intr = (fx, fy, cx, cy); extrinsics [n,4,4] world->camera."""
    keys, tsdf, weight, col = vol.export_blocks(color=True)
    e = np.ascontiguousarray(extrinsics, np.float64).reshape(-1, 4, 4)
    poses = np.ascontiguousarray(np.stack([oracle.inverse4(x) for x in e]) if len(e) else np.zeros((0, 4, 4)))
    k = np.ascontiguousarray(intr, np.float64).reshape(4)
    n, H, W = len(e), int(height), int(width)
    out = {"depth": np.empty((n, H, W), np.float32), "vertex": np.empty((n, H, W, 3), np.float32),
           "normal": np.empty((n, H, W, 3), np.float32), "color": np.empty((n, H, W, 3), np.uint8)}
    p = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    r = int(model().raycast_model(len(keys), p(keys), p(tsdf), p(weight), p(col), vol.voxel_length, vol.sdf_trunc, n, W, H, p(k),
                                  p(poses), depth_min, depth_max, p(out["depth"]), p(out["vertex"]), p(out["normal"]),
                                  p(out["color"])))
    if r < 0:
        raise RuntimeError("bad ray-cast arguments")
    out["n_hits"] = r
    return out


W, H = 160, 120
INTR = (280.0, 280.0, 79.5, 59.5)      # 3.6 mm per pixel at 1 m: finer than the 1 cm voxels
VL, TRUNC = 0.01, 0.04
RGB = np.broadcast_to(np.array([200, 100, 50], np.uint8), (H, W, 3)).copy()


def rays(extrinsic):
    """camera centre and world direction of every pixel (FP64), t = camera z"""
    pose = np.linalg.inv(extrinsic)
    fx, fy, cx, cy = INTR
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    dc = np.stack([(u - cx) / fx, (v - cy) / fy, np.ones_like(u)], -1)
    return pose[:3, 3], dc @ pose[:3, :3].T


def plane_depth(extrinsic, n, c):
    """depth of the plane n.x = c (0 where it is behind the camera)"""
    o, d = rays(extrinsic)
    t = (c - n @ o) / (d @ n)
    return np.where(t > 0, t, 0.0)


def sphere_depth(extrinsic, centre, r):
    o, d = rays(extrinsic)
    oc = o - np.asarray(centre)
    a = (d * d).sum(-1)
    b = 2 * (d @ oc)
    cc = oc @ oc - r * r
    disc = b * b - 4 * a * cc
    t = (-b - np.sqrt(np.maximum(disc, 0))) / (2 * a)
    return np.where((disc > 0) & (t > 0), t, 0.0)


def look(eye, target):
    """world->camera extrinsic of a camera at `eye` looking at `target` (optical frame: z forward, y down)"""
    eye, target = np.asarray(eye, float), np.asarray(target, float)
    z = target - eye
    z /= np.linalg.norm(z)
    up = np.array([0.0, -1.0, 0.0]) if abs(z[1]) < 0.9 else np.array([0.0, 0.0, 1.0])
    x = np.cross(up, z)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    pose = np.eye(4)
    pose[:3, 0], pose[:3, 1], pose[:3, 2], pose[:3, 3] = x, y, z, eye
    return np.linalg.inv(pose)


def volume(depths, extrinsics):
    v = oracle.Volume(VL, TRUNC)
    for dep, e in zip(depths, extrinsics):
        v.integrate(dep.astype(np.float32), RGB, INTR, e)
    return v


def interior(mask, px):
    """pixels at least `px` pixels inside a boolean mask"""
    from scipy.ndimage import binary_erosion
    return binary_erosion(mask, iterations=px, border_value=0)


def angle_deg(a, b):
    cos = (a * b).sum(-1) / (np.linalg.norm(a, axis=-1) * np.linalg.norm(b, axis=-1))
    return np.degrees(np.arccos(np.clip(cos, -1, 1)))


def test_fronto_parallel_plane():
    E = np.eye(4)
    dep = plane_depth(E, np.array([0.0, 0.0, 1.0]), 1.0)
    v = volume([dep], [E])
    out = raycast(v, INTR, E[None], W, H)
    # 2 voxels (plus the normal's +-1 voxel stencil) inside the observed region: 3 voxels = 4.2 px at 1 m
    m = interior(dep > 0, 5)
    got = out["depth"][0]
    assert (got[m] > 0).all()
    assert np.abs(got[m] - 1.0).max() <= 0.1 * VL
    assert angle_deg(out["normal"][0][m], np.array([0.0, 0.0, -1.0])).max() <= 1.0
    assert np.abs(out["vertex"][0][m][:, 2] - 1.0).max() <= 0.1 * VL
    assert (out["color"][0][m] == RGB[0, 0]).all()
    assert out["n_hits"] == int((got > 0).sum())
    assert (out["vertex"][0][got == 0] == 0).all() and (out["normal"][0][got == 0] == 0).all()


def test_tilted_plane():
    E = np.eye(4)
    n = np.array([0.0, np.sin(np.radians(35)), -np.cos(np.radians(35))])
    c = n @ np.array([0.0, 0.0, 1.0])
    dep = plane_depth(E, n, c)
    dep[dep > 2.0] = 0.0
    v = volume([dep], [E])
    out = raycast(v, INTR, E[None], W, H)
    m = interior(dep > 0, 6)
    got = out["depth"][0]
    assert (got[m] > 0).all()
    # metric error along the ray, in voxels
    err = np.abs(got[m] - dep[m]) * np.linalg.norm(rays(E)[1], axis=-1)[m] / VL
    assert err.max() <= 0.25
    assert np.median(angle_deg(out["normal"][0][m], n)) <= 1.0          # n faces the camera: the TSDF grows that way


def test_sphere():
    centre, r = np.array([0.0, 0.0, 1.0]), 0.3
    E = np.eye(4)
    dep = sphere_depth(E, centre, r)
    v = volume([dep], [E])
    out = raycast(v, INTR, E[None], W, H)
    o, d = rays(E)
    nrm = (o + dep[..., None] * d - centre) / r
    cos_inc = -(nrm * d).sum(-1) / np.linalg.norm(d, axis=-1)
    m = interior(dep > 0, 3) & (cos_inc > 0.5)          # away from the grazing rim (incidence below 60 degrees)
    got = out["depth"][0]
    assert (got[m] > 0).all()
    err = np.abs(got[m] - dep[m]) * np.linalg.norm(d, axis=-1)[m] / VL
    assert err.max() <= 0.25
    radial = out["vertex"][0][m].astype(np.float64) - centre
    ang = angle_deg(out["normal"][0][m].astype(np.float64), radial)     # the TSDF grows outward: the gradient points out
    assert np.median(ang) <= 2.0 and np.percentile(ang, 90) <= 3.0


def test_no_hits():
    E = np.eye(4)
    empty = oracle.Volume(VL, TRUNC)
    assert raycast(empty, INTR, E[None], W, H)["n_hits"] == 0
    dep = plane_depth(E, np.array([0.0, 0.0, 1.0]), 1.0)
    v = volume([dep], [E])
    assert raycast(v, INTR, E[None], W, H)["n_hits"] > 0
    assert raycast(v, INTR, E[None], W, H, depth_max=0.9)["n_hits"] == 0     # window ends before the surface
    assert raycast(v, INTR, E[None], W, H, depth_min=1.1)["n_hits"] == 0     # window starts behind it
    away = look([0.0, 0.0, 0.0], [0.0, 0.0, -1.0])                          # facing away from the plane
    out = raycast(v, INTR, away[None], W, H)
    assert out["n_hits"] == 0 and not out["depth"].any() and not out["color"].any()


def test_camera_inside_object_sees_no_back_faces():
    centre, r = np.array([0.0, 0.0, 1.5]), 0.3
    eyes = [centre + 1.2 * np.array(d) for d in ([1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1])]
    exts = [look(e, centre) for e in eyes]
    v = volume([sphere_depth(e, centre, r) for e in exts], exts)
    assert raycast(v, INTR, exts[0][None], W, H)["n_hits"] > 0               # from outside: the sphere
    inside = [look(centre, centre + np.array(d)) for d in ([1, 0, 0], [0, 0, 1], [0, 1, 0])]
    out = raycast(v, INTR, np.stack(inside), W, H, depth_min=0.01)
    assert out["n_hits"] == 0


def test_dda_reaches_a_lone_block():
    """only the blocks around a 9x9-pixel patch exist; rays start 0.9 m before them, in absent blocks"""
    E = np.eye(4)
    dep = plane_depth(E, np.array([0.0, 0.0, 1.0]), 1.0)
    patch = np.zeros_like(dep)
    patch[52:61, 100:109] = dep[52:61, 100:109]
    v = volume([patch], [E])
    assert v.num_blocks() <= 8
    out = raycast(v, INTR, E[None], W, H)
    got = out["depth"][0]
    assert got[56, 104] > 0 and abs(got[56, 104] - 1.0) <= 0.1 * VL
    assert (got[:, :90] == 0).all()
    # an oblique camera whose rays cross several absent blocks sideways before they reach the patch
    side = look([-0.6, 0.0, 0.2], [0.27, -0.02, 1.0])
    o = raycast(v, INTR, side[None], W, H)
    assert o["n_hits"] > 0
    hit = o["depth"][0] > 0
    P = o["vertex"][0][hit]
    assert np.abs(P[:, 2] - 1.0).max() <= 0.25 * VL / np.cos(np.radians(60))


def test_raycast_argument_checks_without_gpu():
    """every argument is checked before any CUDA call (a null volume is checked after the other arguments)"""
    from otslam_b200 import _lib
    L = _lib.lib
    k = np.array(INTR, np.float64)
    e = np.eye(4).reshape(1, 16).copy()
    hits = C.c_int64(123)

    def call(n=1, w=W, h=H, intr=k, ext=e, dmin=0.1, dmax=3.0):
        hits.value = 123
        st = L.otslam_volume_raycast(None, n, w, h, _lib.ptr(intr), _lib.ptr(ext), dmin, dmax, None, None, None, None,
                                     C.byref(hits))
        assert hits.value == 0
        return st, _lib.last_error()

    sing = np.zeros((1, 16))
    nan_e = e.copy()
    nan_e[0, 3] = np.nan
    cases = {
        "n_views": call(n=-1), "width": call(w=0), "height": call(h=-5),
        "null intr": call(intr=None), "fx": call(intr=np.array([0.0, 140, 79.5, 59.5])),
        "fx nan": call(intr=np.array([np.nan, 140, 79.5, 59.5])), "fy inf": call(intr=np.array([140, np.inf, 79.5, 59.5])),
        "cx nan": call(intr=np.array([140, 140, np.nan, 59.5])),
        "dmin 0": call(dmin=0.0), "dmin >= dmax": call(dmin=2.0, dmax=2.0), "dmax inf": call(dmax=np.inf),
        "dmin nan": call(dmin=np.nan), "null ext": call(ext=None), "singular": call(ext=sing), "nan ext": call(ext=nan_e),
        "overflow": call(n=1 << 30, w=1 << 16, h=1 << 16, ext=np.tile(e, (1, 1))),
    }
    for name, (st, msg) in cases.items():
        assert st == _lib.ERR_INVALID, name
        assert "null volume" not in msg, name            # refused for its own reason, before the volume is looked at
    st, msg = call()
    assert st == _lib.ERR_INVALID and "null volume" in msg
    assert L.otslam_volume_raycast(None, 0, W, H, _lib.ptr(k), None, 0.1, 3.0, None, None, None, None, None) == _lib.ERR_INVALID


def test_model_refuses_bad_windows():
    v = oracle.Volume(VL, TRUNC)
    E = np.eye(4)[None]
    with pytest.raises(RuntimeError):
        raycast(v, INTR, E, W, H, depth_min=0.0)
    with pytest.raises(RuntimeError):
        raycast(v, INTR, E, W, H, depth_max=1e6)
