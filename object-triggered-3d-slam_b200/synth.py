"""Analytic synthetic RGB-D sequences in the reference's capture format.

No Gazebo bags or datasets exist offline, so sequences are ray-cast analytically from the scene
vocabulary of the reference's world file
(/root/reference/ros2_ws/src/gazebo_turtlebot3/worlds/cardboard_table_chairs_cones_room.world:249-426:
table, chairs, cones, cardboard box, room) with the reference camera (640x480, fx=fy=565.6009,
cx=320.5, cy=240.5; /root/reference/3d_model/reconstruct_rgbd.py:22-24) and the capture contract
of scanner_node.cpp:260-302: depth = u16 millimetres (NaN / >5 m -> 0, cv::convertTo rounding),
colour RGB8, pose = 4x4 camera(body)->map with 6 decimals, where
`pose_ros @ T_fix` is the optical pose (reconstruct_rgbd.py:29-34,93).

Data generation is plumbing (torch tensor ops, CPU or CUDA); it is not on the measured path.
"""
import math
import os

import numpy as np
import torch

T_FIX = np.array([[0, -1, 0, 0], [0, 0, -1, 0], [1, 0, 0, 0], [0, 0, 0, 1]], dtype=np.float64)
REF_INTRINSICS = (640, 480, 565.6009, 565.6009, 320.5, 240.5)       # reconstruct_rgbd.py:22-24
HD_INTRINSICS = (1280, 720, 1131.2018, 1131.2018, 640.5, 360.5)      # config 4 extension (SURVEY 8d)


# ----------------------------------------------------------------------------- scenes
def _box(cx, cy, z0, z1, sx, sy, color):
    return ("box", (cx - sx / 2, cy - sy / 2, z0), (cx + sx / 2, cy + sy / 2, z1), color)


def table(cx=0.0, cy=0.0, color=(180, 120, 60)):
    prims = [_box(cx, cy, 0.70, 0.75, 1.2, 0.8, color)]
    for sx in (-1, 1):
        for sy in (-1, 1):
            prims.append(_box(cx + sx * 0.55, cy + sy * 0.35, 0.0, 0.70, 0.05, 0.05, (90, 60, 30)))
    return prims


def chair(cx=0.0, cy=0.0, color=(60, 90, 200)):
    prims = [_box(cx, cy, 0.40, 0.45, 0.45, 0.45, color), _box(cx, cy + 0.20, 0.45, 0.90, 0.45, 0.05, color)]
    for sx in (-1, 1):
        for sy in (-1, 1):
            prims.append(_box(cx + sx * 0.20, cy + sy * 0.20, 0.0, 0.40, 0.04, 0.04, (40, 40, 40)))
    return prims


def cone(cx=0.0, cy=0.0, r=0.18, h=0.45, color=(240, 110, 20)):
    return [("cone", (cx, cy, 0.0), (r, h), color)]


def cardboard(cx=0.0, cy=0.0, color=(190, 160, 110)):
    return [_box(cx, cy, 0.0, 0.3, 0.5, 0.4, color)]


def room(sx=8.0, sy=6.0, h=2.5, t=0.1, color=(200, 200, 190)):
    return [_box(0, sy / 2 + t / 2, 0, h, sx + 2 * t, t, color), _box(0, -sy / 2 - t / 2, 0, h, sx + 2 * t, t, color),
            _box(sx / 2 + t / 2, 0, 0, h, t, sy, color), _box(-sx / 2 - t / 2, 0, 0, h, t, sy, color)]


FLOOR_COLOR = (120, 120, 120)

SCENES = {
    "table": lambda: table(),
    "chair_table": lambda: table(0.0, 0.0) + chair(0.0, -0.85),
    "chair": lambda: chair(),
    "cone": lambda: cone(),
    "cardboard": lambda: cardboard(),
    "room": lambda: room() + table(-1.5, 0.8) + chair(-1.5, -0.2) + cone(1.5, 1.0) + cardboard(1.8, -1.2),
}


# ----------------------------------------------------------------------------- trajectories
def look_at(eye, target, up=(0.0, 0.0, 1.0)):
    """4x4 optical-camera -> world pose (z forward, x right, y down)."""
    eye, target, up = (np.asarray(a, np.float64) for a in (eye, target, up))
    f = target - eye
    f /= np.linalg.norm(f)
    r = np.cross(f, up)
    r /= np.linalg.norm(r)
    d = np.cross(f, r)
    T = np.eye(4)
    T[:3, 0], T[:3, 1], T[:3, 2], T[:3, 3] = r, d, f, eye
    return T


def circle(n, radius, height, target=(0.0, 0.0, 0.5), phase=0.0, center=(0.0, 0.0)):
    poses = []
    for k in range(n):
        a = phase + 2 * math.pi * k / n
        eye = (center[0] + radius * math.cos(a), center[1] + radius * math.sin(a), height)
        poses.append(look_at(eye, target))
    return poses


def trajectory(name, n):
    """Named camera trajectories of SURVEY 8(d)."""
    if name == "table":            # config 1: r=2.0 m, h=1.1 m, look-at (0,0,0.5)
        return circle(n, 2.0, 1.1)
    if name == "chair_table":      # config 2: two rings
        n1 = n // 2
        return circle(n1, 1.6, 0.9, (0, -0.4, 0.5)) + circle(n - n1, 2.2, 1.4, (0, -0.4, 0.5), phase=0.1)
    if name in ("chair", "cone", "cardboard"):
        return circle(n, 1.5, 0.9, (0, 0, 0.3))
    if name == "room":             # config 4: lawn-mower + orbit inside the 8x6 room
        poses = []
        n1 = n // 2
        for k in range(n1):
            s = k / max(1, n1 - 1)
            lane = int(s * 4)
            u = s * 4 - lane
            x = -3.0 + 6.0 * (u if lane % 2 == 0 else 1 - u)
            y = -2.0 + lane * 1.3
            yaw = 2 * math.pi * s * 3
            poses.append(look_at((x, y, 1.2), (x + math.cos(yaw), y + math.sin(yaw), 0.9)))
        poses += circle(n - n1, 1.2, 1.3, (0, 0, 0.6))
        return poses
    raise KeyError(name)


def pose_ros_from_optical(T_wo, decimals=6):
    """What scanner_node.cpp:294-298 writes: camera(body)->map, std::fixed 6 decimals."""
    return np.round(T_wo @ np.linalg.inv(T_FIX), decimals)


def extrinsic_from_pose_ros(pose_ros):
    """reconstruct_rgbd.py:93-96."""
    return np.linalg.inv(pose_ros @ T_FIX)


# ----------------------------------------------------------------------------- ray casting
def _checker(P, base, cell=0.08):
    k = torch.floor(P[..., 0] / cell) + torch.floor(P[..., 1] / cell) + torch.floor(P[..., 2] / cell + 0.5)
    shade = torch.where((k.to(torch.int64) & 1) == 0, 1.0, 0.6).to(P.dtype)
    return base.to(P.dtype) * shade[..., None]


def render(prims, T_wo, intr=REF_INTRINSICS, device="cpu", max_range=5.0, floor=True, depth_m=False):
    """Ray-cast one frame. Returns (depth_u16 [H,W], rgb_u8 [H,W,3]) torch tensors on `device`; depth_m=True returns the
    unrounded f64 depth in metres instead of the millimetre image (0 where nothing is hit)."""
    W, H, fx, fy, cx, cy = intr
    dt = torch.float64
    T = torch.as_tensor(T_wo, dtype=dt, device=device)
    j = torch.arange(W, dtype=dt, device=device)
    i = torch.arange(H, dtype=dt, device=device)
    dc = torch.stack(torch.broadcast_tensors(((j - cx) / fx)[None, :], ((i - cy) / fy)[:, None],
                                             torch.ones((), dtype=dt, device=device)), -1)   # z_cam == 1
    D = dc @ T[:3, :3].T                       # world direction, ray parameter == camera z
    O = T[:3, 3]
    best_t = torch.full((H, W), float("inf"), dtype=dt, device=device)
    best_c = torch.zeros((H, W, 3), dtype=dt, device=device)
    eps = 1e-9

    def consider(t, col):
        nonlocal best_t, best_c
        ok = (t > 1e-6) & (t < best_t)
        best_t = torch.where(ok, t, best_t)
        best_c = torch.where(ok[..., None], col, best_c)

    if floor:
        t = -O[2] / torch.where(D[..., 2].abs() < eps, eps, D[..., 2])
        consider(t, torch.tensor(FLOOR_COLOR, dtype=dt, device=device).expand(H, W, 3))
    for p in prims:
        col = torch.tensor(p[3], dtype=dt, device=device).expand(H, W, 3)
        if p[0] == "box":
            lo = torch.tensor(p[1], dtype=dt, device=device)
            hi = torch.tensor(p[2], dtype=dt, device=device)
            inv = 1.0 / torch.where(D.abs() < eps, eps, D)
            t0 = (lo - O) * inv
            t1 = (hi - O) * inv
            tn = torch.minimum(t0, t1).amax(-1)
            tf = torch.maximum(t0, t1).amin(-1)
            hit = (tn <= tf) & (tf > 1e-6)
            t = torch.where(tn > 1e-6, tn, tf)           # inside the box (room walls): exit point
            consider(torch.where(hit, t, float("inf")), col)
        elif p[0] == "cone":                              # apex up, base on z = base z
            bx, by, bz = p[1]
            r, h = p[2]
            k2 = (r / h) ** 2
            ox, oy, oz = O[0] - bx, O[1] - by, O[2] - (bz + h)   # relative to the apex
            a = D[..., 0] ** 2 + D[..., 1] ** 2 - k2 * D[..., 2] ** 2
            b = 2 * (ox * D[..., 0] + oy * D[..., 1] - k2 * oz * D[..., 2])
            c = ox * ox + oy * oy - k2 * oz * oz
            disc = b * b - 4 * a * c
            sq = torch.sqrt(torch.clamp(disc, min=0))
            a_ = torch.where(a.abs() < eps, eps, a)
            for sgn in (-1.0, 1.0):
                t = (-b + sgn * sq) / (2 * a_)
                z = oz + t * D[..., 2]
                ok = (disc >= 0) & (z <= 0) & (z >= -h)
                consider(torch.where(ok, t, float("inf")), col)
            t = (bz - O[2]) / torch.where(D[..., 2].abs() < eps, eps, D[..., 2])   # base cap
            px, py = O[0] + t * D[..., 0] - bx, O[1] + t * D[..., 1] - by
            consider(torch.where(px * px + py * py <= r * r, t, float("inf")), col)
        else:
            raise KeyError(p[0])
    hit = torch.isfinite(best_t) & (best_t <= max_range)          # scanner_node.cpp:277-278
    P = O + best_t.nan_to_num(posinf=0.0)[..., None] * D
    rgb = torch.where(hit[..., None], _checker(P, best_c), torch.zeros_like(best_c))
    if depth_m:
        return torch.where(hit, best_t, torch.zeros_like(best_t)), rgb.round().clamp(0, 255).to(torch.uint8)
    depth = torch.where(hit, torch.round(best_t * 1000.0), torch.zeros_like(best_t))
    depth = depth.clamp(0, 65535).to(torch.int32).to(torch.uint16) if hasattr(torch, "uint16") else depth
    return depth, rgb.round().clamp(0, 255).to(torch.uint8)


class Sequence:
    """depth [N,H,W] u16, rgb [N,H,W,3] u8 (torch, on `device`), pose_ros / extrinsic [N,4,4] f64 (numpy)."""

    def __init__(self, depth, rgb, pose_ros, intr):
        self.depth, self.rgb, self.pose_ros, self.intr = depth, rgb, pose_ros, intr
        self.extrinsic = np.stack([extrinsic_from_pose_ros(p) for p in pose_ros])

    def __len__(self):
        return len(self.pose_ros)

    @property
    def fxfycxcy(self):
        return tuple(self.intr[2:6])

    def numpy(self):
        # torch.uint16 -> numpy via int32 view-safe path
        d = self.depth.cpu()
        d = d.view(torch.int16).numpy().view(np.uint16) if d.dtype == torch.uint16 else d.numpy().astype(np.uint16)
        return d, self.rgb.cpu().numpy()


def make_sequence(scene="table", n_frames=8, intr=REF_INTRINSICS, device="cpu", poses=None, subsample=None):
    """Render `n_frames` of a named scene along its SURVEY 8(d) trajectory.

    subsample=(start, step) keeps frames start::step of the n_frames-long trajectory (so small test
    sequences see the same viewpoints as the full one).
    """
    prims = SCENES[scene]()
    poses = trajectory(scene, n_frames) if poses is None else poses
    if subsample is not None:
        poses = poses[subsample[0]::subsample[1]]
    ds, cs, pr = [], [], []
    for T in poses:
        p_ros = pose_ros_from_optical(T)
        T_used = p_ros @ T_FIX                     # render from the pose the files will carry
        d, c = render(prims, T_used, intr, device)
        ds.append(d)
        cs.append(c)
        pr.append(p_ros)
    return Sequence(torch.stack(ds), torch.stack(cs), np.stack(pr), intr)


def write_capture_tree(seq, base_dir, label="Object_0", start=1):
    """Write color/<label>_<n>.jpg, depth/<label>_<n>.png, poses/<label>_<n>.txt
    (scanner_node.cpp:268-299)."""
    from . import capture
    depth, rgb = seq.numpy()
    for k in range(len(seq)):
        capture.save_frame(base_dir, label, start + k, rgb[k], depth[k], seq.pose_ros[k])


def occupancy_map(w=2000, h=2000, occupied_frac=0.02, seed=0):
    """nav2 map_saver style PGM: 0 occupied, 254 free, 205 unknown
    (/root/reference/fusion/2d_selective_merge.py:64-66)."""
    rng = np.random.default_rng(seed)
    img = np.full((h, w), 254, np.uint8)
    img[rng.random((h, w)) < 0.1] = 205
    img[rng.random((h, w)) < occupied_frac] = 0
    return img
