"""Frame-to-model tracking timings and pose errors on one GPU, single-scale and coarse to fine.  Prints one JSON line.

Legs: configs[1] (1000 frames of the chair+table sequence, 640x480, 5 mm) and the HD geometry of configs[3] (2000 frames of
the large room, 1280x720, 2 mm).  Per leg the volume is integrated from HBM at the true poses, then every captured frame
(a CUDA tensor) is tracked against it in batches of 32, from initial poses moved by 1-3 cm and turned by 1-2 degrees in
seeded random directions, twice from the same starts: single-scale (the defaults of TSDFVolume.track) and with
volume.TRACK_PYRAMID.  One batch of each warms up first.  Reported per run: frames/s from the device time of the calls
(otslam_last_op_device_ms, summed) and from wall time; mean iterations; status counts; and the median, 95th percentile and
maximum translation and rotation error against the true poses, for each status separately.  Single-scale runs also report
the share of device time that the model render takes (the same poses ray cast separately into CUDA tensors with vertex
and normal only: the tracker's render).
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

BATCH = 32


def rot(axis, deg):
    import numpy as np
    a = np.asarray(axis, float) / np.linalg.norm(axis)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    t = np.radians(deg)
    return np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K


def perturb(extrinsic, axis, deg, shift):
    """the extrinsic of the camera moved by `shift` metres and turned by `deg` about `axis`, both in its own frame"""
    import numpy as np
    d = np.eye(4)
    d[:3, :3] = rot(axis, deg)
    d[:3, 3] = shift
    return np.linalg.inv(np.linalg.inv(extrinsic) @ d)


def pose_error(extrinsic, truth):
    """(translation error in metres, rotation error in degrees) between two world->camera extrinsics"""
    import numpy as np
    a, b = np.linalg.inv(extrinsic), np.linalg.inv(truth)
    cos = (np.trace(a[:3, :3] @ b[:3, :3].T) - 1) / 2
    return float(np.linalg.norm(a[:3, 3] - b[:3, 3])), float(np.degrees(np.arccos(np.clip(cos, -1, 1))))


def starts(extrinsics, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    out = []
    for e in extrinsics:
        d = rng.normal(size=3)
        out.append(perturb(e, rng.normal(size=3), rng.uniform(1.0, 2.0) * rng.choice([-1, 1]), d / np.linalg.norm(d) * rng.uniform(0.01, 0.03)))
    return np.stack(out)


def stats(x):
    import numpy as np
    return {"median": float(np.median(x)), "p95": float(np.percentile(x, 95)), "max": float(x.max())} if len(x) else None


def run(vol, d, k, init, ext, W, H, render, **kw):
    """track every frame in batches from `init` with TSDFVolume.track(**kw); timings, status counts and errors by status"""
    import numpy as np
    import torch
    from otslam_b200 import _lib
    frames = len(init)
    vol.track(d[:BATCH], k, init[:BATCH], **kw)                     # warm-up
    torch.cuda.synchronize()
    dev_ms, wall, render_ms = 0.0, 0.0, 0.0
    res = {x: [] for x in ("extrinsic", "status", "iterations")}
    for first in range(0, frames, BATCH):
        t0 = time.perf_counter()
        r = vol.track(d[first:first + BATCH], k, init[first:first + BATCH], **kw)   # returns with the results on the host
        wall += time.perf_counter() - t0
        dev_ms += _lib.last_op_device_ms()
        for x in res:
            res[x].append(r[x])
        if render:
            vol.ray_cast_tensors(k, init[first:first + BATCH], W, H, attributes=("vertex", "normal"))
            render_ms += _lib.last_op_device_ms()
    res = {x: np.concatenate(v) for x, v in res.items()}
    err = np.array([pose_error(x, t) for x, t in zip(res["extrinsic"], ext)])
    out = {"frames_per_s_device": frames / (dev_ms * 1e-3), "frames_per_s_wall": frames / wall,
           "mean_iterations": float(res["iterations"].mean()),
           "status_counts": {str(s): int((res["status"] == s).sum()) for s in range(4)},
           "error_by_status": {str(s): {"translation_mm": stats(err[res["status"] == s, 0] * 1e3),
                                        "rotation_deg": stats(err[res["status"] == s, 1])}
                               for s in range(4) if (res["status"] == s).any()}}
    if render:
        out["render_share_of_device_time"] = render_ms / dev_ms
    return out


def leg(name, scene, frames, intr, voxel, settings):
    import torch
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq = synth.make_sequence(scene, frames, intr=intr, device="cuda:0")
    d, c, ext, k = seq.depth, seq.rgb, seq.extrinsic, seq.fxfycxcy
    W, H = intr[0], intr[1]
    vol = TSDFVolume(voxel, 4 * voxel)
    vol.integrate_batch(d, c, k, ext)
    torch.cuda.synchronize()
    init = starts(ext, 11)
    vol.ray_cast_tensors(k, init[:BATCH], W, H, attributes=("vertex", "normal"))     # warm-up of the separate render
    out = {"workload": name, "frames": frames, "width": W, "height": H, "voxel_mm": voxel * 1000}
    for label, kw in settings.items():
        out[label] = run(vol, d, k, init, ext, W, H, not kw, **kw)
    vol.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--hd-frames", type=int, default=2000, help="0 = skip the HD leg")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("track_bench needs a CUDA device")
    from otslam_b200 import synth
    from otslam_b200.volume import TRACK_PYRAMID
    from raycast_bench import gpu_details
    res = gpu_details()
    res["batch_frames"] = BATCH
    res["initial_error"] = "1-3 cm, 1-2 degrees, seeded directions"
    settings = {"single_scale": {}, "pyramid": dict(TRACK_PYRAMID)}
    res["pyramid"] = settings["pyramid"]
    res["legs"] = [leg("configs[1] chair+table 640x480", "chair_table", a.frames, synth.REF_INTRINSICS, 0.005, settings)]
    if a.hd_frames > 0:
        res["legs"].append(leg("configs[3] geometry: large room 1280x720", "room", a.hd_frames, synth.HD_INTRINSICS, 0.002,
                               settings))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
