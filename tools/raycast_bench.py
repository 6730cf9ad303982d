"""Ray-casting timings and model residuals on one GPU.  Prints one JSON line.

Legs: configs[1] (1000 frames of the chair+table sequence, 640x480, 5 mm) and the HD geometry of configs[3] (2000 frames of
the large room, 1280x720, 2 mm).  Per leg the volume is integrated from HBM (integration ms per frame, wall time), then
every capture pose is rendered in batches of 32 views, twice: into NumPy arrays (host outputs, staged through the
library's bounded device buffers) and into CUDA tensors (device outputs, written in place).  Reported per mode: rays/s and
ms per view from the device time of the render kernels (otslam_last_op_device_ms, summed over the calls) and from wall
time.  One batch of each mode warms up first.  The residual compares each rendered depth map with the captured frame it
was integrated from: median and 95th percentile of |rendered - captured| over pixels valid in both (per frame; the mean
and the maximum over frames are reported), and the hit ratio (pixels with a hit over pixels with a captured depth).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BATCH = 32


def gpu_details():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # noqa: BLE001
        out["power_limit_w"] = f"unavailable: {e}"
    return out


def render_all(vol, k, ext, W, H, device_outputs, residual=None):
    """every pose in batches; returns (device ms, wall ms); residual(first, depth batch) is called per batch"""
    import torch
    from otslam_b200 import _lib
    call = vol.ray_cast_tensors if device_outputs else vol.ray_cast
    call(k, ext[:BATCH], W, H)                                      # warm-up
    torch.cuda.synchronize()
    dev_ms, wall = 0.0, 0.0
    for first in range(0, len(ext), BATCH):
        t0 = time.perf_counter()
        out = call(k, ext[first:first + BATCH], W, H)               # returns with the outputs complete
        wall += time.perf_counter() - t0
        dev_ms += _lib.last_op_device_ms()
        if residual is not None:
            residual(first, out["depth"])
        del out
    return dev_ms, wall * 1e3


def leg(name, scene, frames, intr, voxel):
    import torch
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume
    seq = synth.make_sequence(scene, frames, intr=intr, device="cuda:0")
    d, c, ext, k = seq.depth, seq.rgb, seq.extrinsic, seq.fxfycxcy
    W, H = intr[0], intr[1]
    torch.cuda.synchronize()
    warm = TSDFVolume(voxel, 4 * voxel)
    warm.integrate_batch(d[:64], c[:64], k, ext[:64])
    warm.close()
    vol = TSDFVolume(voxel, 4 * voxel)
    vol.profile(True)
    t0 = time.perf_counter()
    vol.integrate_batch(d, c, k, ext)                               # returns when the device is done
    integ_wall = (time.perf_counter() - t0) * 1e3
    prof = vol.profile(False)
    integ_dev = sum(ms for ms, _ in prof.values())
    out = {"workload": name, "frames": frames, "width": W, "height": H, "voxel_mm": voxel * 1000, "n_blocks": vol.num_blocks(),
           "integrate_ms_per_frame_device": integ_dev / frames, "integrate_ms_per_frame_wall": integ_wall / frames}
    med, p95, hit = [], [], []

    def residual(first, depth):
        got = depth if torch.is_tensor(depth) else torch.from_numpy(depth).cuda()
        cap = (d[first:first + len(got)].view(torch.int16).to(torch.int32) & 0xFFFF).to(torch.float32) / 1000.0
        for g, cp in zip(got, cap):
            both = (g > 0) & (cp > 0)
            r = (g[both] - cp[both]).abs()
            if r.numel():
                q = torch.quantile(r, torch.tensor([0.5, 0.95], device=r.device))
                med.append(float(q[0])); p95.append(float(q[1]))
            hit.append(float(both.sum()) / max(1.0, float((cp > 0).sum())))

    rays = frames * W * H
    for mode, dev in (("host_outputs", False), ("device_outputs", True)):
        dev_ms, wall_ms = render_all(vol, k, ext, W, H, dev, residual if dev else None)
        out[mode] = {"rays_per_s_device": rays / (dev_ms * 1e-3), "ms_per_view_device": dev_ms / frames,
                     "rays_per_s_wall": rays / (wall_ms * 1e-3), "ms_per_view_wall": wall_ms / frames}
    out["residual_m"] = {"median_mean_over_frames": sum(med) / len(med), "median_max_over_frames": max(med),
                         "p95_mean_over_frames": sum(p95) / len(p95), "p95_max_over_frames": max(p95),
                         "hit_ratio_mean": sum(hit) / len(hit), "hit_ratio_min": min(hit)}
    vol.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--hd-frames", type=int, default=2000, help="0 = skip the HD leg")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("raycast_bench needs a CUDA device")
    from otslam_b200 import synth
    res = gpu_details()
    res["batch_views"] = BATCH
    res["legs"] = [leg("configs[1] chair+table 640x480", "chair_table", a.frames, synth.REF_INTRINSICS, 0.005)]
    if a.hd_frames > 0:
        res["legs"].append(leg("configs[3] geometry: large room 1280x720", "room", a.hd_frames, synth.HD_INTRINSICS, 0.002))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
