"""Volume checkpoint timings on one GPU: save and load of the volume bench.py integrates, against re-integrating the same
frames from HBM.  Prints one JSON line.

Legs: configs[1] (1000 frames of the chair+table sequence, 640x480, 5 mm) and the HD geometry of configs[3] (2000 frames of
the large room, 1280x720, 2 mm; its load also grows the block hash several times).  Per leg: device time of the save's
gather + checksum kernels and of the load's filter + verify + insert kernels (CUDA events), both also as GB/s counting
2 x 65536 bytes per block against bench.py's measured 6454 GB/s HBM roofline; device time of the host<->device copies; time
in file reads / writes / fsync; wall time of each call; and the wall time of integrating the same frames into a fresh volume
from HBM.  One save + load round warms up, the second is reported.  Files go to a temporary directory (--dir) and are
deleted; the loaded volume's stats() must equal the original's.  The load reads a file that was just written, so its reads
come from the page cache.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6454.3          # bench.py's measured HBM roofline on a B200 (profiles/bench_r02_n1.json "peak")
BLOCK = 65536


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


def rates(prof, n_blocks):
    gbs = 2 * BLOCK * n_blocks / (prof["kernel_ms"] * 1e-3) / 1e9 if prof["kernel_ms"] > 0 else None
    copy_gbs = BLOCK * n_blocks / (prof["copy_ms"] * 1e-3) / 1e9 if prof["copy_ms"] > 0 else None
    file_gbs = BLOCK * n_blocks / (prof["file_ms"] * 1e-3) / 1e9 if prof["file_ms"] > 0 else None
    return dict(prof, kernel_gbs=gbs, kernel_of_hbm_roofline=gbs / HBM_GBS if gbs else None, copy_gbs=copy_gbs, file_gbs=file_gbs)


def leg(name, scene, frames, intr, voxel, directory):
    import torch
    from otslam_b200 import synth
    from otslam_b200.volume import TSDFVolume, checkpoint_profile
    seq = synth.make_sequence(scene, frames, intr=intr, device="cuda:0")
    d, c, ext, k = seq.depth, seq.rgb, seq.extrinsic, seq.fxfycxcy
    torch.cuda.synchronize()
    src = TSDFVolume(voxel, 4 * voxel)
    src.integrate_batch(d, c, k, ext)                               # also the warm-up of the integration
    n = src.num_blocks()
    out = {"workload": name, "frames": frames, "voxel_mm": voxel * 1000, "n_blocks": n, "file_gb": None}
    need = 4096 * 3 + n * (BLOCK + 20)
    free = shutil.disk_usage(directory).free
    t0 = time.perf_counter()
    again = TSDFVolume(voxel, 4 * voxel)
    again.integrate_batch(d, c, k, ext)                             # returns when the device is done
    out["reintegrate_from_hbm_ms"] = (time.perf_counter() - t0) * 1e3
    again.close()
    if free < need * 1.1:
        out["not_measured"] = f"{need / 1e9:.1f} GB needed in {directory}, {free / 1e9:.1f} GB free"
        src.close()
        return out
    path = os.path.join(directory, f"{scene}_{frames}.otslam")
    want = src.stats()
    for rnd in range(2):
        src.save(path)
        save = checkpoint_profile()
        dst = TSDFVolume(voxel, 4 * voxel)
        loaded = dst.load(path)
        load = checkpoint_profile()
        assert loaded == n and dst.stats() == want, "loaded volume differs from the saved one"
        out["file_gb"] = os.path.getsize(path) / 1e9
        os.remove(path)
        dst.close()
    out["save"], out["load"] = rates(save, n), rates(load, n)
    out["stats_equal"] = True
    src.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dir", default=None, help="directory for the temporary checkpoint files (default: the system's temp dir)")
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--hd-frames", type=int, default=2000, help="0 = skip the HD leg")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("checkpoint_bench needs a CUDA device")
    from otslam_b200 import synth
    tmp = tempfile.mkdtemp(prefix="otslam_ckpt_", dir=a.dir)
    try:
        res = gpu_details()
        res["legs"] = [leg("configs[1] chair+table 640x480", "chair_table", a.frames, synth.REF_INTRINSICS, 0.005, tmp)]
        if a.hd_frames > 0:
            res["legs"].append(leg("configs[3] geometry: large room 1280x720", "room", a.hd_frames, synth.HD_INTRINSICS, 0.002, tmp))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
