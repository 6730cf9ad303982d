"""Normal estimation and point-to-plane ICP on the GPU (DESIGN.md §4 "Normals and point-to-plane registration").

  normals : otslam_cloud_estimate_normals on mesh samples (100 k and 1 M) of the configs[1] volume (chair_table scene,
            every 10th of 300 frames, 1 cm voxels) and on its extract_point_cloud points; k-NN 30 and hybrid (2 cm, 30):
            device ms (CUDA events, otslam_last_op_device_ms, best of --reps) and points/s.  The CPU model's time on this
            host's cores, for scale.
  icp     : the evaluation-shaped problem of test_icp_point_to_point_recovers_a_known_motion: 30 k mesh samples, the
            source = every second one moved by a 0.03 rad / 1 cm motion, threshold 0.05, max_iteration 2000.  Point-to-plane
            (one call, otslam_cloud_icp_point_to_plane) against point-to-point (the compat loop): iterations, wall ms, device
            ms (point-to-plane: the call's events; point-to-point: the sum over its operator calls) and the final transform
            error.

Prints the GPU's name and power limit, then one JSON line.  Writes nothing.
    python tools/registration_bench.py [--reps 5]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("registration_bench needs a CUDA device")
    from otslam_b200 import _lib, synth
    from otslam_b200.volume import TSDFVolume
    import otslam_b200.o3d_compat as o3d
    import normals_icp_ref as ref
    from oracle import oracle

    print("gpu:", gpu_info(), flush=True)
    seq = synth.make_sequence("chair_table", 300, subsample=(0, 10))
    d, c = seq.numpy()
    v = TSDFVolume(0.01, 0.04)
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    verts, cols, nrm, faces, _ = v.extract_triangle_mesh()
    ext, _, _, _ = v.extract_point_cloud(normals=True)
    v.close()
    clouds = {}
    for n in (100_000, 1_000_000):
        clouds[f"samples_{n // 1000}k"] = oracle.sample_uniform(verts, cols, nrm, faces, n, seed=3)[0]
    clouds[f"extracted_{len(ext) // 1000}k"] = ext
    out = {"gpu": gpu_info(), "normals": [], "icp": {}}
    for name, p in clouds.items():
        p = np.ascontiguousarray(p)
        res = np.empty_like(p)
        for mode, radius in (("knn30", float("inf")), ("hybrid_2cm_30", 0.02)):
            ms = []
            for _ in range(a.reps + 1):                        # the first call warms the module and the scratch cache
                _lib.check(_lib.lib.otslam_cloud_estimate_normals(_lib.ptr(p), len(p), None, radius, 30, _lib.ptr(res), 0))
                ms.append(_lib.last_op_device_ms())
            t = time.perf_counter()
            want = ref.estimate_normals(p, radius, 30)
            cpu_ms = (time.perf_counter() - t) * 1e3
            best = min(ms[1:])
            row = {"cloud": name, "points": len(p), "search": mode, "device_ms": round(best, 3),
                   "points_per_s": round(len(p) / best * 1e3), "model_cpu_ms": round(cpu_ms, 1),
                   "equal_to_model": bool((want.view(np.uint64) == res.view(np.uint64)).all())}
            out["normals"].append(row)
            print(row, flush=True)

    sp = oracle.sample_uniform(verts, cols, nrm, faces, 30000, seed=11)[0]
    aa = 0.03
    T_true = np.eye(4)
    T_true[:3, :3] = [[np.cos(aa), -np.sin(aa), 0], [np.sin(aa), np.cos(aa), 0], [0, 0, 1]]
    T_true[:3, 3] = [0.01, -0.008, 0.005]
    reg = o3d.pipelines.registration
    tgt = o3d.geometry.PointCloud(sp)
    tgt.estimate_normals(o3d.geometry.KDTreeSearchParamKNN(30))
    src = o3d.geometry.PointCloud(sp[::2].copy())
    src.transform(np.linalg.inv(T_true))
    crit = reg.ICPConvergenceCriteria(max_iteration=2000)
    for name, est in (("point_to_plane", reg.TransformationEstimationPointToPlane()),
                      ("point_to_point", reg.TransformationEstimationPointToPoint())):
        best = None
        for _ in range(2):
            torch.cuda.synchronize()
            dev = [0.0, 0]
            if name == "point_to_point":              # device time = the sum over the loop's operator calls
                orig = _lib.lib.otslam_cloud_nn_within, _lib.lib.otslam_cloud_transform

                def wrap(f, count):
                    def g(*args):
                        r = f(*args)
                        dev[0] += max(0.0, _lib.last_op_device_ms())
                        dev[1] += count
                        return r
                    return g
                _lib.lib.otslam_cloud_nn_within, _lib.lib.otslam_cloud_transform = wrap(orig[0], 1), wrap(orig[1], 0)
            t = time.perf_counter()
            r = reg.registration_icp(src, tgt, 0.05, np.eye(4), est, crit)
            wall = (time.perf_counter() - t) * 1e3
            if name == "point_to_point":
                _lib.lib.otslam_cloud_nn_within, _lib.lib.otslam_cloud_transform = orig
            else:
                dev[0] = _lib.last_op_device_ms()
            best = (wall, dev[0], r, dev[1] - 1) if best is None or wall < best[0] else best
        wall, dms, r, n_eval = best
        iters = None
        if name == "point_to_plane":
            it = C.c_int32()
            T = np.empty(16)
            pts, tp, tn = (np.ascontiguousarray(np.asarray(x), np.float64) for x in (src.points, tgt.points, tgt.normals))
            _lib.check(_lib.lib.otslam_cloud_icp_point_to_plane(_lib.ptr(pts), len(pts), _lib.ptr(tp), _lib.ptr(tn), len(tp), 0.05,
                                                                _lib.ptr(np.eye(4).reshape(16)), 1e-6, 1e-6, 2000, _lib.ptr(T), None,
                                                                None, C.byref(it), None, 0))
            iters = it.value
        else:
            iters = n_eval                           # one correspondence search per evaluation, the first before any update
        out["icp"][name] = {"iterations": iters, "wall_ms": round(wall, 2), "device_ms": round(dms, 3), "fitness": r.fitness,
                            "transform_err": float(np.abs(r.transformation - T_true).max())}
        print(name, out["icp"][name], flush=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
