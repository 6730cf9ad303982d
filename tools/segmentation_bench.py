"""Plane segmentation and DBSCAN clustering on the GPU (DESIGN.md §4 "Plane segmentation and DBSCAN clustering").

On mesh samples (100 k and 1 M) of the configs[1] volume (chair_table scene, every 10th of 300 frames, 1 cm voxels):
  plane_p1      : otslam_cloud_segment_plane(0.01, 3, 1000, probability = 1): all 1000 hypotheses are evaluated
  plane_default : the same with the default probability 0.99999999 (the break rule stops the search early)
  dbscan        : otslam_cloud_cluster_dbscan(eps 0.02, min_points 10) on the points off the plane
  dense         : DBSCAN of --dense-n points inside a ball of diameter < eps (every pair is a neighbour pair: the union pass
                  is quadratic)
Device ms = otslam_last_op_device_ms (CUDA events around the grid build / waves and kernels), best of --reps after one
warm-up call.  The CPU model's time on this host's cores is given for scale, with whether GPU and model agree bit for bit.
Prints the GPU's name and power limit, then one JSON line.  Writes nothing.
    python tools/segmentation_bench.py [--reps 5] [--dense-n 20000]
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
    ap.add_argument("--dense-n", type=int, default=20000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("segmentation_bench needs a CUDA device")
    from otslam_b200 import _lib, synth
    from otslam_b200.volume import TSDFVolume
    import segment_ref as ref
    from oracle import oracle

    print("gpu:", gpu_info(), flush=True)
    seq = synth.make_sequence("chair_table", 300, subsample=(0, 10))
    d, c = seq.numpy()
    v = TSDFVolume(0.01, 0.04)
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    verts, cols, nrm, faces, _ = v.extract_triangle_mesh()
    v.close()

    def timed(fn):
        ms = []
        for _ in range(a.reps + 1):                  # the first call warms the module and the scratch cache
            out = fn()
            ms.append(_lib.last_op_device_ms())
        return min(ms[1:]), out

    def plane(p, prob):
        plane_ = np.empty(4)
        inl = np.empty(len(p), np.int64)
        m, ev = C.c_int64(), C.c_int32()
        _lib.check(_lib.lib.otslam_cloud_segment_plane(_lib.ptr(p), len(p), 0.01, 3, 1000, prob, C.c_uint64(7), _lib.ptr(plane_),
                                                       _lib.ptr(inl), C.byref(m), C.byref(ev), 0))
        return plane_, inl[:m.value].copy(), ev.value

    def dbscan(p, eps, mp):
        lab = np.empty(len(p), np.int32)
        nc = C.c_int32()
        _lib.check(_lib.lib.otslam_cloud_cluster_dbscan(_lib.ptr(p), len(p), eps, mp, _lib.ptr(lab), C.byref(nc), 0))
        return lab, nc.value

    def model_time(fn):
        t = time.perf_counter()
        r = fn()
        return (time.perf_counter() - t) * 1e3, r

    rows = []
    for n in (100_000, 1_000_000):
        p = np.ascontiguousarray(oracle.sample_uniform(verts, cols, nrm, faces, n, seed=3)[0])
        for case, prob in (("plane_p1", 1.0), ("plane_default", 0.99999999)):
            ms, (pl, inl, ev) = timed(lambda: plane(p, prob))
            cpu_ms, want = model_time(lambda: ref.segment_plane(p, 0.01, 3, 1000, prob, seed=7))
            same = bool((pl.view(np.uint64) == want["plane"].view(np.uint64)).all() and ev == want["n_evaluated"]
                        and np.array_equal(inl, want["inliers"]))
            rows.append({"case": case, "points": n, "hypotheses": ev, "inliers": len(inl), "device_ms": round(ms, 3),
                         "point_tests_per_s": round(ev * n / ms * 1e3), "model_cpu_ms": round(cpu_ms, 1), "equal_to_model": same})
            print(rows[-1], flush=True)
        keep = np.ones(n, bool)
        keep[inl] = False
        rest = np.ascontiguousarray(p[keep])
        ms, (lab, nc) = timed(lambda: dbscan(rest, 0.02, 10))
        cpu_ms, (wl, wn) = model_time(lambda: ref.cluster_dbscan(rest, 0.02, 10))
        rows.append({"case": "dbscan", "points": len(rest), "clusters": nc, "device_ms": round(ms, 3), "model_cpu_ms": round(cpu_ms, 1),
                     "equal_to_model": bool(nc == wn and (lab == wl).all())})
        print(rows[-1], flush=True)
    rng = np.random.default_rng(1)
    ball = rng.normal(size=(a.dense_n, 3))
    ball *= (0.0099 * rng.random(a.dense_n) ** (1 / 3) / np.linalg.norm(ball, axis=1))[:, None]   # radius < eps / 2
    ball = np.ascontiguousarray(ball)
    ms, (lab, nc) = timed(lambda: dbscan(ball, 0.02, 10))
    cpu_ms, (wl, wn) = model_time(lambda: ref.cluster_dbscan(ball, 0.02, 10))
    rows.append({"case": "dense", "points": a.dense_n, "clusters": nc, "device_ms": round(ms, 3),
                 "neighbour_pairs_per_s": round(a.dense_n ** 2 / ms * 1e3), "model_cpu_ms": round(cpu_ms, 1),
                 "equal_to_model": bool(nc == wn and (lab == wl).all())})
    print(rows[-1], flush=True)
    print(json.dumps({"gpu": gpu_info(), "rows": rows}))


if __name__ == "__main__":
    main()
