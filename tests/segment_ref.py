"""ctypes wrapper of tests/models/segment_model.cpp, the CPU restatement of DBSCAN clustering and RANSAC plane segmentation
(DESIGN.md §4 "Plane segmentation and DBSCAN clustering") that the CUDA kernels are compared with bit for bit.  Compiled
like the oracle (g++ -O2 -fopenmp -ffp-contract=off) into a temporary directory on first use."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_MODEL = None


def model():
    global _MODEL
    if _MODEL is None:
        d = tempfile.mkdtemp(prefix="otslam_segment_model_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "segment_model.so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-fopenmp", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-o", so,
                               os.path.join(ROOT, "tests", "models", "segment_model.cpp")])
        lib = C.CDLL(so)
        vp, i64, d_, i, u64 = C.c_void_p, C.c_int64, C.c_double, C.c_int, C.c_uint64
        lib.model_dbscan.argtypes = [vp, i64, d_, i64, vp, vp]
        lib.model_hypothesis_planes.argtypes = [vp, i64, i, u64, i64, i64, vp]
        lib.model_ransac_bound.argtypes = [d_, i, d_, i]
        lib.model_ransac_bound.restype = i64
        lib.model_evaluate.argtypes = [vp, i64, vp, d_, vp, vp]
        lib.model_evaluate.restype = None
        lib.model_segment_plane.argtypes = [vp, i64, d_, i, i, d_, u64, vp, vp, vp, vp]
        _MODEL = lib
    return _MODEL


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pts(a):
    return np.ascontiguousarray(np.asarray(a, np.float64).reshape(-1, 3))


def cluster_dbscan(pts, eps, min_points):
    """(labels int32 [n], number of clusters): Open3D's ClusterDBSCAN loop."""
    p = _pts(pts)
    lab = np.empty(len(p), np.int32)
    nc = C.c_int32()
    if model().model_dbscan(_p(p), len(p), float(eps), int(min_points), _p(lab), C.byref(nc)) != 0:
        raise ValueError("bad arguments")
    return lab, nc.value


def hypothesis_planes(pts, ransac_n, seed, h0, count):
    """[count, 4] planes of hypotheses h0 .. h0 + count - 1 (zeros: invalid)."""
    p = _pts(pts)
    out = np.empty((count, 4), np.float64)
    if model().model_hypothesis_planes(_p(p), len(p), int(ransac_n), C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), int(h0), int(count),
                                       _p(out)) != 0:
        raise ValueError("bad arguments")
    return out


def ransac_bound(fitness, ransac_n, probability, num_iterations):
    return model().model_ransac_bound(float(fitness), int(ransac_n), float(probability), int(num_iterations))


def evaluate(pts, plane, threshold):
    """(inlier count, tree sum of the inlier distances) of one plane."""
    p = _pts(pts)
    pl = np.ascontiguousarray(plane, np.float64)
    c, s = C.c_int64(), C.c_double()
    model().model_evaluate(_p(p), len(p), _p(pl), float(threshold), C.byref(c), C.byref(s))
    return c.value, s.value


def segment_plane(pts, distance_threshold, ransac_n, num_iterations, probability=0.99999999, seed=0):
    """dict: plane [4], inliers int64 (ascending), n_evaluated."""
    p = _pts(pts)
    plane = np.empty(4, np.float64)
    inl = np.empty(len(p), np.int64)
    m, ev = C.c_int64(), C.c_int32()
    if model().model_segment_plane(_p(p), len(p), float(distance_threshold), int(ransac_n), int(num_iterations), float(probability),
                                   C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), _p(plane), _p(inl), C.byref(m), C.byref(ev)) != 0:
        raise ValueError("bad arguments")
    return {"plane": plane, "inliers": inl[:m.value].copy(), "n_evaluated": ev.value}
