"""ctypes wrapper of tests/models/normals_icp_model.cpp, the CPU restatement of normal estimation and point-to-plane ICP
(DESIGN.md §4 "Normals and point-to-plane registration") that the CUDA kernels are compared with bit for bit.  Compiled
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
        d = tempfile.mkdtemp(prefix="otslam_normals_icp_model_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "normals_icp_model.so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-fopenmp", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-o", so,
                               os.path.join(ROOT, "tests", "models", "normals_icp_model.cpp")])
        lib = C.CDLL(so)
        vp, i64, d_, i = C.c_void_p, C.c_int64, C.c_double, C.c_int
        lib.model_neighbours.argtypes = [vp, i64, d_, i, vp, vp]
        lib.model_estimate_normals.argtypes = [vp, i64, vp, d_, i, vp]
        lib.model_icp_point_to_plane.argtypes = [vp, i64, vp, vp, i64, d_, vp, d_, d_, i, vp, vp, vp, vp, vp]
        _MODEL = lib
    return _MODEL


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pts(a):
    return np.ascontiguousarray(np.asarray(a, np.float64).reshape(-1, 3))


def neighbours(pts, radius, max_nn):
    """(idx [n, max_nn] with -1 beyond the count, count [n]): each point's neighbour list in (d2, index) order."""
    p = _pts(pts)
    idx = np.empty((len(p), max_nn), np.int32)
    cnt = np.empty(len(p), np.int32)
    model().model_neighbours(_p(p), len(p), float(radius), int(max_nn), _p(idx), _p(cnt))
    return idx, cnt


def estimate_normals(pts, radius=np.inf, max_nn=30, prior=None):
    p = _pts(pts)
    pr = None if prior is None else _pts(prior)
    out = np.empty_like(p)
    if model().model_estimate_normals(_p(p), len(p), _p(pr), float(radius), int(max_nn), _p(out)) != 0:
        raise ValueError("bad arguments")
    return out


def icp_point_to_plane(source, target, target_normals, max_distance, init=None, relative_fitness=1e-6, relative_rmse=1e-6,
                       max_iteration=30):
    """dict: transformation [4,4], fitness, inlier_rmse, iterations, corr [n_source] (target index or -1)."""
    s, t, tn = _pts(source), _pts(target), _pts(target_normals)
    T0 = np.ascontiguousarray(np.eye(4) if init is None else init, np.float64).reshape(16)
    T = np.empty(16)
    fit, rmse, it = C.c_double(), C.c_double(), C.c_int32()
    corr = np.empty(len(s), np.int32)
    r = model().model_icp_point_to_plane(_p(s), len(s), _p(t), _p(tn), len(t), float(max_distance), _p(T0), float(relative_fitness),
                                         float(relative_rmse), int(max_iteration), _p(T), C.byref(fit), C.byref(rmse), C.byref(it),
                                         _p(corr))
    if r != 0:
        raise ValueError("bad arguments")
    return {"transformation": T.reshape(4, 4), "fitness": fit.value, "inlier_rmse": rmse.value, "iterations": it.value,
            "corr": corr}
