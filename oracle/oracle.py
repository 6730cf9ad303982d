"""ctypes wrapper around oracle/liboracle.so -- TEST INFRASTRUCTURE, not product code.

The oracle restates the Open3D legacy CPU pipeline that the reference scripts call
(/root/reference/3d_model/reconstruct_rgbd.py:79-118 and friends); see oracle.cpp's header for
the "parity unpinned" statement.  Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may
import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    src = os.path.join(_HERE, "oracle.cpp")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(so):
            build()
        L = C.CDLL(so)
        L.oracle_last_error.restype = C.c_char_p
        L.oracle_volume_create.restype = C.c_void_p
        L.oracle_volume_create.argtypes = [C.c_double, C.c_double]
        L.oracle_volume_extract_mesh.restype = C.c_void_p
        for name in ("oracle_volume_halo_export", "oracle_volume_num_blocks", "oracle_volume_extract_points", "oracle_zfilter",
                     "oracle_backproject_rgbd", "oracle_voxel_down_sample", "oracle_remove_statistical_outlier",
                     "oracle_grid_to_points"):
            getattr(L, name).restype = C.c_int64
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _err():
    return RuntimeError(lib().oracle_last_error().decode())


def num_threads():
    return int(lib().oracle_num_threads())


def set_num_threads(n):
    """Use n OpenMP threads from now on (ignores an inherited OMP_NUM_THREADS); returns the count in effect."""
    return int(lib().oracle_set_num_threads(int(n)))


def inverse4(m):
    m = np.ascontiguousarray(m, np.float64)
    out = np.empty((4, 4), np.float64)
    if lib().oracle_inverse4(_p(m), _p(out)) != 0:
        raise _err()
    return out


def depth_convert(depth_u16, depth_scale=1000.0, depth_trunc=3.0):
    d = np.ascontiguousarray(depth_u16, np.uint16)
    out = np.empty(d.shape, np.float32)
    lib().oracle_depth_convert(_p(d), C.c_int64(d.size), C.c_double(depth_scale), C.c_double(depth_trunc), _p(out))
    return out


class Volume:
    """Oracle ScalableTSDFVolume (SURVEY A.3/A.4)."""

    def __init__(self, voxel_length, sdf_trunc, slab=None):
        self.h = C.c_void_p(lib().oracle_volume_create(voxel_length, sdf_trunc))
        if not self.h:
            raise _err()
        self.voxel_length, self.sdf_trunc = voxel_length, sdf_trunc
        if slab is not None:
            axis, thickness, n_ranks, rank = slab[:4]
            halo = slab[4] if len(slab) > 4 else 1
            if lib().oracle_volume_set_slab(self.h, axis, thickness, n_ranks, rank, halo) != 0:
                raise _err()

    def __del__(self):
        if getattr(self, "h", None) and _LIB is not None:
            _LIB.oracle_volume_destroy(self.h)
            self.h = None

    def reset(self):
        lib().oracle_volume_reset(self.h)

    def integrate(self, depth_f32, rgb, intr, extrinsic):
        """intr = (fx, fy, cx, cy); returns (n_touched_blocks, n_updated_voxels)."""
        d = np.ascontiguousarray(depth_f32, np.float32)
        c = np.ascontiguousarray(rgb, np.uint8)
        H, W = d.shape
        assert c.shape == (H, W, 3)
        e = np.ascontiguousarray(extrinsic, np.float64)
        nt, nu = C.c_int64(0), C.c_int64(0)
        r = lib().oracle_volume_integrate(self.h, _p(d), _p(c), W, H, C.c_double(intr[0]), C.c_double(intr[1]),
                                          C.c_double(intr[2]), C.c_double(intr[3]), _p(e), C.byref(nt), C.byref(nu))
        if r != 0:
            raise _err()
        return nt.value, nu.value

    def num_blocks(self):
        return int(lib().oracle_volume_num_blocks(self.h))

    def export_blocks(self, color=True):
        n = self.num_blocks()
        keys = np.empty((n, 3), np.int32)
        tsdf = np.empty((n, 4096), np.float32)
        weight = np.empty((n, 4096), np.float32)
        col = np.empty((n, 4096, 3), np.float64) if color else None
        lib().oracle_volume_export_blocks(self.h, _p(keys), _p(tsdf), _p(weight), _p(col))
        return keys, tsdf, weight, col

    def halo_export(self):
        """(keys [n,4] i32 = block key + piece kind, dest rank [n] i32, pieces): boundary pieces for the halo exchange."""
        n = int(lib().oracle_volume_halo_export(self.h, None, None, None, None, None))
        keys = np.empty((n, 4), np.int32); dest = np.empty(n, np.int32)
        tsdf = np.empty((n, 256), np.float32); w = np.empty((n, 256), np.float32); col = np.empty((n, 256, 3), np.float64)
        lib().oracle_volume_halo_export(self.h, _p(keys), _p(dest), _p(tsdf), _p(w), _p(col))
        # one opaque byte record per block so the exchange code is layout agnostic
        planes = np.concatenate([tsdf.view(np.uint8).reshape(n, -1), w.view(np.uint8).reshape(n, -1),
                                 col.view(np.uint8).reshape(n, -1)], axis=1) if n else np.zeros((0, 256 * 32), np.uint8)
        return keys, dest, np.ascontiguousarray(planes)

    def halo_import(self, keys, planes):
        n = len(keys)
        if n == 0:
            return
        planes = np.ascontiguousarray(planes, np.uint8).reshape(n, 256 * 32)
        tsdf = np.ascontiguousarray(planes[:, :1024]).view(np.float32)
        w = np.ascontiguousarray(planes[:, 1024:2048]).view(np.float32)
        col = np.ascontiguousarray(planes[:, 2048:]).view(np.float64)
        k = np.ascontiguousarray(keys, np.int32)
        lib().oracle_volume_halo_import(self.h, C.c_int64(n), _p(k), _p(tsdf), _p(w), _p(col))

    def import_blocks(self, keys, tsdf, weight, color):
        """Add whole blocks in export_blocks' form (keys [n,3] i32, tsdf / weight [n,4096] f32, colour [n,4096,3] f64 on the
        0..255 scale); a block already present is overwritten."""
        k = np.ascontiguousarray(keys, np.int32).reshape(-1, 3)
        n = len(k)
        t = np.ascontiguousarray(tsdf, np.float32).reshape(n, 4096)
        w = np.ascontiguousarray(weight, np.float32).reshape(n, 4096)
        c = np.ascontiguousarray(color, np.float64).reshape(n, 4096, 3)
        lib().oracle_volume_import_blocks(self.h, C.c_int64(n), _p(k), _p(t), _p(w), _p(c))

    def extract_triangle_mesh(self):
        nv, nf = C.c_int64(0), C.c_int64(0)
        m = C.c_void_p(lib().oracle_volume_extract_mesh(self.h, C.byref(nv), C.byref(nf)))
        verts = np.empty((nv.value, 3), np.float64)
        cols = np.empty((nv.value, 3), np.float64)
        faces = np.empty((nf.value, 3), np.int32)
        ek = np.empty((nv.value, 4), np.int32)
        lib().oracle_mesh_copy(m, _p(verts), _p(cols), _p(faces), _p(ek))
        lib().oracle_mesh_free(m)
        return verts, cols, faces, ek

    def extract_point_cloud(self):
        n = int(lib().oracle_volume_extract_points(self.h, None, None, None))
        pts = np.empty((n, 3), np.float64)
        cols = np.empty((n, 3), np.float64)
        ek = np.empty((n, 4), np.int32)
        lib().oracle_volume_extract_points(self.h, _p(pts), _p(cols), _p(ek))
        return pts, cols, ek

    def point_normals(self, pts):
        """GetNormalAt for each point (the normals extract_point_cloud attaches): normalised central TSDF differences."""
        p = np.ascontiguousarray(pts, np.float64)
        out = np.empty_like(p)
        lib().oracle_volume_point_normals(self.h, _p(p), C.c_int64(len(p)), _p(out))
        return out


def vertex_normals(verts, faces):
    v = np.ascontiguousarray(verts, np.float64)
    f = np.ascontiguousarray(faces, np.int32)
    out = np.empty_like(v)
    lib().oracle_vertex_normals(_p(v), C.c_int64(len(v)), _p(f), C.c_int64(len(f)), _p(out))
    return out


def sample_uniform(verts, colors, normals, faces, n, seed=0):
    v = np.ascontiguousarray(verts, np.float64)
    c = None if colors is None else np.ascontiguousarray(colors, np.float64)
    nr = None if normals is None else np.ascontiguousarray(normals, np.float64)
    f = np.ascontiguousarray(faces, np.int32)
    op = np.empty((n, 3), np.float64)
    oc = None if c is None else np.empty((n, 3), np.float64)
    on = None if nr is None else np.empty((n, 3), np.float64)
    tri = np.empty(n, np.int32)
    r = lib().oracle_sample_uniform(_p(v), _p(c), _p(nr), C.c_int64(len(v)), _p(f), C.c_int64(len(f)), C.c_int64(n),
                                    C.c_uint64(seed), _p(op), _p(oc), _p(on), _p(tri))
    if r != 0:
        raise _err()
    return op, oc, on, tri


def zfilter(pts, cols, zmin):
    p = np.ascontiguousarray(pts, np.float64)
    c = None if cols is None else np.ascontiguousarray(cols, np.float64)
    op = np.empty_like(p)
    oc = None if c is None else np.empty_like(c)
    m = int(lib().oracle_zfilter(_p(p), _p(c), C.c_int64(len(p)), C.c_double(zmin), _p(op), _p(oc)))
    return op[:m], None if oc is None else oc[:m]


def backproject_rgbd(depth_f32, rgb, intr, extrinsic=None):
    d = np.ascontiguousarray(depth_f32, np.float32)
    c = None if rgb is None else np.ascontiguousarray(rgb, np.uint8)
    H, W = d.shape
    e = np.eye(4) if extrinsic is None else np.ascontiguousarray(extrinsic, np.float64)
    pts = np.empty((H * W, 3), np.float64)
    cols = np.empty((H * W, 3), np.float64)
    n = int(lib().oracle_backproject_rgbd(_p(d), _p(c), W, H, C.c_double(intr[0]), C.c_double(intr[1]),
                                          C.c_double(intr[2]), C.c_double(intr[3]), _p(e), _p(pts), _p(cols)))
    if n < 0:
        raise _err()
    return pts[:n].copy(), cols[:n].copy()


def voxel_down_sample(pts, cols, voxel):
    p = np.ascontiguousarray(pts, np.float64)
    c = None if cols is None else np.ascontiguousarray(cols, np.float64)
    n = len(p)
    op = np.empty((n, 3), np.float64)
    oc = np.empty((n, 3), np.float64)
    ok = np.empty((n, 3), np.int32)
    on = np.empty(n, np.int32)
    m = int(lib().oracle_voxel_down_sample(_p(p), _p(c), C.c_int64(n), C.c_double(voxel), _p(op), _p(oc), _p(ok), _p(on)))
    if m < 0:
        raise _err()
    return op[:m].copy(), (None if c is None else oc[:m].copy()), ok[:m].copy(), on[:m].copy()


def remove_statistical_outlier(pts, nb_neighbors, std_ratio):
    p = np.ascontiguousarray(pts, np.float64)
    n = len(p)
    idx = np.empty(n, np.int64)
    dbar = np.empty(n, np.float64)
    m = int(lib().oracle_remove_statistical_outlier(_p(p), C.c_int64(n), int(nb_neighbors), C.c_double(std_ratio),
                                                    _p(idx), _p(dbar)))
    if m < 0:
        raise _err()
    return idx[:m].copy(), dbar


def grid_to_points(img, res, ox, oy, thresh=100):
    g = np.ascontiguousarray(img, np.uint8)
    h, w = g.shape
    n = int(lib().oracle_grid_to_points(_p(g), w, h, C.c_double(res), C.c_double(ox), C.c_double(oy), int(thresh), None))
    out = np.empty((n, 3), np.float64)
    lib().oracle_grid_to_points(_p(g), w, h, C.c_double(res), C.c_double(ox), C.c_double(oy), int(thresh), _p(out))
    return out


def pack_ply_cloud(pts, cols):
    p = np.ascontiguousarray(pts, np.float64)
    c = None if cols is None else np.ascontiguousarray(cols, np.float64)
    out = np.empty((len(p), 27), np.uint8)
    lib().oracle_pack_ply_cloud(_p(p), _p(c), C.c_int64(len(p)), _p(out))
    return out


def transform(pts, nrm, T):
    p = np.ascontiguousarray(pts, np.float64)
    q = None if nrm is None else np.ascontiguousarray(nrm, np.float64)
    op, on = np.empty_like(p), None if q is None else np.empty_like(q)
    lib().oracle_transform(_p(p), _p(q), C.c_int64(len(p)), _p(np.ascontiguousarray(T, np.float64).reshape(16)), _p(op), _p(on))
    return op, on


def center(pts):
    p = np.ascontiguousarray(pts, np.float64)
    c = np.zeros(3)
    lib().oracle_center(_p(p), C.c_int64(len(p)), _p(c))
    return c


def rotate(pts, nrm, R, c):
    p = np.ascontiguousarray(pts, np.float64)
    q = None if nrm is None else np.ascontiguousarray(nrm, np.float64)
    op, on = np.empty_like(p), None if q is None else np.empty_like(q)
    lib().oracle_rotate(_p(p), _p(q), C.c_int64(len(p)), _p(np.ascontiguousarray(R, np.float64).reshape(9)),
                        _p(np.ascontiguousarray(c, np.float64)), _p(op), _p(on))
    return op, on


def smart_paste(base_img, overlay_img, x, y, w, h):
    """/root/reference/fusion/2d_selective_merge.py:58-69, restated (NumPy, in place on a copy)."""
    base_img = base_img.copy()
    h_img, w_img = base_img.shape
    if x < 0 or y < 0 or x + w > w_img or y + h > h_img:
        return base_img
    roi_base = base_img[y:y + h, x:x + w]
    roi_new = overlay_img[y:y + h, x:x + w]
    unknown_pixel, threshold = 205, 5
    has_data_mask = (roi_new < (unknown_pixel - threshold)) | (roi_new > (unknown_pixel + threshold))
    roi_base[has_data_mask] = roi_new[has_data_mask]
    return base_img
