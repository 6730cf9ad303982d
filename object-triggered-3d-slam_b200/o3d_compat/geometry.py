"""o3d.geometry: Image, RGBDImage, PointCloud, TriangleMesh backed by NumPy buffers; the heavy
methods call the CUDA library (no CPU fallback)."""
import ctypes as C

import numpy as np

from .. import _lib
from .utility import Vector3dVector, Vector3iVector

_GLOBAL_SEED = [None]          # o3d.utility.random.seed
_SEED_COUNTER = [0]


def _next_seed(seed):
    if seed is not None:
        return int(seed)
    if _GLOBAL_SEED[0] is not None:
        _SEED_COUNTER[0] += 1
        return _GLOBAL_SEED[0] + _SEED_COUNTER[0] - 1
    return int(np.random.SeedSequence().entropy & 0xFFFFFFFFFFFFFFFF)   # unseeded, like Open3D


def _as_n3(a, dtype=np.float64):
    a = np.ascontiguousarray(a, dtype)
    if a.size == 0:
        return np.zeros((0, 3), dtype)
    if a.ndim != 2 or a.shape[1] != 3:
        raise RuntimeError("expected an (N, 3) array")
    return a


class Image:
    """o3d.geometry.Image: np.asarray(img) is the H x W (x C) buffer."""

    def __init__(self, array=None):
        self._a = None if array is None else np.ascontiguousarray(array)

    def __array__(self, dtype=None, copy=None):
        a = np.zeros((0, 0), np.uint8) if self._a is None else self._a
        return a if dtype is None else a.astype(dtype)

    def is_empty(self):
        return self._a is None or self._a.size == 0

    @property
    def width(self):
        return 0 if self.is_empty() else self._a.shape[1]

    @property
    def height(self):
        return 0 if self.is_empty() else self._a.shape[0]

    def __repr__(self):
        if self.is_empty():
            return "Image of size 0x0, with 0 channels."
        ch = 1 if self._a.ndim == 2 else self._a.shape[2]
        return f"Image of size {self.width}x{self.height}, with {ch} channels."


class RGBDImage:
    """o3d.geometry.RGBDImage.  The depth conversion of create_from_color_and_depth
    (reconstruct_rgbd.py:99-104; u16 -> f32 metres, >= depth_trunc -> 0) is deferred: integrate()
    fuses it into the GPU frame-packing kernel, and `.depth` materialises it with the GPU
    depth_convert kernel on first access."""

    def __init__(self):
        self._color_arr = None
        self._depth_raw = None
        self._depth_is_raw_u16 = False
        self._depth_scale, self._depth_trunc = 1000.0, 3.0
        self._depth_f32 = None

    @staticmethod
    def create_from_color_and_depth(color, depth, depth_scale=1000.0, depth_trunc=3.0, convert_rgb_to_intensity=True):
        c = np.asarray(color)
        d = np.asarray(depth)
        if c.size == 0 or d.size == 0 or c.shape[:2] != d.shape[:2]:
            raise RuntimeError("[CreateFromColorAndDepth] Unsupported image format.")
        r = RGBDImage()
        if convert_rgb_to_intensity and c.ndim == 3:
            # Open3D's default; never used by the reference scripts (they pass False).  Host-side.
            w = np.array([0.2990, 0.5870, 0.1140], np.float32)
            r._color_arr = np.ascontiguousarray((c[..., :3].astype(np.float32) @ w) / np.float32(255.0))
        else:
            r._color_arr = np.ascontiguousarray(c)
        r._depth_scale, r._depth_trunc = float(depth_scale), float(depth_trunc)
        if d.ndim == 3 and d.shape[2] == 1:
            d = d[..., 0]
        if d.dtype == np.uint16 and d.ndim == 2:
            r._depth_raw, r._depth_is_raw_u16 = np.ascontiguousarray(d), True
        elif d.dtype == np.float32 and d.ndim == 2:
            # Open3D applies scale/trunc to float images too; done once here on the GPU is not
            # possible for f32 input through the u16 kernel, so scale on the host (rare path).
            f = d / np.float32(depth_scale)
            f[f.astype(np.float64) >= depth_trunc] = 0
            r._depth_raw, r._depth_is_raw_u16 = np.ascontiguousarray(f, np.float32), False
        else:
            raise RuntimeError("[CreateFromColorAndDepth] Unsupported image format.")
        return r

    @property
    def color(self):
        return Image(self._color_arr)

    @property
    def depth(self):
        if self._depth_raw is None:
            return Image()
        if not self._depth_is_raw_u16:
            return Image(self._depth_raw)
        if self._depth_f32 is None:
            out = np.empty(self._depth_raw.shape, np.float32)
            _lib.check(_lib.lib.otslam_depth_convert(_lib.ptr(self._depth_raw), self._depth_raw.size, self._depth_scale,
                                                     self._depth_trunc, _lib.ptr(out), 0))
            self._depth_f32 = out
        return Image(self._depth_f32)

    def __repr__(self):
        return f"RGBDImage of size \nColor image : {self.color!r}\nDepth image : {self.depth!r}"


class PointCloud:
    def __init__(self, points=None):
        self._points = np.zeros((0, 3), np.float64)
        self._colors = np.zeros((0, 3), np.float64)
        self._normals = np.zeros((0, 3), np.float64)
        if points is not None:
            self.points = points

    points = property(lambda s: s._points, lambda s, v: setattr(s, "_points", _as_n3(v)))
    colors = property(lambda s: s._colors, lambda s, v: setattr(s, "_colors", _as_n3(v)))
    normals = property(lambda s: s._normals, lambda s, v: setattr(s, "_normals", _as_n3(v)))

    def has_points(self):
        return len(self._points) > 0

    def has_colors(self):
        return len(self._points) > 0 and len(self._colors) == len(self._points)

    def has_normals(self):
        return len(self._points) > 0 and len(self._normals) == len(self._points)

    def is_empty(self):
        return not self.has_points()

    def __repr__(self):
        return f"PointCloud with {len(self._points)} points."

    def paint_uniform_color(self, color):
        """fusion/hybrid_map.py:59,88 -- resize colours to N and fill."""
        c = np.asarray(color, np.float64).reshape(3)
        self._colors = np.ascontiguousarray(np.broadcast_to(c, (len(self._points), 3)).copy())
        return self

    def __iadd__(self, other):
        """PointCloud += (fusion/hybrid_map.py:91, SURVEY A.11): keep colours/normals only when both
        sides have them (or self is empty)."""
        n_old = len(self._points)
        keep_c = (n_old == 0 or self.has_colors()) and other.has_colors()
        keep_n = (n_old == 0 or self.has_normals()) and other.has_normals()
        self._colors = np.concatenate([self._colors[:n_old], other._colors]) if keep_c else np.zeros((0, 3))
        self._normals = np.concatenate([self._normals[:n_old], other._normals]) if keep_n else np.zeros((0, 3))
        self._points = np.concatenate([self._points, other._points])
        return self

    def __add__(self, other):
        r = PointCloud()
        r._points, r._colors, r._normals = self._points.copy(), self._colors.copy(), self._normals.copy()
        r += other
        return r

    # ---- rigid-body edits: the key callbacks of fusion/hybrid_map_manual.py:86-119 -----------------
    def transform(self, transformation):
        """obj_pcd.transform(T) (hybrid_map_manual.py:87), in place."""
        T = np.ascontiguousarray(transformation, np.float64)
        if T.shape != (4, 4):
            raise RuntimeError("transform expects a 4x4 matrix")
        n = len(self._points)
        if n:
            hn = self.has_normals()
            op = np.empty((n, 3), np.float64)
            on = np.empty((n, 3), np.float64) if hn else None
            _lib.check(_lib.lib.otslam_cloud_transform(_lib.ptr(self._points), _lib.ptr(self._normals if hn else None), n, _lib.ptr(T),
                                                       _lib.ptr(op), _lib.ptr(on), 0))
            self._points = op
            if hn:
                self._normals = on
        return self

    def get_center(self):
        """obj_pcd.get_center() (hybrid_map_manual.py:110): mean of the points (index-order sums)."""
        c = np.zeros(3, np.float64)
        _lib.check(_lib.lib.otslam_cloud_center(_lib.ptr(self._points), len(self._points), _lib.ptr(c), 0))
        return c

    @staticmethod
    def get_rotation_matrix_from_xyz(rotation):
        """R = Rx(a) @ Ry(b) @ Rz(c) (Open3D: AngleAxis(a, X) * AngleAxis(b, Y) * AngleAxis(c, Z)); the reference
        only ever passes (0, 0, yaw) (hybrid_map_manual.py:111)."""
        a, b, c = (float(x) for x in rotation)
        rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
        ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
        rz = np.array([[np.cos(c), -np.sin(c), 0], [np.sin(c), np.cos(c), 0], [0, 0, 1]])
        return rx @ ry @ rz

    def rotate(self, R, center=None):
        """obj_pcd.rotate(R, center=center) (hybrid_map_manual.py:112), in place; default centre = get_center()."""
        R = np.ascontiguousarray(R, np.float64)
        if R.shape != (3, 3):
            raise RuntimeError("rotate expects a 3x3 matrix")
        c = self.get_center() if center is None else np.ascontiguousarray(center, np.float64).reshape(3)
        n = len(self._points)
        if n:
            hn = self.has_normals()
            op = np.empty((n, 3), np.float64)
            on = np.empty((n, 3), np.float64) if hn else None
            _lib.check(_lib.lib.otslam_cloud_rotate(_lib.ptr(self._points), _lib.ptr(self._normals if hn else None), n, _lib.ptr(R),
                                                    _lib.ptr(c), _lib.ptr(op), _lib.ptr(on), 0))
            self._points = op
            if hn:
                self._normals = on
        return self

    def translate(self, translation, relative=True):
        t = np.asarray(translation, np.float64).reshape(3)
        T = np.eye(4)
        T[:3, 3] = t if relative else t - self.get_center()
        return self.transform(T)

    def select_by_index(self, indices, invert=False):
        idx = np.asarray(indices, np.int64)
        if invert:
            m = np.ones(len(self._points), bool)
            m[idx] = False
            idx = np.nonzero(m)[0]
        r = PointCloud()
        r._points = np.ascontiguousarray(self._points[idx])
        if self.has_colors():
            r._colors = np.ascontiguousarray(self._colors[idx])
        if self.has_normals():
            r._normals = np.ascontiguousarray(self._normals[idx])
        return r

    @staticmethod
    def create_from_rgbd_image(image, intrinsic, extrinsic=None, project_valid_depth_only=True):
        """3d_model/check_one_frame.py:27 (SURVEY A.12)."""
        if not project_valid_depth_only:
            raise RuntimeError("project_valid_depth_only=False is not supported")
        d = np.asarray(image.depth)
        if d.ndim != 2 or d.dtype != np.float32 or d.shape != (intrinsic.height, intrinsic.width):
            raise RuntimeError("[CreatePointCloudFromRGBDImage] Unsupported image format.")
        c = image._color_arr
        rgb = c if (c is not None and c.dtype == np.uint8 and c.shape == d.shape + (3,)) else None
        H, W = d.shape
        pts = np.empty((H * W, 3), np.float64)
        cols = np.empty((H * W, 3), np.float64) if rgb is not None else None
        n = C.c_int64(0)
        k = np.array(intrinsic.fxfycxcy(), np.float64)
        e = None if extrinsic is None else np.ascontiguousarray(extrinsic, np.float64)
        _lib.check(_lib.lib.otslam_backproject_rgbd(_lib.ptr(d), _lib.ptr(rgb), W, H, _lib.ptr(k), _lib.ptr(e), _lib.ptr(pts),
                                                    _lib.ptr(cols), C.byref(n), 0))
        pc = PointCloud()
        pc._points = np.ascontiguousarray(pts[:n.value])
        if cols is not None:
            pc._colors = np.ascontiguousarray(cols[:n.value])
        return pc

    def compute_point_cloud_distance(self, target):
        """Distance from each point of this cloud to its nearest neighbour in `target` (the accuracy /
        completeness metric of /root/reference/eval/eval_table_chair/eval_table_chair.py:106-119)."""
        n = len(self._points)
        out = np.empty(n, np.float64)
        _lib.check(_lib.lib.otslam_cloud_nn_distance(_lib.ptr(self._points), n, _lib.ptr(target._points), len(target._points),
                                                     _lib.ptr(out), 0))
        return out

    def voxel_down_sample(self, voxel_size):
        """check_one_frame.py:28 (SURVEY A.7); output ordered by voxel key."""
        n = len(self._points)
        if voxel_size <= 0:
            raise RuntimeError("[VoxelDownSample] voxel_size <= 0.")
        r = PointCloud()
        if n == 0:
            return r
        op = np.empty((n, 3), np.float64)
        oc = np.empty((n, 3), np.float64) if self.has_colors() else None
        m = C.c_int64(0)
        _lib.check(_lib.lib.otslam_cloud_voxel_down_sample(_lib.ptr(self._points), _lib.ptr(self._colors if self.has_colors() else None),
                                                           n, float(voxel_size), _lib.ptr(op), _lib.ptr(oc), None, None, C.byref(m), 0))
        r._points = np.ascontiguousarray(op[:m.value])
        if oc is not None:
            r._colors = np.ascontiguousarray(oc[:m.value])
        if self.has_normals():
            # Open3D averages normals per voxel exactly like colours (sum in point-index order / count, not re-normalised):
            # the same kernel with the normals in the colour slot gives the same voxels in the same order
            on = np.empty((n, 3), np.float64)
            _lib.check(_lib.lib.otslam_cloud_voxel_down_sample(_lib.ptr(self._points), _lib.ptr(self._normals), n, float(voxel_size),
                                                               _lib.ptr(op), _lib.ptr(on), None, None, C.byref(m), 0))
            r._normals = np.ascontiguousarray(on[:m.value])
        return r

    def remove_statistical_outlier(self, nb_neighbors, std_ratio, print_progress=False):
        """north_star opt-in stage (SURVEY A.8): returns (selected cloud, kept indices)."""
        n = len(self._points)
        idx = np.empty(n, np.int64)
        m = C.c_int64(0)
        _lib.check(_lib.lib.otslam_cloud_remove_statistical_outlier(_lib.ptr(self._points), n, int(nb_neighbors), float(std_ratio),
                                                                    _lib.ptr(idx), C.byref(m), None, 0))
        idx = idx[:m.value].copy()
        return self.select_by_index(idx), idx.tolist()

    # ---- normals: PointCloud.estimate_normals and the orientation helpers (DESIGN.md §4 "Normals and point-to-plane
    # registration"); the normals registration_icp(..., TransformationEstimationPointToPlane()) needs on its target
    def estimate_normals(self, search_param=None, fast_normal_computation=True):
        """Normals from the covariance of each point's neighbours (search_param: KDTreeSearchParamKNN (default, 30
        neighbours) or KDTreeSearchParamHybrid).  A cloud that already has normals orients the new ones along them; one
        without gets the sign that makes the largest-magnitude component positive.  fast_normal_computation is accepted
        for compatibility: there is one eigen solver."""
        radius, max_nn = (search_param or KDTreeSearchParamKNN())._radius_max_nn()
        n = len(self._points)
        prior = self._normals if self.has_normals() else None
        out = np.empty((n, 3), np.float64)
        _lib.check(_lib.lib.otslam_cloud_estimate_normals(_lib.ptr(self._points), n, _lib.ptr(prior), radius, max_nn, _lib.ptr(out), 0))
        self._normals = out

    def _require_normals(self):
        if not self.has_normals():
            raise RuntimeError("No normals in the PointCloud. Call EstimateNormals() first.")

    def orient_normals_to_align_with_direction(self, orientation_reference=(0.0, 0.0, 1.0)):
        """Open3D's rule: a zero normal becomes the reference, one with n . reference < 0 is flipped."""
        self._require_normals()
        ref = np.asarray(orientation_reference, np.float64).reshape(3)
        nrm = self._normals.copy()
        zero = np.linalg.norm(nrm, axis=1) == 0.0
        flip = ~zero & ((nrm @ ref) < 0.0)
        nrm[flip] *= -1.0
        nrm[zero] = ref
        self._normals = nrm

    def orient_normals_towards_camera_location(self, camera_location=(0.0, 0.0, 0.0)):
        """Open3D's rule with reference = camera_location - point: a zero normal becomes the normalised reference ((0, 0,
        1) when that is zero too), one with n . reference < 0 is flipped."""
        self._require_normals()
        ref = np.asarray(camera_location, np.float64).reshape(1, 3) - self._points
        nrm = self._normals.copy()
        zero = np.linalg.norm(nrm, axis=1) == 0.0
        flip = ~zero & (np.einsum("ij,ij->i", nrm, ref) < 0.0)
        nrm[flip] *= -1.0
        rlen = np.linalg.norm(ref, axis=1)
        nrm[zero & (rlen > 0.0)] = ref[zero & (rlen > 0.0)] / rlen[zero & (rlen > 0.0), None]
        nrm[zero & (rlen == 0.0)] = (0.0, 0.0, 1.0)
        self._normals = nrm

    # ---- segmentation (DESIGN.md §4 "Plane segmentation and DBSCAN clustering"): drop the floor, keep the object's cluster
    def segment_plane(self, distance_threshold, ransac_n, num_iterations, probability=0.99999999, seed=None):
        """Open3D's RANSAC plane fit -> (plane [a, b, c, d] with a x + b y + c z + d = 0, inlier indices as a list).
        The hypotheses are drawn from seed (None: the next seed of o3d.utility.random.seed, or an unseeded one)."""
        n = len(self._points)
        plane = np.zeros(4, np.float64)
        idx = np.empty(n, np.int64)
        m = C.c_int64(0)
        _lib.check(_lib.lib.otslam_cloud_segment_plane(_lib.ptr(self._points), n, float(distance_threshold), int(ransac_n),
                                                       int(num_iterations), float(probability),
                                                       C.c_uint64(_next_seed(seed) & 0xFFFFFFFFFFFFFFFF), _lib.ptr(plane),
                                                       _lib.ptr(idx), C.byref(m), None, 0))
        return plane, idx[:m.value].tolist()

    def cluster_dbscan(self, eps, min_points, print_progress=False):
        """DBSCAN labels (int32, -1 = noise), clusters numbered in the order of their smallest point index."""
        n = len(self._points)
        labels = np.empty(n, np.int32)
        _lib.check(_lib.lib.otslam_cloud_cluster_dbscan(_lib.ptr(self._points), n, float(eps), int(min_points), _lib.ptr(labels), None, 0))
        return labels


_MAX_NN = 128          # neighbours a normal estimation may keep (otslam_cloud_estimate_normals)


class KDTreeSearchParamKNN:
    """The knn nearest neighbours (1..128)."""

    def __init__(self, knn=30):
        self.knn = int(knn)

    def _radius_max_nn(self):
        return float("inf"), self.knn


class KDTreeSearchParamHybrid:
    """At most max_nn (1..128) nearest neighbours strictly within radius."""

    def __init__(self, radius, max_nn):
        self.radius, self.max_nn = float(radius), int(max_nn)

    def _radius_max_nn(self):
        return self.radius, self.max_nn


class KDTreeSearchParamRadius:
    def __init__(self, radius):
        raise RuntimeError(f"KDTreeSearchParamRadius (an unbounded neighbour count) is not supported: normal estimation keeps at "
                           f"most {_MAX_NN} neighbours; use KDTreeSearchParamHybrid(radius, max_nn) with max_nn <= {_MAX_NN}")


class _ResidentArray:
    """Stand-in for a mesh array that still lives in HBM (what Open3D exposes as a Vector3dVector):
    len() is free, anything that needs the values (np.asarray, indexing, .shape ...) downloads the mesh."""

    def __init__(self, mesh, name, n):
        self._mesh, self._name, self._n = mesh, name, n

    def __len__(self):
        return self._n

    def _host(self):
        self._mesh._materialize()
        return getattr(self._mesh, "_" + self._name)

    def __array__(self, dtype=None, copy=None):
        a = self._host()
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, i):
        return self._host()[i]

    def __iter__(self):
        return iter(self._host())

    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        return getattr(self._host(), k)


class TriangleMesh:
    def __init__(self):
        self._vertices = np.zeros((0, 3), np.float64)
        self._vertex_colors = np.zeros((0, 3), np.float64)
        self._vertex_normals = np.zeros((0, 3), np.float64)
        self._triangles = np.zeros((0, 3), np.int32)
        self._res = None          # (TSDFVolume, nv, nf, has_colors) while the arrays are still in HBM
        self._res_normals = False  # compute_vertex_normals() was called on the resident mesh

    # ---- device-resident state (set by ScalableTSDFVolume.extract_triangle_mesh) ---------------
    def _attach_resident(self, vol, nv, nf, colors):
        self._res = (vol, nv, nf, colors) if nv > 0 else None
        self._res_normals = False

    def _materialize(self):
        """Download the resident arrays (once) and become an ordinary host mesh."""
        if self._res is None:
            return
        vol, nv, nf, colors = self._res
        self._res = None
        v, c, n, f = vol.mesh_download(nv, nf, normals=self._res_normals)
        self._vertices, self._triangles = v, f
        if colors:
            self._vertex_colors = c
        if self._res_normals:
            self._vertex_normals = n

    def _get(self, name, present=True):
        if self._res is not None:
            nv, nf = self._res[1], self._res[2]
            if not present:
                return np.zeros((0, 3), np.float64)
            return _ResidentArray(self, name, nf if name == "triangles" else nv)
        return getattr(self, "_" + name)

    def _set(self, name, value, dtype=np.float64):
        self._materialize()
        setattr(self, "_" + name, _as_n3(value, dtype))

    vertices = property(lambda s: s._get("vertices"), lambda s, v: s._set("vertices", v))
    vertex_colors = property(lambda s: s._get("vertex_colors", s._res is None or s._res[3]), lambda s, v: s._set("vertex_colors", v))
    vertex_normals = property(lambda s: s._get("vertex_normals", s._res is None or s._res_normals),
                              lambda s, v: s._set("vertex_normals", v))
    triangles = property(lambda s: s._get("triangles"), lambda s, v: s._set("triangles", v, np.int32))

    def has_vertices(self):
        return len(self.vertices) > 0

    def has_triangles(self):
        return len(self.vertices) > 0 and len(self.triangles) > 0

    def has_vertex_colors(self):
        return len(self.vertices) > 0 and len(self.vertex_colors) == len(self.vertices)

    def has_vertex_normals(self):
        return len(self.vertices) > 0 and len(self.vertex_normals) == len(self.vertices)

    def is_empty(self):
        return not self.has_vertices()

    def __repr__(self):
        return f"TriangleMesh with {len(self.vertices)} points and {len(self.triangles)} triangles."

    def compute_vertex_normals(self, normalized=True):
        """reconstruct_rgbd.py:113 (SURVEY A.9)."""
        if self._res is not None:           # extraction already left the normals next to the mesh in HBM
            self._res_normals = True
            return self
        nv, nf = len(self._vertices), len(self._triangles)
        out = np.empty((nv, 3), np.float64)
        _lib.check(_lib.lib.otslam_mesh_vertex_normals(_lib.ptr(self._vertices), nv, _lib.ptr(self._triangles), nf, _lib.ptr(out), 0))
        self._vertex_normals = out
        return self

    def sample_points_uniformly(self, number_of_points=100, use_triangle_normal=False, seed=None):
        """reconstruct_rgbd_filter.py:123 (SURVEY A.10)."""
        if number_of_points <= 0:
            raise RuntimeError("[SamplePointsUniformly] number_of_points <= 0")
        if not self.has_triangles():
            raise RuntimeError("[SamplePointsUniformly] input mesh has no triangles")
        n = int(number_of_points)
        hc, hn = self.has_vertex_colors(), self.has_vertex_normals()
        if self._res is not None:           # sample straight from HBM
            op, oc, on = self._res[0].mesh_sample(n, _next_seed(seed), colors=hc, normals=hn)
            pc = PointCloud()
            pc._points = op
            if hc:
                pc._colors = oc
            if hn:
                pc._normals = on
            return pc
        op = np.empty((n, 3), np.float64)
        oc = np.empty((n, 3), np.float64) if hc else None
        on = np.empty((n, 3), np.float64) if hn else None
        _lib.check(_lib.lib.otslam_mesh_sample_uniform(
            _lib.ptr(self._vertices), _lib.ptr(self._vertex_colors if hc else None), _lib.ptr(self._vertex_normals if hn else None),
            len(self._vertices), _lib.ptr(self._triangles), len(self._triangles), n, C.c_uint64(_next_seed(seed)),
            _lib.ptr(op), _lib.ptr(oc), _lib.ptr(on), 0))
        pc = PointCloud()
        pc._points = op
        if hc:
            pc._colors = oc
        if hn:
            pc._normals = on
        return pc

    @staticmethod
    def create_coordinate_frame(size=1.0, origin=(0.0, 0.0, 0.0)):
        """Only handed to draw_geometries (fusion/hybrid_map.py:128); an empty placeholder suffices."""
        return TriangleMesh()


__all__ = ["Image", "RGBDImage", "PointCloud", "TriangleMesh", "Vector3dVector", "Vector3iVector", "KDTreeSearchParamKNN",
           "KDTreeSearchParamHybrid", "KDTreeSearchParamRadius"]
