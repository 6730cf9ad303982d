"""Device-resident point clouds: the post stage of the filter scripts without PCIe round trips.

The reference's tail (/root/reference/3d_model/reconstruct_rgbd_filter.py:123-134) is
    mesh.sample_points_uniformly(100000) -> points[:, 2] >= 0.03 mask -> (north_star: voxel_down_sample ->
    remove_statistical_outlier) -> write_point_cloud
Through host arrays that chain crosses PCIe once per operator and direction.  The stateless operators of the C ABI accept
DEVICE pointers as well as host pointers (unified addressing), so a DeviceCloud keeps points / colours / normals as CUDA
tensors between them and downloads once, at the end.  Same kernels, same arithmetic and order as the host-buffer calls:
results are bit-identical (tests/test_gpu_resident_mesh.py).
"""
import ctypes as C

import numpy as np

from . import _lib


def _sync():
    import torch
    torch.cuda.synchronize()


class DeviceCloud:
    def __init__(self, points, colors=None, normals=None):
        self.points, self.colors, self.normals = points, colors, normals

    def __len__(self):
        return int(self.points.shape[0])

    @property
    def device_index(self):
        return int(self.points.device.index or 0)

    @staticmethod
    def from_numpy(points, colors=None, normals=None, device=0):
        import torch
        dev = torch.device("cuda", device)
        t = lambda a: None if a is None or len(a) == 0 else torch.from_numpy(np.ascontiguousarray(a, np.float64)).to(dev)  # noqa: E731
        return DeviceCloud(t(points) if len(points) else torch.zeros((0, 3), dtype=torch.float64, device=dev), t(colors), t(normals))

    @staticmethod
    def sample_mesh(volume, n, seed, colors=True, normals=False):
        """mesh.sample_points_uniformly(n) from the mesh the volume's last extraction left in HBM, result left in HBM."""
        import torch
        dev = torch.device("cuda", volume.device)
        n = int(n)
        op = torch.empty((n, 3), dtype=torch.float64, device=dev)
        oc = torch.empty((n, 3), dtype=torch.float64, device=dev) if colors else None
        on = torch.empty((n, 3), dtype=torch.float64, device=dev) if normals else None
        _lib.check(_lib.lib.otslam_volume_mesh_sample(volume._h, n, C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), _lib.ptr(op), _lib.ptr(oc),
                                                      _lib.ptr(on)))
        return DeviceCloud(op, oc, on)

    def zfilter(self, zmin):
        """points[:, 2] >= zmin, order preserved (reconstruct_rgbd_filter.py:126-132; normals are dropped there too)."""
        import torch
        n = len(self)
        op = torch.empty_like(self.points)
        oc = torch.empty_like(self.colors) if self.colors is not None else None
        m = C.c_int64(0)
        _sync()
        _lib.check(_lib.lib.otslam_cloud_zfilter(_lib.ptr(self.points), _lib.ptr(self.colors), n, float(zmin), _lib.ptr(op), _lib.ptr(oc),
                                                 C.byref(m), self.device_index))
        _sync()
        return DeviceCloud(op[:m.value], None if oc is None else oc[:m.value])

    def voxel_down_sample(self, voxel_size):
        """PointCloud.voxel_down_sample (check_one_frame.py:28): per-voxel means of points, colours and normals, by voxel key."""
        import torch
        n = len(self)
        if voxel_size <= 0:
            raise RuntimeError("[VoxelDownSample] voxel_size <= 0.")
        if n == 0:
            return DeviceCloud(self.points)
        op = torch.empty_like(self.points)
        oc = torch.empty_like(self.points) if self.colors is not None else None
        m = C.c_int64(0)
        _sync()
        _lib.check(_lib.lib.otslam_cloud_voxel_down_sample(_lib.ptr(self.points), _lib.ptr(self.colors), n, float(voxel_size), _lib.ptr(op),
                                                           _lib.ptr(oc), None, None, C.byref(m), self.device_index))
        on = None
        if self.normals is not None:      # normals average like colours (Open3D: sum / count, not re-normalised)
            on = torch.empty_like(self.points)
            tmp = torch.empty_like(self.points)
            _lib.check(_lib.lib.otslam_cloud_voxel_down_sample(_lib.ptr(self.points), _lib.ptr(self.normals), n, float(voxel_size),
                                                               _lib.ptr(tmp), _lib.ptr(on), None, None, C.byref(m), self.device_index))
        _sync()
        k = m.value
        return DeviceCloud(op[:k], None if oc is None else oc[:k], None if on is None else on[:k])

    def remove_statistical_outlier(self, nb_neighbors, std_ratio):
        """PointCloud.remove_statistical_outlier -> (kept cloud, kept indices as a CUDA int64 tensor)."""
        import torch
        n = len(self)
        idx = torch.empty(n, dtype=torch.int64, device=self.points.device)
        m = C.c_int64(0)
        _sync()
        _lib.check(_lib.lib.otslam_cloud_remove_statistical_outlier(_lib.ptr(self.points), n, int(nb_neighbors), float(std_ratio),
                                                                    _lib.ptr(idx), C.byref(m), None, self.device_index))
        _sync()
        idx = idx[:m.value]
        take = lambda t: None if t is None else t.index_select(0, idx)  # noqa: E731
        return DeviceCloud(take(self.points), take(self.colors), take(self.normals)), idx

    def select_by_index(self, idx, invert=False):
        """The points (colours, normals) at idx, a CUDA or host integer index; invert=True keeps all the others, in order."""
        import torch
        idx = torch.as_tensor(idx, dtype=torch.int64, device=self.points.device)
        if invert:
            keep = torch.ones(len(self), dtype=torch.bool, device=self.points.device)
            keep[idx] = False
            idx = torch.nonzero(keep).flatten()
        take = lambda t: None if t is None else t.index_select(0, idx)  # noqa: E731
        return DeviceCloud(take(self.points), take(self.colors), take(self.normals))

    def segment_plane(self, distance_threshold, ransac_n, num_iterations, probability=0.99999999, seed=0):
        """PointCloud.segment_plane -> (plane as a float64 ndarray [4], inlier indices as a CUDA int64 tensor)."""
        import torch
        n = len(self)
        plane = np.zeros(4, np.float64)
        idx = torch.empty(n, dtype=torch.int64, device=self.points.device)
        m = C.c_int64(0)
        _sync()
        _lib.check(_lib.lib.otslam_cloud_segment_plane(_lib.ptr(self.points), n, float(distance_threshold), int(ransac_n),
                                                       int(num_iterations), float(probability), C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF),
                                                       _lib.ptr(plane), _lib.ptr(idx), C.byref(m), None, self.device_index))
        _sync()
        return plane, idx[:m.value]

    def cluster_dbscan(self, eps, min_points):
        """PointCloud.cluster_dbscan -> labels as a CUDA int32 tensor (-1 = noise)."""
        import torch
        labels = torch.empty(len(self), dtype=torch.int32, device=self.points.device)
        _sync()
        _lib.check(_lib.lib.otslam_cloud_cluster_dbscan(_lib.ptr(self.points), len(self), float(eps), int(min_points), _lib.ptr(labels),
                                                        None, self.device_index))
        _sync()
        return labels

    def to_numpy(self):
        from .slab import to_host
        ts = [t for t in (self.points, self.colors, self.normals) if t is not None]
        out = list(to_host(ts))
        p = out.pop(0)
        c = out.pop(0) if self.colors is not None else None
        nrm = out.pop(0) if self.normals is not None else None
        return p, c, nrm

    def to_pointcloud(self):
        """Download once into a compat PointCloud (what o3d.io.write_point_cloud takes)."""
        from .o3d_compat import geometry
        p, c, nrm = self.to_numpy()
        pc = geometry.PointCloud()
        pc._points = np.ascontiguousarray(p)
        if c is not None:
            pc._colors = np.ascontiguousarray(c)
        if nrm is not None:
            pc._normals = np.ascontiguousarray(nrm)
        return pc
