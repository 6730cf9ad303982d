"""o3d.pipelines.integration: ScalableTSDFVolume on the GPU (reconstruct_rgbd.py:79-83,107,112)."""
import ctypes as C
import enum
import os
import types

import numpy as np

from .. import _lib
from ..volume import TSDFVolume, checkpoint_info
from . import geometry

_FMT = "[ScalableTSDFVolume::Integrate] Unsupported image format."


class TSDFVolumeColorType(enum.Enum):
    NoColor = 0
    RGB8 = 1
    Gray32 = 2


class ScalableTSDFVolume:
    def __init__(self, voxel_length, sdf_trunc, color_type, volume_unit_resolution=16, depth_sampling_stride=4,
                 device=0, slab=None):
        if volume_unit_resolution != 16 or depth_sampling_stride != 4:
            raise RuntimeError("otslam_b200 supports volume_unit_resolution=16, depth_sampling_stride=4 (the Open3D "
                               "defaults the reference relies on)")
        if color_type == TSDFVolumeColorType.Gray32:
            raise RuntimeError("TSDFVolumeColorType.Gray32 is not supported (the reference uses RGB8)")
        self.voxel_length, self.sdf_trunc, self.color_type = float(voxel_length), float(sdf_trunc), color_type
        self._vol = TSDFVolume(voxel_length, sdf_trunc, color=(color_type == TSDFVolumeColorType.RGB8), device=device,
                               slab=slab)

    # -- reference API -------------------------------------------------------------------------
    def reset(self):
        self._vol.reset()

    def integrate(self, image, intrinsic, extrinsic):
        """volume.integrate(rgbd, intrinsics, extrinsic) -- reconstruct_rgbd.py:107."""
        depth_raw, color = image._depth_raw, image._color_arr
        if depth_raw is None or depth_raw.ndim != 2:
            raise RuntimeError(_FMT)
        H, W = depth_raw.shape
        if (W, H) != (intrinsic.width, intrinsic.height):
            raise RuntimeError(_FMT)
        rgb = None
        if self.color_type == TSDFVolumeColorType.RGB8:
            if color is None or color.dtype != np.uint8 or color.shape != (H, W, 3):
                raise RuntimeError(_FMT)
            rgb = color
        ext = np.asarray(extrinsic, np.float64)
        if ext.shape != (4, 4):
            raise RuntimeError("extrinsic must be a 4x4 matrix")
        if image._depth_is_raw_u16:
            self._vol.integrate_u16(depth_raw, rgb, intrinsic.fxfycxcy(), ext, image._depth_scale, image._depth_trunc)
        elif depth_raw.dtype == np.float32:
            self._vol.integrate_f32(depth_raw, rgb, intrinsic.fxfycxcy(), ext)
        else:
            raise RuntimeError(_FMT)

    def extract_triangle_mesh(self):
        """reconstruct_rgbd.py:112.  The mesh (often ~100 MB) stays in HBM: the returned TriangleMesh
        downloads its arrays only when they are read (np.asarray(mesh.vertices), write_triangle_mesh);
        len(mesh.vertices), compute_vertex_normals() and sample_points_uniformly() work on the device."""
        m = geometry.TriangleMesh()
        nv, nf = self._vol.extract_mesh_resident(owner=m)
        m._attach_resident(self._vol, nv, nf, colors=self.color_type != TSDFVolumeColorType.NoColor)
        return m

    def extract_point_cloud(self):
        """ScalableTSDFVolume.extract_point_cloud(): zero crossings along +x/+y/+z with colours and TSDF-gradient normals."""
        p, c, _, n = self._vol.extract_point_cloud(normals=True)
        pc = geometry.PointCloud()
        pc.points = p
        pc.normals = n
        if self.color_type != TSDFVolumeColorType.NoColor:
            pc.colors = c
        return pc

    # -- batched extension: the whole frame loop in one call (frame order preserved) ------------
    def integrate_sequence(self, depths, colors, intrinsic, extrinsics, depth_scale=1000.0, depth_trunc=3.0):
        n = len(extrinsics)
        if n == 0:
            return
        if tuple(depths.shape[1:]) != (intrinsic.height, intrinsic.width):
            raise RuntimeError(_FMT)
        self._vol.integrate_batch(depths, colors if self.color_type == TSDFVolumeColorType.RGB8 else None,
                                  intrinsic.fxfycxcy(), extrinsics, depth_scale, depth_trunc)

    # -- checkpoint extension (the names of Open3D's tensor VoxelBlockGrid; the file format is this library's own) ----
    def save(self, file_name):
        """Write the volume's voxel state to `file_name`; ScalableTSDFVolume.load continues from it bit for bit."""
        self._vol.save(file_name)

    @staticmethod
    def load(file_name, device=0):
        """A new volume holding a checkpoint (or, given a list, the part files of a sharded volume), with the voxel
        parameters stored in the file."""
        first = file_name if isinstance(file_name, (str, bytes, os.PathLike)) else file_name[0]
        info = checkpoint_info(first)
        color = TSDFVolumeColorType.RGB8 if info["color"] else TSDFVolumeColorType.NoColor
        vol = ScalableTSDFVolume(info["voxel_length"], info["sdf_trunc"], color, device=device)
        vol._vol.load(file_name)
        return vol

    # -- ray-casting extension (named after Open3D's tensor VoxelBlockGrid.ray_cast) ---------------------------------------
    def ray_cast(self, intrinsic, extrinsic, depth_min=0.1, depth_max=3.0):
        """Render the volume from one camera (a PinholeCameraIntrinsic and a world->camera 4x4 extrinsic): a dict of
        NumPy arrays depth [H,W] f32 metres, vertex / normal [H,W,3] f32 world, color [H,W,3] u8 (0 where nothing is hit).
        depth_max defaults to the reference's depth_trunc of 3.0."""
        return self._vol.ray_cast(intrinsic.fxfycxcy(), extrinsic, intrinsic.width, intrinsic.height, depth_min, depth_max)

    # -- tracking extension (named after Open3D's tensor SLAM Model.track_frame_to_model) -------------------------------
    def track_frame_to_model(self, image, intrinsic, extrinsic, depth_min=0.1, depth_max=3.0, depth_diff=0.07,
                             max_iterations=20):
        """Refine the pose of one frame (an RGBDImage with raw u16 depth; its depth scale is used) against the volume by
        point-to-plane ICP on its ray-cast model, starting from `extrinsic` (world->camera 4x4).  Unlike Open3D, whose
        result holds a camera-to-camera correction, OdometryResult.transformation IS the refined world->camera extrinsic:
        what integrate() takes.  depth_diff and max_iterations may be per-level sequences (coarse-to-fine tracking over a
        depth pyramid, as TSDFVolume.track; volume.TRACK_PYRAMID is the recommended setting).  The volume is only read."""
        if image._depth_raw is None or not image._depth_is_raw_u16:
            raise RuntimeError("track_frame_to_model needs an RGBDImage made from raw u16 depth")
        r = self._vol.track(image._depth_raw, intrinsic.fxfycxcy(), extrinsic, image._depth_scale, depth_min, depth_max,
                            depth_diff, max_iterations)
        return OdometryResult(r["extrinsic"], float(r["fitness"]), float(r["inlier_rmse"]), int(r["status"]) == 0)


class OdometryResult:
    """Result of ScalableTSDFVolume.track_frame_to_model: the refined world->camera extrinsic, fitness (inliers / valid
    pixels), inlier_rmse (metres) and whether the iteration converged."""

    def __init__(self, transformation, fitness, inlier_rmse, converged):
        self.transformation, self.fitness, self.inlier_rmse, self.converged = transformation, fitness, inlier_rmse, converged

    def __repr__(self):
        return f"OdometryResult with fitness={self.fitness:e}, inlier_rmse={self.inlier_rmse:e}, converged={self.converged}"


integration = types.SimpleNamespace(ScalableTSDFVolume=ScalableTSDFVolume, TSDFVolumeColorType=TSDFVolumeColorType)


# ---------------------------------------------------------------------------------------------------------------------
# o3d.pipelines.registration: point-to-point ICP as the reference's evaluation scripts call it
# (/root/reference/eval/eval_table_chair/eval_table_chair.py:90-104; SURVEY 8f row 3).  Correspondence search and the rigid
# update of the source run on the GPU (otslam_cloud_nn_within, otslam_cloud_transform); the 3x3 SVD of the Umeyama step
# and the convergence test are host arithmetic, as in Open3D.
# ---------------------------------------------------------------------------------------------------------------------
class TransformationEstimationPointToPoint:
    def __init__(self, with_scaling=False):
        if with_scaling:
            raise RuntimeError("TransformationEstimationPointToPoint(with_scaling=True) is not supported")
        self.with_scaling = False

    @staticmethod
    def compute_transformation(src, dst):
        """Eigen::umeyama(src, dst, false): least-squares rigid transform src -> dst."""
        ms, md = src.mean(axis=0), dst.mean(axis=0)
        cov = (dst - md).T @ (src - ms) / len(src)
        U, _, Vt = np.linalg.svd(cov)
        S = np.eye(3)
        if np.linalg.det(U) * np.linalg.det(Vt) < 0:
            S[2, 2] = -1.0
        T = np.eye(4)
        T[:3, :3] = U @ S @ Vt
        T[:3, 3] = md - T[:3, :3] @ ms
        return T


class TransformationEstimationPointToPlane:
    """Point-to-plane estimation: registration_icp runs the whole loop on the GPU in one call
    (otslam_cloud_icp_point_to_plane); the target needs normals (PointCloud.estimate_normals)."""

    def __init__(self, kernel=None):
        if kernel is not None:
            raise RuntimeError("TransformationEstimationPointToPlane(kernel=...): robust kernels are not supported")
        self.kernel = None


class ICPConvergenceCriteria:
    def __init__(self, relative_fitness=1e-6, relative_rmse=1e-6, max_iteration=30):
        self.relative_fitness, self.relative_rmse, self.max_iteration = float(relative_fitness), float(relative_rmse), int(max_iteration)


class RegistrationResult:
    def __init__(self):
        self.transformation = np.eye(4)
        self.fitness, self.inlier_rmse = 0.0, 0.0
        self.correspondence_set = np.zeros((0, 2), np.int32)

    def __repr__(self):
        return (f"RegistrationResult with fitness={self.fitness:e}, inlier_rmse={self.inlier_rmse:e}, and "
                f"correspondence_set size of {len(self.correspondence_set)}")


def _correspondences(src_pts, tgt_pts, max_dist):
    n = len(src_pts)
    idx = np.empty(n, np.int32)
    d2 = np.empty(n, np.float64)
    _lib.check(_lib.lib.otslam_cloud_nn_within(_lib.ptr(src_pts), n, _lib.ptr(tgt_pts), len(tgt_pts), float(max_dist), _lib.ptr(idx),
                                               _lib.ptr(d2), 0))
    sel = np.nonzero(idx >= 0)[0]
    return sel, idx[sel], d2[sel]


def evaluate_registration(source, target, max_correspondence_distance, transformation=None):
    """o3d.pipelines.registration.evaluate_registration: fitness = inliers / |source|, inlier_rmse over the inliers."""
    src = geometry.PointCloud(np.asarray(source.points))
    if transformation is not None:
        src.transform(transformation)
    r = RegistrationResult()
    r.transformation = np.eye(4) if transformation is None else np.array(transformation, np.float64)
    tgt = np.ascontiguousarray(np.asarray(target.points), np.float64)
    sel, ti, d2 = _correspondences(np.ascontiguousarray(src.points), tgt, max_correspondence_distance)
    if len(sel):
        r.fitness = len(sel) / len(src.points)
        r.inlier_rmse = float(np.sqrt(d2.sum() / len(sel)))
        r.correspondence_set = np.stack([sel.astype(np.int32), ti.astype(np.int32)], 1)
    return r


def registration_icp(source, target, max_correspondence_distance, init=None, estimation_method=None, criteria=None):
    """registration_icp(source, target, threshold, init, TransformationEstimationPointToPoint() or
    TransformationEstimationPointToPlane(), ICPConvergenceCriteria(...))."""
    estimation_method = estimation_method or TransformationEstimationPointToPoint()
    criteria = criteria or ICPConvergenceCriteria()
    if not isinstance(estimation_method, (TransformationEstimationPointToPoint, TransformationEstimationPointToPlane)):
        raise RuntimeError("only TransformationEstimationPointToPoint and TransformationEstimationPointToPlane are supported")
    if max_correspondence_distance <= 0:
        raise RuntimeError("[RegistrationICP] Invalid max_correspondence_distance.")
    if isinstance(estimation_method, TransformationEstimationPointToPlane):
        return _registration_icp_point_to_plane(source, target, max_correspondence_distance, init, criteria)
    T = np.eye(4) if init is None else np.array(init, np.float64)
    tgt = np.ascontiguousarray(np.asarray(target.points), np.float64)
    pcd = geometry.PointCloud(np.asarray(source.points))
    pcd.transform(T)

    def evaluate():
        r = RegistrationResult()
        sel, ti, d2 = _correspondences(np.ascontiguousarray(pcd.points), tgt, max_correspondence_distance)
        if len(sel):
            r.fitness = len(sel) / len(pcd.points)
            r.inlier_rmse = float(np.sqrt(d2.sum() / len(sel)))
            r.correspondence_set = np.stack([sel.astype(np.int32), ti.astype(np.int32)], 1)
        return r

    result = evaluate()
    for _ in range(criteria.max_iteration):
        if len(result.correspondence_set) < 3:
            break
        cs = result.correspondence_set
        update = estimation_method.compute_transformation(np.asarray(pcd.points)[cs[:, 0]], tgt[cs[:, 1]])
        T = update @ T
        pcd.transform(update)
        backup, result = result, evaluate()
        if abs(backup.fitness - result.fitness) < criteria.relative_fitness and \
                abs(backup.inlier_rmse - result.inlier_rmse) < criteria.relative_rmse:
            break
    result.transformation = T
    return result


def _registration_icp_point_to_plane(source, target, max_correspondence_distance, init, criteria):
    if not target.has_normals():
        raise RuntimeError("TransformationEstimationPointToPlane and TransformationEstimationColoredICP "
                           "require pre-computed normal vectors for target PointCloud.")
    src = np.ascontiguousarray(np.asarray(source.points), np.float64)
    tgt = np.ascontiguousarray(np.asarray(target.points), np.float64)
    tn = np.ascontiguousarray(np.asarray(target.normals), np.float64)
    T0 = np.ascontiguousarray(np.eye(4) if init is None else init, np.float64).reshape(16)
    T = np.empty(16)
    fit, rmse, it = C.c_double(), C.c_double(), C.c_int32()
    corr = np.empty(len(src), np.int32)
    _lib.check(_lib.lib.otslam_cloud_icp_point_to_plane(
        _lib.ptr(src), len(src), _lib.ptr(tgt), _lib.ptr(tn), len(tgt), float(max_correspondence_distance), _lib.ptr(T0),
        criteria.relative_fitness, criteria.relative_rmse, criteria.max_iteration, _lib.ptr(T), C.byref(fit), C.byref(rmse),
        C.byref(it), _lib.ptr(corr), 0))
    r = RegistrationResult()
    r.transformation = T.reshape(4, 4)
    r.fitness, r.inlier_rmse = fit.value, rmse.value
    sel = np.nonzero(corr >= 0)[0]
    r.correspondence_set = np.stack([sel.astype(np.int32), corr[sel]], 1) if len(sel) else np.zeros((0, 2), np.int32)
    return r


registration = types.SimpleNamespace(registration_icp=registration_icp, evaluate_registration=evaluate_registration,
                                     TransformationEstimationPointToPoint=TransformationEstimationPointToPoint,
                                     TransformationEstimationPointToPlane=TransformationEstimationPointToPlane,
                                     ICPConvergenceCriteria=ICPConvergenceCriteria, RegistrationResult=RegistrationResult)
