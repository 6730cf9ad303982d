"""Host-side handle of one GPU ScalableTSDFVolume (thin wrapper over the C ABI).

Mirrors o3d.pipelines.integration.ScalableTSDFVolume as used at
/root/reference/3d_model/reconstruct_rgbd.py:79-83,107,112.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import _lib


def checkpoint_info(path):
    """Header of a checkpoint written by TSDFVolume.save, validated on the host (no GPU needed)."""
    vl, tr = C.c_double(0), C.c_double(0)
    ct = C.c_int32(0)
    frames, nb = C.c_int64(0), C.c_int64(0)
    _lib.check(_lib.lib.otslam_checkpoint_info(os.fsencode(path), C.byref(vl), C.byref(tr), C.byref(ct), C.byref(frames), C.byref(nb)))
    return {"voxel_length": vl.value, "sdf_trunc": tr.value, "color": ct.value == _lib.COLOR_RGB8, "frames": frames.value,
            "n_blocks": nb.value}


def checkpoint_profile():
    """Timings of this thread's last save / load: device ms of kernels and of copies, ms in file I/O, wall ms."""
    out = np.zeros(4, np.float64)
    _lib.check(_lib.lib.otslam_checkpoint_profile(_lib.ptr(out)))
    return {"kernel_ms": float(out[0]), "copy_ms": float(out[1]), "file_ms": float(out[2]), "wall_ms": float(out[3])}


# Recommended coarse-to-fine setting of TSDFVolume.track (index = pyramid level, 0 = full resolution), chosen from
# tools/track_bench.py on a B200 (DESIGN.md §4 "Frame-to-model tracking"): vol.track(..., **TRACK_PYRAMID).
TRACK_PYRAMID = {"depth_diff": (0.07, 0.1, 0.2, 0.4), "max_iterations": (20, 10, 10, 10)}


class TSDFVolume:
    def __init__(self, voxel_length, sdf_trunc, color=True, device=0, slab=None):
        self.voxel_length, self.sdf_trunc, self.device = float(voxel_length), float(sdf_trunc), int(device)
        self._h = C.c_void_p()
        spec = None
        self.n_ranks = 1
        if slab is not None:
            axis, thickness, n_ranks, rank = (int(x) for x in slab[:4])
            halo = int(slab[4]) if len(slab) > 4 else 1
            spec = C.byref(_lib.SlabSpec(axis, thickness, n_ranks, rank, halo))
            self.n_ranks = max(1, n_ranks)
        _lib.check(_lib.lib.otslam_volume_create(self.voxel_length, self.sdf_trunc,
                                                 _lib.COLOR_RGB8 if color else _lib.COLOR_NONE, self.device, spec,
                                                 C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            self._detach_resident_mesh()
            _lib.lib.otslam_volume_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:       # noqa: BLE001 -- interpreter shutdown
            pass

    def reset(self):
        self._detach_resident_mesh()
        _lib.check(_lib.lib.otslam_volume_reset(self._h))

    # ---- the extracted mesh stays in HBM; a compat TriangleMesh may refer to it lazily ------------
    def _detach_resident_mesh(self):
        """The resident mesh is about to be replaced / freed: a lazy TriangleMesh still pointing at it
        downloads its arrays first."""
        ref = getattr(self, "_lazy_mesh", None)
        self._lazy_mesh = None
        m = ref() if ref is not None else None
        if m is not None:
            m._materialize()

    def extract_mesh_resident(self, owner=None):
        """extract_triangle_mesh + compute_vertex_normals on the device, result left in HBM.
        Returns (n_vertices, n_faces); `owner` (a lazy TriangleMesh) is told before the result dies."""
        self._detach_resident_mesh()
        nv, nf = C.c_int64(0), C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_extract_mesh(self._h, C.byref(nv), C.byref(nf)))
        if owner is not None:
            self._lazy_mesh = weakref.ref(owner)
        return nv.value, nf.value

    def mesh_download(self, nv, nf, normals=True):
        verts = np.empty((nv, 3), np.float64)
        cols = np.empty((nv, 3), np.float64)
        nrm = np.empty((nv, 3), np.float64) if normals else None
        faces = np.empty((nf, 3), np.int32)
        _lib.check(_lib.lib.otslam_volume_mesh_copy(self._h, _lib.ptr(verts), _lib.ptr(cols), _lib.ptr(nrm), _lib.ptr(faces), None))
        return verts, cols, nrm, faces

    def mesh_sample(self, n, seed, colors=True, normals=False):
        """sample_points_uniformly straight from the resident mesh (no mesh download / re-upload)."""
        op = np.empty((n, 3), np.float64)
        oc = np.empty((n, 3), np.float64) if colors else None
        on = np.empty((n, 3), np.float64) if normals else None
        _lib.check(_lib.lib.otslam_volume_mesh_sample(self._h, int(n), C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), _lib.ptr(op),
                                                      _lib.ptr(oc), _lib.ptr(on)))
        return op, oc, on

    def set_stream(self, cuda_stream):
        _lib.check(_lib.lib.otslam_volume_set_stream(self._h, C.c_void_p(int(cuda_stream) if cuda_stream else 0)))

    def wait_stream(self, cuda_stream):
        """Order the volume's streams after everything queued so far on `cuda_stream` (a raw cudaStream_t value; 0 = the
        legacy default stream): the contract for buffers in HBM that another stream produced (INTEGRATION.md)."""
        _lib.check(_lib.lib.otslam_volume_wait_stream(self._h, C.c_void_p(int(cuda_stream) if cuda_stream else 0)))

    def _after_torch_stream(self, tensor):
        """A CUDA torch tensor is about to be read by the volume's own streams: wait for torch's current stream."""
        import torch
        self.wait_stream(torch.cuda.current_stream(tensor.device).cuda_stream)

    def set_batch(self, n):
        _lib.check(_lib.lib.otslam_volume_set_batch(self._h, int(n)))

    def set_zsplit(self, zs):
        _lib.check(_lib.lib.otslam_volume_set_zsplit(self._h, int(zs)))

    def profile(self, enable=None):
        """Per-kernel CUDA-event totals {pack, alloc, integrate}: (ms, launches) accumulated so far.
        enable=True (re)starts recording from zero, False stops it, None only reads."""
        ms = np.zeros(4, np.float64)
        ln = np.zeros(4, np.int64)
        _lib.check(_lib.lib.otslam_volume_profile(self._h, -1 if enable is None else int(bool(enable)), _lib.ptr(ms), _lib.ptr(ln)))
        names = ("pack", "alloc", "integrate")
        return {k: (float(ms[i]), int(ln[i])) for i, k in enumerate(names)}

    @staticmethod
    def _intr(intr):
        return np.ascontiguousarray(intr, np.float64).reshape(4)

    def integrate_u16(self, depth, rgb, intr, extrinsic, depth_scale=1000.0, depth_trunc=3.0):
        d = np.ascontiguousarray(depth, np.uint16)
        c = None if rgb is None else np.ascontiguousarray(rgb, np.uint8)
        H, W = d.shape
        if c is not None and c.shape != (H, W, 3):
            raise RuntimeError("[ScalableTSDFVolume::Integrate] Unsupported image format.")
        k, e = self._intr(intr), np.ascontiguousarray(extrinsic, np.float64).reshape(16)
        _lib.check(_lib.lib.otslam_volume_integrate_u16(self._h, _lib.ptr(d), _lib.ptr(c), W, H, _lib.ptr(k), _lib.ptr(e),
                                                        float(depth_scale), float(depth_trunc)))

    def integrate_f32(self, depth_m, rgb, intr, extrinsic):
        d = np.ascontiguousarray(depth_m, np.float32)
        c = None if rgb is None else np.ascontiguousarray(rgb, np.uint8)
        H, W = d.shape
        if c is not None and c.shape != (H, W, 3):
            raise RuntimeError("[ScalableTSDFVolume::Integrate] Unsupported image format.")
        k, e = self._intr(intr), np.ascontiguousarray(extrinsic, np.float64).reshape(16)
        _lib.check(_lib.lib.otslam_volume_integrate_f32(self._h, _lib.ptr(d), _lib.ptr(c), W, H, _lib.ptr(k), _lib.ptr(e)))

    # ---- multi-object arena (config 3): several objects' volumes in one block hash, object id in the block key -----------
    def set_objects(self, n_objects):
        """Turn this (empty) volume into an arena of n_objects independent objects (otslam_volume_set_objects)."""
        _lib.check(_lib.lib.otslam_volume_set_objects(self._h, int(n_objects)))
        self.n_objects = int(n_objects)

    def select_object(self, obj):
        """The object that extraction / export_blocks / stats / num_blocks address from now on."""
        _lib.check(_lib.lib.otslam_volume_select_object(self._h, int(obj)))

    def integrate_batch(self, depth, rgb, intr, extrinsics, depth_scale=1000.0, depth_trunc=3.0, object_ids=None):
        """depth [n,H,W] u16, rgb [n,H,W,3] u8: numpy arrays / CPU torch tensors (host path, copies
        pipelined inside the call) or CUDA torch tensors (already resident in HBM).  object_ids [n] i32 (arenas only):
        the object each frame belongs to."""
        n, H, W = int(depth.shape[0]), int(depth.shape[1]), int(depth.shape[2])
        on_dev = hasattr(depth, "is_cuda") and depth.is_cuda
        if isinstance(depth, np.ndarray):
            depth = np.ascontiguousarray(depth, np.uint16)
            rgb = None if rgb is None else np.ascontiguousarray(rgb, np.uint8)
        else:
            assert depth.is_contiguous() and (rgb is None or rgb.is_contiguous())
            assert depth.element_size() == 2
            assert rgb is None or (rgb.element_size() == 1 and bool(rgb.is_cuda) == bool(on_dev))
        if rgb is not None and tuple(rgb.shape) != (n, H, W, 3):
            raise RuntimeError("[ScalableTSDFVolume::Integrate] Unsupported image format.")
        k = self._intr(intr)
        e = np.ascontiguousarray(extrinsics, np.float64).reshape(n, 16)
        if on_dev:
            self._after_torch_stream(depth)       # frames produced on a torch stream (copy, NCCL gather, rendering)
        if object_ids is not None:
            ids = np.ascontiguousarray(object_ids, np.int32).reshape(n)
            _lib.check(_lib.lib.otslam_volume_integrate_batch_objects(
                self._h, n, _lib.ptr(depth), _lib.ptr(rgb), W, H, _lib.ptr(k), _lib.ptr(e), _lib.ptr(ids), float(depth_scale),
                float(depth_trunc), _lib.MEM_DEVICE if on_dev else _lib.MEM_HOST))
            return
        _lib.check(_lib.lib.otslam_volume_integrate_batch(self._h, n, _lib.ptr(depth), _lib.ptr(rgb), W, H, _lib.ptr(k),
                                                          _lib.ptr(e), float(depth_scale), float(depth_trunc),
                                                          _lib.MEM_DEVICE if on_dev else _lib.MEM_HOST))

    def num_blocks(self):
        n = C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_num_blocks(self._h, C.byref(n)))
        return n.value

    def export_blocks(self, color=True):
        n = self.num_blocks()
        keys = np.empty((n, 3), np.int32)
        tsdf = np.empty((n, 4096), np.float32)
        weight = np.empty((n, 4096), np.float32)
        col = np.empty((n, 4096, 3), np.float32) if color else None
        _lib.check(_lib.lib.otslam_volume_export_blocks(self._h, _lib.ptr(keys), _lib.ptr(tsdf), _lib.ptr(weight), _lib.ptr(col)))
        return keys, tsdf, weight, col

    def stats(self):
        nb, ws, no = C.c_int64(0), C.c_uint64(0), C.c_uint64(0)
        _lib.check(_lib.lib.otslam_volume_stats(self._h, C.byref(nb), C.byref(ws), C.byref(no)))
        return {"n_blocks": nb.value, "weight_sum": ws.value, "n_observed": no.value}

    # ---- checkpoints (otslam_volume_save / _load; format in DESIGN.md §4) ---------------------------------------------
    def save(self, path):
        """Write this volume's blocks to `path` (a slab rank: its owned blocks; an arena: the selected object)."""
        _lib.check(_lib.lib.otslam_volume_save(self._h, os.fsencode(path)))

    def load(self, paths):
        """Add the blocks of one checkpoint file or of several part files (e.g. every rank's part of a sharded volume);
        a slab rank keeps the blocks its spec keeps.  Each file is checked completely before any of its blocks is
        inserted: a bad file raises and leaves the volume as it was.  Returns the number of blocks added."""
        self._detach_resident_mesh()
        total = 0
        for p in [paths] if isinstance(paths, (str, bytes, os.PathLike)) else paths:
            n = C.c_int64(0)
            _lib.check(_lib.lib.otslam_volume_load(self._h, os.fsencode(p), C.byref(n)))
            total += n.value
        return total

    def halo_export(self):
        """(keys [n,4] i32 = block key + piece kind, dest rank [n] i32, pieces [n,4096] u8) for the slab halo exchange."""
        n = C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_halo_export(self._h, C.byref(n), None, None, None))
        keys = np.empty((n.value, 4), np.int32)
        dest = np.empty(n.value, np.int32)
        planes = np.empty((n.value, 4096), np.uint8)
        if n.value:
            _lib.check(_lib.lib.otslam_volume_halo_export(self._h, C.byref(n), _lib.ptr(keys), _lib.ptr(dest), _lib.ptr(planes)))
        return keys, dest, planes

    def halo_import(self, keys, planes):
        """keys [n,4] i32 / planes [n,4096] u8: numpy arrays or (contiguous) torch tensors, host or CUDA."""
        if isinstance(keys, np.ndarray):
            keys = np.ascontiguousarray(keys, np.int32)
            planes = np.ascontiguousarray(planes, np.uint8)
        else:
            assert keys.is_contiguous() and planes.is_contiguous() and keys.element_size() == 4 and planes.element_size() == 1
            if keys.is_cuda:
                self._after_torch_stream(keys)    # e.g. pieces that an NCCL recv just wrote
        _lib.check(_lib.lib.otslam_volume_halo_import(self._h, len(keys), _lib.ptr(keys), _lib.ptr(planes)))

    # ---- device-resident forms for the multi-GPU exchange (slab.py): torch tensors on this volume's GPU, no host copy
    def halo_pack_tensors(self):
        """(keys [n,4] i32, planes [n,4096] u8, pieces per destination rank [n_ranks]) -- packed in HBM, grouped by
        destination rank, ready for ncclSend."""
        import torch
        n = C.c_int64(0)
        counts = np.zeros(self.n_ranks, np.int64)
        _lib.check(_lib.lib.otslam_volume_halo_pack(self._h, C.byref(n), _lib.ptr(counts)))
        dev = torch.device("cuda", self.device)
        keys = torch.empty((n.value, 4), dtype=torch.int32, device=dev)
        planes = torch.empty((n.value, 4096), dtype=torch.uint8, device=dev)
        if n.value:
            _lib.check(_lib.lib.otslam_volume_halo_fetch(self._h, _lib.ptr(keys), _lib.ptr(planes)))
        return keys, planes, counts

    def extract_point_cloud_tensors(self):
        """extract_point_cloud() with the result as torch CUDA tensors (points, colours f64 [n,3]; edge keys i32 [n,4])."""
        import torch
        n = C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_extract_points(self._h, C.byref(n)))
        dev = torch.device("cuda", self.device)
        pts = torch.empty((n.value, 3), dtype=torch.float64, device=dev)
        cols = torch.empty((n.value, 3), dtype=torch.float64, device=dev)
        ek = torch.empty((n.value, 4), dtype=torch.int32, device=dev)
        _lib.check(_lib.lib.otslam_volume_points_copy(self._h, _lib.ptr(pts), _lib.ptr(cols), _lib.ptr(ek)))
        return pts, cols, ek

    def extract_mesh_tensors(self):
        """extract_triangle_mesh() as torch CUDA tensors (vertices, colours f64 [nv,3]; faces i32 [nf,3]; edge keys i32 [nv,4])."""
        import torch
        self._detach_resident_mesh()
        nv, nf = C.c_int64(0), C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_extract_mesh(self._h, C.byref(nv), C.byref(nf)))
        dev = torch.device("cuda", self.device)
        verts = torch.empty((nv.value, 3), dtype=torch.float64, device=dev)
        cols = torch.empty((nv.value, 3), dtype=torch.float64, device=dev)
        faces = torch.empty((nf.value, 3), dtype=torch.int32, device=dev)
        ek = torch.empty((nv.value, 4), dtype=torch.int32, device=dev)
        _lib.check(_lib.lib.otslam_volume_mesh_copy(self._h, _lib.ptr(verts), _lib.ptr(cols), None, _lib.ptr(faces), _lib.ptr(ek)))
        return verts, cols, faces, ek

    def extract_triangle_mesh(self, normals=True):
        self._detach_resident_mesh()
        nv, nf = C.c_int64(0), C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_extract_mesh(self._h, C.byref(nv), C.byref(nf)))
        verts = np.empty((nv.value, 3), np.float64)
        cols = np.empty((nv.value, 3), np.float64)
        nrm = np.empty((nv.value, 3), np.float64) if normals else None
        faces = np.empty((nf.value, 3), np.int32)
        ek = np.empty((nv.value, 4), np.int32)
        _lib.check(_lib.lib.otslam_volume_mesh_copy(self._h, _lib.ptr(verts), _lib.ptr(cols), _lib.ptr(nrm), _lib.ptr(faces), _lib.ptr(ek)))
        return verts, cols, nrm, faces, ek

    def extract_point_cloud(self, normals=False):
        """(points, colours, edge keys[, normals]) of volume.extract_point_cloud(); normals = TSDF gradient at the points."""
        n = C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_extract_points(self._h, C.byref(n)))
        pts = np.empty((n.value, 3), np.float64)
        cols = np.empty((n.value, 3), np.float64)
        ek = np.empty((n.value, 4), np.int32)
        _lib.check(_lib.lib.otslam_volume_points_copy(self._h, _lib.ptr(pts), _lib.ptr(cols), _lib.ptr(ek)))
        if not normals:
            return pts, cols, ek
        nrm = np.empty((n.value, 3), np.float64)
        if n.value:
            _lib.check(_lib.lib.otslam_volume_points_normals(self._h, _lib.ptr(nrm)))
        return pts, cols, ek, nrm

    # ---- ray casting (otslam_volume_raycast; arithmetic in DESIGN.md §4 "Ray casting") --------------------------------
    RAY_CAST_ATTRIBUTES = ("depth", "color", "normal", "vertex")

    def _ray_cast(self, intr, extrinsics, width, height, depth_min, depth_max, attributes, alloc):
        attributes = tuple(attributes)
        bad = [a for a in attributes if a not in self.RAY_CAST_ATTRIBUTES]
        if bad:
            raise ValueError(f"unknown ray-cast attributes {bad}; choose from {self.RAY_CAST_ATTRIBUTES}")
        e = np.ascontiguousarray(extrinsics, np.float64)
        single = e.shape == (4, 4)
        e = e.reshape(-1, 16)
        n, H, W = len(e), int(height), int(width)
        shapes = {"depth": ((n, H, W), "f4"), "vertex": ((n, H, W, 3), "f4"), "normal": ((n, H, W, 3), "f4"),
                  "color": ((n, H, W, 3), "u1")}
        out = {a: alloc(*shapes[a]) for a in attributes}
        hits = C.c_int64(0)
        _lib.check(_lib.lib.otslam_volume_raycast(self._h, n, W, H, _lib.ptr(self._intr(intr)), _lib.ptr(e), float(depth_min),
                                                  float(depth_max), _lib.ptr(out.get("depth")), _lib.ptr(out.get("vertex")),
                                                  _lib.ptr(out.get("normal")), _lib.ptr(out.get("color")), C.byref(hits)))
        if single:
            out = {k: a[0] for k, a in out.items()}
        return out, hits.value

    def ray_cast(self, intr, extrinsics, width, height, depth_min=0.1, depth_max=3.0,
                 attributes=("depth", "color", "normal", "vertex")):
        """Render the volume from camera poses (after Open3D's VoxelBlockGrid.ray_cast).  intr = (fx, fy, cx, cy);
        extrinsics = one world->camera 4x4 (unbatched results) or [n,4,4].  Returns a dict of NumPy arrays: depth [n,H,W]
        f32 metres (camera z), vertex / normal [n,H,W,3] f32 world, color [n,H,W,3] u8; 0 where a ray hits nothing.  The
        volume is only read."""
        out, _ = self._ray_cast(intr, extrinsics, width, height, depth_min, depth_max, attributes,
                                lambda shape, dt: np.empty(shape, dt))
        return out

    def ray_cast_tensors(self, intr, extrinsics, width, height, depth_min=0.1, depth_max=3.0,
                         attributes=("depth", "color", "normal", "vertex")):
        """ray_cast() with the maps rendered straight into torch CUDA tensors on this volume's GPU (no host copy).  The
        tensors are complete when this returns."""
        import torch
        dev = torch.device("cuda", self.device)
        dts = {"f4": torch.float32, "u1": torch.uint8}
        self.wait_stream(torch.cuda.current_stream(dev).cuda_stream)   # the outputs may reuse memory torch still uses
        out, _ = self._ray_cast(intr, extrinsics, width, height, depth_min, depth_max, attributes,
                                lambda shape, dt: torch.empty(shape, dtype=dts[dt], device=dev))
        return out

    # ---- frame-to-model tracking (otslam_volume_track; DESIGN.md §4 "Frame-to-model tracking") ---------------------------
    def track(self, depth, intr, init_extrinsics, depth_scale=1000.0, depth_min=0.1, depth_max=3.0, depth_diff=0.07,
              max_iterations=20):
        """Refine the world->camera poses of raw u16 depth frames against this volume by point-to-plane ICP on its
        ray-cast model (after Open3D's tensor SLAM Model.track_frame_to_model).  depth: a NumPy array or a CUDA torch
        tensor, [n,H,W] or [H,W]; intr = (fx, fy, cx, cy); init_extrinsics [n,4,4] or one 4x4.  Each frame is tracked
        independently against the volume as it is; the volume is only read.  Returns a dict: extrinsic [n,4,4] (refined),
        status [n] (0 converged, 1 reached max_iterations, 2 fewer than 64 inliers, 3 degenerate; 2 and 3 keep the last
        pose), iterations [n], fitness [n] (inliers / valid pixels) and inlier_rmse [n] (metres); unbatched for one
        [H,W] frame.

        depth_diff and max_iterations may each be a sequence of per-level values (index = level, 0 = full resolution):
        the frames are then tracked coarse to fine over a depth pyramid of that many levels (1..4), and a scalar beside a
        sequence applies to every level.  status is then level 0's and iterations the sum over the levels.
        TRACK_PYRAMID is the recommended setting for starts a few centimetres and degrees off."""
        levels = {len(x) for x in (depth_diff, max_iterations) if np.ndim(x) > 0}
        if len(levels) > 1:
            raise ValueError(f"depth_diff and max_iterations give different level counts {sorted(levels)}")
        on_dev = hasattr(depth, "is_cuda") and depth.is_cuda
        if on_dev:
            assert depth.is_contiguous() and depth.element_size() == 2
        else:
            depth = np.ascontiguousarray(depth, np.uint16)
        single = depth.ndim == 2
        if single:
            depth = depth[None]
        n, H, W = int(depth.shape[0]), int(depth.shape[1]), int(depth.shape[2])
        e = np.ascontiguousarray(init_extrinsics, np.float64).reshape(n, 16)
        out = {"extrinsic": np.empty((n, 4, 4)), "status": np.empty(n, np.int32), "iterations": np.empty(n, np.int32),
               "fitness": np.empty(n), "inlier_rmse": np.empty(n)}
        if on_dev:
            self._after_torch_stream(depth)
        outs = (_lib.ptr(out["extrinsic"]), _lib.ptr(out["status"]), _lib.ptr(out["iterations"]), _lib.ptr(out["fitness"]),
                _lib.ptr(out["inlier_rmse"]), _lib.MEM_DEVICE if on_dev else _lib.MEM_HOST)
        k = self._intr(intr)                # kept alive across the call: only its address goes into `head`
        head = (self._h, n, _lib.ptr(depth), W, H, _lib.ptr(k), _lib.ptr(e), float(depth_scale), float(depth_min),
                float(depth_max))
        if levels:
            L = levels.pop()
            dd = np.ascontiguousarray(np.broadcast_to(np.asarray(depth_diff, np.float64), (L,)))
            mi = np.ascontiguousarray(np.broadcast_to(np.asarray(max_iterations, np.int32), (L,)))
            _lib.check(_lib.lib.otslam_volume_track_pyramid(*head, L, _lib.ptr(dd), _lib.ptr(mi), *outs))
        else:
            _lib.check(_lib.lib.otslam_volume_track(*head, float(depth_diff), int(max_iterations), *outs))
        if single:
            out = {k: a[0] for k, a in out.items()}
        return out




class ArenaView:
    """One object of a multi-object arena, with the interface of a TSDFVolume of its own: what the compat
    ScalableTSDFVolume of a config-3 job is re-bound to after pipeline.integrate_many (the objects' frames went through
    ONE work list / integration launch per batch; extraction, export and statistics address this object only)."""

    def __init__(self, arena, obj):
        self._arena, self._obj = arena, int(obj)
        self.voxel_length, self.sdf_trunc, self.device = arena.voxel_length, arena.sdf_trunc, arena.device

    def __getattr__(self, name):
        attr = getattr(self._arena, name)
        if not callable(attr):
            return attr

        def call(*a, **k):
            self._arena.select_object(self._obj)
            return attr(*a, **k)
        return call

    def integrate_batch(self, depth, rgb, intr, extrinsics, depth_scale=1000.0, depth_trunc=3.0):
        self._arena.integrate_batch(depth, rgb, intr, extrinsics, depth_scale, depth_trunc,
                                    object_ids=np.full(int(depth.shape[0]), self._obj, np.int32))

    def integrate_u16(self, depth, rgb, intr, extrinsic, depth_scale=1000.0, depth_trunc=3.0):
        d = np.ascontiguousarray(depth, np.uint16)[None]
        c = None if rgb is None else np.ascontiguousarray(rgb, np.uint8)[None]
        self.integrate_batch(d, c, intr, np.asarray(extrinsic, np.float64).reshape(1, 4, 4), depth_scale, depth_trunc)

    def integrate_f32(self, *a, **k):
        raise RuntimeError("an arena object integrates raw u16 depth only")

    def reset(self):
        raise RuntimeError("objects of a multi-object arena cannot be reset individually")

    def close(self):
        pass            # the arena lives as long as one of its views does
