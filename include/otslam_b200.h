/* otslam_b200.h -- C ABI of the B200-native RGB-D reconstruction hot path.
 *
 * The reference (TakiRyo/object-triggered-3D-SLAM) has no FFI of its own for this path: its four
 * scripts reach the arithmetic through the `open3d` Python package.  Each entry point below names
 * the reference call site (file:line under /root/reference) whose work it replaces; the binding a
 * maintainer adds is the ctypes shim shown in INTEGRATION.md (shipped as
 * object-triggered-3d-slam_b200/_lib.py + o3d_compat/).
 *
 * Conventions: plain pointers and sizes only; every function returns 0 (OTSLAM_OK) or a negative
 * status, with a message available from otslam_last_error() (thread-local).  Matrices are 4x4
 * row-major FP64.  Unless a function says "device", pointers are HOST pointers and the call is
 * synchronous (results visible on return).  There is no CPU fallback: every call fails with
 * OTSLAM_ERR_CUDA when no sm_100 GPU is usable.
 */
#ifndef OTSLAM_B200_H
#define OTSLAM_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define OTSLAM_OK 0
#define OTSLAM_ERR_INVALID (-1)   /* bad argument */
#define OTSLAM_ERR_FORMAT (-2)    /* "[ScalableTSDFVolume::Integrate] Unsupported image format."; malformed checkpoint file */
#define OTSLAM_ERR_CUDA (-3)      /* CUDA runtime / no device */
#define OTSLAM_ERR_NOMEM (-4)     /* device memory exhausted */
#define OTSLAM_ERR_OVERFLOW (-5)  /* per-voxel frame-count limit (65535) or key range exceeded */

#define OTSLAM_MEM_HOST 0
#define OTSLAM_MEM_DEVICE 1

#define OTSLAM_COLOR_NONE 0       /* TSDFVolumeColorType.NoColor */
#define OTSLAM_COLOR_RGB8 1       /* TSDFVolumeColorType.RGB8 (reconstruct_rgbd.py:82) */

typedef struct otslam_volume otslam_volume;

/* Spatial slab sharding of the block grid across the GPUs of one box (SURVEY 8e): a block is owned by rank
 * (floor(c / thickness) mod n_ranks), where c is its key on `axis` (0 / 1 / 2) or kx + ky for axis = 3
 * ("diagonal" slabs: axis-aligned walls and floors spread over all ranks; needs halo = 0).  Extraction needs
 * the +1 neighbour voxels of owned blocks: halo = 1 integrates the +1 neighbour blocks redundantly on this rank
 * (no exchange at all); halo = 0 integrates owned blocks only and the ranks exchange boundary pieces once
 * before extraction (otslam_volume_halo_export / _import).  n_ranks == 1: keep everything. */
typedef struct {
    int32_t axis, thickness, n_ranks, rank, halo;
} otslam_slab_spec;

const char* otslam_last_error(void);
int otslam_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py "gpu_launches") */
int64_t otslam_launch_count(void);
/* device-side duration (CUDA events, ms) of the kernel section of the last stateless operator or
 * extraction call made by this thread, host<->device copies excluded; -1 if none (bench.py's
 * post-stage rooflines) */
double otslam_last_op_device_ms(void);
/* operators keep their device temporaries in a per-device cache (cudaMalloc / cudaFree cost more
 * than their kernels); this returns the cached blocks to the driver */
int otslam_trim_scratch(void);
/* page-locked host staging memory for the frame loop's inputs (otslam_volume_integrate_batch copies from pinned
 * memory at PCIe speed and truly asynchronously; from pageable memory the driver stages through its own buffer) */
int otslam_host_alloc(uint64_t bytes, void** out);
int otslam_host_free(void* p);

/* device self-test of the integration kernel's shared-reciprocal division and ALU floor against
 * the IEEE intrinsics (__fdiv_rn, F2I) on n pseudo-random operand triples; *mismatches must be 0. */
int otslam_selftest_division(uint64_t n, uint64_t seed, uint64_t* mismatches, int device);

/* device self-test of the parallel sequential-order FP64 accumulation (csrc/ordered_sum.cu) against
 * the scalar left-to-right loop on n generated terms: totals and every prefix must agree bit for bit.
 * pattern 0 = triangle-area-like, 1 = 2^-64..2^64 magnitudes, 2 = coarse grid (frequent exact ties),
 * 3 = zeros and jumps, 4 = with negative / infinite terms. */
int otslam_selftest_ordered_sum(int64_t n, uint64_t seed, int pattern, uint64_t* mismatches, int device);

/* ---- volume life cycle: o3d.pipelines.integration.ScalableTSDFVolume(voxel_length, sdf_trunc,
 *      color_type) (3d_model/reconstruct_rgbd.py:79-83); volume_unit_resolution = 16,
 *      depth_sampling_stride = 4 as in Open3D. `slab` may be NULL.  A failed allocation returns OTSLAM_ERR_NOMEM,
 *      as in every other entry point. */
int otslam_volume_create(double voxel_length, double sdf_trunc, int color_type, int device,
                         const otslam_slab_spec* slab, otslam_volume** out);
int otslam_volume_destroy(otslam_volume* v);
int otslam_volume_reset(otslam_volume* v);                       /* ScalableTSDFVolume.reset() */
/* run this volume's kernels on a caller-owned cudaStream_t (e.g. torch's current stream) */
int otslam_volume_set_stream(otslam_volume* v, void* cuda_stream);
/* Stream contract for DEVICE buffers (OTSLAM_MEM_DEVICE frames, device halo pieces): the volume works on its own
 * non-blocking streams, so buffers produced on another stream (a torch stream, an NCCL collective) must either be
 * complete (that stream synchronised) or ordered with this call: everything queued on `producer_stream` (NULL = the
 * legacy default stream) so far will finish before any work the volume queues afterwards. */
int otslam_volume_wait_stream(otslam_volume* v, void* producer_stream);
/* frames fused per block residency in integrate_batch (1..32, default 32) */
int otslam_volume_set_batch(otslam_volume* v, int frames_per_batch);

/* CTAs per block along z in the integration kernel: 0 = default (2), 1, 2, 4 or 8; results are bit-identical for
 * every setting */
int otslam_volume_set_zsplit(otslam_volume* v, int zsplit);

/* kernel timing with CUDA events on the volume's stream (bench.py roofline): enable > 0 switches
 * recording on and zeroes the accumulators, 0 switches it off, < 0 only reads; out_ms /
 * out_launches (nullable, 4 entries: 0 = depth pack, 1 = block allocation, 2 = integration,
 * 3 = reserved) return the totals accumulated before this call. */
int otslam_volume_profile(otslam_volume* v, int enable, double* out_ms, int64_t* out_launches);

/* ---- per-frame integration: RGBDImage.create_from_color_and_depth(depth_scale, depth_trunc,
 *      convert_rgb_to_intensity=False) + volume.integrate(rgbd, intrinsic, extrinsic)
 *      (3d_model/reconstruct_rgbd.py:99-107).  depth: H*W u16 (raw units), rgb: H*W*3 u8,
 *      intr = {fx, fy, cx, cy}, extrinsic = world->camera. */
int otslam_volume_integrate_u16(otslam_volume* v, const uint16_t* depth, const uint8_t* rgb, int width, int height,
                                const double intr[4], const double extrinsic[16], double depth_scale,
                                double depth_trunc);
/* same with an already converted f32 metre depth image (what RGBDImage.depth holds) */
int otslam_volume_integrate_f32(otslam_volume* v, const float* depth_m, const uint8_t* rgb, int width, int height,
                                const double intr[4], const double extrinsic[16]);
/* the whole frame loop of reconstruct_object() (reconstruct_rgbd.py:86-109) in one call:
 * n frames, frame order preserved; depth [n][H][W], rgb [n][H][W][3], extrinsics [n][16].
 * memory = OTSLAM_MEM_HOST (pinned or pageable; copies are pipelined with compute) or
 * OTSLAM_MEM_DEVICE (buffers already resident in HBM). */
int otslam_volume_integrate_batch(otslam_volume* v, int n_frames, const uint16_t* depth, const uint8_t* rgb,
                                  int width, int height, const double intr[4], const double* extrinsics,
                                  double depth_scale, double depth_trunc, int memory);

/* ---- multi-object arenas: BASELINE configs[2] = 3d_model/multi_reconstruct_rgbd_filter.py:139-145 (several objects, each its
 *      own ScalableTSDFVolume, reconstructed one after the other).  An arena holds up to 8 such volumes in ONE block hash /
 *      pool with the object id folded into the block key, so that a batch of frames drawn from several objects is one work
 *      list and one integration launch over the union of their touched blocks (small per-object volumes cannot fill 148 SMs
 *      on their own).  set_objects on an empty, un-sharded volume; object_ids [n_frames] says which object each frame
 *      belongs to (frame order is preserved per object, which is all the running means depend on); select_object chooses
 *      the object that extract_mesh / extract_points / export_blocks / num_blocks / stats address.  Every object's result
 *      is bit-identical to integrating its frames into a volume of its own.  |block x key| < 2^17 inside an arena. */
int otslam_volume_set_objects(otslam_volume* v, int n_objects);
int otslam_volume_select_object(otslam_volume* v, int object_id);
int otslam_volume_integrate_batch_objects(otslam_volume* v, int n_frames, const uint16_t* depth, const uint8_t* rgb,
                                          int width, int height, const double intr[4], const double* extrinsics,
                                          const int32_t* object_ids, double depth_scale, double depth_trunc, int memory);

/* ---- inspection / checkpoint (parity dumps) */
int otslam_volume_num_blocks(otslam_volume* v, int64_t* n_blocks);
/* blocks sorted lexicographically by key; voxel index x*256+y*16+z; colour on the 0..255 scale.
 * keys [n][3], tsdf/weight [n][4096], color [n][4096][3]; any pointer may be NULL. */
int otslam_volume_export_blocks(otslam_volume* v, int32_t* keys, float* tsdf, float* weight, float* color);
/* sum of all voxel weights (== number of voxel updates since reset) and voxels with weight > 0 */
int otslam_volume_stats(otslam_volume* v, int64_t* n_blocks, uint64_t* weight_sum, uint64_t* n_observed);

/* ---- checkpoints (file format version 1, DESIGN.md §4): a volume's voxel records written verbatim, so that a loaded
 *      volume continues integrating bit for bit as if it had never been saved.
 * save writes the blocks this volume is responsible for: all blocks of a plain volume; the OWNED blocks of a slab rank
 * (halo-imported pieces and halo = 1 neighbour blocks are left out, so the part files of N ranks partition the volume);
 * the selected object of an arena, with the object's key offset removed.  The file is written under a temporary name,
 * synced and renamed.
 * load adds a file's blocks to a volume (which may hold blocks already): voxel_length / sdf_trunc / color_type must equal
 * the volume's bit for bit; a slab rank keeps what its spec keeps (owned blocks, plus the +1 neighbours when halo = 1), so
 * loading every part file of N ranks into M ranks reshards the volume; an arena loads into the selected object
 * (|kx| >= 2^17: OTSLAM_ERR_OVERFLOW).  The frame count becomes max(volume's, file's).  Every check (header, size, key order
 * and duplicates, keys already present, checksums, record validity) runs before anything is inserted: on any error the
 * volume is unchanged.  Malformed files: OTSLAM_ERR_FORMAT.  *n_loaded (nullable) = blocks added. */
int otslam_volume_save(otslam_volume* v, const char* path);
int otslam_volume_load(otslam_volume* v, const char* path, int64_t* n_loaded);
/* header of a checkpoint, validated on the host (no GPU needed); outputs nullable */
int otslam_checkpoint_info(const char* path, double* voxel_length, double* sdf_trunc, int32_t* color_type, int64_t* frames,
                           int64_t* n_blocks);
/* this thread's last save / load: [0] device ms of its kernels (save: gather + checksum; load: key filter + verify +
 * insert), [1] device ms of its host<->device copies, [2] ms spent in file reads / writes / fsync (summed over the I/O
 * thread's calls), [3] wall ms of the whole call */
int otslam_checkpoint_profile(double out[4]);

/* ---- halo exchange for slab.halo == 0 (the path's only inter-GPU exchange of voxel data besides the final
 *      gather): export the low-side boundary pieces (256 voxel records of 16 bytes each, opaque) of every
 *      owned block whose -axis neighbour block belongs to another rank, with that rank as destination.
 *      keys [n][4] = block key + piece kind: 0 / 1 / 2 = the plane x / y / z = 0, 3 = the column x = y = 0.
 *      Axis slabs send one plane per boundary block; diagonal slabs send the x and the y plane to the owner
 *      of the -x / -y neighbours and the column to the owner of the -x-y neighbour.  import inserts received
 *      pieces into (non-owned) blocks.  Call export with NULL buffers to get the count. */
int otslam_volume_halo_export(otslam_volume* v, int64_t* n, int32_t* keys, int32_t* dest_rank, void* planes);
/* keys / planes may be HOST or DEVICE pointers (unified addressing); device sources must be complete on the volume's
 * stream (otslam_volume_wait_stream) or on a synchronised stream */
int otslam_volume_halo_import(otslam_volume* v, int64_t n, const int32_t* keys, const void* planes);
/* The device-resident form of the export, for the NCCL exchange (no host copy of voxel data): pack selects and packs the
 * pieces inside HBM, grouped by destination rank ((key, kind) order inside a group) and returns the total and the
 * per-destination counts (counts_per_rank [n_ranks], nullable); fetch copies the packed keys [n][4] / planes [n][4096]
 * into caller buffers, which may be DEVICE pointers (e.g. torch CUDA tensors handed to ncclSend) or host pointers. */
int otslam_volume_halo_pack(otslam_volume* v, int64_t* n_pieces, int64_t* counts_per_rank);
int otslam_volume_halo_fetch(otslam_volume* v, int32_t* keys, void* planes);

/* ---- surface extraction: volume.extract_triangle_mesh() (reconstruct_rgbd.py:112) followed by
 *      mesh.compute_vertex_normals() (reconstruct_rgbd.py:113).  extract runs the kernels and
 *      keeps the result on the device; copy fetches it.  edge_keys [nv][4] = global voxel (X,Y,Z)
 *      + axis of each vertex's lattice edge (canonical order for comparisons); nullable outputs. */
int otslam_volume_extract_mesh(otslam_volume* v, int64_t* n_vertices, int64_t* n_faces);
int otslam_volume_mesh_copy(otslam_volume* v, double* vertices, double* colors, double* normals, int32_t* faces,
                            int32_t* edge_keys);   /* destinations: host or device pointers */
/* mesh.sample_points_uniformly(n) (reconstruct_rgbd_filter.py:123) straight from the mesh the last
 * otslam_volume_extract_mesh left in HBM: no download + re-upload of the (often ~100 MB) mesh when the
 * caller only wants the samples.  Same arithmetic and sample order as otslam_mesh_sample_uniform;
 * out_colors / out_normals nullable. */
int otslam_volume_mesh_sample(otslam_volume* v, int64_t n_samples, uint64_t seed, double* out_points,
                              double* out_colors, double* out_normals);
/* volume.extract_point_cloud() (named by north_star; zero crossings along +x/+y/+z) */
int otslam_volume_extract_points(otslam_volume* v, int64_t* n_points);
int otslam_volume_points_copy(otslam_volume* v, double* points, double* colors, int32_t* edge_keys);   /* host or device */
/* the normals extract_point_cloud() attaches: normalised central differences (+-0.99 voxel) of the trilinearly interpolated
 * TSDF at every point of the last extraction (Open3D GetNormalAt / GetTSDFAt); normals [n][3], host or device */
int otslam_volume_points_normals(otslam_volume* v, double* normals);

/* ---- ray casting: render the volume from n camera poses (the ray-cast half of a KinectFusion-style system; interface
 *      after Open3D's tensor VoxelBlockGrid.ray_cast, arithmetic in DESIGN.md §4 "Ray casting").  Pixel (u, v) of view i
 *      follows the ray that integration projects onto (u, v), from the camera centre of inverse4(extrinsics[i]); depth is
 *      the camera z of the first front-face (+ -> -) zero crossing of two consecutive observed samples with
 *      depth_min <= t < depth_max.  Outputs (each nullable, host or device pointer): depth [n][H][W] f32 metres, vertex and
 *      normal [n][H][W][3] f32 world (normal = GetNormalAt at the vertex, as extract_point_cloud's), color [n][H][W][3] u8
 *      (trilinear over the observed voxels, renormalised; 0 for a NoColor volume); 0 where a ray hits nothing.
 *      *n_hits (nullable) = pixels with a hit.  An arena renders its selected object only; slab-sharded volumes are refused
 *      (load the part files into one volume).  The volume is read only: no result, block list or epoch changes.  Bad
 *      arguments give OTSLAM_ERR_INVALID before any CUDA call.  otslam_last_op_device_ms() = device ms of the render. */
int otslam_volume_raycast(otslam_volume* v, int n_views, int width, int height, const double intr[4],
                          const double* extrinsics, double depth_min, double depth_max, float* depth, float* vertex,
                          float* normal, uint8_t* color, int64_t* n_hits);

/* ---- frame-to-model tracking: refine the world->camera poses of n depth frames against the volume by projective
 *      point-to-plane ICP on its ray-cast model (interface after Open3D's tensor SLAM Model.track_frame_to_model,
 *      arithmetic in DESIGN.md §4 "Frame-to-model tracking").  Each frame is tracked independently against the volume as
 *      it is: its model (vertex and normal maps over [depth_min, depth_max)) is rendered once at init_extrinsics[i], and
 *      its pixels (depth = raw / depth_scale, valid when > 0 and < depth_max) are associated projectively into that view
 *      and gated by depth_diff metres.  depth [n][H][W] u16 in `memory` (OTSLAM_MEM_HOST or OTSLAM_MEM_DEVICE, as
 *      integrate_batch); init_extrinsics [n][16] on the host.  Host outputs (all but extrinsics_out nullable):
 *      extrinsics_out [n][16] refined world->camera; status [n] 0 = converged, 1 = reached max_iterations (1..100),
 *      2 = fewer than 64 inliers, 3 = degenerate system (2 and 3 keep the last pose); iterations [n]; fitness [n] =
 *      inliers / valid pixels and inlier_rmse [n] = point-to-plane RMS over the inliers, both at the returned pose.  An
 *      arena tracks against its selected object; slab-sharded volumes are refused (load the part files into one volume).
 *      The volume is read only.  Bad arguments give OTSLAM_ERR_INVALID before any CUDA call.
 *      otslam_last_op_device_ms() = device ms of the whole call. */
int otslam_volume_track(otslam_volume* v, int n_frames, const uint16_t* depth, int width, int height, const double intr[4],
                        const double* init_extrinsics, double depth_scale, double depth_min, double depth_max,
                        double depth_diff, int max_iterations, double* extrinsics_out, int32_t* status,
                        int32_t* iterations, double* fitness, double* inlier_rmse, int memory);
/* ---- coarse-to-fine frame-to-model tracking: otslam_volume_track over a depth pyramid of n_levels (1..4) levels, index
 *      = level, 0 = full resolution.  Level l + 1 halves level l (an odd last column or row dropped; intrinsics fx / 2,
 *      fy / 2, (cx - 0.5) / 2, (cy - 0.5) / 2); a coarse pixel averages the valid depths of its 2x2 block that lie within
 *      4 voxels of the block's nearest.  Each level has its own model render at init_extrinsics[i], its own gate
 *      depth_diff[l] (metres, finite and > 0) and its own max_iterations[l] (1..100).  Levels run from the coarsest to 0,
 *      each from the pose the coarser level returned, whatever its status.  status is level 0's; iterations are summed
 *      over the levels; fitness and inlier_rmse are level 0's at the returned pose.  With more than one level the
 *      coarsest must be at least 16x8 pixels.  n_levels = 1 is otslam_volume_track, bit for bit.  Other arguments,
 *      outputs and checks as otslam_volume_track. */
int otslam_volume_track_pyramid(otslam_volume* v, int n_frames, const uint16_t* depth, int width, int height,
                                const double intr[4], const double* init_extrinsics, double depth_scale,
                                double depth_min, double depth_max, int n_levels, const double* depth_diff,
                                const int32_t* max_iterations, double* extrinsics_out, int32_t* status,
                                int32_t* iterations, double* fitness, double* inlier_rmse, int memory);

/* ---- stateless image / cloud operators.  Every pointer argument may be a HOST pointer or a DEVICE pointer of `device`
 *      (unified addressing; the copies inside become device-to-device): a caller that keeps its clouds in HBM between
 *      operators (otslam_b200/cloud.py: DeviceCloud) never crosses PCIe.  Device inputs must be complete (producer stream
 *      synchronised); results are complete on return. */
/* RGBDImage.create_from_color_and_depth depth half (reconstruct_rgbd.py:99-104) */
int otslam_depth_convert(const uint16_t* depth, int64_t n, double depth_scale, double depth_trunc, float* out,
                         int device);
/* PointCloud.create_from_rgbd_image (3d_model/check_one_frame.py:27); points/colors sized H*W*3 */
int otslam_backproject_rgbd(const float* depth_m, const uint8_t* rgb, int width, int height, const double intr[4],
                            const double extrinsic[16], double* points, double* colors, int64_t* n_points,
                            int device);
/* TriangleMesh.compute_vertex_normals (reconstruct_rgbd.py:113) */
int otslam_mesh_vertex_normals(const double* vertices, int64_t n_vertices, const int32_t* faces, int64_t n_faces,
                               double* normals, int device);
/* TriangleMesh.sample_points_uniformly(number_of_points) (reconstruct_rgbd_filter.py:123);
 * colors / normals (and their outputs) nullable */
int otslam_mesh_sample_uniform(const double* vertices, const double* colors, const double* normals,
                               int64_t n_vertices, const int32_t* faces, int64_t n_faces, int64_t n_samples,
                               uint64_t seed, double* out_points, double* out_colors, double* out_normals,
                               int device);
/* mask = points[:,2] >= zmin; rebuild (reconstruct_rgbd_filter.py:126-132) */
int otslam_cloud_zfilter(const double* points, const double* colors, int64_t n, double zmin, double* out_points,
                         double* out_colors, int64_t* n_out, int device);
/* PointCloud.voxel_down_sample (check_one_frame.py:28); outputs sized n, sorted by voxel key */
int otslam_cloud_voxel_down_sample(const double* points, const double* colors, int64_t n, double voxel_size,
                                   double* out_points, double* out_colors, int32_t* out_keys, int32_t* out_counts,
                                   int64_t* n_out, int device);
/* PointCloud.remove_statistical_outlier(nb_neighbors, std_ratio) (north_star); out_indices sized n */
int otslam_cloud_remove_statistical_outlier(const double* points, int64_t n, int nb_neighbors, double std_ratio,
                                            int64_t* out_indices, int64_t* n_out, double* mean_dist, int device);
/* PointCloud.compute_point_cloud_distance(target): distance from every source point to its nearest
 * target point -- the accuracy / completeness metric of the reference's evaluation scripts
 * (eval/eval_table_chair/eval_table_chair.py:106-119; SURVEY 8f "next" row 3) */
int otslam_cloud_nn_distance(const double* source, int64_t n_source, const double* target, int64_t n_target,
                             double* out_dist, int device);
/* correspondence search of o3d.pipelines.registration.registration_icp (eval/eval_table_chair/eval_table_chair.py:90-104):
 * for every source point the index of the nearest target point strictly closer than `radius`, or -1; out_dist2 (nullable)
 * = the squared distance.  The ICP loop around it (Umeyama update, convergence test) is host code in
 * o3d_compat/pipelines.py. */
int otslam_cloud_nn_within(const double* source, int64_t n_source, const double* target, int64_t n_target, double radius,
                           int32_t* out_index, double* out_dist2, int device);
/* PointCloud.estimate_normals(KDTreeSearchParamHybrid(radius, max_nn)) (radius = +inf: KDTreeSearchParamKNN(max_nn)), for
 * clouds that come without normals (a ground-truth scan, a cloud read from PLY).  Arithmetic in DESIGN.md §4 "Normals and
 * point-to-plane registration":
 *   neighbours of point i = the min(max_nn, m) points with the smallest squared distance among the m points with
 *     d2 < radius^2, point i itself included (d2 = 0); d2 = (dx^2 + dy^2) + dz^2 in FP64, the list ordered by (d2, index)
 *     ascending, so that the set and the summation order do not depend on the search structure (lattices, duplicated and
 *     identical points included);
 *   covariance = Open3D's ComputeCovariance: the nine cumulants x, y, z, xx, xy, xz, yy, yz, zz summed in neighbour order,
 *     divided by the count, C = E[x x^T] - mu mu^T; C = I with fewer than 3 neighbours;
 *   normal = the unit eigenvector of C's smallest eigenvalue by a cyclic Jacobi (+ - * / sqrt only, C scaled by its largest
 *     |entry|; among equal eigenvalues the highest index, so C = I gives (0, 0, 1)); a zero vector becomes the prior
 *     normal, or (0, 0, 1) without priors;
 *   sign: with prior_normals (nullable; a cloud's existing normals) flipped when n . prior < 0; without, flipped so that
 *     the largest-magnitude component (the first of equal ones) is positive.
 * out_normals [n][3].  1 <= max_nn <= 128, radius > 0 (finite, or +inf), n < 2^31, non-null points and out_normals:
 * otherwise OTSLAM_ERR_INVALID before any CUDA call.  otslam_last_op_device_ms() = device ms of search and kernel. */
int otslam_cloud_estimate_normals(const double* points, int64_t n, const double* prior_normals, double radius, int max_nn,
                                  double* out_normals, int device);
/* o3d.pipelines.registration.registration_icp(source, target, max_distance, init,
 * TransformationEstimationPointToPlane(), ICPConvergenceCriteria(relative_fitness, relative_rmse, max_iteration)) in one
 * call: Open3D's RegistrationICP loop, correspondences by otslam_cloud_nn_within's rule (nearest target strictly within
 * max_distance, ties to the lower index) on a grid of the target built once.  The source is moved by init, evaluated, then
 * each iteration solves J^T J x = -J^T r (r = n . (s - t), J = [s x n, n], n = the target's normal; FP64 sums by fixed
 * trees, the tracking's Cholesky and degeneracy rule), turns x into R = Rz(x2) Ry(x1) Rx(x0), t = x[3..5] (identity when
 * the solve fails or nothing corresponds), sets T <- update * T, moves the source by the update and evaluates again; it stops
 * after max_iteration (>= 0) iterations or when |d fitness| < relative_fitness and |d rmse| < relative_rmse.
 * fitness = inliers / n_source, inlier_rmse = sqrt(sum d2 / inliers) (0 without inliers), both at the returned transform;
 * corr_index [n_source] (nullable) = each source point's target index or -1 from the last evaluation.  source, target,
 * target_normals and corr_index may be device pointers; init, transform_out [16] and the scalar outputs (nullable) are host
 * pointers.  n_source = 0 returns init with 0 iterations.  Bad arguments give OTSLAM_ERR_INVALID before any CUDA call.
 * otslam_last_op_device_ms() = device ms from the grid build to the last evaluation. */
int otslam_cloud_icp_point_to_plane(const double* source, int64_t n_source, const double* target, const double* target_normals,
                                    int64_t n_target, double max_distance, const double init[16], double relative_fitness,
                                    double relative_rmse, int max_iteration, double transform_out[16], double* fitness,
                                    double* inlier_rmse, int32_t* iterations, int32_t* corr_index, int device);
/* PointCloud.cluster_dbscan(eps, min_points) (no reference call site): separates the objects of a cloud.  Rule in DESIGN.md
 * §4 "Plane segmentation and DBSCAN clustering":
 *   neighbours of point i = the points j with d2 < eps^2, d2 = (dx^2 + dy^2) + dz^2 in FP64 without FMA (otslam_cloud_nn_within's
 *     arithmetic), point i itself included;
 *   core point = at least min_points neighbours; clusters = the connected components of the core points (two core points
 *     joined when d2 < eps^2), labelled 0, 1, ... in increasing order of their smallest point index;
 *   a non-core point with a core neighbour takes the smallest label among its core neighbours, any other point -1.
 * This is what Open3D's ClusterDBSCAN loop computes.  out_labels [n]; *n_clusters (nullable) = the number of clusters.
 * points and out_labels may be device pointers.  eps finite and > 0, min_points >= 0, 0 <= n < 2^31, non-null points and
 * out_labels when n > 0: otherwise OTSLAM_ERR_INVALID before any CUDA call.  otslam_last_op_device_ms() = device ms of the
 * grid build and the kernels.  No neighbour list is stored; when every point lies within eps of every other the cost grows
 * with n^2 (as Open3D's does). */
int otslam_cloud_cluster_dbscan(const double* points, int64_t n, double eps, int64_t min_points, int32_t* out_labels, int32_t* n_clusters,
                                int device);
/* PointCloud.segment_plane(distance_threshold, ransac_n, num_iterations, probability) (no reference call site): the
 * dominant plane by RANSAC, Open3D's SegmentPlane run over hypotheses h = 0 .. num_iterations - 1 in order.  Rule in
 * DESIGN.md §4 "Plane segmentation and DBSCAN clustering":
 *   sample: r = ransac_n distinct indices by Floyd's algorithm, for k = 0 .. r-1: j = n - r + k,
 *     t = min(floor(u01(seed, h r + k) (j + 1)), j), j instead when t was drawn already (u01: the mesh sampler's RNG);
 *   plane: r = 3 Open3D's ComputeTrianglePlane ((p1 - p0) x (p2 - p0) normalised, d = -abc.p0; invalid when the cross
 *     product is 0), r > 3 GetPlaneFromPoints over the sample in draw order;
 *   evaluation: dist = |((a x + b y) + c z) + d|, inlier when dist < distance_threshold, fitness = count / n,
 *     rmse = sum dist / sqrt(count) (0 without inliers), the sum by the fixed tree of DESIGN.md;
 *   selection: h > B is skipped (B starts unbounded), invalid planes are skipped, a hypothesis replaces the best one when
 *     its fitness is greater or equal with a strictly smaller rmse; then B = 0 when fitness = 1, else
 *     q = log(1 - probability) / log(1 - fitness^r) and B = floor(q) when 0 <= q < num_iterations, num_iterations otherwise;
 *   result: out_inliers [n] = the best hypothesis's inliers ascending (*n_inliers of them), plane_out = GetPlaneFromPoints
 *     over them (sums by fixed trees); (0, 0, 0, 0) and no inliers without a valid best plane.
 * *n_evaluated (nullable) = the hypotheses not skipped by B, invalid ones included.  points and out_inliers may be device
 * pointers; plane_out and the scalars are host pointers.  distance_threshold finite and >= 0, 3 <= ransac_n <= 16,
 * num_iterations >= 0, 0 < probability <= 1, ransac_n <= n < 2^31: otherwise OTSLAM_ERR_INVALID before any CUDA call
 * (n < ransac_n: "There must be at least 'ransac_n' points.").  otslam_last_op_device_ms() = device ms of the search and
 * the refit. */
int otslam_cloud_segment_plane(const double* points, int64_t n, double distance_threshold, int ransac_n, int num_iterations,
                               double probability, uint64_t seed, double plane_out[4], int64_t* out_inliers, int64_t* n_inliers,
                               int32_t* n_evaluated, int device);
/* create_map_cloud's pixel loop (fusion/hybrid_map.py:45-55); out sized w*h*3 (or NULL to count) */
int otslam_grid_to_points(const uint8_t* gray, int width, int height, double resolution, double origin_x,
                          double origin_y, int threshold, double* out_points, int64_t* n_out, int device);
/* paint_uniform_color + `+=` concat + PLY vertex packing (fusion/hybrid_map.py:59,88-91,115,121):
 * n_clouds clouds of counts[i] points; paint[i] = RGB in 0..1 (3 doubles per cloud) or, when
 * paint == NULL, per-point colours colors[i]; writes 27-byte binary-PLY records. */
int otslam_cloud_merge_pack(int n_clouds, const double* const* points, const double* const* colors,
                            const int64_t* counts, const double* paint, uint8_t* out_records, int device);


/* ---- SURVEY 8(f) row 4: the steps either side of hybrid_map.py, non-interactive */
/* PointCloud.transform(T) (fusion/hybrid_map_manual.py:86-90, the W/S/A/D keys): p' = (T*[p,1]).xyz / w,
 * normals rotated by T's 3x3 block; normals / out_normals nullable */
int otslam_cloud_transform(const double* points, const double* normals, int64_t n, const double transform[16],
                           double* out_points, double* out_normals, int device);
/* PointCloud.get_center() (fusion/hybrid_map_manual.py:110): mean of the points, summed in index order */
int otslam_cloud_center(const double* points, int64_t n, double center[3], int device);
/* PointCloud.rotate(R, center) (fusion/hybrid_map_manual.py:112, the Z/C keys): p' = R*(p - center) + center */
int otslam_cloud_rotate(const double* points, const double* normals, int64_t n, const double rotation[9],
                        const double center[3], double* out_points, double* out_normals, int device);
/* smart_paste(base_img, overlay_img, x, y, w, h) (fusion/2d_selective_merge.py:58-69): inside the rectangle,
 * overlay pixels that are not within `threshold` of `unknown_pixel` replace the base map's; in place on
 * `base`; a rectangle that leaves the image changes nothing (as in the reference) */
int otslam_grid_smart_paste(uint8_t* base, const uint8_t* overlay, int width, int height, int x, int y, int w, int h,
                            int unknown_pixel, int threshold, int device);

/* ---- SURVEY 8(f) row 1: the readers in front of the frame loop.  o3d.io.read_image(color_path) and
 * o3d.io.read_image(depth_path) (3d_model/reconstruct_rgbd.py:88-89, reconstruct_rgbd_filter.py:91-92) decode the files
 * ScannerNode::save_files wrote with cv::imwrite (ros2_ws/src/system_manager/src/scanner_node.cpp:268-283: baseline JPEG
 * colour, 16-bit grey PNG depth; the gt_ / plain capture tools write 8-bit RGB PNG colour).  A decoder object takes a chunk of
 * such files -- as paths or as bytes already in memory --, uploads the COMPRESSED bytes and runs inflate / PNG filters /
 * Huffman / IDCT / upsampling / colour conversion on the GPU, into frame slots 0..n-1 kept in device memory, ready for
 * otslam_decoder_integrate.  Results equal the stock decoders' (libpng; libjpeg's default islow IDCT + fancy upsampling) bit
 * for bit.  Per-file status: 0 = decoded; 1 = a valid file of a kind the GPU decoders do not cover (progressive / grey /
 * CMYK JPEG, interlaced or palette PNG, another image size ...): decode it with the stock decoder and otslam_decoder_put it;
 * 2 = missing or damaged (CRC / structure), the reference's "Read image failed". */
typedef struct otslam_decoder otslam_decoder;
/* a stream or event that cannot be created for lack of memory returns OTSLAM_ERR_NOMEM, as in every other entry point */
int otslam_decoder_create(int device, int height, int width, int max_frames, otslam_decoder** out);
int otslam_decoder_destroy(otslam_decoder* d);
/* n <= max_frames files per kind, read by host threads; either path array may be NULL (kind not wanted) */
int otslam_decoder_decode_files(otslam_decoder* d, int n, const char* const* color_paths, const char* const* depth_paths,
                                int32_t* color_status, int32_t* depth_status);
/* the same for bytes in host memory: file i of a kind = blob[offsets[i] .. offsets[i + 1]) (empty = missing) */
int otslam_decoder_decode(otslam_decoder* d, int n, const uint8_t* color_blob, const int64_t* color_offsets,
                          const uint8_t* depth_blob, const int64_t* depth_offsets, int32_t* color_status, int32_t* depth_status);
/* overwrite a slot with arrays decoded elsewhere (u16 [H][W], RGB8 [H][W][3]; host or device; either nullable) */
int otslam_decoder_put(otslam_decoder* d, int slot, const uint16_t* depth, const uint8_t* rgb);
/* copy slots [first, first + count) out (host or device pointers; either nullable) */
int otslam_decoder_fetch(otslam_decoder* d, int first, int count, uint16_t* depth, uint8_t* rgb);
/* volume.integrate(rgbd, intrinsic, extrinsic) (reconstruct_rgbd.py:99-107) for the slots listed (ascending), in that order;
 * object_ids nullable (multi-object arenas).  The slots' contents are consumed (holes are closed in place). */
int otslam_decoder_integrate(otslam_decoder* d, otslam_volume* v, int n_keep, const int32_t* slots, const double intr[4],
                             const double* extrinsics, double depth_scale, double depth_trunc, const int32_t* object_ids);
/* np.loadtxt(pose_path) (reconstruct_rgbd.py:90) for n pose files at once (host threads; no GPU involved): poses[n][16]
 * row-major.  status 0 = 16 plain decimal numbers, converted with correctly rounded strtod (the same doubles np.loadtxt
 * yields); 1 = anything else (comments, commas, other counts, inf / nan ...): parse it with np.loadtxt; 2 = unreadable. */
int otslam_read_pose_files(int n, const char* const* paths, double* poses, int32_t* status);
/* device times (CUDA events, ms) of the last decode: [0] inflate, [1] PNG filters + emit, [2] JPEG Huffman, [3] IDCT,
 * [4] upsampling + colour; [5] = compressed bytes uploaded */
int otslam_decoder_profile(otslam_decoder* d, double out[6]);

#ifdef __cplusplus
}
#endif
#endif
