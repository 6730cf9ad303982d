// raycast.cuh -- the ray caster's internal interface (raycast.cu), shared by otslam_volume_raycast and the frame-to-model
// tracker (track.cu), which renders its model's vertex and normal maps with the same kernel.
#pragma once
#include "volume_lookup.cuh"

namespace otslam {

struct RayView {
    float R[9];      // rows 0..2, cols 0..2 of camera_pose = inverse4(extrinsic), cast to f32
    float o[3];      // camera centre (column 3 of camera_pose), f32
};

struct RayArgs {
    ExtractCtx c;
    const RayView* views;   // [chunk]
    int W, H;
    float cx, cy, ifx, ify; // ifx = 1.0f / (float)fx, as the integration's multiplier table (SURVEY A.2)
    float vl, ktr;          // (float)voxel_length, (float)(k * sdf_trunc)
    float dmin, dmax;
    int cap;                // iterations per ray (host: raycast_cap)
    int color;              // volume keeps colour
    double gap;             // 0.99 voxel (GetNormalAt)
    float* depth;           // outputs of this chunk, [chunk][H][W](...) or null
    float* vertex;
    float* normal;
    uint8_t* rgb;
    unsigned long long* hits;
};

// The ray-cast view of a world->camera extrinsic; false if it is not finite or is singular.  No CUDA call.
bool ray_view(const double* extrinsic, RayView* out);

// Kernel arguments of a render of volume v (all but views, outputs and the hit counter).  Checks what needs the volume:
// slab sharding, the arena's selection and the depth window's bound; the intrinsics and 0 < depth_min < depth_max are the
// caller's to check first.  `op` prefixes the error messages.  No CUDA call.
int ray_args(const otslam_volume* v, int width, int height, const double intr[4], double depth_min, double depth_max,
             const char* op, RayArgs* a);

// Renders n_views views (d_views on the device) into device outputs (each nullable, [n_views][H][W](...)) on stream s;
// a.hits must point to a device counter.
int raycast_launch(RayArgs a, const RayView* d_views, int n_views, float* depth, float* vertex, float* normal, uint8_t* rgb,
                   cudaStream_t s);

}  // namespace otslam
