// track.cu -- frame-to-model camera tracking on sm_100a: projective point-to-plane ICP of raw u16 depth frames against
// vertex and normal maps ray cast from the volume (the model for the interface is Open3D's tensor SLAM
// Model.track_frame_to_model), coarse to fine over a depth pyramid.  The arithmetic is DESIGN.md §4 "Frame-to-model
// tracking" and is restated on the CPU by tests/models/track_model.cpp (one level) and
// tests/models/track_pyramid_model.cpp (the pyramid); they agree bit for bit.  All FP64 arithmetic is
// explicit round-to-nearest, no FMA.
//
//   track_pyrdown_kernel  one thread per coarse pixel: level l + 1 of the depth pyramid from level l (the u16 frame and
//                         its scale at level 0, float metres above)
//   raycast_launch        (raycast.cu) the model: vertex and normal maps of each frame at its initial pose E0, once per
//                         level, at that level's size and intrinsics
//   track_assoc_kernel    one thread per source pixel, a 16x8 pixel tile per CTA, one grid z slice per frame: back-project
//                         with the current pose T, project into E0, gate, and form the 30 terms of the pixel; the CTA sums
//                         its 128 pixels by a fixed pairwise tree and writes one partial per tile
//   track_solve_kernel    one CTA per frame: sums the tile partials by a fixed pairwise tree (in place, in global memory),
//                         then one thread solves the 6x6 system and updates the frame's pose and status
//   track_arm_kernel      re-arms every frame's flag and step history before the next finer level
// The levels and iterations are queued with no host round trip; a converged or failed frame's later CTAs of a level exit on
// its device flag.
#include <cmath>
#include <vector>

#include "cta_ops.cuh"
#include "icp_solve.h"
#include "raycast.cuh"

namespace otslam {

constexpr int kTrackChunk = 32;                     // frames whose maps are rendered at once
constexpr size_t kTrackMapBytes = 512ull << 20;     // bound of the chunk's vertex + normal maps
constexpr int kTileW = 16, kTileH = 8, kTilePx = kTileW * kTileH;
constexpr int kTerms = 30;                          // 21 JtJ (upper triangle, row-major), 6 Jtr, r^2, inliers, valid pixels
constexpr int kSolveThreads = 256;
constexpr double kMinInliers = 64.0;
constexpr double kConverged = 1e-6;                 // max |xi_i| (radians, metres) of a converged step
constexpr double kStalled = 1e-5;                   // ... or a step this small that is not smaller than the one before
constexpr int kMaxLevels = 4;                       // pyramid levels, 0 = full resolution
constexpr double kPyrBand = 4.0;                    // a coarse pixel averages depths within 4 voxels of its block's nearest

struct TrackFrame {
    double T[16];        // current camera pose (camera -> world)
    double E[16];        // its extrinsic, inverse4(T); the returned pose
    double E0[16];       // initial extrinsic: the view of the model maps
    double fitness, rmse;
    double last_step;    // max |xi_i| of the previous step (infinity before the first)
    int status, iters, active;
};

struct TrackArgs {
    const uint16_t* depth;   // [chunk][H][W], level 0
    const float* fdepth;     // [chunk][H][W] metres, levels >= 1 (the pyramid)
    const float* vertex;     // [chunk][H][W][3] model maps at E0
    const float* normal;
    TrackFrame* frames;      // [chunk]
    double* partials;        // [chunk][kTerms][P]
    int W, H, tiles_x, n_tiles, P;
    float scale;             // (float)depth_scale
    double dmax, ddiff2;     // depth_max, depth_diff * depth_diff
    double fx, fy, cx, cy;
};

__device__ __forceinline__ double dm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double da(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double ds(double a, double b) { return __dsub_rn(a, b); }

// the shared cofactor inverse (inverse4 in volume.cu), restated with explicit round-to-nearest operations
__device__ bool inverse4_rn(const double* m, double* o) {
    const double a00 = m[0], a01 = m[1], a02 = m[2], a03 = m[3], a10 = m[4], a11 = m[5], a12 = m[6], a13 = m[7],
                 a20 = m[8], a21 = m[9], a22 = m[10], a23 = m[11], a30 = m[12], a31 = m[13], a32 = m[14], a33 = m[15];
    const double s0 = ds(dm(a00, a11), dm(a01, a10)), s1 = ds(dm(a00, a12), dm(a02, a10)), s2 = ds(dm(a00, a13), dm(a03, a10)),
                 s3 = ds(dm(a01, a12), dm(a02, a11)), s4 = ds(dm(a01, a13), dm(a03, a11)), s5 = ds(dm(a02, a13), dm(a03, a12)),
                 c0 = ds(dm(a20, a31), dm(a21, a30)), c1 = ds(dm(a20, a32), dm(a22, a30)), c2 = ds(dm(a20, a33), dm(a23, a30)),
                 c3 = ds(dm(a21, a32), dm(a22, a31)), c4 = ds(dm(a21, a33), dm(a23, a31)), c5 = ds(dm(a22, a33), dm(a23, a32));
    const double det = da(ds(da(da(ds(dm(s0, c5), dm(s1, c4)), dm(s2, c3)), dm(s3, c2)), dm(s4, c1)), dm(s5, c0));
    if (det == 0.0 || !isfinite(det)) return false;
    const double id = __ddiv_rn(1.0, det);
    o[0] = dm(da(ds(dm(a11, c5), dm(a12, c4)), dm(a13, c3)), id);
    o[1] = dm(ds(ds(dm(a02, c4), dm(a01, c5)), dm(a03, c3)), id);
    o[2] = dm(da(ds(dm(a31, s5), dm(a32, s4)), dm(a33, s3)), id);
    o[3] = dm(ds(ds(dm(a22, s4), dm(a21, s5)), dm(a23, s3)), id);
    o[4] = dm(ds(ds(dm(a12, c2), dm(a10, c5)), dm(a13, c1)), id);
    o[5] = dm(da(ds(dm(a00, c5), dm(a02, c2)), dm(a03, c1)), id);
    o[6] = dm(ds(ds(dm(a32, s2), dm(a30, s5)), dm(a33, s1)), id);
    o[7] = dm(da(ds(dm(a20, s5), dm(a22, s2)), dm(a23, s1)), id);
    o[8] = dm(da(ds(dm(a10, c4), dm(a11, c2)), dm(a13, c0)), id);
    o[9] = dm(ds(ds(dm(a01, c2), dm(a00, c4)), dm(a03, c0)), id);
    o[10] = dm(da(ds(dm(a30, s4), dm(a31, s2)), dm(a33, s0)), id);
    o[11] = dm(ds(ds(dm(a21, s2), dm(a20, s4)), dm(a23, s0)), id);
    o[12] = dm(ds(ds(dm(a11, c1), dm(a10, c3)), dm(a12, c0)), id);
    o[13] = dm(da(ds(dm(a00, c3), dm(a01, c1)), dm(a02, c0)), id);
    o[14] = dm(ds(ds(dm(a31, s1), dm(a30, s3)), dm(a32, s0)), id);
    o[15] = dm(da(ds(dm(a20, s3), dm(a21, s1)), dm(a22, s0)), id);
    return true;
}

// rows 0..2 of M p, in the integration's product order ((M0 x + M1 y) + M2 z) + M3
__device__ __forceinline__ void affine(const double* M, const double p[3], double out[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) out[r] = da(da(da(dm(M[4 * r], p[0]), dm(M[4 * r + 1], p[1])), dm(M[4 * r + 2], p[2])), M[4 * r + 3]);
}

// report = 0: one Gauss-Newton iteration's association (frames no longer active exit); report = 1: the final pass.
// kCoarse: the source is a pyramid level's float depth (valid iff > 0, and every such value is < depth_max); else the
// level-0 u16 frame, converted as integration's K1 does.
template <bool kCoarse>
__global__ void __launch_bounds__(kTilePx) track_assoc_kernel(const TrackArgs a, int report) {
    __shared__ double sm[kTerms][kTilePx];
    const TrackFrame& f = a.frames[blockIdx.z];
    if (!report && !f.active) return;
    const int lane = threadIdx.x;
    const int u = blockIdx.x * kTileW + (lane % kTileW), v = blockIdx.y * kTileH + (lane / kTileW);
    double t[kTerms];
#pragma unroll
    for (int k = 0; k < kTerms; ++k) t[k] = 0.0;
    if (u < a.W && v < a.H) {
        const size_t px = (size_t)a.W * a.H;
        const size_t i = blockIdx.z * px + (size_t)v * a.W + u;
        const float d = kCoarse ? a.fdepth[i] : __fdiv_rn((float)a.depth[i], a.scale);
        if (d > 0.f && (double)d < a.dmax) {
            t[29] = 1.0;
            const double z = (double)d;
            const double pc[3] = {dm(__ddiv_rn(ds((double)u, a.cx), a.fx), z), dm(__ddiv_rn(ds((double)v, a.cy), a.fy), z), z};
            double p[3], q[3];
            affine(f.T, pc, p);
            affine(f.E0, p, q);
            if (q[2] > 0.0) {
                const double uf = floor(da(da(__ddiv_rn(dm(a.fx, q[0]), q[2]), a.cx), 0.5));
                const double vf = floor(da(da(__ddiv_rn(dm(a.fy, q[1]), q[2]), a.cy), 0.5));
                if (uf >= 0.0 && uf < (double)a.W && vf >= 0.0 && vf < (double)a.H) {
                    const size_t m = 3 * (blockIdx.z * px + (size_t)vf * a.W + (size_t)uf);
                    const double N[3] = {(double)a.normal[m], (double)a.normal[m + 1], (double)a.normal[m + 2]};
                    if (N[0] != 0.0 || N[1] != 0.0 || N[2] != 0.0) {
                        const double e[3] = {ds(p[0], (double)a.vertex[m]), ds(p[1], (double)a.vertex[m + 1]),
                                             ds(p[2], (double)a.vertex[m + 2])};
                        if (da(da(dm(e[0], e[0]), dm(e[1], e[1])), dm(e[2], e[2])) <= a.ddiff2)
                            point_to_plane_terms(p, N, e, t, 1);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < kTerms; ++k) sm[k][lane] = t[k];
    cta_halving_tree(sm);                // absent pixels add 0
    if (lane < kTerms) a.partials[((size_t)blockIdx.z * kTerms + lane) * a.P + blockIdx.y * a.tiles_x + blockIdx.x] = sm[lane][0];
}

__global__ void __launch_bounds__(kSolveThreads) track_solve_kernel(const TrackArgs a, int it, int max_it, int report) {
    TrackFrame& f = a.frames[blockIdx.x];
    if (!report && !f.active) return;
    double* buf = a.partials + (size_t)blockIdx.x * kTerms * a.P;
    cta_tree_rows<kSolveThreads>(buf, kTerms, a.n_tiles, a.P);
    if (threadIdx.x != 0) return;
    double S[kTerms];
    for (int k = 0; k < kTerms; ++k) S[k] = buf[(size_t)k * a.P];
    if (report) {
        f.fitness = S[29] > 0.0 ? __ddiv_rn(S[28], S[29]) : 0.0;
        f.rmse = S[28] > 0.0 ? __dsqrt_rn(__ddiv_rn(S[27], S[28])) : 0.0;
        return;
    }
    f.iters += 1;                                   // summed over the levels
    if (S[28] < kMinInliers) { f.status = 2; f.active = 0; return; }
    double xi[6];
    if (!solve6(S, xi)) { f.status = 3; f.active = 0; return; }
    // Cayley rotation: a = w / 2, dR = I + 2 / (1 + |a|^2) ([a]x + [a]x^2); dT = [dR | t]; T <- dT T; E = inverse4(T)
    const double h[3] = {dm(0.5, xi[0]), dm(0.5, xi[1]), dm(0.5, xi[2])};
    const double n2 = da(da(dm(h[0], h[0]), dm(h[1], h[1])), dm(h[2], h[2]));
    const double c = __ddiv_rn(2.0, da(1.0, n2));
    const double K[9] = {0.0, -h[2], h[1], h[2], 0.0, -h[0], -h[1], h[0], 0.0};
    double D[16];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            double k2 = dm(h[i], h[j]);
            if (i == j) k2 = ds(k2, n2);
            D[4 * i + j] = da(i == j ? 1.0 : 0.0, dm(c, da(K[3 * i + j], k2)));
        }
        D[4 * i + 3] = xi[3 + i];
    }
    D[12] = 0.0; D[13] = 0.0; D[14] = 0.0; D[15] = 1.0;
    double T[16], E[16];
    for (int r = 0; r < 4; ++r)
        for (int cc = 0; cc < 4; ++cc)
            T[4 * r + cc] = da(da(da(dm(D[4 * r], f.T[cc]), dm(D[4 * r + 1], f.T[4 + cc])), dm(D[4 * r + 2], f.T[8 + cc])),
                               dm(D[4 * r + 3], f.T[12 + cc]));
    if (!inverse4_rn(T, E)) { f.status = 3; f.active = 0; return; }
    for (int k = 0; k < 16; ++k) { f.T[k] = T[k]; f.E[k] = E[k]; }
    double step = 0.0;
    for (int k = 0; k < 6; ++k)
        if (fabs(xi[k]) > step) step = fabs(xi[k]);
    // A step that stops shrinking near the association's resolution is a 2-cycle of pixel associations flipping at
    // depth edges (DESIGN §4): converged too.
    const bool stalled = step <= kStalled && step >= f.last_step;
    f.last_step = step;
    if (step <= kConverged || stalled) { f.status = 0; f.active = 0; }
    else if (it + 1 >= max_it) { f.status = 1; f.active = 0; }
}

// Level l + 1 of the depth pyramid from level l (DESIGN §4): coarse pixel (u, v) takes the valid depths of the 2x2 block
// at (2u, 2v) -- at level 0 d = raw / scale, valid iff d > 0 and (double)d < dmax; above, valid iff d > 0 -- keeps those
// within `band` metres of the block's smallest, sums them in FP64 in raster order, divides by their count and rounds to
// FP32; 0 when none is valid.  The sum of at most four such floats is exact, so the result depends on no order.
template <bool kFromU16>
__global__ void track_pyrdown_kernel(const uint16_t* src16, const float* srcf, float* dst, int Ws, int Hs, int Wd, int Hd,
                                     float scale, double dmax, double band) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Wd * Hd) return;
    const int u = i % Wd, v = i / Wd;
    const size_t base = (size_t)blockIdx.y * Ws * Hs + (size_t)(2 * v) * Ws + 2 * u;
    const size_t at[4] = {base, base + 1, base + Ws, base + Ws + 1};
    float d[4];
    bool ok[4];
    float lo = INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (kFromU16) {
            d[k] = __fdiv_rn((float)src16[at[k]], scale);
            ok[k] = d[k] > 0.f && (double)d[k] < dmax;
        } else {
            d[k] = srcf[at[k]];
            ok[k] = d[k] > 0.f;
        }
        if (ok[k] && d[k] < lo) lo = d[k];
    }
    double sum = 0.0;
    int n = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (ok[k] && ds((double)d[k], (double)lo) <= band) { sum = da(sum, (double)d[k]); ++n; }
    dst[(size_t)blockIdx.y * Wd * Hd + i] = n ? __double2float_rn(__ddiv_rn(sum, (double)n)) : 0.f;
}

// before a finer level: every frame of the chunk iterates again from the pose the coarser level returned
__global__ void track_arm_kernel(TrackFrame* frames, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    frames[i].active = 1;
    frames[i].status = 1;
    frames[i].last_step = INFINITY;
}

static bool finite_all(const double* p, int n) {
    for (int i = 0; i < n; ++i)
        if (!std::isfinite(p[i])) return false;
    return true;
}

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_volume_track_pyramid(otslam_volume* v, int n_frames, const uint16_t* depth, int width, int height,
                                const double intr[4], const double* init_extrinsics, double depth_scale, double depth_min,
                                double depth_max, int n_levels, const double* depth_diff, const int32_t* max_iterations,
                                double* extrinsics_out, int32_t* status, int32_t* iterations, double* fitness,
                                double* inlier_rmse, int memory) {
    // ---- every argument is checked before any CUDA call
    if (n_frames < 0) return set_error(OTSLAM_ERR_INVALID, "track: n_frames < 0");
    if (width <= 0 || height <= 0) return set_error(OTSLAM_ERR_INVALID, "track: width and height must be > 0");
    if (!intr) return set_error(OTSLAM_ERR_INVALID, "track: null intrinsics");
    if (!finite_all(intr, 4) || !(intr[0] > 0.0) || !(intr[1] > 0.0))
        return set_error(OTSLAM_ERR_INVALID, "track: fx and fy must be finite and > 0, cx and cy finite");
    if (!std::isfinite(depth_min) || !std::isfinite(depth_max) || !(depth_min > 0.0) || !(depth_min < depth_max))
        return set_error(OTSLAM_ERR_INVALID, "track: need finite 0 < depth_min < depth_max");
    if (!std::isfinite(depth_scale) || !(depth_scale > 0.0)) return set_error(OTSLAM_ERR_INVALID, "track: depth_scale must be finite and > 0");
    if (n_levels < 1 || n_levels > kMaxLevels) return set_error(OTSLAM_ERR_INVALID, "track: n_levels must be in 1..4");
    if (!depth_diff || !max_iterations) return set_error(OTSLAM_ERR_INVALID, "track: null depth_diff or max_iterations");
    for (int l = 0; l < n_levels; ++l) {
        if (!std::isfinite(depth_diff[l]) || !(depth_diff[l] > 0.0))
            return set_error(OTSLAM_ERR_INVALID, "track: depth_diff must be finite and > 0");
        if (max_iterations[l] < 1 || max_iterations[l] > 100)
            return set_error(OTSLAM_ERR_INVALID, "track: max_iterations must be in 1..100");
    }
    if (n_levels > 1 && ((width >> (n_levels - 1)) < kTileW || (height >> (n_levels - 1)) < kTileH))
        return set_error(OTSLAM_ERR_INVALID, "track: the coarsest pyramid level must be at least 16x8 pixels");
    if (memory != OTSLAM_MEM_HOST && memory != OTSLAM_MEM_DEVICE) return set_error(OTSLAM_ERR_INVALID, "track: bad memory kind");
    if (n_frames > 0 && (!depth || !init_extrinsics || !extrinsics_out))
        return set_error(OTSLAM_ERR_INVALID, "track: null depth, init_extrinsics or extrinsics_out");
    std::vector<TrackFrame> frames((size_t)n_frames);
    std::vector<RayView> views((size_t)n_frames);
    for (int i = 0; i < n_frames; ++i) {
        const double* e = init_extrinsics + 16 * (size_t)i;
        TrackFrame& f = frames[i];
        f = TrackFrame{};
        if (!ray_view(e, &views[i]) || !inverse4(e, f.T))
            return set_error(OTSLAM_ERR_INVALID, "track: initial extrinsic is not finite or is singular");
        for (int k = 0; k < 16; ++k) f.E[k] = f.E0[k] = e[k];
        f.last_step = INFINITY;
        f.status = 1; f.active = 1;
    }
    // level l + 1: half the size (an odd last column or row dropped), fx / 2, fy / 2, (cx - 0.5) / 2, (cy - 0.5) / 2 in
    // FP64, so that coarse pixel u' looks along the ray through the centre 2u' + 0.5 of the 2x2 block it covers
    RayArgs ra[kMaxLevels];
    TrackArgs a[kMaxLevels];
    double li[4] = {intr[0], intr[1], intr[2], intr[3]};
    size_t frame_bytes = 0;                      // every level's maps and the coarse levels' depth, per frame
    for (int l = 0; l < n_levels; ++l) {
        if (l > 0) li[0] = li[0] / 2.0, li[1] = li[1] / 2.0, li[2] = (li[2] - 0.5) / 2.0, li[3] = (li[3] - 0.5) / 2.0;
        const int W = width >> l, H = height >> l;
        OT_TRY(ray_args(v, W, H, li, depth_min, depth_max, "track", &ra[l]));
        TrackArgs& t = a[l];
        t = TrackArgs{};
        t.W = W; t.H = H;
        t.tiles_x = (W + kTileW - 1) / kTileW;
        t.n_tiles = t.tiles_x * ((H + kTileH - 1) / kTileH);
        t.P = pow2_at_least(t.n_tiles);
        t.scale = (float)depth_scale;
        t.dmax = depth_max; t.ddiff2 = depth_diff[l] * depth_diff[l];
        t.fx = li[0]; t.fy = li[1]; t.cx = li[2]; t.cy = li[3];
        frame_bytes += (l ? 28 : 24) * (size_t)W * H;
    }
    if (n_frames == 0) return OTSLAM_OK;

    OT_TRY(use_device(v->device));
    cudaStream_t s = v->stream;
    const int chunk = (int)std::min<size_t>(std::min(kTrackChunk, n_frames), std::max<size_t>(1, kTrackMapBytes / frame_bytes));
    const double band = kPyrBand * v->voxel_length;
    DevBuf<RayView> d_views;
    DevBuf<TrackFrame> d_frames;
    DevBuf<float> d_maps;                        // per level: vertex [chunk][H][W][3], normal, then (l >= 1) depth [chunk][H][W]
    DevBuf<double> d_partials;
    DevBuf<uint16_t> d_depth;
    DevBuf<unsigned long long> d_hits;
    OT_CUDA(d_views.alloc((size_t)n_frames)); OT_CUDA(d_frames.alloc((size_t)n_frames)); OT_CUDA(d_hits.alloc(1));
    OT_CUDA(d_maps.alloc(frame_bytes / sizeof(float) * chunk));
    OT_CUDA(d_partials.alloc((size_t)kTerms * a[0].P * chunk));
    if (memory == OTSLAM_MEM_HOST) OT_CUDA(d_depth.alloc((size_t)width * height * chunk));
    float *vtx[kMaxLevels], *nrm[kMaxLevels], *fd[kMaxLevels] = {};
    {
        float* m = d_maps.p;
        for (int l = 0; l < n_levels; ++l) {
            const size_t px = (size_t)a[l].W * a[l].H * chunk;
            vtx[l] = m; nrm[l] = m + 3 * px; m += 6 * px;
            if (l > 0) { fd[l] = m; m += px; }
            a[l].vertex = vtx[l]; a[l].normal = nrm[l]; a[l].fdepth = fd[l];
            a[l].partials = d_partials.p;
            ra[l].hits = d_hits.p;
        }
    }
    const size_t px0 = (size_t)width * height;
    {
        OpTimer timer(s);
        OT_CUDA(cudaMemcpyAsync(d_views.p, views.data(), sizeof(RayView) * views.size(), cudaMemcpyHostToDevice, s));
        OT_CUDA(cudaMemcpyAsync(d_frames.p, frames.data(), sizeof(TrackFrame) * frames.size(), cudaMemcpyHostToDevice, s));
        for (int first = 0; first < n_frames; first += chunk) {
            const int nf = std::min(chunk, n_frames - first);
            if (memory == OTSLAM_MEM_HOST) {
                OT_CUDA(cudaMemcpyAsync(d_depth.p, depth + px0 * first, 2 * px0 * nf, cudaMemcpyHostToDevice, s));
                a[0].depth = d_depth.p;
            } else {
                a[0].depth = depth + px0 * first;
            }
            for (int l = 0; l < n_levels; ++l) {
                a[l].frames = d_frames.p + first;
                if (l > 0) {
                    const TrackArgs& f = a[l - 1];
                    const dim3 grid((unsigned)((a[l].W * a[l].H + 255) / 256), (unsigned)nf);
                    if (l == 1)
                        track_pyrdown_kernel<true><<<grid, 256, 0, s>>>(f.depth, nullptr, fd[l], f.W, f.H, a[l].W, a[l].H, f.scale,
                                                                        depth_max, band);
                    else
                        track_pyrdown_kernel<false><<<grid, 256, 0, s>>>(nullptr, fd[l - 1], fd[l], f.W, f.H, a[l].W, a[l].H, f.scale,
                                                                         depth_max, band);
                    OT_LAUNCHED();
                }
                OT_TRY(raycast_launch(ra[l], d_views.p + first, nf, nullptr, vtx[l], nrm[l], nullptr, s));
            }
            for (int l = n_levels - 1; l >= 0; --l) {
                if (l < n_levels - 1) {
                    track_arm_kernel<<<(nf + 127) / 128, 128, 0, s>>>(a[l].frames, nf);
                    OT_LAUNCHED();
                }
                const dim3 grid((unsigned)a[l].tiles_x, (unsigned)((a[l].H + kTileH - 1) / kTileH), (unsigned)nf);
                const int max_it = max_iterations[l];
                for (int it = 0; it <= max_it; ++it) {
                    const int report = it == max_it;   // level 0's last pass reports fitness and RMSE at the returned pose
                    if (report && l > 0) break;
                    if (l > 0) track_assoc_kernel<true><<<grid, kTilePx, 0, s>>>(a[l], report);
                    else track_assoc_kernel<false><<<grid, kTilePx, 0, s>>>(a[l], report);
                    OT_LAUNCHED();
                    track_solve_kernel<<<nf, kSolveThreads, 0, s>>>(a[l], it, max_it, report);
                    OT_LAUNCHED();
                }
            }
        }
        OT_CUDA(cudaMemcpyAsync(frames.data(), d_frames.p, sizeof(TrackFrame) * frames.size(), cudaMemcpyDeviceToHost, s));
        timer.stop();
    }
    OT_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < n_frames; ++i) {
        const TrackFrame& f = frames[i];
        for (int k = 0; k < 16; ++k) extrinsics_out[16 * (size_t)i + k] = f.E[k];
        if (status) status[i] = f.status;
        if (iterations) iterations[i] = f.iters;
        if (fitness) fitness[i] = f.fitness;
        if (inlier_rmse) inlier_rmse[i] = f.rmse;
    }
    return OTSLAM_OK;
}

int otslam_volume_track(otslam_volume* v, int n_frames, const uint16_t* depth, int width, int height, const double intr[4],
                        const double* init_extrinsics, double depth_scale, double depth_min, double depth_max, double depth_diff,
                        int max_iterations, double* extrinsics_out, int32_t* status, int32_t* iterations, double* fitness,
                        double* inlier_rmse, int memory) {
    const int32_t it = max_iterations;
    return otslam_volume_track_pyramid(v, n_frames, depth, width, height, intr, init_extrinsics, depth_scale, depth_min, depth_max,
                                       1, &depth_diff, &it, extrinsics_out, status, iterations, fitness, inlier_rmse, memory);
}

}  // extern "C"
