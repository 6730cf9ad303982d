// raycast.cu -- rendering a TSDF volume from camera poses on sm_100a: depth, world vertex, world normal and colour maps,
// the ray-cast half of a KinectFusion-style system (the model for the interface is Open3D's tensor
// VoxelBlockGrid.ray_cast; the legacy ScalableTSDFVolume has none).  The arithmetic is DESIGN.md §4 "Ray casting" and is
// restated on the CPU by tests/models/raycast_model.cpp; the two agree bit for bit (colour: within one level).
//
//   raycast_kernel  one thread per pixel, a 16x8 pixel tile per CTA (a warp's rays cross the same blocks), one grid z
//                   slice per view.  FP32 march: absent block -> jump to the block's exit (DDA over the block grid),
//                   unobserved voxel -> one voxel, observed f > 0 -> max(k f sdf_trunc, vl), else one voxel; the first
//                   + -> - crossing of two consecutive observed samples is the surface, refined with the trilinear TSDF.  The block key and its slot stay
//                   in registers, so the hash is probed only when a ray enters a new block (about every 16 samples).
//                   Normal (FP64 GetNormalAt) and trilinear colour run at the hit only.
// Host outputs are rendered into two bounded device staging buffers, chunk by chunk; the copy of chunk k (copy stream)
// overlaps the render of chunk k + 1.  Device outputs are written in place.  raycast_launch (raycast.cuh) is the one launch
// path, shared with the frame-to-model tracker (track.cu), which renders its model maps with it.
#include <cmath>
#include <vector>

#include "raycast.cuh"

namespace otslam {

constexpr float kStepFactor = 0.5f;             // k: observed f > 0 steps max(k f sdf_trunc, vl) (DESIGN §4 "Ray casting")
constexpr int kViewsPerChunk = 32;
constexpr size_t kStagingBytes = 256ull << 20;  // per staging buffer (two of them) for host outputs
constexpr int kTileW = 16, kTileH = 8;
constexpr double kMaxWindowVoxels = 4194304.0;  // 2^22: depth_max * max|d_c| / vl, keeps one-voxel steps >= 2 ulp(t)

// trilinear colour at a world point over the observed corners only, renormalised; voxel colour = exact sum / count
__device__ __forceinline__ void color_at(const RayArgs& a, const double p[3], uint8_t out[3]) {
    int g0[3];
    double r[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double pv = __ddiv_rn(__dsub_rn(p[i], a.c.half), a.c.vl);
        const double fl = floor(pv);
        g0[i] = (int)fl;
        r[i] = __dsub_rn(pv, fl);
    }
    double acc[3] = {0.0, 0.0, 0.0}, wsum = 0.0;
    for (int q = 0; q < 8; ++q) {
        const int sx = q & 1, sy = (q >> 1) & 1, sz = q >> 2;
        const int g[3] = {g0[0] + sx, g0[1] + sy, g0[2] + sz};
        const int s = block_slot(a.c, g[0] >> 4, g[1] >> 4, g[2] >> 4);
        if (s < 0) continue;
        const uint4 rec = __ldg(block_ptr(a.c.chunks, s) + rec_index(g[0] & 15, g[1] & 15, g[2] & 15));
        const uint32_t w = rec_weight(rec);
        if (w == 0) continue;
        const double wq = __dmul_rn(__dmul_rn(sx ? r[0] : __dsub_rn(1.0, r[0]), sy ? r[1] : __dsub_rn(1.0, r[1])),
                                    sz ? r[2] : __dsub_rn(1.0, r[2]));
        const uint32_t sum[3] = {rec.y & 0xFFFFFFu, rec.z & 0xFFFFFFu, rec.w & 0xFFFFFFu};
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] = __dadd_rn(acc[k], __dmul_rn(wq, __ddiv_rn((double)sum[k], (double)w)));
        wsum = __dadd_rn(wsum, wq);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double c = wsum > 0.0 ? floor(__dadd_rn(__ddiv_rn(acc[k], wsum), 0.5)) : 0.0;
        out[k] = (uint8_t)fmin(fmax(c, 0.0), 255.0);
    }
}

__device__ __forceinline__ void normal_at_hit(const RayArgs& a, const double p[3], float out[3]) {
    double n[3];
    normal_at(a.c, p, a.gap, n);
#pragma unroll
    for (int k = 0; k < 3; ++k) out[k] = (float)n[k];
}

__global__ void __launch_bounds__(kTileW * kTileH) raycast_kernel(const RayArgs a) {
    const int u = blockIdx.x * kTileW + (threadIdx.x % kTileW), v = blockIdx.y * kTileH + (threadIdx.x / kTileW);
    const bool inside = u < a.W && v < a.H;
    const RayView& view = a.views[blockIdx.z];
    bool hit = false;
    float t_hit = 0.f, P[3] = {0.f, 0.f, 0.f};
    if (inside) {
        // the pixel's ray: d_c = ((u - cx) / fx, (v - cy) / fy, 1) as the multiplier table forms it, d_w = R d_c
        const float xc = __fmul_rn(__fsub_rn((float)u, a.cx), a.ifx), yc = __fmul_rn(__fsub_rn((float)v, a.cy), a.ify);
        const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(xc, xc), __fmul_rn(yc, yc)), 1.0f));   // metres per unit t
        float o[3], d[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            o[r] = view.o[r];
            d[r] = __fadd_rn(__fadd_rn(__fmul_rn(view.R[3 * r], xc), __fmul_rn(view.R[3 * r + 1], yc)), view.R[3 * r + 2]);
        }
        const float dt_vox = __fdiv_rn(a.vl, len);
        float t = a.dmin, t_prev = 0.f, f_prev = 0.f, f_hit = 0.f;
        bool have_prev = false;
        uint64_t cur_key = kEmptyKey;
        int cur_slot = -1;
        for (int it = 0; it < a.cap && t < a.dmax; ++it) {
            float q[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) q[r] = floorf(__fdiv_rn(__fadd_rn(o[r], __fmul_rn(t, d[r])), a.vl));
            float tn;
            if (!(fabsf(q[0]) < 16777216.f && fabsf(q[1]) < 16777216.f && fabsf(q[2]) < 16777216.f)) {
                have_prev = false;                                // beyond the key range: one voxel
                tn = __fadd_rn(t, dt_vox);
            } else {
                const int g[3] = {(int)q[0], (int)q[1], (int)q[2]};
                const int b[3] = {g[0] >> 4, g[1] >> 4, g[2] >> 4};
                // |q| < 2^24 keeps every b within [-2^20, 2^20), where the packed key tells blocks apart even when the arena
                // offset takes x outside the key range (block_slot then finds the block absent)
                const uint64_t key = pack_key(b[0] + a.c.x_off, b[1], b[2]);
                if (key != cur_key) { cur_key = key; cur_slot = block_slot(a.c, b[0], b[1], b[2]); }
                const int slot = cur_slot;
                if (slot < 0) {
                    // absent block: to where the ray leaves it (the nearest exit plane), at least one voxel
                    have_prev = false;
                    float t_exit = INFINITY;
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        if (d[r] == 0.f) continue;
                        const float plane = __fmul_rn((float)(16 * (d[r] > 0.f ? b[r] + 1 : b[r])), a.vl);
                        t_exit = fminf(t_exit, __fdiv_rn(__fsub_rn(plane, o[r]), d[r]));
                    }
                    tn = fmaxf(t_exit, __fadd_rn(t, dt_vox));
                } else {
                    const uint4 rec = __ldg(block_ptr(a.c.chunks, slot) + rec_index(g[0] & 15, g[1] & 15, g[2] & 15));
                    if (rec_weight(rec) == 0) {                   // unobserved: one voxel, no crossing across it
                        have_prev = false;
                        tn = __fadd_rn(t, dt_vox);
                    } else {
                        const float f = __uint_as_float(rec.x);
                        if (have_prev && f_prev > 0.f && f <= 0.f) {   // front face between t_prev and t
                            t_hit = t; f_hit = f;
                            hit = true;
                            break;
                        }
                        have_prev = true; f_prev = f; t_prev = t;
                        tn = f > 0.f ? __fadd_rn(t, __fdiv_rn(fmaxf(__fmul_rn(f, a.ktr), a.vl), len)) : __fadd_rn(t, dt_vox);
                    }
                }
            }
            t = tn > t ? tn : nextafterf(t, INFINITY);
        }
        if (hit) {
            // Refinement: the zero of the trilinear TSDF (GetTSDFAt) interpolated linearly on the segment [t_prev, t]; if
            // the trilinear values say the zero lies one segment earlier (F(t_prev) <= 0: the nearest voxel of t_prev sat
            // half a voxel away, on the + side) or later (F(t) > 0), on the one-voxel segment before t_prev or after t.
            // The nearest-voxel values that detected the crossing when no segment brackets zero.
            const float t1 = t_hit;
            auto F = [&](float tt) {
                double p[3];
#pragma unroll
                for (int r = 0; r < 3; ++r) p[r] = (double)__fadd_rn(o[r], __fmul_rn(tt, d[r]));
                return tsdf_at(a.c, p);
            };
            float ta = t_prev, tb = t1;
            double Fa = F(ta), Fb = F(tb);
            bool ok = Fa > 0.0 && Fb <= 0.0;
            if (Fa <= 0.0) {
                const float tz = __fsub_rn(t_prev, dt_vox);
                if (tz >= a.dmin) {
                    const double Fz = F(tz);
                    if (Fz > 0.0) { tb = ta; Fb = Fa; ta = tz; Fa = Fz; ok = true; }
                }
            } else if (Fb > 0.0) {
                const float tz = __fadd_rn(t1, dt_vox);
                if (tz < a.dmax) {
                    const double Fz = F(tz);
                    if (Fz <= 0.0) { ta = tb; Fa = Fb; tb = tz; Fb = Fz; ok = true; }
                }
            }
            if (ok) {
                t_hit = __double2float_rn(__dadd_rn((double)ta, __dmul_rn(__dsub_rn((double)tb, (double)ta), __ddiv_rn(Fa, __dsub_rn(Fa, Fb)))));
            } else {
                ta = t_prev; tb = t1;
                t_hit = __fadd_rn(t_prev, __fdiv_rn(__fmul_rn(__fsub_rn(t1, t_prev), f_prev), __fsub_rn(f_prev, f_hit)));
            }
            t_hit = fminf(fmaxf(t_hit, ta), tb);
#pragma unroll
            for (int r = 0; r < 3; ++r) P[r] = __fadd_rn(o[r], __fmul_rn(t_hit, d[r]));
        }
    }
    const unsigned hits_warp = __ballot_sync(0xffffffffu, hit);
    if ((threadIdx.x & 31) == 0 && hits_warp) atomicAdd(a.hits, (unsigned long long)__popc(hits_warp));
    if (!inside) return;
    const size_t idx = ((size_t)blockIdx.z * a.H + v) * a.W + u;
    if (a.depth) a.depth[idx] = hit ? t_hit : 0.f;
    if (a.vertex) {
#pragma unroll
        for (int r = 0; r < 3; ++r) a.vertex[3 * idx + r] = P[r];
    }
    const double Pd[3] = {(double)P[0], (double)P[1], (double)P[2]};
    if (a.normal) {
        float n[3] = {0.f, 0.f, 0.f};
        if (hit) normal_at_hit(a, Pd, n);
#pragma unroll
        for (int r = 0; r < 3; ++r) a.normal[3 * idx + r] = n[r];
    }
    if (a.rgb) {
        uint8_t c[3] = {0, 0, 0};
        if (hit && a.color) color_at(a, Pd, c);
#pragma unroll
        for (int r = 0; r < 3; ++r) a.rgb[3 * idx + r] = c[r];
    }
}

static bool finite_all(const double* p, int n) {
    for (int i = 0; i < n; ++i)
        if (!std::isfinite(p[i])) return false;
    return true;
}

// Iteration cap of a ray (DESIGN §4).  Every iteration moves t by at least dt_vox = vl / |d_c| in exact arithmetic:
// one-voxel steps add it, truncation steps add more, absent-block jumps take the larger of it and the exit distance.
// The host refuses windows with depth_max * max|d_c| / vl > 2^22, so dt_vox >= 2 ulp(t) for every t < depth_max and the
// rounded sum fl(t + dt) >= t + dt - ulp(t) >= t + dt_vox / 2 (dt itself is rounded by at most 2^-24 relative).  A ray
// that marches its whole window [depth_min, depth_max) therefore needs at most
//   (depth_max - depth_min) / (dt_vox / 2) + 1 <= 2 (depth_max - depth_min) max|d_c| / vl + 1
// iterations; the cap adds 4 more.  A ray that reaches it (none can, by this argument) is a miss.
static int64_t raycast_cap(double dmin, double dmax, double max_len, double vl) {
    return (int64_t)std::ceil(2.0 * (dmax - dmin) * max_len / vl) + 5;
}

// FP32 |d_c| exactly as the kernel forms it; the maximum over an image is at one of its corners
static float ray_len(int u, int v, float cx, float cy, float ifx, float ify) {
    const float xc = ((float)u - cx) * ifx, yc = ((float)v - cy) * ify;
    return std::sqrt((xc * xc + yc * yc) + 1.0f);
}

bool ray_view(const double* e, RayView* out) {
    double pose[16];
    if (!finite_all(e, 16) || !inverse4(e, pose)) return false;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) out->R[3 * r + c] = (float)pose[4 * r + c];
        out->o[r] = (float)pose[4 * r + 3];
    }
    return true;
}

int ray_args(const otslam_volume* v, int width, int height, const double intr[4], double depth_min, double depth_max,
             const char* op, RayArgs* out) {
    const std::string p(op);
    if (!v) return set_error(OTSLAM_ERR_INVALID, p + ": null volume");
    if (v->slab.n_ranks > 1)
        return set_error(OTSLAM_ERR_INVALID, p + ": slab-sharded volumes are not ray cast; load every rank's part file into one "
                                                 "volume (otslam_volume_load) and ray cast that");
    if (v->n_objects > 0 && v->sel_obj < 0) return set_error(OTSLAM_ERR_INVALID, "multi-object arena: otslam_volume_select_object first");
    RayArgs a{};
    a.W = width; a.H = height;
    a.cx = (float)intr[2]; a.cy = (float)intr[3];
    a.ifx = 1.0f / (float)intr[0]; a.ify = 1.0f / (float)intr[1];
    a.vl = (float)v->voxel_length;
    a.ktr = (float)((double)kStepFactor * v->sdf_trunc);
    a.dmin = (float)depth_min; a.dmax = (float)depth_max;
    float max_len = 0.f;
    for (int u : {0, width - 1})
        for (int vv : {0, height - 1}) max_len = std::max(max_len, ray_len(u, vv, a.cx, a.cy, a.ifx, a.ify));
    if (!(depth_max * max_len / v->voxel_length <= kMaxWindowVoxels))
        return set_error(OTSLAM_ERR_INVALID, p + ": depth_max * max|d_c| / voxel_length exceeds 2^22");
    a.cap = (int)raycast_cap(depth_min, depth_max, max_len, v->voxel_length);
    a.color = v->color_type == OTSLAM_COLOR_RGB8;
    a.gap = 0.99 * v->voxel_length;
    a.c.table = volume_hash(v); a.c.chunks = v->d_chunks.p;
    a.c.bkeys = nullptr; a.c.bslots = nullptr; a.c.n = 0; a.c.slab = v->slab;
    a.c.vl = v->voxel_length; a.c.half = 0.5 * v->voxel_length; a.c.unit = v->unit_length;
    a.c.x_off = v->n_objects > 0 ? obj_key_offset(v->sel_obj) : 0;
    a.c.arena = v->n_objects > 0;
    *out = a;
    return OTSLAM_OK;
}

int raycast_launch(RayArgs a, const RayView* d_views, int n_views, float* depth, float* vertex, float* normal, uint8_t* rgb,
                   cudaStream_t s) {
    a.views = d_views;
    a.depth = depth; a.vertex = vertex; a.normal = normal; a.rgb = rgb;
    const dim3 grid((unsigned)((a.W + kTileW - 1) / kTileW), (unsigned)((a.H + kTileH - 1) / kTileH), (unsigned)n_views);
    raycast_kernel<<<grid, kTileW * kTileH, 0, s>>>(a);
    OT_LAUNCHED();
    return OTSLAM_OK;
}

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_volume_raycast(otslam_volume* v, int n_views, int width, int height, const double intr[4], const double* extrinsics,
                          double depth_min, double depth_max, float* depth, float* vertex, float* normal, uint8_t* color,
                          int64_t* n_hits) {
    // ---- every argument is checked before any CUDA call
    if (n_hits) *n_hits = 0;
    if (n_views < 0) return set_error(OTSLAM_ERR_INVALID, "raycast: n_views < 0");
    if (width <= 0 || height <= 0) return set_error(OTSLAM_ERR_INVALID, "raycast: width and height must be > 0");
    if (!intr) return set_error(OTSLAM_ERR_INVALID, "raycast: null intrinsics");
    if (!finite_all(intr, 4) || !(intr[0] > 0.0) || !(intr[1] > 0.0))
        return set_error(OTSLAM_ERR_INVALID, "raycast: fx and fy must be finite and > 0, cx and cy finite");
    if (!std::isfinite(depth_min) || !std::isfinite(depth_max) || !(depth_min > 0.0) || !(depth_min < depth_max))
        return set_error(OTSLAM_ERR_INVALID, "raycast: need finite 0 < depth_min < depth_max");
    if (n_views > 0 && !extrinsics) return set_error(OTSLAM_ERR_INVALID, "raycast: null extrinsics");
    const int64_t px = (int64_t)width * height;
    if (n_views > 0 && px > INT64_MAX / 12 / n_views) return set_error(OTSLAM_ERR_INVALID, "raycast: output size overflows int64");
    std::vector<RayView> views((size_t)n_views);
    for (int i = 0; i < n_views; ++i)
        if (!ray_view(extrinsics + 16 * (size_t)i, &views[i]))
            return set_error(OTSLAM_ERR_INVALID, "raycast: extrinsic is not finite or is singular");
    RayArgs a{};
    OT_TRY(ray_args(v, width, height, intr, depth_min, depth_max, "raycast", &a));
    if (n_views == 0) return OTSLAM_OK;

    OT_TRY(use_device(v->device));
    cudaStream_t s = v->stream, cs = v->copy_stream;
    // which outputs live in host memory (staged) and which on the device (written in place)
    void* outs[4] = {depth, vertex, normal, color};
    const size_t elem[4] = {4, 12, 12, 3};
    bool host[4] = {false, false, false, false};
    size_t host_bytes_per_view = 0;
    for (int k = 0; k < 4; ++k) {
        if (!outs[k]) continue;
        cudaPointerAttributes at;
        OT_CUDA(cudaPointerGetAttributes(&at, outs[k]));
        host[k] = !(at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged);
        if (host[k]) host_bytes_per_view += elem[k] * (size_t)px;
    }
    const int chunk = host_bytes_per_view ? (int)std::max<size_t>(1, std::min<size_t>(kViewsPerChunk, kStagingBytes / host_bytes_per_view))
                                          : kViewsPerChunk;
    DevBuf<RayView> d_views;
    DevBuf<unsigned long long> d_hits;
    DevBuf<uint8_t> staging[2];
    OT_CUDA(d_views.alloc((size_t)n_views)); OT_CUDA(d_hits.alloc(1));
    if (host_bytes_per_view)
        for (auto& b : staging) OT_CUDA(b.alloc(host_bytes_per_view * (size_t)std::min(chunk, n_views)));
    Event rendered[2], copied[2];
    if (host_bytes_per_view)
        for (int b = 0; b < 2; ++b) {
            OT_CUDA(rendered[b].create(cudaEventDisableTiming));
            OT_CUDA(copied[b].create(cudaEventDisableTiming));
        }
    OT_CUDA(cudaMemcpyAsync(d_views.p, views.data(), sizeof(RayView) * views.size(), cudaMemcpyHostToDevice, s));
    OT_CUDA(cudaMemsetAsync(d_hits.p, 0, 8, s));
    a.hits = d_hits.p;
    {
        OpTimer timer(s);
        for (int first = 0, k = 0; first < n_views; first += chunk, ++k) {
            const int nv = std::min(chunk, n_views - first);
            const int buf = k & 1;
            if (host_bytes_per_view && k >= 2) OT_CUDA(cudaStreamWaitEvent(s, copied[buf], 0));   // staging buffer free again
            uint8_t* stage = host_bytes_per_view ? staging[buf].p : nullptr;
            uint8_t* dst[4];
            size_t off = 0;
            for (int j = 0; j < 4; ++j) {
                dst[j] = nullptr;
                if (!outs[j]) continue;
                if (host[j]) { dst[j] = stage + off; off += elem[j] * (size_t)px * nv; }
                else dst[j] = (uint8_t*)outs[j] + elem[j] * (size_t)px * first;
            }
            OT_TRY(raycast_launch(a, d_views.p + first, nv, (float*)dst[0], (float*)dst[1], (float*)dst[2], dst[3], s));
            if (host_bytes_per_view) {
                OT_CUDA(cudaEventRecord(rendered[buf], s));
                OT_CUDA(cudaStreamWaitEvent(cs, rendered[buf], 0));
                for (int j = 0; j < 4; ++j)
                    if (outs[j] && host[j])
                        OT_CUDA(cudaMemcpyAsync((uint8_t*)outs[j] + elem[j] * (size_t)px * first, dst[j], elem[j] * (size_t)px * nv,
                                                cudaMemcpyDeviceToHost, cs));
                OT_CUDA(cudaEventRecord(copied[buf], cs));
            }
        }
        timer.stop();
    }
    unsigned long long total = 0;
    OT_CUDA(cudaMemcpyAsync(&total, d_hits.p, 8, cudaMemcpyDeviceToHost, s));
    OT_CUDA(cudaStreamSynchronize(s));
    OT_CUDA(cudaStreamSynchronize(cs));
    if (n_hits) *n_hits = (int64_t)total;
    return OTSLAM_OK;
}

}  // extern "C"
