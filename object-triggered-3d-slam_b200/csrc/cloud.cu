// cloud.cu -- stateless image / mesh / cloud operators of the path on sm_100a.
//
//   backproject_rgbd   PointCloud.create_from_rgbd_image   (/root/reference/3d_model/check_one_frame.py:27, SURVEY A.12)
//   vertex_normals     TriangleMesh.compute_vertex_normals (3d_model/reconstruct_rgbd.py:113, A.9)
//   sample_uniform     TriangleMesh.sample_points_uniformly (3d_model/reconstruct_rgbd_filter.py:123, A.10)
//   zfilter            points[:,2] >= Z_FILTER_THRESHOLD + rebuild (reconstruct_rgbd_filter.py:126-132)
//   grid_to_points     create_map_cloud's per-pixel loop   (fusion/hybrid_map.py:45-55)
//   merge_pack         paint_uniform_color + `+=` + binary-PLY vertex records (fusion/hybrid_map.py:59,88-91,115,121)
//
// All of them are order-preserving stream compactions or maps; FP64 arithmetic is written with
// explicit round-to-nearest intrinsics in the reference's operation order so results are
// bit-identical to the CPU restatement.
#include <algorithm>
#include <vector>

#include "cta_ops.cuh"
#include "volume.cuh"

namespace otslam {

// ---- back-projection
struct BackprojArgs {
    const float* depth;
    const uint8_t* rgb;
    int W, H;
    double fx, fy, cx, cy;
    double pose[12];
};

__global__ void __launch_bounds__(256) backproject_kernel(BackprojArgs a, const int64_t* __restrict__ base, int* __restrict__ counts,
                                                          double* __restrict__ pts, double* __restrict__ cols) {
    __shared__ int warp_sum[8];
    const int64_t n = (int64_t)a.W * a.H;
    const int64_t p0 = (int64_t)blockIdx.x * kItemsPerCta + threadIdx.x * kItemsPerThread;
    float d[kItemsPerThread];
    int mine = 0;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        d[k] = (p0 + k < n) ? __ldg(a.depth + p0 + k) : 0.f;
        mine += (d[k] > 0.f);
    }
    int total;
    const int rank = cta_exclusive_scan<int, 8>(mine, warp_sum, &total);
    if (!base) {
        if (threadIdx.x == 0) counts[blockIdx.x] = total;
        return;
    }
    int64_t o = base[blockIdx.x] + rank;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        if (!(d[k] > 0.f)) continue;
        const int64_t p = p0 + k;
        const int i = (int)(p / a.W), j = (int)(p - (int64_t)i * a.W);
        const double z = (double)d[k];
        const double x = __ddiv_rn(__dmul_rn(__dsub_rn((double)j, a.cx), z), a.fx);
        const double y = __ddiv_rn(__dmul_rn(__dsub_rn((double)i, a.cy), z), a.fy);
#pragma unroll
        for (int r = 0; r < 3; ++r)
            pts[3 * o + r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.pose[4 * r], x), __dmul_rn(a.pose[4 * r + 1], y)),
                                                 __dmul_rn(a.pose[4 * r + 2], z)),
                                       a.pose[4 * r + 3]);
        if (a.rgb && cols) {
#pragma unroll
            for (int r = 0; r < 3; ++r) cols[3 * o + r] = __ddiv_rn((double)a.rgb[3 * p + r], 255.0);
        }
        ++o;
    }
}

// ---- z filter
__global__ void __launch_bounds__(256) zfilter_kernel(const double* __restrict__ pts, const double* __restrict__ cols, int64_t n,
                                                      double zmin, const int64_t* __restrict__ base, int* __restrict__ counts,
                                                      double* __restrict__ out_pts, double* __restrict__ out_cols) {
    __shared__ int warp_sum[8];
    const int64_t p0 = (int64_t)blockIdx.x * kItemsPerCta + threadIdx.x * kItemsPerThread;
    bool keep[kItemsPerThread];
    int mine = 0;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        keep[k] = (p0 + k < n) && (pts[3 * (p0 + k) + 2] >= zmin);
        mine += keep[k];
    }
    int total;
    const int rank = cta_exclusive_scan<int, 8>(mine, warp_sum, &total);
    if (!base) {
        if (threadIdx.x == 0) counts[blockIdx.x] = total;
        return;
    }
    int64_t o = base[blockIdx.x] + rank;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        if (!keep[k]) continue;
        const int64_t p = p0 + k;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            out_pts[3 * o + r] = pts[3 * p + r];
            if (cols) out_cols[3 * o + r] = cols[3 * p + r];
        }
        ++o;
    }
}

// ---- occupancy grid -> points
__global__ void __launch_bounds__(256) grid_points_kernel(const uint8_t* __restrict__ img, int W, int H, double res, double ox,
                                                          double oy, int thresh, const int64_t* __restrict__ base,
                                                          int* __restrict__ counts, double* __restrict__ out) {
    __shared__ int warp_sum[8];
    const int64_t n = (int64_t)W * H;
    const int64_t p0 = (int64_t)blockIdx.x * kItemsPerCta + threadIdx.x * kItemsPerThread;
    bool occ[kItemsPerThread];
    int mine = 0;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        occ[k] = (p0 + k < n) && ((int)img[p0 + k] < thresh);
        mine += occ[k];
    }
    int total;
    const int rank = cta_exclusive_scan<int, 8>(mine, warp_sum, &total);
    if (!base) {
        if (threadIdx.x == 0) counts[blockIdx.x] = total;
        return;
    }
    int64_t o = base[blockIdx.x] + rank;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        if (!occ[k]) continue;
        const int64_t p = p0 + k;
        const int r = (int)(p / W), c = (int)(p - (int64_t)r * W);
        out[3 * o] = __dadd_rn(ox, __dmul_rn((double)c, res));                 // wx = ox + c*res
        out[3 * o + 1] = __dadd_rn(oy, __dmul_rn((double)(H - 1 - r), res));   // wy = oy + (h-1-r)*res
        out[3 * o + 2] = 0.0;
        ++o;
    }
}

// ---- mesh sampling
__global__ void __launch_bounds__(256) tri_area_kernel(const double* __restrict__ v, const int32_t* __restrict__ f, int64_t nf,
                                                       double* __restrict__ area) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const double *a = v + 3 * (size_t)f[3 * t], *b = v + 3 * (size_t)f[3 * t + 1], *c = v + 3 * (size_t)f[3 * t + 2];
    double e1[3], e2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { e1[k] = __dsub_rn(b[k], a[k]); e2[k] = __dsub_rn(c[k], a[k]); }
    const double x0 = __dsub_rn(__dmul_rn(e1[1], e2[2]), __dmul_rn(e1[2], e2[1]));
    const double x1 = __dsub_rn(__dmul_rn(e1[2], e2[0]), __dmul_rn(e1[0], e2[2]));
    const double x2 = __dsub_rn(__dmul_rn(e1[0], e2[1]), __dmul_rn(e1[1], e2[0]));
    area[t] = __dmul_rn(0.5, __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(x0, x0), __dmul_rn(x1, x1)), __dmul_rn(x2, x2))));
}

// triangle t owns samples [end[t-1], end[t]) with end[t] = llround(cdf[t]*n) (last forced to n)
__global__ void __launch_bounds__(256) sample_kernel(const double* __restrict__ v, const double* __restrict__ col,
                                                     const double* __restrict__ nrm, const int32_t* __restrict__ f, int64_t nf,
                                                     const double* __restrict__ cdf, int64_t n, uint64_t seed,
                                                     double* __restrict__ op, double* __restrict__ oc, double* __restrict__ on) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    // smallest t with idx < end[t]
    int64_t lo = 0, hi = nf - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int64_t end = (mid == nf - 1) ? n : llround(__dmul_rn(cdf[mid], (double)n));
        if (idx < end) hi = mid; else lo = mid + 1;
    }
    const int32_t* tri = f + 3 * lo;
    const double r1 = u01(seed, 2 * (uint64_t)idx), r2 = u01(seed, 2 * (uint64_t)idx + 1);
    const double s = __dsqrt_rn(r1);
    const double a = __dsub_rn(1.0, s), b = __dmul_rn(s, __dsub_rn(1.0, r2)), c = __dmul_rn(s, r2);
    const size_t i0 = 3 * (size_t)tri[0], i1 = 3 * (size_t)tri[1], i2 = 3 * (size_t)tri[2];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        op[3 * idx + k] = __dadd_rn(__dadd_rn(__dmul_rn(a, v[i0 + k]), __dmul_rn(b, v[i1 + k])), __dmul_rn(c, v[i2 + k]));
        if (col && oc) oc[3 * idx + k] = __dadd_rn(__dadd_rn(__dmul_rn(a, col[i0 + k]), __dmul_rn(b, col[i1 + k])), __dmul_rn(c, col[i2 + k]));
        if (nrm && on) on[3 * idx + k] = __dadd_rn(__dadd_rn(__dmul_rn(a, nrm[i0 + k]), __dmul_rn(b, nrm[i1 + k])), __dmul_rn(c, nrm[i2 + k]));
    }
}

// ---- rigid-body edits (fusion/hybrid_map_manual.py:86-119) and the 2-D map paste (fusion/2d_selective_merge.py:58-69)
// mode 0: p' = (T[4x4] * [p,1]).xyz / w, n' = T[0:3,0:3] * n;  mode 1: p' = R[3x3] * (p - c) + c, n' = R * n.
// Product order ((m0*x + m1*y) + m2*z) + m3, as the oracle defines it.
struct RigidArgs {
    double m[16];       // mode 0: T row-major; mode 1: R in m[0..8], centre in m[9..11]
    int mode;
};
__global__ void __launch_bounds__(256) rigid_kernel(const double* __restrict__ pts, const double* __restrict__ nrm, int64_t n, RigidArgs a,
                                                    double* __restrict__ out_pts, double* __restrict__ out_nrm) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
    if (a.mode == 0) {
        double h[4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
            h[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.m[4 * r], x), __dmul_rn(a.m[4 * r + 1], y)), __dmul_rn(a.m[4 * r + 2], z)), a.m[4 * r + 3]);
#pragma unroll
        for (int r = 0; r < 3; ++r) out_pts[3 * i + r] = __ddiv_rn(h[r], h[3]);
    } else {
        x = __dsub_rn(x, a.m[9]); y = __dsub_rn(y, a.m[10]); z = __dsub_rn(z, a.m[11]);
#pragma unroll
        for (int r = 0; r < 3; ++r)
            out_pts[3 * i + r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.m[3 * r], x), __dmul_rn(a.m[3 * r + 1], y)), __dmul_rn(a.m[3 * r + 2], z)), a.m[9 + r]);
    }
    if (nrm && out_nrm) {
        const double p = nrm[3 * i], q = nrm[3 * i + 1], w = nrm[3 * i + 2];
        const int st = a.mode == 0 ? 4 : 3;
#pragma unroll
        for (int r = 0; r < 3; ++r)
            out_nrm[3 * i + r] = __dadd_rn(__dadd_rn(__dmul_rn(a.m[st * r], p), __dmul_rn(a.m[st * r + 1], q)), __dmul_rn(a.m[st * r + 2], w));
    }
}

// p' = (T * [p, 1]).xyz / w on device buffers (otslam_cloud_transform's arithmetic), queued on stream s; the cloud ICP
// moves its source by each update with it
int device_rigid_transform(const double* d_in, int64_t n, const double T[16], double* d_out, cudaStream_t s) {
    if (n <= 0) return OTSLAM_OK;
    RigidArgs a;
    for (int i = 0; i < 16; ++i) a.m[i] = T[i];
    a.mode = 0;
    rigid_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_in, nullptr, n, a, d_out, nullptr);
    OT_LAUNCHED();
    return OTSLAM_OK;
}

__global__ void __launch_bounds__(256) axis_extract_kernel(const double* __restrict__ pts, int64_t n, int axis, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = pts[3 * i + axis];
}

// one thread per pixel of the rectangle: overlay pixels that hold data (not within `threshold` of the
// "unknown" grey) replace the base map's
__global__ void __launch_bounds__(256) smart_paste_kernel(uint8_t* __restrict__ base, const uint8_t* __restrict__ overlay, int width, int x0,
                                                          int y0, int w, int h, int unknown, int threshold) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= w * h) return;
    const size_t p = (size_t)(y0 + i / w) * width + (x0 + i % w);
    const int v = overlay[p];
    if (v < unknown - threshold || v > unknown + threshold) base[p] = (uint8_t)v;
}

// ---- merge + paint + PLY record packing: 256 points per CTA staged through SMEM so that the
// 27-byte records leave as coalesced 16-byte stores.
struct MergeArgs {
    const double* const* pts;     // device array of per-cloud device pointers
    const double* const* cols;    // idem or null
    const int64_t* offsets;       // [n_clouds+1] exclusive prefix of counts
    const uint8_t* paint;         // [n_clouds][3] bytes, or null
    int n_clouds;
    int64_t total;
};

__device__ __forceinline__ uint8_t color_byte(double c) {
    c = fmin(1.0, fmax(0.0, c));
    return (uint8_t)floor(__dadd_rn(__dmul_rn(c, 255.0), 0.5));
}

__global__ void __launch_bounds__(256) merge_pack_kernel(MergeArgs a, uint8_t* __restrict__ out) {
    __shared__ __align__(16) uint8_t stage[256 * 27];
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p < a.total) {
        int lo = 0, hi = a.n_clouds - 1;
        while (lo < hi) {   // cloud of point p: largest c with offsets[c] <= p
            const int mid = (lo + hi + 1) >> 1;
            if (a.offsets[mid] <= p) lo = mid; else hi = mid - 1;
        }
        const int64_t q = p - a.offsets[lo];
        const double* src = a.pts[lo] + 3 * q;
        uint8_t* dst = stage + threadIdx.x * 27;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const unsigned long long bits = (unsigned long long)__double_as_longlong(src[k]);
#pragma unroll
            for (int b = 0; b < 8; ++b) dst[8 * k + b] = (uint8_t)(bits >> (8 * b));
        }
        if (a.paint) {
            dst[24] = a.paint[3 * lo]; dst[25] = a.paint[3 * lo + 1]; dst[26] = a.paint[3 * lo + 2];
        } else if (a.cols && a.cols[lo]) {
            const double* cs = a.cols[lo] + 3 * q;
            dst[24] = color_byte(cs[0]); dst[25] = color_byte(cs[1]); dst[26] = color_byte(cs[2]);
        } else {
            dst[24] = dst[25] = dst[26] = 0;
        }
    }
    __syncthreads();
    const int64_t first = (int64_t)blockIdx.x * 256;
    const int64_t npts = min((int64_t)256, a.total - first);
    const int64_t nbytes = npts * 27;
    uint8_t* o = out + first * 27;   // 256*27 = 6912 = 432*16: every CTA starts 16-byte aligned
    const int64_t nvec = nbytes / 16;
    for (int64_t i = threadIdx.x; i < nvec; i += 256)
        reinterpret_cast<uint4*>(o)[i] = reinterpret_cast<const uint4*>(stage)[i];
    for (int64_t i = nvec * 16 + threadIdx.x; i < nbytes; i += 256) o[i] = stage[i];
}

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_backproject_rgbd(const float* depth_m, const uint8_t* rgb, int width, int height, const double intr[4],
                            const double extrinsic[16], double* points, double* colors, int64_t* n_points, int device) {
    if (!depth_m || !intr || !n_points || width <= 0 || height <= 0) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    OT_TRY(use_device(device));
    const int64_t n = (int64_t)width * height;
    BackprojArgs a;
    double ident[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1}, pose[16];
    if (!inverse4(extrinsic ? extrinsic : ident, pose)) return set_error(OTSLAM_ERR_INVALID, "extrinsic matrix is singular");
    for (int i = 0; i < 12; ++i) a.pose[i] = pose[i];
    a.W = width; a.H = height; a.fx = intr[0]; a.fy = intr[1]; a.cx = intr[2]; a.cy = intr[3];
    DevBuf<float> dd;
    DevBuf<uint8_t> dc;
    OT_CUDA(dd.upload(depth_m, n));
    if (rgb) OT_CUDA(dc.upload(rgb, n * 3));
    a.depth = dd.p; a.rgb = rgb ? dc.p : nullptr;
    DevBuf<int> counts;
    DevBuf<int64_t> base;
    DevBuf<double> dp, dcol;
    cudaStream_t s = 0;
    auto launch = [&](int n_cta, const int64_t* b, int* cnt) -> int {
        backproject_kernel<<<n_cta, 256, 0, s>>>(a, b, cnt, dp.p, dcol.p);
        OT_LAUNCHED();
        return OTSLAM_OK;
    };
    int64_t m = 0;
    OT_TRY(compact_two_pass(n, s, &m, counts, base, launch));
    *n_points = m;
    if (m == 0 || !points) return OTSLAM_OK;
    OT_CUDA(dp.alloc(m * 3));
    if (rgb && colors) OT_CUDA(dcol.alloc(m * 3));
    OT_TRY(launch((int)((n + kItemsPerCta - 1) / kItemsPerCta), base.p, nullptr));
    OT_CUDA(dp.download(points, m * 3));
    if (rgb && colors) OT_CUDA(dcol.download(colors, m * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_mesh_vertex_normals(const double* vertices, int64_t n_vertices, const int32_t* faces, int64_t n_faces,
                               double* normals, int device) {
    if (n_vertices < 0 || n_faces < 0 || (n_vertices && (!vertices || !normals)) || (n_faces && !faces))
        return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    if (n_vertices == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    DevBuf<double> dv, dn;
    DevBuf<int32_t> df;
    OT_CUDA(dv.upload(vertices, n_vertices * 3)); OT_CUDA(dn.alloc(n_vertices * 3));
    OT_CUDA(n_faces ? df.upload(faces, n_faces * 3) : df.alloc(0));
    OT_TRY(device_vertex_normals(dv.p, n_vertices, df.p, n_faces, dn.p, 0));
    OT_CUDA(dn.download(normals, n_vertices * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_mesh_sample_uniform(const double* vertices, const double* colors, const double* normals, int64_t n_vertices,
                               const int32_t* faces, int64_t n_faces, int64_t n_samples, uint64_t seed, double* out_points,
                               double* out_colors, double* out_normals, int device) {
    if (n_samples <= 0) return set_error(OTSLAM_ERR_INVALID, "[SamplePointsUniformly] number_of_points <= 0");
    if (n_faces <= 0 || n_vertices <= 0 || !vertices || !faces) return set_error(OTSLAM_ERR_INVALID, "[SamplePointsUniformly] input mesh has no triangles");
    if (!out_points) return set_error(OTSLAM_ERR_INVALID, "null output");
    OT_TRY(use_device(device));
    DevBuf<double> dv, dc, dn, area, total, op, oc, on;
    DevBuf<int32_t> df;
    OT_CUDA(dv.upload(vertices, n_vertices * 3)); OT_CUDA(df.upload(faces, n_faces * 3)); OT_CUDA(area.alloc(n_faces)); OT_CUDA(total.alloc(1));
    const bool has_c = colors && out_colors, has_n = normals && out_normals;
    if (has_c) { OT_CUDA(dc.upload(colors, n_vertices * 3)); OT_CUDA(oc.alloc(n_samples * 3)); }
    if (has_n) { OT_CUDA(dn.upload(normals, n_vertices * 3)); OT_CUDA(on.alloc(n_samples * 3)); }
    OT_CUDA(op.alloc(n_samples * 3));
    OpTimer timer;
    tri_area_kernel<<<(unsigned)((n_faces + 255) / 256), 256>>>(dv.p, df.p, n_faces, area.p);
    OT_LAUNCHED();
    OT_TRY(device_ordered_sum(area.p, n_faces, 0, nullptr, 0.0, total.p, 0));
    OT_TRY(device_ordered_sum(area.p, n_faces, 1, total.p, 0.0, nullptr, 0));
    sample_kernel<<<(unsigned)((n_samples + 255) / 256), 256>>>(dv.p, has_c ? dc.p : nullptr, has_n ? dn.p : nullptr, df.p, n_faces,
                                                               area.p, n_samples, seed, op.p, oc.p, on.p);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(op.download(out_points, n_samples * 3));
    if (has_c) OT_CUDA(oc.download(out_colors, n_samples * 3));
    if (has_n) OT_CUDA(on.download(out_normals, n_samples * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_volume_mesh_sample(otslam_volume* v, int64_t n_samples, uint64_t seed, double* out_points, double* out_colors,
                              double* out_normals) {
    if (!v) return set_error(OTSLAM_ERR_INVALID, "null volume");
    if (n_samples <= 0) return set_error(OTSLAM_ERR_INVALID, "[SamplePointsUniformly] number_of_points <= 0");
    const MeshResult& m = v->mesh;
    if (m.nf <= 0 || m.nv <= 0) return set_error(OTSLAM_ERR_INVALID, "[SamplePointsUniformly] input mesh has no triangles");
    if (!out_points) return set_error(OTSLAM_ERR_INVALID, "null output");
    OT_TRY(use_device(v->device));
    cudaStream_t s = v->stream;
    DevBuf<double> area, total, op, oc, on;
    OT_CUDA(area.alloc(m.nf)); OT_CUDA(total.alloc(1)); OT_CUDA(op.alloc(n_samples * 3));
    if (out_colors) OT_CUDA(oc.alloc(n_samples * 3));
    if (out_normals) OT_CUDA(on.alloc(n_samples * 3));
    {
        OpTimer timer(s);
        tri_area_kernel<<<(unsigned)((m.nf + 255) / 256), 256, 0, s>>>(m.verts.p, m.faces.p, m.nf, area.p);
        OT_LAUNCHED();
        OT_TRY(device_ordered_sum(area.p, m.nf, 0, nullptr, 0.0, total.p, s));
        OT_TRY(device_ordered_sum(area.p, m.nf, 1, total.p, 0.0, nullptr, s));
        sample_kernel<<<(unsigned)((n_samples + 255) / 256), 256, 0, s>>>(m.verts.p, out_colors ? m.colors.p : nullptr,
                                                                          out_normals ? m.normals.p : nullptr, m.faces.p, m.nf, area.p,
                                                                          n_samples, seed, op.p, oc.p, on.p);
        OT_LAUNCHED();
    }
    OT_CUDA(cudaMemcpyAsync(out_points, op.p, n_samples * 24, cudaMemcpyDefault, s));
    if (out_colors) OT_CUDA(cudaMemcpyAsync(out_colors, oc.p, n_samples * 24, cudaMemcpyDefault, s));
    if (out_normals) OT_CUDA(cudaMemcpyAsync(out_normals, on.p, n_samples * 24, cudaMemcpyDefault, s));
    OT_CUDA(cudaStreamSynchronize(s));
    return OTSLAM_OK;
}

int otslam_cloud_zfilter(const double* points, const double* colors, int64_t n, double zmin, double* out_points,
                         double* out_colors, int64_t* n_out, int device) {
    if (n < 0 || !n_out || (n && (!points || !out_points))) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    *n_out = 0;
    if (n == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    DevBuf<double> dp, dc, op, oc;
    OT_CUDA(dp.upload(points, n * 3));
    const bool has_c = colors && out_colors;
    if (has_c) OT_CUDA(dc.upload(colors, n * 3));
    DevBuf<int> counts;
    DevBuf<int64_t> base;
    cudaStream_t s = 0;
    OpTimer timer;
    auto launch = [&](int n_cta, const int64_t* b, int* cnt) -> int {
        zfilter_kernel<<<n_cta, 256, 0, s>>>(dp.p, has_c ? dc.p : nullptr, n, zmin, b, cnt, op.p, oc.p);
        OT_LAUNCHED();
        return OTSLAM_OK;
    };
    int64_t m = 0;
    OT_TRY(compact_two_pass(n, s, &m, counts, base, launch));
    *n_out = m;
    if (m == 0) return OTSLAM_OK;
    OT_CUDA(op.alloc(m * 3));
    if (has_c) OT_CUDA(oc.alloc(m * 3));
    OT_TRY(launch((int)((n + kItemsPerCta - 1) / kItemsPerCta), base.p, nullptr));
    timer.stop();
    OT_CUDA(op.download(out_points, m * 3));
    if (has_c) OT_CUDA(oc.download(out_colors, m * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_grid_to_points(const uint8_t* gray, int width, int height, double resolution, double origin_x, double origin_y,
                          int threshold, double* out_points, int64_t* n_out, int device) {
    if (!gray || !n_out || width <= 0 || height <= 0) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    OT_TRY(use_device(device));
    const int64_t n = (int64_t)width * height;
    DevBuf<uint8_t> di;
    OT_CUDA(di.upload(gray, n));
    DevBuf<int> counts;
    DevBuf<int64_t> base;
    DevBuf<double> op;
    cudaStream_t s = 0;
    OpTimer timer;
    auto launch = [&](int n_cta, const int64_t* b, int* cnt) -> int {
        grid_points_kernel<<<n_cta, 256, 0, s>>>(di.p, width, height, resolution, origin_x, origin_y, threshold, b, cnt, op.p);
        OT_LAUNCHED();
        return OTSLAM_OK;
    };
    int64_t m = 0;
    OT_TRY(compact_two_pass(n, s, &m, counts, base, launch));
    *n_out = m;
    if (m == 0 || !out_points) return OTSLAM_OK;
    OT_CUDA(op.alloc(m * 3));
    OT_TRY(launch((int)((n + kItemsPerCta - 1) / kItemsPerCta), base.p, nullptr));
    timer.stop();
    OT_CUDA(op.download(out_points, m * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

static int rigid_apply(const double* points, const double* normals, int64_t n, const RigidArgs& a, double* out_points, double* out_normals,
                       int device) {
    if (n < 0 || (n && (!points || !out_points))) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    if (n == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    DevBuf<double> dp, dn, op, on;
    OT_CUDA(dp.upload(points, n * 3)); OT_CUDA(op.alloc(n * 3));
    const bool has_n = normals && out_normals;
    if (has_n) { OT_CUDA(dn.upload(normals, n * 3)); OT_CUDA(on.alloc(n * 3)); }
    OpTimer timer;
    rigid_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dp.p, has_n ? dn.p : nullptr, n, a, op.p, has_n ? on.p : nullptr);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(op.download(out_points, n * 3));
    if (has_n) OT_CUDA(on.download(out_normals, n * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_cloud_transform(const double* points, const double* normals, int64_t n, const double transform[16], double* out_points,
                           double* out_normals, int device) {
    if (!transform) return set_error(OTSLAM_ERR_INVALID, "null transform");
    RigidArgs a;
    for (int i = 0; i < 16; ++i) a.m[i] = transform[i];
    a.mode = 0;
    return rigid_apply(points, normals, n, a, out_points, out_normals, device);
}

int otslam_cloud_rotate(const double* points, const double* normals, int64_t n, const double rotation[9], const double center[3],
                        double* out_points, double* out_normals, int device) {
    if (!rotation || !center) return set_error(OTSLAM_ERR_INVALID, "null rotation / center");
    RigidArgs a;
    for (int i = 0; i < 9; ++i) a.m[i] = rotation[i];
    for (int i = 0; i < 3; ++i) a.m[9 + i] = center[i];
    for (int i = 12; i < 16; ++i) a.m[i] = 0.0;
    a.mode = 1;
    return rigid_apply(points, normals, n, a, out_points, out_normals, device);
}

int otslam_cloud_center(const double* points, int64_t n, double center[3], int device) {
    if (n < 0 || !center || (n && !points)) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    center[0] = center[1] = center[2] = 0.0;
    if (n == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    DevBuf<double> dp, ax, tot;
    OT_CUDA(dp.upload(points, n * 3)); OT_CUDA(ax.alloc(n)); OT_CUDA(tot.alloc(3));
    OpTimer timer;
    for (int a = 0; a < 3; ++a) {     // coordinates may be negative: the exact chain replays such chunks scalar-wise, still in index order
        axis_extract_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dp.p, n, a, ax.p);
        OT_LAUNCHED();
        OT_TRY(device_ordered_sum(ax.p, n, 0, nullptr, 0.0, tot.p + a, 0));
    }
    timer.stop();
    double h[3];
    OT_CUDA(cudaMemcpy(h, tot.p, 24, cudaMemcpyDefault));
    for (int a = 0; a < 3; ++a) center[a] = h[a] / (double)n;
    return OTSLAM_OK;
}

int otslam_grid_smart_paste(uint8_t* base, const uint8_t* overlay, int width, int height, int x, int y, int w, int h, int unknown_pixel,
                            int threshold, int device) {
    if (!base || !overlay || width <= 0 || height <= 0 || w < 0 || h < 0) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    if (x < 0 || y < 0 || (int64_t)x + w > width || (int64_t)y + h > height || w == 0 || h == 0) return OTSLAM_OK;   // reference: returns the base map unchanged
    OT_TRY(use_device(device));
    const size_t n = (size_t)width * height;
    DevBuf<uint8_t> db, dov;
    OT_CUDA(db.upload(base, n)); OT_CUDA(dov.upload(overlay, n));
    OpTimer timer;
    smart_paste_kernel<<<(unsigned)(((int64_t)w * h + 255) / 256), 256>>>(db.p, dov.p, width, x, y, w, h, unknown_pixel, threshold);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(db.download(base, n));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_cloud_merge_pack(int n_clouds, const double* const* points, const double* const* colors, const int64_t* counts,
                            const double* paint, uint8_t* out_records, int device) {
    if (n_clouds < 0 || (n_clouds && (!points || !counts)) || !out_records) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    if (n_clouds == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    std::vector<int64_t> off(n_clouds + 1, 0);
    for (int i = 0; i < n_clouds; ++i) {
        if (counts[i] < 0) return set_error(OTSLAM_ERR_INVALID, "negative point count");
        off[i + 1] = off[i] + counts[i];
    }
    const int64_t total = off[n_clouds];
    if (total == 0) return OTSLAM_OK;
    // inputs are uploaded cloud by cloud (one cudaMemcpyAsync each), output comes back in one copy
    std::vector<DevBuf<double>> dp(n_clouds), dc(n_clouds);
    std::vector<const double*> hp(n_clouds, nullptr), hc(n_clouds, nullptr);
    cudaStream_t s = 0;
    for (int i = 0; i < n_clouds; ++i) {
        if (counts[i] == 0) continue;
        OT_CUDA(dp[i].alloc(counts[i] * 3));
        OT_CUDA(cudaMemcpyAsync(dp[i].p, points[i], counts[i] * 24, cudaMemcpyDefault, s));
        hp[i] = dp[i].p;
        if (!paint && colors && colors[i]) {
            OT_CUDA(dc[i].alloc(counts[i] * 3));
            OT_CUDA(cudaMemcpyAsync(dc[i].p, colors[i], counts[i] * 24, cudaMemcpyDefault, s));
            hc[i] = dc[i].p;
        }
    }
    DevBuf<const double*> dpp, dcp;
    DevBuf<int64_t> doff;
    DevBuf<uint8_t> dpaint, dout;
    OT_CUDA(dpp.alloc(n_clouds)); OT_CUDA(dcp.alloc(n_clouds)); OT_CUDA(doff.alloc(n_clouds + 1)); OT_CUDA(dout.alloc(total * 27));
    OT_CUDA(cudaMemcpyAsync(dpp.p, hp.data(), n_clouds * sizeof(double*), cudaMemcpyDefault, s));
    OT_CUDA(cudaMemcpyAsync(dcp.p, hc.data(), n_clouds * sizeof(double*), cudaMemcpyDefault, s));
    OT_CUDA(cudaMemcpyAsync(doff.p, off.data(), (n_clouds + 1) * 8, cudaMemcpyDefault, s));
    std::vector<uint8_t> pb;
    if (paint) {
        pb.resize(3 * n_clouds);
        for (int i = 0; i < 3 * n_clouds; ++i) {
            const double c = std::min(1.0, std::max(0.0, paint[i]));
            pb[i] = (uint8_t)std::floor(c * 255.0 + 0.5);
        }
        OT_CUDA(dpaint.alloc(3 * n_clouds));
        OT_CUDA(cudaMemcpyAsync(dpaint.p, pb.data(), 3 * n_clouds, cudaMemcpyDefault, s));
    }
    MergeArgs a;
    a.pts = dpp.p; a.cols = dcp.p; a.offsets = doff.p; a.paint = paint ? dpaint.p : nullptr; a.n_clouds = n_clouds; a.total = total;
    OpTimer timer;
    merge_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(a, dout.p);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(cudaMemcpyAsync(out_records, dout.p, total * 27, cudaMemcpyDefault, s));
    OT_CUDA(cudaStreamSynchronize(s));
    return OTSLAM_OK;
}

}  // extern "C"
