// segment.cu -- PointCloud.cluster_dbscan and PointCloud.segment_plane on sm_100a (DESIGN.md §4 "Plane segmentation and
// DBSCAN clustering").
//
//   cluster_dbscan  the points within eps are found by knn.cu's 27-cell walk on a grid with cell ~ eps; no neighbour list
//                   is stored.  Core points are counted (walk stopped at min_points), joined by a lock-free union-find
//                   whose roots hook under the smaller index (the root of a component is its smallest index for every
//                   thread schedule), roots are ranked by a scan, border points take the smallest root among their core
//                   neighbours.
//   segment_plane   RANSAC in waves of hypotheses: one thread per hypothesis samples and fits, each CTA of the evaluation
//                   kernel holds a tile of points in registers and tests it against every plane of the wave, fixed trees
//                   sum the distances; the host applies Open3D's selection and break rule between waves.
#include <algorithm>
#include <cmath>
#include <cstdint>

#include "cta_ops.cuh"
#include "knn_grid.cuh"

namespace otslam {

// ---------------------------------------------------------------------------------------------
// DBSCAN
// ---------------------------------------------------------------------------------------------
constexpr int kDbThreads = 128;

// neighbours of the walk: d2 < eps^2 (point i itself included, d2 = 0)
__global__ void __launch_bounds__(kDbThreads) dbscan_count_kernel(KnnGrid g, const double* __restrict__ pts, int64_t n, double r2,
                                                                  int64_t min_points, int* __restrict__ core, int* __restrict__ parent) {
    const int64_t t = (int64_t)blockIdx.x * kDbThreads + threadIdx.x;
    if (t >= n) return;
    const int i = g.idx[t];                 // visit queries cell by cell: neighbouring threads share cells
    const double q[3] = {pts[3 * (size_t)i], pts[3 * (size_t)i + 1], pts[3 * (size_t)i + 2]};
    int64_t cnt = 0;
    if (min_points > 0)
        grid_walk27(g, pts, q, [&](int, double d2) { return !(d2 < r2 && ++cnt >= min_points); });
    core[i] = cnt >= min_points;
    parent[i] = i;
}

// parent[x] <= x always holds, so every pointer leads to a smaller index; the path is halved as it is walked (each store
// points a node at one of its ancestors, which stays true while trees merge)
__device__ __forceinline__ int uf_find(volatile int* parent, int x) {
    int cur = parent[x];
    if (cur == x) return x;
    int prev = x, next;
    while (cur > (next = parent[cur])) {
        parent[prev] = next;
        prev = cur;
        cur = next;
    }
    return cur;
}

// join the sets of roots-or-members a and b: the larger root is hooked under the smaller one by compare-and-swap; a failed
// swap means that root gained a parent meanwhile, and the loop continues from that parent
__device__ __forceinline__ void uf_hook(int* parent, int a, int b) {
    while (a != b) {
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicCAS(parent + b, b, a);
        if (old == b) return;
        b = old;
    }
}

__global__ void __launch_bounds__(kDbThreads) dbscan_union_kernel(KnnGrid g, const double* __restrict__ pts, int64_t n, double r2,
                                                                  const int* __restrict__ core, int* parent) {
    const int64_t t = (int64_t)blockIdx.x * kDbThreads + threadIdx.x;
    if (t >= n) return;
    const int i = g.idx[t];
    if (!core[i]) return;
    const double q[3] = {pts[3 * (size_t)i], pts[3 * (size_t)i + 1], pts[3 * (size_t)i + 2]};
    grid_walk27(g, pts, q, [&](int j, double d2) {
        if (j < i && d2 < r2 && core[j]) {          // each pair once, from its larger index
            const int rj = uf_find(parent, j), ri = uf_find(parent, i);
            if (ri != rj) uf_hook(parent, ri, rj);
        }
        return true;
    });
}

// root[i] = the root of core point i's component (= its smallest index); flag[i] = 1 for roots.  The roots go to an array
// of their own: the finds still halve paths in parent, and such a store may land on a node after a compressed root was
// stored there, so parent is not the result
__global__ void __launch_bounds__(256) dbscan_compress_kernel(int64_t n, const int* __restrict__ core, int* parent, int* __restrict__ root,
                                                              int* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    int f = 0;
    if (core[i]) {
        const int r = uf_find(parent, (int)i);
        root[i] = r;
        f = r == (int)i;
    }
    flag[i] = f;
}

// label = rank of the root; a non-core point takes the smallest root among its core neighbours (ranks follow root order,
// so this is the smallest label), or -1
__global__ void __launch_bounds__(kDbThreads, 4) dbscan_label_kernel(KnnGrid g, const double* __restrict__ pts, int64_t n, double r2,
                                                                  const int* __restrict__ core, const int* __restrict__ root,
                                                                  const int64_t* __restrict__ rank, int32_t* __restrict__ labels) {
    const int64_t t = (int64_t)blockIdx.x * kDbThreads + threadIdx.x;
    if (t >= n) return;
    const int i = g.idx[t];
    if (core[i]) {
        labels[i] = (int32_t)rank[root[i]];
        return;
    }
    const double q[3] = {pts[3 * (size_t)i], pts[3 * (size_t)i + 1], pts[3 * (size_t)i + 2]};
    int best = 0x7fffffff;
    grid_walk27(g, pts, q, [&](int j, double d2) {
        if (d2 < r2 && core[j]) best = min(best, root[j]);
        return true;
    });
    labels[i] = best == 0x7fffffff ? -1 : (int32_t)rank[best];
}

// ---------------------------------------------------------------------------------------------
// RANSAC plane segmentation
// ---------------------------------------------------------------------------------------------
constexpr int kSegThreads = 256;
constexpr int kSegItems = 8;                              // points per thread
constexpr int kSegTile = kSegThreads * kSegItems;         // points per CTA: position c * kSegTile + k * 256 + thread
constexpr int kWave = 64;                                 // hypotheses per wave
constexpr int kMaxRansacN = 16;

// Open3D's GetPlaneFromPoints from the centroid and the centred second moments xx, xy, xz, yy, yz, zz; false (and a zero
// plane) when the points do not span a plane
__host__ __device__ inline bool plane_from_moments(const double c[3], const double m[6], double out[4]) {
    const double xx = m[0], xy = m[1], xz = m[2], yy = m[3], yz = m[4], zz = m[5];
    const double det_x = yy * zz - yz * yz, det_y = xx * zz - xz * xz, det_z = xx * yy - xy * xy;
    double a, b, cc;
    if (det_x > det_y && det_x > det_z) { a = det_x; b = xz * yz - xy * zz; cc = xy * yz - xz * yy; }
    else if (det_y > det_z) { a = xz * yz - xy * zz; b = det_y; cc = xy * xz - yz * xx; }
    else { a = xy * yz - xz * yy; b = xy * xz - yz * xx; cc = det_z; }
    const double norm = sqrt((a * a + b * b) + cc * cc);
    if (norm == 0.0) { out[0] = out[1] = out[2] = out[3] = 0.0; return false; }
    a = a / norm; b = b / norm; cc = cc / norm;
    out[0] = a; out[1] = b; out[2] = cc;
    out[3] = -((a * c[0] + b * c[1]) + cc * c[2]);
    return true;
}

// one thread per hypothesis h = h0 + w: r distinct indices by Floyd's algorithm on u01(seed, h * r + k), then the plane
// (Open3D's ComputeTrianglePlane for r = 3, GetPlaneFromPoints over the sample in draw order for r > 3); invalid = zero
__global__ void __launch_bounds__(kWave) ransac_hypothesis_kernel(const double* __restrict__ pts, int64_t n, int r, uint64_t seed,
                                                                  int64_t h0, int w_count, double4* __restrict__ planes) {
    const int w = threadIdx.x;
    if (w >= w_count) return;
    const uint64_t h = (uint64_t)(h0 + w);
    int64_t s[kMaxRansacN];
    for (int k = 0; k < r; ++k) {
        const int64_t j = n - r + k;
        int64_t t = (int64_t)floor(__dmul_rn(u01(seed, h * (uint64_t)r + (uint64_t)k), (double)(j + 1)));
        if (t > j) t = j;
        for (int e = 0; e < k; ++e)
            if (s[e] == t) { t = j; break; }
        s[k] = t;
    }
    double pl[4];
    if (r == 3) {
        const double* p0 = pts + 3 * s[0];
        const double* p1 = pts + 3 * s[1];
        const double* p2 = pts + 3 * s[2];
        const double e0[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]}, e1[3] = {p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2]};
        double a = e0[1] * e1[2] - e0[2] * e1[1], b = e0[2] * e1[0] - e0[0] * e1[2], c = e0[0] * e1[1] - e0[1] * e1[0];
        const double norm = sqrt((a * a + b * b) + c * c);
        if (norm == 0.0) {
            pl[0] = pl[1] = pl[2] = pl[3] = 0.0;
        } else {
            a = a / norm; b = b / norm; c = c / norm;
            pl[0] = a; pl[1] = b; pl[2] = c;
            pl[3] = -((a * p0[0] + b * p0[1]) + c * p0[2]);
        }
    } else {
        double cen[3] = {0.0, 0.0, 0.0}, m[6] = {0, 0, 0, 0, 0, 0};
        for (int k = 0; k < r; ++k)
            for (int a = 0; a < 3; ++a) cen[a] = cen[a] + pts[3 * s[k] + a];
        for (int a = 0; a < 3; ++a) cen[a] = cen[a] / (double)r;
        for (int k = 0; k < r; ++k) {
            const double x = pts[3 * s[k]] - cen[0], y = pts[3 * s[k] + 1] - cen[1], z = pts[3 * s[k] + 2] - cen[2];
            m[0] = m[0] + x * x; m[1] = m[1] + x * y; m[2] = m[2] + x * z;
            m[3] = m[3] + y * y; m[4] = m[4] + y * z; m[5] = m[5] + z * z;
        }
        plane_from_moments(cen, m, pl);
    }
    planes[w] = make_double4(pl[0], pl[1], pl[2], pl[3]);
}

// point-to-plane distance of the evaluation, the final inlier test and the rule: |((a x + b y) + c z) + d|
__device__ __forceinline__ double plane_dist(const double4& p, double x, double y, double z) {
    return fabs(((p.x * x + p.y * y) + p.z * z) + p.w);
}

// the fixed tree inside a warp: lane l += lane l + 16, + 8, ..., + 1 (xor partners compute the same sums)
__device__ __forceinline__ double warp_tree(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = v + __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_isum(int v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// ... and over the 8 warp sums of a CTA: w += w + 4, + 2, + 1
__device__ __forceinline__ double cta_tree8(const double* ws) {
    double v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = ws[k];
#pragma unroll
    for (int o = 4; o; o >>= 1)
#pragma unroll
        for (int k = 0; k < o; ++k) v[k] = v[k] + v[k + o];
    return v[0];
}

// each CTA: a tile of kSegTile points in registers against the w_count planes of the wave; partials[w][cta] = the tile's
// inlier count (-1 for an invalid plane, so that its total is negative), partials[w_count + w][cta] = the tile's sum of
// inlier distances (thread: items in k order, then the trees)
__global__ void __launch_bounds__(kSegThreads) ransac_eval_kernel(const double* __restrict__ pts, int64_t n, const double4* __restrict__ planes,
                                                                  int w_count, double thr, double* __restrict__ partials, int P) {
    __shared__ double4 sp[kWave];
    __shared__ double ssum[kWave][8];
    __shared__ int scnt[kWave][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < w_count) sp[threadIdx.x] = planes[threadIdx.x];
    double x[kSegItems], y[kSegItems], z[kSegItems];
    bool ok[kSegItems];
    const int64_t base = (int64_t)blockIdx.x * kSegTile + threadIdx.x;
#pragma unroll
    for (int k = 0; k < kSegItems; ++k) {
        const int64_t p = base + (int64_t)k * kSegThreads;
        ok[k] = p < n;
        x[k] = ok[k] ? pts[3 * p] : 0.0;
        y[k] = ok[k] ? pts[3 * p + 1] : 0.0;
        z[k] = ok[k] ? pts[3 * p + 2] : 0.0;
    }
    __syncthreads();
    for (int w = 0; w < w_count; ++w) {
        const double4 pl = sp[w];
        double s = 0.0;
        int c = 0;
#pragma unroll
        for (int k = 0; k < kSegItems; ++k) {
            const double d = plane_dist(pl, x[k], y[k], z[k]);
            const bool in = ok[k] && d < thr;
            s = s + (in ? d : 0.0);
            c += in;
        }
        s = warp_tree(s);
        c = warp_isum(c);
        if (lane == 0) { ssum[w][warp] = s; scnt[w][warp] = c; }
    }
    __syncthreads();
    if (threadIdx.x < w_count) {
        const int w = threadIdx.x;
        int c = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) c += scnt[w][k];
        const double4 pl = sp[w];
        const bool valid = pl.x != 0.0 || pl.y != 0.0 || pl.z != 0.0 || pl.w != 0.0;
        partials[(size_t)w * P + blockIdx.x] = valid ? (double)c : -1.0;
        partials[(size_t)(w_count + w) * P + blockIdx.x] = cta_tree8(ssum[w]);
    }
}

// an inlier of the selected plane, by the test of its evaluation
struct PlaneInlier {
    const double* pts;
    const double4* plane;
    double thr;
    __device__ bool operator()(int64_t p) const {
        return plane_dist(*plane, pts[3 * p], pts[3 * p + 1], pts[3 * p + 2]) < thr;
    }
};

// the refit's sums over the m inliers, positions as in ransac_eval_kernel: mode 0 the 3 coordinate sums, mode 1 the 6
// centred moments xx, xy, xz, yy, yz, zz about cen; partials[term][cta]
__global__ void __launch_bounds__(kSegThreads) refit_sum_kernel(const double* __restrict__ pts, const int64_t* __restrict__ idx, int64_t m,
                                                                int mode, double cx, double cy, double cz, double* __restrict__ partials, int P) {
    __shared__ double ws[6][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_terms = mode == 0 ? 3 : 6;
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const int64_t base = (int64_t)blockIdx.x * kSegTile + threadIdx.x;
#pragma unroll
    for (int k = 0; k < kSegItems; ++k) {
        const int64_t p = base + (int64_t)k * kSegThreads;
        double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (p < m) {
            const int64_t i = idx[p];
            const double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
            if (mode == 0) { v[0] = x; v[1] = y; v[2] = z; }
            else {
                const double rx = x - cx, ry = y - cy, rz = z - cz;
                v[0] = rx * rx; v[1] = rx * ry; v[2] = rx * rz; v[3] = ry * ry; v[4] = ry * rz; v[5] = rz * rz;
            }
        }
#pragma unroll
        for (int t = 0; t < 6; ++t) acc[t] = acc[t] + v[t];
    }
#pragma unroll
    for (int t = 0; t < 6; ++t) {
        const double s = warp_tree(acc[t]);
        if (lane == 0) ws[t][warp] = s;
    }
    __syncthreads();
    if (threadIdx.x < n_terms) partials[(size_t)threadIdx.x * P + blockIdx.x] = cta_tree8(ws[threadIdx.x]);
}

// the rows' fixed-tree totals of n_terms partial rows -> host
static int refit_sums(const double* d_pts, const int64_t* d_idx, int64_t m, int mode, const double cen[3], double* h_out) {
    const int n_cta = (int)((m + kSegTile - 1) / kSegTile), P = pow2_at_least(n_cta), n_terms = mode == 0 ? 3 : 6;
    DevBuf<double> part, tot;
    OT_CUDA(part.alloc((size_t)n_terms * P)); OT_CUDA(tot.alloc(n_terms));
    refit_sum_kernel<<<n_cta, kSegThreads>>>(d_pts, d_idx, m, mode, cen[0], cen[1], cen[2], part.p, P);
    OT_LAUNCHED();
    tree_rows_kernel<256><<<n_terms, 256>>>(part.p, n_cta, P, tot.p);
    OT_LAUNCHED();
    OT_CUDA(cudaMemcpy(h_out, tot.p, n_terms * sizeof(double), cudaMemcpyDeviceToHost));
    return OTSLAM_OK;
}

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_cloud_cluster_dbscan(const double* points, int64_t n, double eps, int64_t min_points, int32_t* out_labels, int32_t* n_clusters,
                                int device) {
    // ---- every argument is checked before any CUDA call
    if (!(eps > 0.0) || !std::isfinite(eps)) return set_error(OTSLAM_ERR_INVALID, "cluster_dbscan: eps must be finite and > 0");
    if (min_points < 0) return set_error(OTSLAM_ERR_INVALID, "cluster_dbscan: min_points < 0");
    if (n < 0 || n > 0x7fffffffLL) return set_error(OTSLAM_ERR_INVALID, "cluster_dbscan: n must be in [0, 2^31)");
    if (n && (!points || !out_labels)) return set_error(OTSLAM_ERR_INVALID, "cluster_dbscan: null points or out_labels");
    if (n_clusters) *n_clusters = 0;
    if (n == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    DevBuf<double> dp;
    DevBuf<int> core, parent, root, flag;
    DevBuf<int64_t> rank;
    DevBuf<int32_t> dl;
    OT_CUDA(dp.upload(points, n * 3)); OT_CUDA(core.alloc(n)); OT_CUDA(parent.alloc(n)); OT_CUDA(root.alloc(n)); OT_CUDA(flag.alloc(n));
    OT_CUDA(rank.alloc(n + 1)); OT_CUDA(dl.alloc(n));
    OpTimer timer;
    double mn[3], mx[3];
    OT_TRY(cloud_minmax(dp.p, n, mn, mx));
    // the cell is eps enlarged by 2^-20: two points with a computed d2 < eps^2 then lie in adjacent cells whatever the
    // rounding of their cell coordinates, so the 27-cell walk sees every neighbour (build_grid may enlarge it further)
    GridBuffers b;
    KnnGrid g;
    OT_TRY(build_grid(dp.p, n, mn, mx, eps * (1.0 + 1.0 / 1048576.0), 1 << 20, b, g));
    const double r2 = eps * eps;
    const unsigned grid = (unsigned)((n + kDbThreads - 1) / kDbThreads), grid256 = (unsigned)((n + 255) / 256);
    dbscan_count_kernel<<<grid, kDbThreads>>>(g, dp.p, n, r2, min_points, core.p, parent.p);
    OT_LAUNCHED();
    dbscan_union_kernel<<<grid, kDbThreads>>>(g, dp.p, n, r2, core.p, parent.p);
    OT_LAUNCHED();
    dbscan_compress_kernel<<<grid256, 256>>>(n, core.p, parent.p, root.p, flag.p);
    OT_LAUNCHED();
    OT_TRY(device_exclusive_scan(flag.p, rank.p, (int)n, 0));
    dbscan_label_kernel<<<grid, kDbThreads>>>(g, dp.p, n, r2, core.p, root.p, rank.p, dl.p);
    OT_LAUNCHED();
    timer.stop();
    int64_t total = 0;
    OT_CUDA(cudaMemcpy(&total, rank.p + n, 8, cudaMemcpyDeviceToHost));
    OT_CUDA(dl.download(out_labels, n));
    OT_CUDA(cudaDeviceSynchronize());
    if (n_clusters) *n_clusters = (int32_t)total;
    return OTSLAM_OK;
}

int otslam_cloud_segment_plane(const double* points, int64_t n, double distance_threshold, int ransac_n, int num_iterations,
                               double probability, uint64_t seed, double plane_out[4], int64_t* out_inliers, int64_t* n_inliers,
                               int32_t* n_evaluated, int device) {
    // ---- every argument is checked before any CUDA call
    if (!plane_out || !n_inliers) return set_error(OTSLAM_ERR_INVALID, "segment_plane: null plane_out or n_inliers");
    if (n < 0 || n > 0x7fffffffLL) return set_error(OTSLAM_ERR_INVALID, "segment_plane: n must be in [0, 2^31)");
    if (n && (!points || !out_inliers)) return set_error(OTSLAM_ERR_INVALID, "segment_plane: null points or out_inliers");
    if (!(distance_threshold >= 0.0) || !std::isfinite(distance_threshold))
        return set_error(OTSLAM_ERR_INVALID, "segment_plane: distance_threshold must be finite and >= 0");
    if (ransac_n < 3) return set_error(OTSLAM_ERR_INVALID, "ransac_n should be set to higher than or equal to 3.");
    if (ransac_n > kMaxRansacN) return set_error(OTSLAM_ERR_INVALID, "segment_plane: ransac_n > 16 is not supported");
    if (num_iterations < 0) return set_error(OTSLAM_ERR_INVALID, "segment_plane: num_iterations < 0");
    if (!(probability > 0.0 && probability <= 1.0)) return set_error(OTSLAM_ERR_INVALID, "Probability must be > 0 or <= 1.0");
    if (n < ransac_n) return set_error(OTSLAM_ERR_INVALID, "There must be at least 'ransac_n' points.");
    for (int k = 0; k < 4; ++k) plane_out[k] = 0.0;
    *n_inliers = 0;
    if (n_evaluated) *n_evaluated = 0;
    OT_TRY(use_device(device));
    const int n_cta = (int)((n + kSegTile - 1) / kSegTile), P = pow2_at_least(n_cta);
    DevBuf<double> dp, part, res;
    DevBuf<double4> planes, best_plane;
    OT_CUDA(dp.upload(points, n * 3)); OT_CUDA(part.alloc((size_t)2 * kWave * P)); OT_CUDA(res.alloc(2 * kWave));
    OT_CUDA(planes.alloc(kWave)); OT_CUDA(best_plane.alloc(1));
    OpTimer timer;
    // Open3D's selection in hypothesis order: skip h > B; replace on a greater fitness, or an equal one with a smaller rmse
    int64_t B = INT64_MAX;
    bool have_best = false;
    double best_fit = 0.0, best_rmse = 0.0;
    int32_t evaluated = 0;
    double h_res[2 * kWave];
    for (int64_t h0 = 0; h0 < num_iterations && h0 <= B; h0 += kWave) {
        const int wn = (int)std::min<int64_t>(kWave, num_iterations - h0);
        ransac_hypothesis_kernel<<<1, kWave>>>(dp.p, n, ransac_n, seed, h0, wn, planes.p);
        OT_LAUNCHED();
        ransac_eval_kernel<<<n_cta, kSegThreads>>>(dp.p, n, planes.p, wn, distance_threshold, part.p, P);
        OT_LAUNCHED();
        tree_rows_kernel<256><<<2 * wn, 256>>>(part.p, n_cta, P, res.p);
        OT_LAUNCHED();
        OT_CUDA(cudaMemcpy(h_res, res.p, 2 * wn * sizeof(double), cudaMemcpyDeviceToHost));
        for (int w = 0; w < wn; ++w) {
            const int64_t h = h0 + w;
            if (h > B) break;
            ++evaluated;
            const double count = h_res[w], fit = count / (double)n;
            if (count < 0.0) continue;              // invalid plane
            const double rmse = count > 0.0 ? h_res[wn + w] / std::sqrt(count) : 0.0;
            if (fit > best_fit || (fit == best_fit && rmse < best_rmse)) {
                best_fit = fit;
                best_rmse = rmse;
                have_best = true;
                OT_CUDA(cudaMemcpy(best_plane.p, planes.p + w, sizeof(double4), cudaMemcpyDeviceToDevice));
                if (fit < 1.0) {
                    const double q = std::log(1.0 - probability) / std::log(1.0 - std::pow(fit, (double)ransac_n));
                    B = (q >= 0.0 && q < (double)num_iterations) ? (int64_t)std::floor(q) : (int64_t)num_iterations;
                } else {
                    B = 0;
                }
            }
        }
    }
    if (n_evaluated) *n_evaluated = evaluated;
    if (!have_best) return OTSLAM_OK;
    // the best plane's inliers (the same test as its evaluation), then GetPlaneFromPoints over them by the fixed trees
    DevBuf<int64_t> oidx;
    int64_t m = 0;
    OT_TRY(select_indices(PlaneInlier{dp.p, best_plane.p, distance_threshold}, n, 0, oidx, &m));
    double sum[3], mom[6], cen[3] = {0.0, 0.0, 0.0};
    OT_TRY(refit_sums(dp.p, oidx.p, m, 0, cen, sum));
    for (int a = 0; a < 3; ++a) cen[a] = sum[a] / (double)m;
    OT_TRY(refit_sums(dp.p, oidx.p, m, 1, cen, mom));
    timer.stop();
    plane_from_moments(cen, mom, plane_out);
    OT_CUDA(oidx.download(out_inliers, m));
    OT_CUDA(cudaDeviceSynchronize());
    *n_inliers = m;
    return OTSLAM_OK;
}

}  // extern "C"
