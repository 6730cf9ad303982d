// knn_grid.cuh -- the uniform grid of knn.cu (points bucketed by cell, cell -> bucket hash) as seen by the other
// translation units that search it: the DBSCAN passes of segment.cu walk the same 27 cells with the same arithmetic.
#pragma once
#include "volume.cuh"

namespace otslam {

// key = floor((p - origin) / cell) per axis packed as kx << sh_x | ky << sh_y | kz with just enough
// bits per axis (the host sizes them from the bounding box), so the sort needs few passes and
// key order == lexicographic (x, y, z)
struct KeyLayout {
    int sh_x, sh_y, bits;
    uint64_t mask_y, mask_z;
};
__host__ __device__ inline uint64_t layout_key(const KeyLayout& L, int x, int y, int z) {
    return ((uint64_t)(uint32_t)x << L.sh_x) | ((uint64_t)(uint32_t)y << L.sh_y) | (uint64_t)(uint32_t)z;
}

// one level of the search structure: points bucketed by uniform-grid cell (sorted by cell key), cell -> bucket hash
struct KnnGrid {
    const int32_t* idx;         // sorted position -> original index
    const int32_t* seg_start;   // [n_seg+1]
    HashTable cells;            // cell key -> segment id
    double mn[3], cell;
    int dim[3];
    KeyLayout L;
};

// ---- host side of the search structure
struct GridBuffers {
    DevBuf<uint64_t> k0, k1, hk;
    DevBuf<int32_t> i0, i1, seg, hv;
    int64_t n_seg = 0;
};

// exact per-axis min / max of n FP64 points on the device
int cloud_minmax(const double* d_pts, int64_t n, double* mn, double* mx);
// bucket the n points of d_pts on a grid of `cell`-sized cells over [mn, mx] (at most max_dim cells per axis: the cell
// may grow, never shrink)
int build_grid(const double* d_pts, int64_t n, const double mn[3], const double mx[3], double cell, int max_dim, GridBuffers& b,
               KnnGrid& g);

// Calls f(pi, d2) for every point pi of the 27 cells around q, d2 = (dx^2 + dy^2) + dz^2 in FP64 without FMA, cells in
// (z, y, x) order and points in bucket order; f returns false to stop the walk.  With cell >= r, the points with d2 < r^2
// are all among them.
template <typename F>
__device__ __forceinline__ void grid_walk27(const KnnGrid& g, const double* __restrict__ pts, const double (&q)[3], F&& f) {
    int c[3];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax)      // may lie outside the grid: clamp to one cell beyond it (still "no cell in range")
        c[ax] = (int)fmin(fmax(floor(__ddiv_rn(__dsub_rn(q[ax], g.mn[ax]), g.cell)), -2.0), (double)g.dim[ax] + 1.0);
    for (int dz = -1; dz <= 1; ++dz)
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                const int x = c[0] + dx, y = c[1] + dy, z = c[2] + dz;
                if (x < 0 || x >= g.dim[0] || y < 0 || y >= g.dim[1] || z < 0 || z >= g.dim[2]) continue;
                const int seg = hash_find(g.cells, layout_key(g.L, x, y, z));
                if (seg < 0) continue;
                for (int j = g.seg_start[seg]; j < g.seg_start[seg + 1]; ++j) {
                    const int pi = g.idx[j];
                    const double ex = __dsub_rn(q[0], pts[3 * (size_t)pi]), ey = __dsub_rn(q[1], pts[3 * (size_t)pi + 1]),
                                 ez = __dsub_rn(q[2], pts[3 * (size_t)pi + 2]);
                    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
                    if (!f(pi, d2)) return;
                }
            }
}

// ---- correspondence search of point-to-point ICP (o3d.pipelines.registration.registration_icp,
// /root/reference/eval/eval_table_chair/eval_table_chair.py:90-104): for every source point the nearest target point
// strictly closer than `radius` (KDTree SearchHybrid(point, radius, 1)), or -1.  The radius bounds the search, so a uniform
// grid with cell = radius needs the 27 cells around the query only: one thread per query, exact FP64 squared distances in
// the (dx^2 + dy^2) + dz^2 order, ties broken towards the lower target index (deterministic).
__device__ __forceinline__ void nn_within_search(const KnnGrid& g, const double* __restrict__ pts, const double (&q)[3], double r2,
                                                 int& bi, double& best) {
    best = r2;
    bi = -1;
    grid_walk27(g, pts, q, [&](int pi, double d2) {
        if (d2 < best || (d2 == best && bi >= 0 && pi < bi)) { best = d2; bi = pi; }
        return true;
    });
}

}  // namespace otslam
