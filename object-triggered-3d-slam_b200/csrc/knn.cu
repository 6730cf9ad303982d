// knn.cu -- voxel_down_sample and statistical outlier removal on sm_100a.
//
//   voxel_down_sample          PointCloud.voxel_down_sample (/root/reference/3d_model/check_one_frame.py:28, SURVEY A.7)
//   remove_statistical_outlier PointCloud.remove_statistical_outlier (north_star; SURVEY A.8)
//
// Both need "sum in point-index order" semantics to be bit-identical to the CPU algorithm, so the
// points are bucketed with a STABLE radix sort (voxel / cell key, point index) and every bucket is
// reduced sequentially.  The k-NN search is one warp per query over a hashed uniform grid: lanes
// look up the cells of a ring in parallel, the warp scans their points cooperatively and keeps the
// k best squared distances (exact FP64, the reference's (dx^2+dy^2)+dz^2 order) in shared memory.
// The stable LSD radix sort (8-bit digits, only as many passes as the keys have significant bits)
// is hand-written below as well: per-tile histogram -> scan -> stable scatter with warp-level
// __match_any_sync ranking.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "cta_ops.cuh"
#include "icp_solve.h"
#include "knn_grid.cuh"

namespace otslam {

// ---- exact min / max of FP64 coordinates via order-preserving integer keys
__device__ __forceinline__ unsigned long long d2key(double d) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
static double key2d(unsigned long long k) {
    const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    double d;
    memcpy(&d, &b, 8);
    return d;
}

__global__ void __launch_bounds__(256) minmax_kernel(const double* __restrict__ pts, int64_t n, unsigned long long* mm /*[6]: min xyz, max xyz*/) {
    unsigned long long lo[3] = {~0ull, ~0ull, ~0ull}, hi[3] = {0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const unsigned long long k = d2key(pts[3 * i + a]);
            lo[a] = min(lo[a], k);
            hi[a] = max(hi[a], k);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o; o >>= 1) {
            lo[a] = min(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = max(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(mm + a, lo[a]);
            atomicMax(mm + 3 + a, hi[a]);
        }
    }
}

int cloud_minmax(const double* d_pts, int64_t n, double* mn, double* mx) {
    DevBuf<unsigned long long> mm;
    OT_CUDA(mm.alloc(6));
    unsigned long long init[6] = {~0ull, ~0ull, ~0ull, 0, 0, 0};
    OT_CUDA(cudaMemcpy(mm.p, init, sizeof(init), cudaMemcpyDefault));
    minmax_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8), 256>>>(d_pts, n, mm.p);
    OT_LAUNCHED();
    unsigned long long h[6];
    OT_CUDA(cudaMemcpy(h, mm.p, sizeof(h), cudaMemcpyDefault));
    for (int a = 0; a < 3; ++a) { mn[a] = key2d(h[a]); mx[a] = key2d(h[3 + a]); }
    return OTSLAM_OK;
}

static int nbits_for(double n_cells) {
    int b = 1;
    while (b < 62 && (double)(1ull << b) < n_cells) ++b;
    return b;
}
static KeyLayout make_layout(double nx, double ny, double nz) {
    const int bx = nbits_for(nx), by = nbits_for(ny), bz = nbits_for(nz);
    KeyLayout L;
    L.sh_y = bz; L.sh_x = by + bz; L.bits = bx + by + bz;
    L.mask_y = (1ull << by) - 1; L.mask_z = (1ull << bz) - 1;
    return L;
}

__global__ void __launch_bounds__(256) cell_key_kernel(const double* __restrict__ pts, int64_t n, double ox, double oy, double oz,
                                                       double cell, int clamp_hi_x, int clamp_hi_y, int clamp_hi_z, KeyLayout L,
                                                       uint64_t* __restrict__ keys, int32_t* __restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int kx = (int)floor(__ddiv_rn(__dsub_rn(pts[3 * i], ox), cell));
    int ky = (int)floor(__ddiv_rn(__dsub_rn(pts[3 * i + 1], oy), cell));
    int kz = (int)floor(__ddiv_rn(__dsub_rn(pts[3 * i + 2], oz), cell));
    if (clamp_hi_x >= 0) {   // k-NN grid: clamp into the grid (voxel_down_sample passes -1: exact keys)
        kx = min(max(kx, 0), clamp_hi_x); ky = min(max(ky, 0), clamp_hi_y); kz = min(max(kz, 0), clamp_hi_z);
    }
    keys[i] = layout_key(L, kx, ky, kz);
    idx[i] = (int32_t)i;
}

// ---------------------------------------------------------------------------------------------
// stable LSD radix sort of (u64 key, i32 value) pairs
// ---------------------------------------------------------------------------------------------
constexpr int kSortItems = 8;                         // keys per thread
constexpr int kSortTile = 256 * kSortItems;           // keys per CTA

__global__ void __launch_bounds__(256) radix_hist_kernel(const uint64_t* __restrict__ keys, int64_t n, int shift, int n_cta,
                                                         int* __restrict__ hist /*[256][n_cta]*/) {
    __shared__ int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kSortTile;
#pragma unroll
    for (int r = 0; r < kSortItems; ++r) {
        const int64_t i = base + r * 256 + threadIdx.x;
        if (i < n) atomicAdd(&h[(int)((keys[i] >> shift) & 0xFF)], 1);
    }
    __syncthreads();
    hist[threadIdx.x * n_cta + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(256) radix_scatter_kernel(const uint64_t* __restrict__ keys, const int32_t* __restrict__ vals,
                                                            int64_t n, int shift, int n_cta, const int64_t* __restrict__ offs,
                                                            uint64_t* __restrict__ out_keys, int32_t* __restrict__ out_vals) {
    __shared__ int warp_cnt[8][256];                  // this round: keys per (warp, digit)
    __shared__ int64_t digit_base[256];               // global offset of this tile's next key of each digit
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    digit_base[t] = offs[(int64_t)t * n_cta + blockIdx.x];
    const int64_t base = (int64_t)blockIdx.x * kSortTile;
    for (int r = 0; r < kSortItems; ++r) {
#pragma unroll
        for (int w = 0; w < 8; ++w) warp_cnt[w][t] = 0;
        __syncthreads();
        const int64_t i = base + r * 256 + t;
        const bool valid = i < n;
        uint64_t key = 0;
        int val = 0, digit = 256 + lane;              // invalid lanes never match anybody
        if (valid) { key = keys[i]; val = vals[i]; digit = (int)((key >> shift) & 0xFF); }
        // lanes of the warp holding the same digit, in lane (= index) order: stable rank inside the warp
        const unsigned peers = __match_any_sync(0xffffffffu, digit);
        const int rank_in_warp = __popc(peers & ((1u << lane) - 1u));
        if (valid && rank_in_warp == 0) warp_cnt[wid][digit] = __popc(peers);
        __syncthreads();
        int64_t pos = 0;
        if (valid) {
            int before = 0;
            for (int w = 0; w < wid; ++w) before += warp_cnt[w][digit];
            pos = digit_base[digit] + before + rank_in_warp;
        }
        __syncthreads();
        {   // advance the per-digit bases by this round's totals (thread t owns digit t)
            int tot = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) tot += warp_cnt[w][t];
            digit_base[t] += tot;
        }
        if (valid) { out_keys[pos] = key; out_vals[pos] = val; }
        __syncthreads();
    }
}

// sorts by the low `bits` bits of the keys on stream s; the result ends up in (kb, vb); (ka, va) are clobbered
int device_sort_pairs(uint64_t* ka_in, int32_t* va_in, uint64_t* kb_out, int32_t* vb_out, int64_t n, int bits, cudaStream_t s) {
    if (n <= 0) return OTSLAM_OK;
    const int n_cta = (int)((n + kSortTile - 1) / kSortTile);
    const int passes = std::max(1, (bits + 7) / 8);
    DevBuf<int> hist;
    DevBuf<int64_t> offs;
    OT_CUDA(hist.alloc((size_t)256 * n_cta));
    OT_CUDA(offs.alloc((size_t)256 * n_cta + 1));
    uint64_t *ka = ka_in, *kb = kb_out;
    int32_t *va = va_in, *vb = vb_out;
    for (int p = 0; p < passes; ++p) {
        radix_hist_kernel<<<n_cta, 256, 0, s>>>(ka, n, 8 * p, n_cta, hist.p);
        OT_LAUNCHED();
        OT_TRY(device_exclusive_scan(hist.p, offs.p, 256 * n_cta, s));   // digit-major: all tiles of digit 0, then digit 1, ...
        radix_scatter_kernel<<<n_cta, 256, 0, s>>>(ka, va, n, 8 * p, n_cta, offs.p, kb, vb);
        OT_LAUNCHED();
        std::swap(ka, kb);
        std::swap(va, vb);
    }
    if (ka != kb_out) {   // an even number of passes leaves the result in the input buffers
        OT_CUDA(cudaMemcpyAsync(kb_out, ka, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
        OT_CUDA(cudaMemcpyAsync(vb_out, va, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
    }
    // hist / offs go back to the scratch cache on return; the caller's later allocations are used on the same stream
    // (stream order protects them) and every operator synchronises before it returns
    return OTSLAM_OK;
}
// segment heads of the sorted keys: the first key of each run of equal keys
struct SegmentHead {
    const uint64_t* keys;
    __device__ bool operator()(int64_t p) const { return p == 0 || keys[p] != keys[p - 1]; }
};

// seg_start[0..n_seg) = the segment heads in order, seg_start[n_seg] = n
static int find_segments(const uint64_t* d_keys, int64_t n, DevBuf<int32_t>& seg_start, int64_t* n_seg) {
    OT_TRY(select_indices(SegmentHead{d_keys}, n, 0, seg_start, n_seg, 1));
    const int32_t nn = (int32_t)n;
    OT_CUDA(cudaMemcpy(seg_start.p + *n_seg, &nn, 4, cudaMemcpyDefault));
    return OTSLAM_OK;
}

// one thread per voxel: sequential FP64 sums in point-index order (stable sort => ascending indices)
__global__ void __launch_bounds__(128) voxel_mean_kernel(const double* __restrict__ pts, const double* __restrict__ cols,
                                                         const uint64_t* __restrict__ keys, const int32_t* __restrict__ idx,
                                                         const int32_t* __restrict__ seg_start, int64_t n_seg, KeyLayout L,
                                                         double* __restrict__ out_pts, double* __restrict__ out_cols,
                                                         int32_t* __restrict__ out_keys, int32_t* __restrict__ out_counts) {
    const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_seg) return;
    const int b = seg_start[m], e = seg_start[m + 1];
    double sp[3] = {0, 0, 0}, sc[3] = {0, 0, 0};
    for (int j = b; j < e; ++j) {
        const size_t i = (size_t)idx[j];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            sp[a] = __dadd_rn(sp[a], pts[3 * i + a]);
            if (cols) sc[a] = __dadd_rn(sc[a], cols[3 * i + a]);
        }
    }
    const double cnt = (double)(e - b);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        out_pts[3 * m + a] = __ddiv_rn(sp[a], cnt);
        if (cols && out_cols) out_cols[3 * m + a] = __ddiv_rn(sc[a], cnt);
    }
    const uint64_t k = keys[b];
    if (out_keys) {
        out_keys[3 * m] = (int32_t)(k >> L.sh_x);
        out_keys[3 * m + 1] = (int32_t)((k >> L.sh_y) & L.mask_y);
        out_keys[3 * m + 2] = (int32_t)(k & L.mask_z);
    }
    if (out_counts) out_counts[m] = e - b;
}

// ---- k-NN grid hash: cell key -> segment id
__global__ void __launch_bounds__(256) cell_hash_build_kernel(const uint64_t* __restrict__ sorted_keys, const int32_t* __restrict__ seg_start,
                                                              int64_t n_seg, HashTable t) {
    const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m < n_seg) hash_insert_absent(t, sorted_keys[seg_start[m]], (int32_t)m);
}


// Two levels.  Scanned clouds are surfaces: a grid sized for ~2 points per cell of the bounding-box VOLUME
// puts hundreds of points into every occupied cell (1 M points on a table: ~200), and each query then
// computes thousands of distances for its 20 neighbours.  The fine level is sized from the measured
// occupancy so that an occupied cell holds ~8 points and serves the first `fine_rings` rings; a query that
// cannot finish there (outliers, sparse regions: ring r costs ~24 r^2 hash probes) restarts on the coarse
// level, whose larger cells reach far with few rings; a query that is still searching after `coarse_rings`
// rings there (an isolated point far from everything: ring r costs ~24 r^2 probes, and ONE such warp
// crawling through 30 rings was 40 % of the kernel's duration) restarts on the top level (cells 8x larger).
// The result is the exact k smallest squared distances on any level (conservative ring termination), so
// it does not depend on the cell sizes.
struct KnnArgs {
    const double* pts;          // target cloud, original order
    const double* qpts;         // query points (== pts for the outlier filter)
    const int32_t* qidx;        // query visit order -> query index (null: identity)
    int64_t nq;
    int mode;                   // 0: dbar = mean of the k sqrt distances (A.8); 1: nearest-neighbour distance
    int64_t n;
    int k;
    int fine_rings;             // 0: no fine level
    int coarse_rings;           // ring limit on the coarse level when a top level exists (else unlimited)
    KnnGrid lv[3];              // fine, coarse, top
    double* dbar;               // [n] original order
};

constexpr int kKnnWarps = 8;
constexpr int kKnnMaxK = 128;
constexpr int kKnnTableRings = 3;                       // shells of rings 0..3: 1 + 26 + 98 + 218 = 343 cells
__constant__ int c_shell_offsets[343];                  // dx | dy << 8 | dz << 16 (signed bytes), ring by ring
__constant__ int c_shell_start[kKnnTableRings + 2];

__device__ __forceinline__ void warp_argmax(const double* best, int cnt, int lane, double& vmax, int& pmax) {
    double v = -1.0;
    int p = 0;
    for (int e = lane; e < cnt; e += 32) {
        const double b = best[e];
        if (b > v) { v = b; p = e; }
    }
    for (int o = 16; o; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int op = __shfl_xor_sync(0xffffffffu, p, o);
        if (ov > v || (ov == v && op < p)) { v = ov; p = op; }
    }
    vmax = v; pmax = p;
}

// (d2, index) order of the normal estimation's neighbour lists
__device__ __forceinline__ bool pair_less(double d, int i, double e, int j) { return d < e || (d == e && i < j); }

// the largest (d2, index) of the list: its value, index and position
__device__ __forceinline__ void warp_argmax_idx(const double* best, const int* bidx, int cnt, int lane, double& vmax, int& imax,
                                                int& pmax) {
    double v = -1.0;
    int i = -1, p = 0;
    for (int e = lane; e < cnt; e += 32)
        if (pair_less(v, i, best[e], bidx[e])) { v = best[e]; i = bidx[e]; p = e; }
    for (int o = 16; o; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        const int op = __shfl_xor_sync(0xffffffffu, p, o);
        if (pair_less(v, i, ov, oi)) { v = ov; i = oi; p = op; }
    }
    vmax = v; imax = i; pmax = p;
}

// The k best of a query on one level of the search structure.  kIdx = false (statistical outlier removal, nearest
// distance): the k smallest squared distances, a newcomer inserted after its equals.  kIdx = true (normal estimation):
// the k smallest (d2, index) pairs among the points with d2 < r2, the index carried beside each distance (reg_idx in
// registers for k <= 32, bidx in shared memory up to 128), and the ring walk also ends once the scanned box reaches
// beyond the radius.  True when the k best are final (ring termination, radius reached or whole grid covered), false
// when `last_ring` was scanned without reaching that point.
template <bool kIdx>
__device__ __forceinline__ bool knn_search_level(const KnnGrid& g, const double* __restrict__ pts, const double (&q)[3], int k,
                                                 int last_ring, int lane, double* best, int* bidx, double& reg_best, int& reg_idx,
                                                 int& found, double& thr, int& thr_idx, int& pos, double r2) {
    int c[3];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        const int v = (int)floor(__ddiv_rn(__dsub_rn(q[ax], g.mn[ax]), g.cell));
        c[ax] = min(max(v, 0), g.dim[ax] - 1);
    }
    const int maxring = max(g.dim[0], max(g.dim[1], g.dim[2]));
    for (int ring = 0; ring <= maxring; ++ring) {
        if ((found >= k || (kIdx && r2 < INFINITY)) && ring >= 1) {
            // distance from q to the nearest face of the already scanned box that still has grid behind it
            double reach = 1e300;
#pragma unroll
            for (int ax = 0; ax < 3; ++ax) {
                if (c[ax] - (ring - 1) > 0) reach = fmin(reach, q[ax] - (g.mn[ax] + (double)(c[ax] - (ring - 1)) * g.cell));
                if (c[ax] + ring < g.dim[ax]) reach = fmin(reach, (g.mn[ax] + (double)(c[ax] + ring) * g.cell) - q[ax]);
            }
            if (reach == 1e300) return true;           // the box covers the whole grid
            reach -= 1e-9 * g.cell;                    // conservative against rounding of the cell boundaries
            // strictly beyond the k-th: an unscanned point cannot tie with it (kIdx: a tie with a lower index would enter)
            if (found >= k && reach > 0.0 && reach * reach > thr) return true;
            if (kIdx && reach > 0.0 && reach * reach >= r2) return true;
        }
        if (ring > last_ring) return false;
        // enumerate the shell cells of this ring, 32 at a time (one hash lookup per lane)
        const int side = 2 * ring + 1;
        const int ncell = ring == 0 ? 1 : side * side * side - (side - 2) * (side - 2) * (side - 2);
        for (int c0 = 0; c0 < ncell; c0 += 32) {
            const int ci = c0 + lane;
            int seg = -1;
            if (ci < ncell) {
                int dx, dy, dz;
                if (ring <= kKnnTableRings) {              // precomputed offsets: no integer divisions on the common path
                    const int o = c_shell_offsets[c_shell_start[ring] + ci];
                    dx = (int)(signed char)(o & 0xFF); dy = (int)(signed char)((o >> 8) & 0xFF); dz = (int)(signed char)((o >> 16) & 0xFF);
                } else {
                    // shell = two full z-caps (side*side each) + side walls: (side-2) z-layers of a square ring (4*side-4)
                    const int cap = side * side;
                    if (ci < 2 * cap) {
                        const int w = ci % cap;
                        dz = (ci < cap) ? -ring : ring;
                        dx = w / side - ring; dy = w % side - ring;
                    } else {
                        const int r = ci - 2 * cap, per = 4 * side - 4;
                        dz = r / per - ring + 1;
                        const int w = r % per;
                        if (w < side) { dx = -ring; dy = w - ring; }
                        else if (w < 2 * side) { dx = ring; dy = w - side - ring; }
                        else if (w < 3 * side - 2) { dy = -ring; dx = w - 2 * side - ring + 1; }
                        else { dy = ring; dx = w - (3 * side - 2) - ring + 1; }
                    }
                }
                const int x = c[0] + dx, y = c[1] + dy, z = c[2] + dz;
                if (x >= 0 && x < g.dim[0] && y >= 0 && y < g.dim[1] && z >= 0 && z < g.dim[2]) {
                    seg = hash_find(g.cells, layout_key(g.L, x, y, z));
                }
            }
            unsigned have = __ballot_sync(0xffffffffu, seg >= 0);
            while (have) {
                const int src = __ffs(have) - 1;
                have &= have - 1;
                const int sg = __shfl_sync(0xffffffffu, seg, src);
                const int b = g.seg_start[sg], e = g.seg_start[sg + 1];
                for (int j0 = b; j0 < e; j0 += 32) {
                    const int j = j0 + lane;
                    double d2 = 0.0;
                    int pidx = 0;
                    bool cand = false;
                    if (j < e) {
                        pidx = g.idx[j];
                        const size_t pi = (size_t)pidx;
                        const double dx = __dsub_rn(q[0], pts[3 * pi]), dy = __dsub_rn(q[1], pts[3 * pi + 1]),
                                     dz = __dsub_rn(q[2], pts[3 * pi + 2]);
                        d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
                        cand = !kIdx || d2 < r2;
                    }
                    unsigned todo = __ballot_sync(0xffffffffu, cand && (found < k || (kIdx ? pair_less(d2, pidx, thr, thr_idx) : d2 < thr)));
                    if (k <= 32) {
                        // k best kept sorted ascending, one per lane (lanes >= found hold +inf): an insert is a
                        // ballot (rank of the newcomer), one shuffle (shift the tail up) and a select
                        while (todo) {
                            const int L = __ffs(todo) - 1;
                            todo &= todo - 1;
                            const double d = __shfl_sync(0xffffffffu, d2, L);
                            if (kIdx) {
                                const int di = __shfl_sync(0xffffffffu, pidx, L);
                                if (found == k && !pair_less(d, di, thr, thr_idx)) continue;             // warp-uniform
                                const int rank = __popc(__ballot_sync(0xffffffffu, pair_less(reg_best, reg_idx, d, di)));
                                const double up = __shfl_up_sync(0xffffffffu, reg_best, 1);
                                const int upi = __shfl_up_sync(0xffffffffu, reg_idx, 1);
                                if (lane == rank) { reg_best = d; reg_idx = di; }
                                else if (lane > rank) { reg_best = up; reg_idx = upi; }
                                if (found < k) ++found;
                                if (lane >= k) { reg_best = INFINITY; reg_idx = 0x7fffffff; }
                                if (found == k) { thr = __shfl_sync(0xffffffffu, reg_best, k - 1); thr_idx = __shfl_sync(0xffffffffu, reg_idx, k - 1); }
                            } else {
                                if (found == k && !(d < thr)) continue;                      // warp-uniform
                                const int rank = __popc(__ballot_sync(0xffffffffu, reg_best <= d));   // ties: after its equals
                                const double up = __shfl_up_sync(0xffffffffu, reg_best, 1);
                                if (lane == rank) reg_best = d;
                                else if (lane > rank) reg_best = up;
                                if (found < k) ++found;
                                if (lane >= k) reg_best = INFINITY;
                                if (found == k) thr = __shfl_sync(0xffffffffu, reg_best, k - 1);
                            }
                        }
                    } else {
                        while (todo) {
                            const int L = __ffs(todo) - 1;
                            todo &= todo - 1;
                            const double d = __shfl_sync(0xffffffffu, d2, L);
                            if (kIdx) {
                                const int di = __shfl_sync(0xffffffffu, pidx, L);
                                if (found < k) {
                                    if (lane == 0) { best[found] = d; bidx[found] = di; }
                                    ++found;
                                    __syncwarp();
                                    if (found == k) warp_argmax_idx(best, bidx, k, lane, thr, thr_idx, pos);
                                } else if (pair_less(d, di, thr, thr_idx)) {
                                    if (lane == 0) { best[pos] = d; bidx[pos] = di; }
                                    __syncwarp();
                                    warp_argmax_idx(best, bidx, k, lane, thr, thr_idx, pos);
                                }
                            } else if (found < k) {
                                if (lane == 0) best[found] = d;
                                ++found;
                                __syncwarp();
                                if (found == k) warp_argmax(best, k, lane, thr, pos);
                            } else if (d < thr) {
                                if (lane == 0) best[pos] = d;
                                __syncwarp();
                                warp_argmax(best, k, lane, thr, pos);
                            }
                        }
                    }
                }
            }
        }
    }
    return true;
}

__global__ void __launch_bounds__(kKnnWarps * 32) knn_mean_dist_kernel(KnnArgs a) {
    __shared__ double s_best[kKnnWarps][kKnnMaxK];
    __shared__ double s_sorted[kKnnWarps][kKnnMaxK];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t qpos = (int64_t)blockIdx.x * kKnnWarps + wid;
    if (qpos >= a.nq) return;
    double* best = s_best[wid];
    double* sorted = s_sorted[wid];
    const int64_t qi = a.qidx ? (int64_t)a.qidx[qpos] : qpos;
    const double q[3] = {a.qpts[3 * (size_t)qi], a.qpts[3 * (size_t)qi + 1], a.qpts[3 * (size_t)qi + 2]};
    const int k = a.k;
    int found = 0;
    double thr = 0.0;   // current k-th best (valid when found == k)
    int pos = 0;
    double reg_best = INFINITY;                    // k <= 32: the sorted k best, one per lane
    int reg_idx = 0, thr_idx = 0;                  // unused without the index (kIdx = false)
    // one copy of the search code for the three levels (three inlined copies thrashed the instruction cache:
    // ncu showed no_instruction stalls of 2 warps per issue slot)
    bool done = false;
#pragma unroll 1
    for (int level = a.fine_rings > 0 ? 0 : 1; level < 3 && !done; ++level) {
        const int last = level == 0 ? a.fine_rings : (level == 1 ? a.coarse_rings : 0x3fffffff);
        found = 0; thr = 0.0; pos = 0; reg_best = INFINITY;    // a coarser level's buckets contain the finer level's finds again
        __syncwarp();
        done = knn_search_level<false>(a.lv[level], a.pts, q, k, last, lane, best, nullptr, reg_best, reg_idx, found, thr, thr_idx, pos,
                                       INFINITY);
    }
    if (k <= 32 && lane < found) best[lane] = reg_best;
    __syncwarp();
    // ascending order, then the sequential sum of square roots (SURVEY A.8)
    for (int e = lane; e < found; e += 32) {
        const double v = best[e];
        int rank = 0;
        for (int i = 0; i < found; ++i) {
            const double o = best[i];
            rank += (o < v) || (o == v && i < e);
        }
        sorted[rank] = v;
    }
    __syncwarp();
    if (lane == 0) {
        double s = 0.0;
        for (int j = 0; j < found; ++j) s = __dadd_rn(s, __dsqrt_rn(sorted[j]));
        if (a.mode == 1) a.dbar[qi] = found > 0 ? __dsqrt_rn(sorted[0]) : -1.0;
        else a.dbar[qi] = found > 0 ? __ddiv_rn(s, (double)found) : -1.0;
    }
}

// ---- normal estimation (PointCloud.estimate_normals, DESIGN.md §4 "Normals and point-to-plane registration")
constexpr int kJacobiSweeps = 16;

// one Jacobi rotation of the symmetric A zeroing A[p][q]; V accumulates the rotations (its columns are the eigenvectors)
__device__ __forceinline__ void jacobi_rotate(double (&A)[3][3], double (&V)[3][3], int p, int q) {
    const double apq = A[p][q];
    if (apq == 0.0) return;
    const int r = 3 - p - q;
    const double theta = __ddiv_rn(__dsub_rn(A[q][q], A[p][p]), __dmul_rn(2.0, apq));
    double t;
    if (fabs(theta) > 1e150) t = __ddiv_rn(0.5, theta);      // theta^2 would overflow; t = 1 / (2 theta) to working precision
    else {
        t = __ddiv_rn(1.0, __dadd_rn(fabs(theta), __dsqrt_rn(__dadd_rn(__dmul_rn(theta, theta), 1.0))));
        if (theta < 0.0) t = -t;
    }
    const double c = __ddiv_rn(1.0, __dsqrt_rn(__dadd_rn(__dmul_rn(t, t), 1.0))), s = __dmul_rn(t, c);
    const double app = __dsub_rn(A[p][p], __dmul_rn(t, apq)), aqq = __dadd_rn(A[q][q], __dmul_rn(t, apq));
    const double arp = A[r][p], arq = A[r][q];
    A[r][p] = A[p][r] = __dsub_rn(__dmul_rn(c, arp), __dmul_rn(s, arq));
    A[r][q] = A[q][r] = __dadd_rn(__dmul_rn(s, arp), __dmul_rn(c, arq));
    A[p][p] = app; A[q][q] = aqq; A[p][q] = A[q][p] = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double vp = V[i][p], vq = V[i][q];
        V[i][p] = __dsub_rn(__dmul_rn(c, vp), __dmul_rn(s, vq));
        V[i][q] = __dadd_rn(__dmul_rn(s, vp), __dmul_rn(c, vq));
    }
}

// unit eigenvector of the smallest eigenvalue of the symmetric C = {c00, c01, c02, c11, c12, c22} with + - * / sqrt only:
// C scaled by its largest |entry| (a zero matrix gives the zero vector), cyclic Jacobi over (0,1), (0,2), (1,2) until the
// off-diagonal is exactly zero or kJacobiSweeps sweeps; among equal eigenvalues the highest index (C = I gives (0, 0, 1))
__device__ void smallest_eigenvector(const double (&C)[6], double (&n)[3]) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) s = fmax(s, fabs(C[i]));
    if (!(s > 0.0)) { n[0] = n[1] = n[2] = 0.0; return; }
    const double a00 = __ddiv_rn(C[0], s), a01 = __ddiv_rn(C[1], s), a02 = __ddiv_rn(C[2], s), a11 = __ddiv_rn(C[3], s),
                 a12 = __ddiv_rn(C[4], s), a22 = __ddiv_rn(C[5], s);
    double A[3][3] = {{a00, a01, a02}, {a01, a11, a12}, {a02, a12, a22}};
    double V[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
    for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
        if (A[0][1] == 0.0 && A[0][2] == 0.0 && A[1][2] == 0.0) break;
        jacobi_rotate(A, V, 0, 1);
        jacobi_rotate(A, V, 0, 2);
        jacobi_rotate(A, V, 1, 2);
    }
    int m = 0;
    if (A[1][1] <= A[m][m]) m = 1;
    if (A[2][2] <= A[m][m]) m = 2;
    const double x = V[0][m], y = V[1][m], z = V[2][m];
    const double len = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)));
    n[0] = __ddiv_rn(x, len); n[1] = __ddiv_rn(y, len); n[2] = __ddiv_rn(z, len);
}

// one warp per query: the neighbour list in (d2, index) order, Open3D's ComputeCovariance (nine cumulants summed in
// neighbour order by lanes 0..8, over the count; C = I below 3 neighbours), the smallest eigenvector, then the fallbacks
// and the sign of Open3D's EstimateNormals
__global__ void __launch_bounds__(kKnnWarps * 32) normals_kernel(KnnArgs a, const double* __restrict__ prior, double r2,
                                                                 double* __restrict__ out) {
    __shared__ double s_best[kKnnWarps][kKnnMaxK];
    __shared__ int s_bidx[kKnnWarps][kKnnMaxK];
    __shared__ int s_nbr[kKnnWarps][kKnnMaxK];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t qpos = (int64_t)blockIdx.x * kKnnWarps + wid;
    if (qpos >= a.nq) return;
    double* best = s_best[wid];
    int* bidx = s_bidx[wid];
    int* nbr = s_nbr[wid];
    const int64_t qi = a.qidx ? (int64_t)a.qidx[qpos] : qpos;
    const double q[3] = {a.qpts[3 * (size_t)qi], a.qpts[3 * (size_t)qi + 1], a.qpts[3 * (size_t)qi + 2]};
    const int k = a.k;
    int found = 0, pos = 0, reg_idx = 0x7fffffff, thr_idx = 0;
    double thr = 0.0, reg_best = INFINITY;
    bool done = false;
#pragma unroll 1
    for (int level = a.fine_rings > 0 ? 0 : 1; level < 3 && !done; ++level) {
        const int last = level == 0 ? a.fine_rings : (level == 1 ? a.coarse_rings : 0x3fffffff);
        found = 0; thr = 0.0; thr_idx = 0; pos = 0; reg_best = INFINITY; reg_idx = 0x7fffffff;
        __syncwarp();
        done = knn_search_level<true>(a.lv[level], a.pts, q, k, last, lane, best, bidx, reg_best, reg_idx, found, thr, thr_idx, pos, r2);
    }
    if (k <= 32) {
        if (lane < found) nbr[lane] = reg_idx;
    } else {
        __syncwarp();
        for (int e = lane; e < found; e += 32) {
            const double v = best[e];
            const int vi = bidx[e];
            int rank = 0;
            for (int i = 0; i < found; ++i) rank += pair_less(best[i], bidx[i], v, vi);
            nbr[rank] = vi;
        }
    }
    __syncwarp();
    // lane c < 9 sums cumulant c: x, y, z, xx, xy, xz, yy, yz, zz (nibble c of U / V; V = 0xF: first order)
    double cum = 0.0;
    if (lane < 9) {
        const int u = (int)((0x211000210ull >> (4 * lane)) & 0xF), v = (int)((0x221210FFFull >> (4 * lane)) & 0xF);
        for (int j = 0; j < found; ++j) {
            const size_t p = 3 * (size_t)nbr[j];
            const double x = a.pts[p + u];
            cum = __dadd_rn(cum, v == 0xF ? x : __dmul_rn(x, a.pts[p + v]));
        }
        cum = __ddiv_rn(cum, (double)found);
    }
    double m[9];
#pragma unroll
    for (int c = 0; c < 9; ++c) m[c] = __shfl_sync(0xffffffffu, cum, c);
    if (lane != 0) return;
    double C[6] = {1.0, 0.0, 0.0, 1.0, 0.0, 1.0};
    if (found >= 3) {
        C[0] = __dsub_rn(m[3], __dmul_rn(m[0], m[0]));
        C[1] = __dsub_rn(m[4], __dmul_rn(m[0], m[1]));
        C[2] = __dsub_rn(m[5], __dmul_rn(m[0], m[2]));
        C[3] = __dsub_rn(m[6], __dmul_rn(m[1], m[1]));
        C[4] = __dsub_rn(m[7], __dmul_rn(m[1], m[2]));
        C[5] = __dsub_rn(m[8], __dmul_rn(m[2], m[2]));
    }
    double n[3];
    smallest_eigenvector(C, n);
    const double* pr = prior ? prior + 3 * (size_t)qi : nullptr;
    if (n[0] == 0.0 && n[1] == 0.0 && n[2] == 0.0) {
        if (pr) { n[0] = pr[0]; n[1] = pr[1]; n[2] = pr[2]; }
        else { n[2] = 1.0; }
    } else if (pr) {
        if (__dadd_rn(__dadd_rn(__dmul_rn(n[0], pr[0]), __dmul_rn(n[1], pr[1])), __dmul_rn(n[2], pr[2])) < 0.0) {
            n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2];
        }
    } else {
        int b = 0;
        if (fabs(n[1]) > fabs(n[b])) b = 1;
        if (fabs(n[2]) > fabs(n[b])) b = 2;
        if (n[b] < 0.0) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }
    }
    out[3 * (size_t)qi] = n[0]; out[3 * (size_t)qi + 1] = n[1]; out[3 * (size_t)qi + 2] = n[2];
}

// sum over buckets of size^2: sum / n = the number of points sharing a cell with a typical point
__global__ void __launch_bounds__(256) crowding_kernel(const int32_t* __restrict__ seg_start, int64_t n_seg, unsigned long long* out) {
    const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long v = 0;
    if (m < n_seg) { const unsigned long long c = (unsigned long long)(seg_start[m + 1] - seg_start[m]); v = c * c; }
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, v);
}

static int upload_shell_table() {
    static bool done[64] = {};
    int dev = 0;
    OT_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && done[dev]) return OTSLAM_OK;
    std::vector<int> off, start;
    for (int ring = 0; ring <= kKnnTableRings; ++ring) {
        start.push_back((int)off.size());
        const int side = 2 * ring + 1;
        const int ncell = ring == 0 ? 1 : side * side * side - (side - 2) * (side - 2) * (side - 2);
        for (int ci = 0; ci < ncell; ++ci) {          // the kernel's arithmetic enumeration, verbatim
            int dx, dy, dz;
            if (ring == 0) { dx = dy = dz = 0; }
            else {
                const int cap = side * side;
                if (ci < 2 * cap) {
                    const int w = ci % cap;
                    dz = (ci < cap) ? -ring : ring;
                    dx = w / side - ring; dy = w % side - ring;
                } else {
                    const int r = ci - 2 * cap, per = 4 * side - 4;
                    dz = r / per - ring + 1;
                    const int w = r % per;
                    if (w < side) { dx = -ring; dy = w - ring; }
                    else if (w < 2 * side) { dx = ring; dy = w - side - ring; }
                    else if (w < 3 * side - 2) { dy = -ring; dx = w - 2 * side - ring + 1; }
                    else { dy = ring; dx = w - (3 * side - 2) - ring + 1; }
                }
            }
            off.push_back((dx & 0xFF) | ((dy & 0xFF) << 8) | ((dz & 0xFF) << 16));
        }
    }
    start.push_back((int)off.size());
    if (off.size() != 343) return set_error(OTSLAM_ERR_INVALID, "shell table size");
    OT_CUDA(cudaMemcpyToSymbol(c_shell_offsets, off.data(), off.size() * sizeof(int)));
    OT_CUDA(cudaMemcpyToSymbol(c_shell_start, start.data(), start.size() * sizeof(int)));
    if (dev >= 0 && dev < 64) done[dev] = true;
    return OTSLAM_OK;
}

// bucket the n points of d_pts on a grid of `cell`-sized cells over [mn, mx] (at most max_dim cells per axis)
int build_grid(const double* d_pts, int64_t n, const double mn[3], const double mx[3], double cell, int max_dim, GridBuffers& b,
               KnnGrid& g) {
    const double ext[3] = {mx[0] - mn[0], mx[1] - mn[1], mx[2] - mn[2]};
    const double maxext = std::max(ext[0], std::max(ext[1], ext[2]));
    cell = std::max(cell, maxext / (double)max_dim);
    if (!(cell > 0.0) || !std::isfinite(cell)) cell = 1.0;
    g.cell = cell;
    for (int ax = 0; ax < 3; ++ax) { g.mn[ax] = mn[ax]; g.dim[ax] = std::max(1, (int)std::floor(ext[ax] / cell) + 1); }
    g.L = make_layout(g.dim[0], g.dim[1], g.dim[2]);
    OT_CUDA(b.k0.alloc(n)); OT_CUDA(b.k1.alloc(n)); OT_CUDA(b.i0.alloc(n)); OT_CUDA(b.i1.alloc(n));
    cell_key_kernel<<<(unsigned)((n + 255) / 256), 256>>>(d_pts, n, mn[0], mn[1], mn[2], cell, g.dim[0] - 1, g.dim[1] - 1, g.dim[2] - 1,
                                                         g.L, b.k0.p, b.i0.p);
    OT_LAUNCHED();
    OT_TRY(device_sort_pairs(b.k0.p, b.i0.p, b.k1.p, b.i1.p, n, g.L.bits, 0));
    OT_TRY(find_segments(b.k1.p, n, b.seg, &b.n_seg));
    uint32_t cap = 1024;
    while (!hash_fits(b.n_seg, cap)) cap <<= 1;
    OT_CUDA(b.hk.alloc(cap)); OT_CUDA(b.hv.alloc(cap));
    OT_CUDA(cudaMemset(b.hk.p, 0xFF, (size_t)cap * 8));
    g.cells = {b.hk.p, b.hv.p, cap - 1};
    cell_hash_build_kernel<<<(unsigned)((b.n_seg + 255) / 256), 256>>>(b.k1.p, b.seg.p, b.n_seg, g.cells);
    OT_LAUNCHED();
    g.idx = b.i1.p; g.seg_start = b.seg.p;
    return OTSLAM_OK;
}

constexpr double kKnnFineOccupancy = 16.0;    // target points per occupied fine cell (measured best of 4..64 on 1 M surface points, k = 20)
constexpr int kKnnFineRings = 3;

// coarse level (~2 points per cell of the bounding-box volume) + fine level when the occupied cells are crowded
constexpr int kKnnCoarseRings = 6;
constexpr double kKnnTopFactor = 8.0;

static int build_search(const double* d_pts, int64_t n, GridBuffers& bc, GridBuffers& bf, GridBuffers& bt, KnnArgs& a) {
    double mn[3], mx[3];
    OT_TRY(cloud_minmax(d_pts, n, mn, mx));
    const double ext[3] = {mx[0] - mn[0], mx[1] - mn[1], mx[2] - mn[2]};
    const double vol = std::max(ext[0], 1e-9) * std::max(ext[1], 1e-9) * std::max(ext[2], 1e-9);
    const double cell = std::cbrt(vol / std::max(1.0, (double)n / 2.0));
    OT_TRY(build_grid(d_pts, n, mn, mx, cell, 1024, bc, a.lv[1]));
    a.coarse_rings = 0x3fffffff;
    if (std::max(a.lv[1].dim[0], std::max(a.lv[1].dim[1], a.lv[1].dim[2])) > 4 * kKnnCoarseRings) {
        OT_TRY(build_grid(d_pts, n, mn, mx, a.lv[1].cell * kKnnTopFactor, 1024, bt, a.lv[2]));
        a.coarse_rings = kKnnCoarseRings;
    }
    OT_TRY(upload_shell_table());
    a.fine_rings = 0;
    // crowding seen by a typical point (mean bucket size weighted by the points in it); isolated outliers,
    // which open many near-empty cells, do not dilute it the way n / n_cells would
    DevBuf<unsigned long long> sq;
    OT_CUDA(sq.alloc(1));
    OT_CUDA(cudaMemset(sq.p, 0, 8));
    crowding_kernel<<<(unsigned)((bc.n_seg + 255) / 256), 256>>>(bc.seg.p, bc.n_seg, sq.p);
    OT_LAUNCHED();
    unsigned long long hsq = 0;
    OT_CUDA(cudaMemcpy(&hsq, sq.p, 8, cudaMemcpyDefault));
    const double occ = (double)hsq / (double)n;
    static const double target = getenv("OTSLAM_KNN_OCC") ? atof(getenv("OTSLAM_KNN_OCC")) : kKnnFineOccupancy;   // dev knobs
    static const int rings = getenv("OTSLAM_KNN_RINGS") ? atoi(getenv("OTSLAM_KNN_RINGS")) : kKnnFineRings;
    if (occ > 2.0 * target && rings > 0) {
        // surface-like data: points per occupied cell scale with cell^2
        const double fine_cell = a.lv[1].cell * std::sqrt(target / occ);
        OT_TRY(build_grid(d_pts, n, mn, mx, fine_cell, 1 << 16, bf, a.lv[0]));
        a.fine_rings = std::min(rings, kKnnTableRings);
        if (getenv("OTSLAM_KNN_DEBUG"))
            fprintf(stderr, "knn: n %lld coarse cell %.4g (%lld cells, crowding %.1f) fine cell %.4g (%lld cells)\n", (long long)n,
                    a.lv[1].cell, (long long)bc.n_seg, occ, a.lv[0].cell, (long long)bf.n_seg);
    }
    return OTSLAM_OK;
}

// the points remove_statistical_outlier keeps: 0 < dbar < thr
struct SorKeep {
    const double* dbar;
    double thr;
    __device__ bool operator()(int64_t p) const { return dbar[p] > 0.0 && dbar[p] < thr; }
};

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_cloud_voxel_down_sample(const double* points, const double* colors, int64_t n, double voxel_size, double* out_points,
                                   double* out_colors, int32_t* out_keys, int32_t* out_counts, int64_t* n_out, int device) {
    if (!n_out || n < 0 || (n && !points)) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    *n_out = 0;
    if (!(voxel_size > 0.0)) return set_error(OTSLAM_ERR_INVALID, "[VoxelDownSample] voxel_size <= 0.");
    if (n == 0) return OTSLAM_OK;
    if (n > 0x7fffffffLL) return set_error(OTSLAM_ERR_OVERFLOW, "more than 2^31 points");
    OT_TRY(use_device(device));
    DevBuf<double> dp, dc;
    OT_CUDA(dp.upload(points, n * 3));
    if (colors) OT_CUDA(dc.upload(colors, n * 3));
    OpTimer timer;
    double mn[3], mx[3];
    OT_TRY(cloud_minmax(dp.p, n, mn, mx));
    double vmin[3];
    for (int a = 0; a < 3; ++a) {
        vmin[a] = mn[a] - voxel_size * 0.5;
        const double vmax = mx[a] + voxel_size * 0.5;
        if (voxel_size * 2147483647.0 < vmax - vmin[a]) return set_error(OTSLAM_ERR_INVALID, "[VoxelDownSample] voxel_size is too small.");
    }
    const KeyLayout L = make_layout(std::floor((mx[0] - vmin[0]) / voxel_size) + 1.0, std::floor((mx[1] - vmin[1]) / voxel_size) + 1.0,
                                    std::floor((mx[2] - vmin[2]) / voxel_size) + 1.0);
    if (L.bits > 63) return set_error(OTSLAM_ERR_OVERFLOW, "[VoxelDownSample] voxel grid needs more than 63 key bits on the GPU path");
    DevBuf<uint64_t> k0, k1;
    DevBuf<int32_t> i0, i1;
    OT_CUDA(k0.alloc(n)); OT_CUDA(k1.alloc(n)); OT_CUDA(i0.alloc(n)); OT_CUDA(i1.alloc(n));
    cell_key_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dp.p, n, vmin[0], vmin[1], vmin[2], voxel_size, -1, -1, -1, L, k0.p, i0.p);
    OT_LAUNCHED();
    OT_TRY(device_sort_pairs(k0.p, i0.p, k1.p, i1.p, n, L.bits, 0));
    DevBuf<int32_t> seg;
    int64_t m = 0;
    OT_TRY(find_segments(k1.p, n, seg, &m));
    *n_out = m;
    if (!out_points) return OTSLAM_OK;
    DevBuf<double> op, oc;
    DevBuf<int32_t> ok, on;
    OT_CUDA(op.alloc(m * 3)); OT_CUDA(oc.alloc(m * 3)); OT_CUDA(ok.alloc(m * 3)); OT_CUDA(on.alloc(m));
    voxel_mean_kernel<<<(unsigned)((m + 127) / 128), 128>>>(dp.p, colors ? dc.p : nullptr, k1.p, i1.p, seg.p, m, L, op.p, oc.p, ok.p, on.p);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(op.download(out_points, m * 3));
    if (colors && out_colors) OT_CUDA(oc.download(out_colors, m * 3));
    if (out_keys) OT_CUDA(ok.download(out_keys, m * 3));
    if (out_counts) OT_CUDA(on.download(out_counts, m));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_cloud_remove_statistical_outlier(const double* points, int64_t n, int nb_neighbors, double std_ratio,
                                            int64_t* out_indices, int64_t* n_out, double* mean_dist, int device) {
    if (!n_out || n < 0 || (n && (!points || !out_indices))) return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    *n_out = 0;
    if (nb_neighbors < 1 || !(std_ratio > 0.0))
        return set_error(OTSLAM_ERR_INVALID, "[RemoveStatisticalOutliers] Illegal input parameters, the number of neighbors and "
                                             "standard deviation ratio must be positive.");
    if (n == 0) return OTSLAM_OK;
    if (n > 0x7fffffffLL) return set_error(OTSLAM_ERR_OVERFLOW, "more than 2^31 points");
    const int k = (int)std::min<int64_t>(nb_neighbors, n);
    if (k > kKnnMaxK) return set_error(OTSLAM_ERR_INVALID, "nb_neighbors > 128 is not supported on the GPU path");
    OT_TRY(use_device(device));
    DevBuf<double> dp;
    OT_CUDA(dp.upload(points, n * 3));
    OpTimer timer;
    KnnArgs a;
    GridBuffers bc, bf, bt;
    OT_TRY(build_search(dp.p, n, bc, bf, bt, a));
    DevBuf<double> dbar, scal;
    OT_CUDA(dbar.alloc(n)); OT_CUDA(scal.alloc(1));
    a.pts = dp.p; a.qpts = dp.p; a.qidx = a.fine_rings ? a.lv[0].idx : a.lv[1].idx;   // visit queries cell by cell: neighbours share cache lines
    a.nq = n; a.mode = 0; a.n = n; a.k = k; a.dbar = dbar.p;
    knn_mean_dist_kernel<<<(unsigned)((n + kKnnWarps - 1) / kKnnWarps), kKnnWarps * 32>>>(a);
    OT_LAUNCHED();
    if (mean_dist) OT_CUDA(dbar.download(mean_dist, n));
    // global statistics in sequential index order; scalars finished on the host in FP64
    double sum = 0.0, sq = 0.0;
    OT_TRY(device_ordered_sum(dbar.p, n, 2, nullptr, 0.0, scal.p, 0));
    OT_CUDA(cudaMemcpy(&sum, scal.p, 8, cudaMemcpyDefault));
    const int64_t valid = n;   // the query point is its own first neighbour, so every point has >= 1
    const double mean = sum / (double)valid;
    OT_TRY(device_ordered_sum(dbar.p, n, 3, nullptr, mean, scal.p, 0));
    OT_CUDA(cudaMemcpy(&sq, scal.p, 8, cudaMemcpyDefault));
    const double sd = valid > 1 ? std::sqrt(sq / (double)(valid - 1)) : 0.0;
    const double thr = mean + std_ratio * sd;
    DevBuf<int64_t> oidx;
    int64_t m = 0;
    OT_TRY(select_indices(SorKeep{dbar.p, thr}, n, 0, oidx, &m));
    *n_out = m;
    timer.stop();
    if (m > 0) OT_CUDA(oidx.download(out_indices, m));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}


__global__ void __launch_bounds__(128) nn_within_kernel(KnnGrid g, const double* __restrict__ pts, const double* __restrict__ qpts,
                                                        int64_t nq, double r2, int32_t* __restrict__ out_idx, double* __restrict__ out_d2) {
    const int64_t qi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    const double q[3] = {qpts[3 * qi], qpts[3 * qi + 1], qpts[3 * qi + 2]};
    int bi;
    double best;
    nn_within_search(g, pts, q, r2, bi, best);
    out_idx[qi] = bi;
    if (out_d2) out_d2[qi] = bi >= 0 ? best : -1.0;
}

// ---- point-to-plane ICP (o3d.pipelines.registration.registration_icp with TransformationEstimationPointToPlane)
constexpr int kIcpThreads = 128;        // source points per CTA
constexpr int kIcpTerms = 30;           // 21 JtJ (upper triangle, row-major), 6 Jtr, r^2, inliers, Euclidean d^2 of the match
constexpr int kIcpSumThreads = 256;

// one thread per source point at the current pose: its correspondence (nn_within_kernel's rule), r = n.(s - t) and
// J = [s x n, n] with the target's normal n, and the CTA's sum of the 30 terms by a fixed halving tree in source order
__global__ void __launch_bounds__(kIcpThreads) icp_assoc_kernel(KnnGrid g, const double* __restrict__ tgt, const double* __restrict__ tn,
                                                                int has_target, const double* __restrict__ src, int64_t n, double r2,
                                                                int32_t* __restrict__ corr, double* __restrict__ partials, int P) {
    __shared__ double sm[kIcpTerms][kIcpThreads];
    const int lane = threadIdx.x;
    const int64_t i = (int64_t)blockIdx.x * kIcpThreads + lane;
    bool matched = false;
    if (i < n) {
        const double p[3] = {src[3 * i], src[3 * i + 1], src[3 * i + 2]};
        int bi = -1;
        double d2 = 0.0;
        if (has_target) nn_within_search(g, tgt, p, r2, bi, d2);
        corr[i] = bi;
        if (bi >= 0) {
            const size_t m = 3 * (size_t)bi;
            const double N[3] = {tn[m], tn[m + 1], tn[m + 2]};
            const double e[3] = {__dsub_rn(p[0], tgt[m]), __dsub_rn(p[1], tgt[m + 1]), __dsub_rn(p[2], tgt[m + 2])};
            point_to_plane_terms(p, N, e, &sm[0][lane], kIcpThreads);
            sm[29][lane] = d2;
            matched = true;
        }
    }
    if (!matched)                        // no point or no correspondence: its terms are 0
#pragma unroll
        for (int k = 0; k < kIcpTerms; ++k) sm[k][lane] = 0.0;
    cta_halving_tree(sm);                // absent points add 0
    if (lane < kIcpTerms) partials[(size_t)lane * P + blockIdx.x] = sm[lane][0];
}

int otslam_cloud_nn_within(const double* source, int64_t n_source, const double* target, int64_t n_target, double radius,
                           int32_t* out_index, double* out_dist2, int device) {
    if (n_source < 0 || n_target < 0 || (n_source && (!source || !out_index)) || (n_target && !target) || !(radius > 0.0))
        return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    if (n_source == 0) return OTSLAM_OK;
    if (n_target > 0x7fffffffLL || n_source > 0x7fffffffLL) return set_error(OTSLAM_ERR_OVERFLOW, "more than 2^31 points");
    OT_TRY(use_device(device));
    DevBuf<double> dt, dsrc, dd2;
    DevBuf<int32_t> di;
    OT_CUDA(dsrc.upload(source, n_source * 3)); OT_CUDA(di.alloc(n_source)); OT_CUDA(dd2.alloc(n_source));
    if (n_target == 0) {
        OT_CUDA(cudaMemset(di.p, 0xFF, (size_t)n_source * 4));
    } else {
        OT_CUDA(dt.upload(target, n_target * 3));
        OpTimer timer;
        double mn[3], mx[3];
        OT_TRY(cloud_minmax(dt.p, n_target, mn, mx));
        GridBuffers b;
        KnnGrid g;
        OT_TRY(build_grid(dt.p, n_target, mn, mx, radius, 1 << 20, b, g));
        // build_grid may have enlarged the cell (never shrinks it): 27 cells of size >= radius still cover the ball
        nn_within_kernel<<<(unsigned)((n_source + 127) / 128), 128>>>(g, dt.p, dsrc.p, n_source, radius * radius, di.p, dd2.p);
        OT_LAUNCHED();
        timer.stop();
    }
    OT_CUDA(di.download(out_index, n_source));
    if (out_dist2 && n_target) OT_CUDA(dd2.download(out_dist2, n_source));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_cloud_nn_distance(const double* source, int64_t n_source, const double* target, int64_t n_target, double* out_dist,
                             int device) {
    if (n_source < 0 || n_target < 0 || (n_source && (!source || !out_dist)) || (n_target && !target))
        return set_error(OTSLAM_ERR_INVALID, "bad arguments");
    if (n_source == 0) return OTSLAM_OK;
    if (n_target == 0) return set_error(OTSLAM_ERR_INVALID, "[ComputePointCloudDistance] target cloud is empty");
    if (n_target > 0x7fffffffLL || n_source > 0x7fffffffLL) return set_error(OTSLAM_ERR_OVERFLOW, "more than 2^31 points");
    OT_TRY(use_device(device));
    DevBuf<double> dt, dsrc, dout;
    OT_CUDA(dt.upload(target, n_target * 3)); OT_CUDA(dsrc.upload(source, n_source * 3)); OT_CUDA(dout.alloc(n_source));
    OpTimer timer;
    KnnArgs a;
    GridBuffers bc, bf, bt;
    OT_TRY(build_search(dt.p, n_target, bc, bf, bt, a));
    a.pts = dt.p; a.qpts = dsrc.p; a.qidx = nullptr; a.nq = n_source; a.mode = 1; a.n = n_target; a.k = 1; a.dbar = dout.p;
    knn_mean_dist_kernel<<<(unsigned)((n_source + kKnnWarps - 1) / kKnnWarps), kKnnWarps * 32>>>(a);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(dout.download(out_dist, n_source));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_cloud_estimate_normals(const double* points, int64_t n, const double* prior_normals, double radius, int max_nn,
                                  double* out_normals, int device) {
    // ---- every argument is checked before any CUDA call
    if (n < 0) return set_error(OTSLAM_ERR_INVALID, "estimate_normals: n < 0");
    if (n > 0x7fffffffLL) return set_error(OTSLAM_ERR_INVALID, "estimate_normals: more than 2^31 - 1 points");
    if (n && (!points || !out_normals)) return set_error(OTSLAM_ERR_INVALID, "estimate_normals: null points or out_normals");
    if (max_nn < 1 || max_nn > kKnnMaxK) return set_error(OTSLAM_ERR_INVALID, "estimate_normals: max_nn must be in 1..128");
    if (!(radius > 0.0)) return set_error(OTSLAM_ERR_INVALID, "estimate_normals: radius must be > 0 (finite, or +inf for a k-NN search)");
    if (n == 0) return OTSLAM_OK;
    OT_TRY(use_device(device));
    DevBuf<double> dp, dprior, dout;
    OT_CUDA(dp.upload(points, n * 3)); OT_CUDA(dout.alloc(n * 3));
    if (prior_normals) OT_CUDA(dprior.upload(prior_normals, n * 3));
    OpTimer timer;
    KnnArgs a;
    GridBuffers bc, bf, bt;
    OT_TRY(build_search(dp.p, n, bc, bf, bt, a));
    a.pts = dp.p; a.qpts = dp.p; a.qidx = a.fine_rings ? a.lv[0].idx : a.lv[1].idx;   // visit queries cell by cell
    a.nq = n; a.mode = 0; a.n = n; a.k = (int)std::min<int64_t>(max_nn, n); a.dbar = nullptr;
    normals_kernel<<<(unsigned)((n + kKnnWarps - 1) / kKnnWarps), kKnnWarps * 32>>>(a, prior_normals ? dprior.p : nullptr,
                                                                                    radius * radius, dout.p);
    OT_LAUNCHED();
    timer.stop();
    OT_CUDA(dout.download(out_normals, n * 3));
    OT_CUDA(cudaDeviceSynchronize());
    return OTSLAM_OK;
}

int otslam_cloud_icp_point_to_plane(const double* source, int64_t n_source, const double* target, const double* target_normals,
                                    int64_t n_target, double max_distance, const double init[16], double relative_fitness,
                                    double relative_rmse, int max_iteration, double transform_out[16], double* fitness,
                                    double* inlier_rmse, int32_t* iterations, int32_t* corr_index, int device) {
    // ---- every argument is checked before any CUDA call
    if (n_source < 0 || n_target < 0) return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: negative point count");
    if (n_source > 0x7fffffffLL || n_target > 0x7fffffffLL)
        return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: more than 2^31 - 1 points");
    if (n_source && !source) return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: null source");
    if (n_target && (!target || !target_normals)) return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: null target or target_normals");
    if (!init || !transform_out) return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: null init or transform_out");
    if (!(max_distance > 0.0) || !std::isfinite(max_distance))
        return set_error(OTSLAM_ERR_INVALID, "[RegistrationICP] Invalid max_correspondence_distance.");
    for (int k = 0; k < 16; ++k)
        if (!std::isfinite(init[k])) return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: init is not finite");
    if (!(relative_fitness >= 0.0) || !(relative_rmse >= 0.0))
        return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: relative_fitness and relative_rmse must be >= 0");
    if (max_iteration < 0) return set_error(OTSLAM_ERR_INVALID, "icp_point_to_plane: max_iteration < 0");
    double T[16];
    for (int k = 0; k < 16; ++k) T[k] = init[k];
    if (n_source == 0) {
        for (int k = 0; k < 16; ++k) transform_out[k] = T[k];
        if (fitness) *fitness = 0.0;
        if (inlier_rmse) *inlier_rmse = 0.0;
        if (iterations) *iterations = 0;
        return OTSLAM_OK;
    }
    OT_TRY(use_device(device));
    const int64_t n = n_source;
    const int n_cta = (int)((n + kIcpThreads - 1) / kIcpThreads);
    const int P = pow2_at_least(n_cta);
    DevBuf<double> ds0, ds1, dt, dtn, dpart, dsum;
    DevBuf<int32_t> dcorr;
    OT_CUDA(ds0.upload(source, n * 3)); OT_CUDA(ds1.alloc(n * 3)); OT_CUDA(dcorr.alloc(n));
    OT_CUDA(dpart.alloc((size_t)kIcpTerms * P)); OT_CUDA(dsum.alloc(kIcpTerms));
    if (n_target) { OT_CUDA(dt.upload(target, n_target * 3)); OT_CUDA(dtn.upload(target_normals, n_target * 3)); }
    OpTimer timer;
    // the target's grid once per call, cell = max_distance (otslam_cloud_nn_within's)
    KnnGrid g = {};
    GridBuffers b;
    if (n_target) {
        double mn[3], mx[3];
        OT_TRY(cloud_minmax(dt.p, n_target, mn, mx));
        OT_TRY(build_grid(dt.p, n_target, mn, mx, max_distance, 1 << 20, b, g));
    }
    const double r2 = max_distance * max_distance;
    double* cur = ds1.p;
    double* other = ds0.p;
    OT_TRY(device_rigid_transform(ds0.p, n, T, ds1.p, 0));
    double S[kIcpTerms];
    auto evaluate = [&](double& fit, double& rmse) -> int {
        icp_assoc_kernel<<<n_cta, kIcpThreads>>>(g, dt.p, dtn.p, n_target > 0, cur, n, r2, dcorr.p, dpart.p, P);
        OT_LAUNCHED();
        tree_rows_kernel<kIcpSumThreads><<<kIcpTerms, kIcpSumThreads>>>(dpart.p, n_cta, P, dsum.p);
        OT_LAUNCHED();
        OT_CUDA(cudaMemcpy(S, dsum.p, sizeof(S), cudaMemcpyDeviceToHost));
        fit = S[28] / (double)n;
        rmse = S[28] > 0.0 ? std::sqrt(S[29] / S[28]) : 0.0;
        return OTSLAM_OK;
    };
    double fit = 0.0, rmse = 0.0;
    OT_TRY(evaluate(fit, rmse));
    int it = 0;
    while (it < max_iteration) {
        // RegistrationICP: update = the solve's transform, or the identity when it fails or there is no correspondence
        double U[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1}, xi[6], Tn[16];
        if (S[28] > 0.0 && solve6(S, xi)) euler_update(xi, U);
        matmul4(U, T, Tn);
        for (int k = 0; k < 16; ++k) T[k] = Tn[k];
        OT_TRY(device_rigid_transform(cur, n, U, other, 0));
        std::swap(cur, other);
        const double fit0 = fit, rmse0 = rmse;
        OT_TRY(evaluate(fit, rmse));
        ++it;
        if (std::fabs(fit0 - fit) < relative_fitness && std::fabs(rmse0 - rmse) < relative_rmse) break;
    }
    timer.stop();
    if (corr_index) { OT_CUDA(dcorr.download(corr_index, n)); OT_CUDA(cudaDeviceSynchronize()); }
    for (int k = 0; k < 16; ++k) transform_out[k] = T[k];
    if (fitness) *fitness = fit;
    if (inlier_rmse) *inlier_rmse = rmse;
    if (iterations) *iterations = it;
    return OTSLAM_OK;
}

}  // extern "C"
