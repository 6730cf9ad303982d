// scan.cu -- exclusive prefix sum int32 -> int64 (out[n] = total) used by every count -> scan -> emit
// compaction of the path and by the radix sort.  Three phases over tiles of 2048 items (256 threads x
// 8 consecutive items, coalesced 16-byte loads): per-tile sums, scan of the tile sums (one CTA), per-tile
// scan with the tile's base.  Inputs that fit one tile take a single launch.
#include "cta_ops.cuh"

namespace otslam {

constexpr int kScanItems = 8;
constexpr int kScanTile = 256 * kScanItems;

__device__ __forceinline__ void scan_load(const int* __restrict__ in, int64_t base, int64_t n, int (&v)[kScanItems]) {
    if (base + kScanItems <= n && ((reinterpret_cast<uintptr_t>(in + base) & 15) == 0)) {
        const int4 a = *reinterpret_cast<const int4*>(in + base), b = *reinterpret_cast<const int4*>(in + base + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) v[k] = (base + k < n) ? in[base + k] : 0;
    }
}

__global__ void __launch_bounds__(256) scan_tile_sum_kernel(const int* __restrict__ in, int64_t n, int64_t* __restrict__ tile_sum) {
    __shared__ int64_t ws[8];
    int v[kScanItems];
    scan_load(in, (int64_t)blockIdx.x * kScanTile + threadIdx.x * kScanItems, n, v);
    int64_t s = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) s += v[k];
    int64_t tot;
    cta_exclusive_scan<int64_t, 8>(s, ws, &tot);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = tot;
}

// exclusive scan of the tile sums in place (one CTA, 256 per round with a running carry); grand total -> *total
__global__ void __launch_bounds__(256) scan_tile_base_kernel(int64_t* __restrict__ tile_sum, int64_t n_tiles, int64_t* __restrict__ total) {
    __shared__ int64_t ws[8];
    __shared__ int64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < n_tiles; base += 256) {
        const int64_t i = base + threadIdx.x;
        const int64_t v = i < n_tiles ? tile_sum[i] : 0;
        int64_t tot;
        const int64_t ex = cta_exclusive_scan<int64_t, 8>(v, ws, &tot);
        if (i < n_tiles) tile_sum[i] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(256) scan_tile_kernel(const int* __restrict__ in, int64_t n, const int64_t* __restrict__ tile_base,
                                                        int64_t* __restrict__ out) {
    __shared__ int64_t ws[8];
    const int64_t base = (int64_t)blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    int v[kScanItems];
    scan_load(in, base, n, v);
    int64_t s = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) s += v[k];
    int64_t tot;
    int64_t acc = cta_exclusive_scan<int64_t, 8>(s, ws, &tot) + (tile_base ? tile_base[blockIdx.x] : 0);
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        if (base + k < n) out[base + k] = acc;
        acc += v[k];
    }
    if (!tile_base && threadIdx.x == 0) out[n] = tot;          // single-tile launch: total straight away
}

int device_exclusive_scan(const int* d_in, int64_t* d_out, int n, cudaStream_t s) {
    if (n <= 0) {
        OT_CUDA(cudaMemsetAsync(d_out, 0, 8, s));
        return OTSLAM_OK;
    }
    if (n <= kScanTile) {
        scan_tile_kernel<<<1, 256, 0, s>>>(d_in, n, nullptr, d_out);
        OT_LAUNCHED();
        return OTSLAM_OK;
    }
    const int64_t n_tiles = ((int64_t)n + kScanTile - 1) / kScanTile;
    DevBuf<int64_t> tiles;       // returned to the scratch cache at exit; later users are ordered behind us on the stream
    OT_CUDA(tiles.alloc(n_tiles));
    scan_tile_sum_kernel<<<(unsigned)n_tiles, 256, 0, s>>>(d_in, n, tiles.p);
    OT_LAUNCHED();
    scan_tile_base_kernel<<<1, 256, 0, s>>>(tiles.p, n_tiles, d_out + n);
    OT_LAUNCHED();
    scan_tile_kernel<<<(unsigned)n_tiles, 256, 0, s>>>(d_in, n, tiles.p, d_out);
    OT_LAUNCHED();
    return OTSLAM_OK;
}

}  // namespace otslam
