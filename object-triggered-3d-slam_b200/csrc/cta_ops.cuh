// cta_ops.cuh -- the CTA-level building blocks of the operator kernels: the intra-CTA exclusive scan, the ordered
// count -> scan -> emit compaction, and the fixed-order FP64 trees.  The trees fix the order of every addition, so results
// are bit-identical to the CPU models (tests/models/) whatever the schedule; each exists once, here, so that a change to
// an order reaches every operator that uses it.
#pragma once
#include "common.cuh"

namespace otslam {

// Exclusive scan of one value per thread over a CTA of kWarps full warps (a shuffle scan in each warp, then the warp sums
// through warp_sums[kWarps] in shared memory); *total (when not null) = the CTA's sum.  Every thread of the CTA calls it.
template <typename T, int kWarps>
__device__ __forceinline__ T cta_exclusive_scan(T mine, T* warp_sums, T* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    T inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    T before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        const T s = warp_sums[w];
        if (w < wid) before += s;
        tot += s;
    }
    if (total) *total = tot;
    return before + inc - mine;
}

// ---- ordered compaction: each CTA of 256 threads handles 1024 consecutive items (4 per thread, consecutive); a count
// pass writes each CTA's count, a scan over the CTAs gives their bases, an emit pass writes at base + intra-CTA rank.
constexpr int kItemsPerThread = 4;
constexpr int kItemsPerCta = 256 * kItemsPerThread;

// The count pass and the scan on stream s: launch(n_cta, nullptr, counts) runs the count pass; base[0..n_cta] = the
// scanned counts, *n_out = their total (synchronised).  The caller then sizes its outputs and runs
// launch(n_cta, base.p, nullptr), the emit pass.
template <typename F>
int compact_two_pass(int64_t n_items, cudaStream_t s, int64_t* n_out, DevBuf<int>& counts, DevBuf<int64_t>& base, F launch) {
    const int n_cta = (int)((n_items + kItemsPerCta - 1) / kItemsPerCta);
    *n_out = 0;
    if (n_cta == 0) return OTSLAM_OK;
    OT_CUDA(counts.alloc(n_cta));
    OT_CUDA(base.alloc(n_cta + 1));
    OT_TRY(launch(n_cta, (const int64_t*)nullptr, counts.p));
    OT_TRY(device_exclusive_scan(counts.p, base.p, n_cta, s));
    OT_CUDA(cudaMemcpyAsync(n_out, base.p + n_cta, 8, cudaMemcpyDefault, s));
    OT_CUDA(cudaStreamSynchronize(s));
    return OTSLAM_OK;
}

// Both passes of "emit index p < n where keep(p)", in ascending order.  Keep is a small functor struct with
// `__device__ bool operator()(int64_t p) const`.
template <typename Keep, typename Idx>
__global__ void __launch_bounds__(256) select_indices_kernel(const Keep keep, int64_t n, const int64_t* __restrict__ base,
                                                             int* __restrict__ counts, Idx* __restrict__ out) {
    __shared__ int warp_sum[8];
    const int64_t p0 = (int64_t)blockIdx.x * kItemsPerCta + threadIdx.x * kItemsPerThread;
    bool sel[kItemsPerThread];
    int mine = 0;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k) {
        sel[k] = p0 + k < n && keep(p0 + k);
        mine += sel[k];
    }
    int total;
    const int rank = cta_exclusive_scan<int, 8>(mine, warp_sum, &total);
    if (!base) {
        if (threadIdx.x == 0) counts[blockIdx.x] = total;
        return;
    }
    int64_t o = base[blockIdx.x] + rank;
#pragma unroll
    for (int k = 0; k < kItemsPerThread; ++k)
        if (sel[k]) out[o++] = (Idx)(p0 + k);
}

// The indices p < n with keep(p), ascending, into `out` on stream s; *n_out = their number.  `out` is allocated to
// *n_out + tail elements (not at all when that is 0); the tail is the caller's.
template <typename Keep, typename Idx>
int select_indices(const Keep& keep, int64_t n, cudaStream_t s, DevBuf<Idx>& out, int64_t* n_out, int64_t tail = 0) {
    DevBuf<int> counts;
    DevBuf<int64_t> base;
    auto launch = [&](int n_cta, const int64_t* b, int* cnt) -> int {
        select_indices_kernel<<<n_cta, 256, 0, s>>>(keep, n, b, cnt, out.p);
        OT_LAUNCHED();
        return OTSLAM_OK;
    };
    OT_TRY(compact_two_pass(n, s, n_out, counts, base, launch));
    if (*n_out + tail == 0) return OTSLAM_OK;
    OT_CUDA(out.alloc(*n_out + tail));
    if (*n_out == 0) return OTSLAM_OK;
    return launch((int)((n + kItemsPerCta - 1) / kItemsPerCta), base.p, nullptr);
}

// ---- fixed-order FP64 trees

// the smallest power of two >= x: the padded length of a row of the row tree
inline int pow2_at_least(int64_t x) {
    int P = 1;
    while (P < x) P *= 2;
    return P;
}

// The row tree, in place: rows[0 .. n_rows) of P = pow2_at_least(n_valid) partials each (row k at rows + k * P), entries
// i >= n_valid read as 0.0; i += i + P/2, then i + P/4, ..., + 1, so that rows[k * P] ends as row k's total.  The
// kThreads threads of the CTA stride over (row, i); every one of them calls it.
template <int kThreads>
__device__ __forceinline__ void cta_tree_rows(double* rows, int n_rows, int n_valid, int P) {
    for (int h = P / 2; h > 0; h >>= 1) {
        for (int j = threadIdx.x; j < n_rows * h; j += kThreads) {
            const int k = j / h, i = j - k * h;
            const double x = i < n_valid ? rows[(size_t)k * P + i] : 0.0;
            const double y = i + h < n_valid ? rows[(size_t)k * P + i + h] : 0.0;
            rows[(size_t)k * P + i] = __dadd_rn(x, y);
        }
        __syncthreads();
    }
}

// one CTA per row of buf (rows of P partials, n_valid real): out[row] = the row's total by the row tree
template <int kThreads>
__global__ void __launch_bounds__(kThreads) tree_rows_kernel(double* __restrict__ buf, int n_valid, int P, double* __restrict__ out) {
    double* row = buf + (size_t)blockIdx.x * P;
    cta_tree_rows<kThreads>(row, 1, n_valid, P);
    if (threadIdx.x == 0) out[blockIdx.x] = row[0];
}

// The halving tree over the columns of sm[kTerms][kThreads] in shared memory, one column per thread: column i += column
// i + kThreads/2, then i + kThreads/4, ..., + 1, so that sm[k][0] ends as term k's total.  Every thread calls it after
// writing its column; it synchronises before it returns.
template <int kTerms, int kThreads>
__device__ __forceinline__ void cta_halving_tree(double (&sm)[kTerms][kThreads]) {
    for (int s = kThreads / 2; s > 0; s >>= 1) {
        __syncthreads();
        for (int j = threadIdx.x; j < kTerms * s; j += kThreads) {
            const int k = j / s, i = j - k * s;
            sm[k][i] = __dadd_rn(sm[k][i], sm[k][i + s]);
        }
    }
    __syncthreads();
}

}  // namespace otslam
