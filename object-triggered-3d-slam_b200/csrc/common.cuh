// common.cuh -- shared host/device helpers for the otslam_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <string>
#include <utility>

#include "../../include/otslam_b200.h"

namespace otslam {

extern thread_local std::string g_last_error;
extern std::atomic<int64_t> g_launches;
extern thread_local double g_last_op_ms;

extern thread_local uint64_t g_error_count;
inline int set_error(int code, const std::string& msg) {
    g_last_error = msg;
    ++g_error_count;
    return code;
}

#define OT_CUDA(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            int _code = (_e == cudaErrorMemoryAllocation) ? OTSLAM_ERR_NOMEM : OTSLAM_ERR_CUDA;        \
            return otslam::set_error(_code, std::string(#expr) + ": " + cudaGetErrorString(_e));       \
        }                                                                                               \
    } while (0)

#define OT_LAUNCHED()                                                                                   \
    do {                                                                                                \
        otslam::g_launches.fetch_add(1, std::memory_order_relaxed);                                     \
        OT_CUDA(cudaGetLastError());                                                                    \
    } while (0)

#define OT_TRY(expr)                                                                                    \
    do {                                                                                                \
        int _r = (expr);                                                                                \
        if (_r != OTSLAM_OK) return _r;                                                                 \
    } while (0)

// select the device (fails loudly when there is no usable GPU: the product has no CPU path)
int use_device(int device);

// General 4x4 inverse by cofactors, FP64 row-major.  Open3D inverts the extrinsic with Eigen
// (SURVEY A.3 "camera_pose = extrinsic.inverse()"); this routine defines camera_pose for the
// product.  (tests compare it with the oracle's restatement bit for bit.)
bool inverse4(const double* m, double* o);

constexpr int kRes = 16;                  // volume_unit_resolution
constexpr int kVox = kRes * kRes * kRes;  // 4096 voxels per block
constexpr int kStride = 4;                // depth_sampling_stride
constexpr uint64_t kEmptyKey = ~0ull;
constexpr int kKeyBias = 1 << 20;         // 21 bits per axis

__host__ __device__ inline uint64_t pack_key(int x, int y, int z) {
    return ((uint64_t)(uint32_t)(x + kKeyBias) << 42) | ((uint64_t)(uint32_t)(y + kKeyBias) << 21) |
           (uint64_t)(uint32_t)(z + kKeyBias);
}
__host__ __device__ inline void unpack_key(uint64_t k, int& x, int& y, int& z) {
    x = (int)((k >> 42) & 0x1FFFFF) - kKeyBias;
    y = (int)((k >> 21) & 0x1FFFFF) - kKeyBias;
    z = (int)(k & 0x1FFFFF) - kKeyBias;
}
__host__ __device__ inline bool key_in_range(int x, int y, int z) {
    return x >= -kKeyBias && x < kKeyBias && y >= -kKeyBias && y < kKeyBias && z >= -kKeyBias && z < kKeyBias;
}
__host__ __device__ inline uint32_t hash_key(uint64_t k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return (uint32_t)k;
}
// splitmix64 finaliser: the mesh sampler's counter-based RNG (cloud.cu) and the checkpoint checksums (checkpoint.cu)
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// uniform double in [0, 1) from (seed, counter): the mesh sampler's RNG (cloud.cu) and RANSAC's sampling (segment.cu)
__device__ __forceinline__ double u01(uint64_t seed, uint64_t ctr) {
    return __dmul_rn((double)(splitmix64(seed * 0xD1342543DE82EF95ull + ctr) >> 11), 1.0 / 9007199254740992.0);
}

// ---- multi-object arenas (config 3: multi_reconstruct_rgbd_filter.py, several objects, each "its own volume"): the
// objects share ONE block hash / pool / per-batch work list, so that one integration launch covers the union of their
// touched blocks.  The object id lives in the block key: object o (0..7) owns the x-key window
// [o * 2^18 - 2^20 + 0, +2^18), i.e. its true block coordinate kx in [-2^17, 2^17) is stored as kx + obj_key_offset(o).
// Sorting by key groups the blocks by object.  The stored key one past an object's last block (true kx = 2^17 - 1) is the
// next object's first block (true kx = -2^17): readers go through block_slot() (volume_lookup.cuh), which checks the window.
constexpr int kObjShift = 18;
constexpr int kMaxObjects = 8;
constexpr int kObjHalf = 1 << (kObjShift - 1);            // |true kx| limit inside an arena
__host__ __device__ inline int obj_key_offset(int o) { return (o << kObjShift) + kObjHalf - kKeyBias; }
__host__ __device__ inline int obj_of_key_x(int kx_stored) { return (kx_stored + kKeyBias) >> kObjShift; }

// ---------------------------------------------------------------------------------------------
// Voxel record: 16 bytes = ONE 128-bit transaction per voxel.
//   .x            tsdf, f32 running mean exactly as the reference computes it (SURVEY A.4)
//   .y/.z/.w      low 24 bits: integer sums of the R / G / B samples (exact; colour = sum / weight)
//   .y/.z         high 8 bits: low / high byte of the 16-bit integration count (weight); .w's high byte is 0
// Exact integer colour sums stay within 24 bits for <= 65535 integrations of a voxel
// (255 * 65535 < 2^24), which is also what the 16-bit count holds; the host refuses more frames per
// volume (OTSLAM_ERR_OVERFLOW).  All-zero bits == the reference's freshly opened voxel (tsdf 0, weight 0,
// colour 0).  (Round 1 spread a 24-bit count over all three words: two more shifts / masks per update and a
// second carry level for a range the frame limit never reaches.)
__host__ __device__ inline uint32_t rec_weight(const uint4& r) {
    return (r.y >> 24) | ((r.z >> 24) << 8);
}
__host__ __device__ inline uint4 rec_pack(float tsdf, uint32_t w, uint32_t rs, uint32_t gs, uint32_t bs) {
    uint4 r;
#ifdef __CUDA_ARCH__
    r.x = __float_as_uint(tsdf);
#else
    union { float f; uint32_t u; } c; c.f = tsdf; r.x = c.u;
#endif
    r.y = rs | ((w & 0xFFu) << 24);
    r.z = gs | (((w >> 8) & 0xFFu) << 24);
    r.w = bs;
    return r;
}
constexpr int kMaxFramesPerVolume = 65535;

// voxel (x,y,z) -> record index inside a block.  z-major so that the 256 (x,y) columns a CTA's
// threads own are contiguous: a warp touches 32 consecutive 16-byte records per z step.
__host__ __device__ inline int rec_index(int x, int y, int z) { return z * 256 + x * 16 + y; }

constexpr int kChunkBlocksLog2 = 9;                       // 512 blocks = 32 MiB per pool chunk
constexpr int kChunkBlocks = 1 << kChunkBlocksLog2;
constexpr int kMaxChunks = 8192;                          // 4 Mi blocks = 256 GiB of voxels

__device__ inline uint4* block_ptr(uint4* const* chunks, int slot) {
    return chunks[slot >> kChunkBlocksLog2] + (size_t)(slot & (kChunkBlocks - 1)) * kVox;
}

struct SlabSpec {
    int axis, thickness, n_ranks, rank, halo;
};
__host__ __device__ inline int floordiv_i(int a, int b) {
    int q = a / b, r = a % b;
    return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}
__host__ __device__ inline int slab_owner(const SlabSpec& s, int k) {
    int m = floordiv_i(k, s.thickness) % s.n_ranks;
    return m < 0 ? m + s.n_ranks : m;
}
// the coordinate that decides ownership: one block axis (0/1/2), or kx + ky for axis 3 ("diagonal" slabs:
// any axis-aligned wall or floor then spreads over all ranks, which single-axis slabs cannot do for planes
// perpendicular to their axis)
__host__ __device__ inline int slab_coord(const SlabSpec& s, int kx, int ky, int kz) {
    return s.axis == 0 ? kx : (s.axis == 1 ? ky : (s.axis == 2 ? kz : kx + ky));
}
__host__ __device__ inline bool slab_owns(const SlabSpec& s, int kx, int ky, int kz) {
    if (s.n_ranks <= 1) return true;
    return slab_owner(s, slab_coord(s, kx, ky, kz)) == s.rank;
}
// the same on the ownership coordinate alone
__host__ __device__ inline bool slab_keeps_coord(const SlabSpec& s, int a) {
    return slab_owner(s, a) == s.rank || (s.halo && slab_owner(s, a - 1) == s.rank);
}
__host__ __device__ inline bool slab_keeps(const SlabSpec& s, int kx, int ky, int kz) {
    if (s.n_ranks <= 1) return true;
    return slab_keeps_coord(s, slab_coord(s, kx, ky, kz));
}

// Scratch cache for the operators' temporaries and results: cudaMalloc / cudaFree cost 0.1-0.5 ms each
// (and cudaFree synchronises the device), which dominated the post-stage operators (a dozen buffers
// per call, kernels of a few hundred microseconds).  Freed blocks go to a per-device free list and
// are handed out again to requests of similar size.  Every operator synchronises before it returns
// (and the volume synchronises its stream before it replaces a result), so a released block is idle
// -- except on an error return, which is why a release that follows an error (the thread's error
// count moved since the allocation) drains the device first.
// otslam_trim_scratch() releases the cache.
extern thread_local uint64_t g_error_count;
cudaError_t scratch_alloc(void** p, size_t bytes);
void scratch_free(void* p);

// RAII device buffer from the scratch cache: the operators' temporaries and results, and the volume's mesh, points,
// sorted block list and halo pieces
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    uint64_t err_epoch = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n), err_epoch(o.err_epoch) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { release(); std::swap(p, o.p); std::swap(n, o.n); std::swap(err_epoch, o.err_epoch); }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (!p) return;
        if (err_epoch != g_error_count) cudaDeviceSynchronize();
        scratch_free(p);
        p = nullptr;
        n = 0;
    }
    cudaError_t alloc(size_t count) {
        release();
        n = count;
        err_epoch = g_error_count;
        return scratch_alloc((void**)&p, (count ? count : 1) * sizeof(T));
    }
    // alloc(count), then count elements from src; src and dst may be host or device pointers (unified addressing).  A
    // device-to-device cudaMemcpy may return before it completes: an operator synchronises before it returns.
    cudaError_t upload(const T* src, size_t count) {
        const cudaError_t e = alloc(count);
        return e != cudaSuccess ? e : cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyDefault);
    }
    cudaError_t download(T* dst, size_t count) const { return cudaMemcpy(dst, p, count * sizeof(T), cudaMemcpyDefault); }
};

// ---- owning handles for the long-lived resources (the volume, the decoder, checkpoint staging): move-only, released by
// the destructor.  Unlike DevBuf they bypass the scratch cache: cudaMalloc / cudaHostAlloc, freed when the owner goes.
// DeviceArray<T> / PinnedArray<T>: an array's capacity is 0 whenever its pointer is null.
template <typename T, bool kPinned, unsigned kHostFlags = cudaHostAllocDefault>
struct CudaArray {
    T* p = nullptr;
    size_t cap = 0;
    CudaArray() = default;
    CudaArray(CudaArray&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    CudaArray& operator=(CudaArray&& o) noexcept {
        if (this != &o) { release(); std::swap(p, o.p); std::swap(cap, o.cap); }
        return *this;
    }
    ~CudaArray() { release(); }
    void release() {
        if (p) { if constexpr (kPinned) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr;
        cap = 0;
    }
    // room for n elements: with less, frees the old allocation and allocates max(n, want) ({nullptr, 0} if that fails)
    cudaError_t reserve(size_t n, size_t want = 0) {
        if (n <= cap) return cudaSuccess;
        release();
        want = std::max(n, want);
        cudaError_t e;
        if constexpr (kPinned) e = cudaHostAlloc((void**)&p, want * sizeof(T), kHostFlags);
        else e = cudaMalloc((void**)&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        else p = nullptr;
        return e;
    }
};
template <typename T>
using DeviceArray = CudaArray<T, false>;
template <typename T, unsigned kHostFlags = cudaHostAllocDefault>
using PinnedArray = CudaArray<T, true, kHostFlags>;

// Event / Stream: null until create() succeeds; convert to the raw handle
template <typename H, cudaError_t (*kDestroy)(H)>
struct CudaHandle {
    H h = nullptr;
    CudaHandle() = default;
    CudaHandle(CudaHandle&& o) noexcept : h(o.h) { o.h = nullptr; }
    ~CudaHandle() { reset(); }
    void reset(H n = nullptr) {
        if (h) kDestroy(h);
        h = n;
    }
    operator H() const { return h; }
};
struct Event : CudaHandle<cudaEvent_t, cudaEventDestroy> {
    cudaError_t create(unsigned flags = cudaEventDefault) {
        cudaEvent_t e = nullptr;
        const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
        if (r == cudaSuccess) reset(e);
        return r;
    }
};
struct Stream : CudaHandle<cudaStream_t, cudaStreamDestroy> {
    cudaError_t create(unsigned flags, int priority = 0) {   // 0: the default priority
        cudaStream_t s = nullptr;
        const cudaError_t r = cudaStreamCreateWithPriority(&s, flags, priority);
        if (r == cudaSuccess) reset(s);
        return r;
    }
};

// Device-side duration of a stateless operator's kernel section (uploads before it and downloads
// after it excluded): events on the operators' stream, read back by otslam_last_op_device_ms().
struct OpTimer {
    Event a, b;
    bool stopped = false;
    cudaStream_t st;
    explicit OpTimer(cudaStream_t s = 0) : st(s) {
        g_last_op_ms = -1.0;
        if (a.create() == cudaSuccess && b.create() == cudaSuccess) cudaEventRecord(a, st);
    }
    void stop() {
        if (!stopped && b) cudaEventRecord(b, st);
        stopped = true;
    }
    ~OpTimer() {
        stop();
        float ms = 0.f;
        if (b && cudaEventSynchronize(b) == cudaSuccess && cudaEventElapsedTime(&ms, a, b) == cudaSuccess) g_last_op_ms = ms;
    }
};

// ---- device routines shared between translation units; each queues its work on stream s
// scan.cu: exclusive prefix sum of n int32 into int64, the total at d_out[n]
int device_exclusive_scan(const int* d_in, int64_t* d_out, int n, cudaStream_t s);
// knn.cu: stable LSD radix sort of (u64 key, i32 value) pairs by the low `bits` bits; result in (kb, vb), (ka, va) clobbered
int device_sort_pairs(uint64_t* ka, int32_t* va, uint64_t* kb, int32_t* vb, int64_t n, int bits, cudaStream_t s);
// ordered_sum.cu: the left-to-right FP64 chain over the terms of d_x[0..n), bit-identical to the scalar loop; term mode 0:
// x, 2: x > 0 ? x : 0, 3: x > 0 ? (x - mean)^2 : 0, the sum into *d_out; mode 1: x / *d_div, d_x becomes the inclusive prefix
int device_ordered_sum(double* d_x, int64_t n, int mode, const double* d_div, double mean, double* d_out, cudaStream_t s);
// cloud.cu: p' = (T * [p, 1]).xyz / w of n points, otslam_cloud_transform's arithmetic
int device_rigid_transform(const double* d_in, int64_t n, const double T[16], double* d_out, cudaStream_t s);
// extract.cu: compute_vertex_normals of a device mesh, each vertex's face normals added in triangle order
int device_vertex_normals(const double* d_verts, int64_t nv, const int32_t* d_faces, int64_t nf, double* d_normals,
                          cudaStream_t s);

}  // namespace otslam
