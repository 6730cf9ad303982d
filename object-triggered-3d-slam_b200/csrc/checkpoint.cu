// checkpoint.cu -- volume checkpoints: otslam_volume_save / otslam_volume_load / otslam_checkpoint_info.
//
// A checkpoint holds the voxel records of a volume's blocks verbatim (the 16-byte records of common.cuh, exact
// integer colour sums and counts included), so "integrate A, save, load, integrate B" gives the same bits as
// "integrate A then B".  File format version 1 (DESIGN.md §4 "Checkpoints"), all little-endian:
//   [0, 4096)        header (CkptHeader)
//   keys_off = 4096  i32 [n][3] block keys, strictly ascending (x, y, z): the export_blocks order; padded to 4 KiB
//   cks_off          u64 [n] block checksums; padded to 4 KiB
//   rec_off          n x 65536 bytes: each block's 4096 records as they lie in the pool (in-block order rec_index)
// Block checksum  c = mix(pack_key(x, y, z)) + sum_{i < 8192} mix(w[i] ^ (i * 0x9E3779B97F4A7C15))  mod 2^64, w[i] the
// i-th u64 word of the block and mix = splitmix64; the header checksum is the same sum over the header's first 511 words.
// Any change to the record layout needs a new format version.
//
//   save: ckpt_own_kernel + scan + ckpt_select_kernel pick the blocks the volume is responsible for, in key order;
//         ckpt_gather_kernel (one CTA per block) copies each block into a staging buffer and sums its checksum;
//         chunks of 1024 blocks go D2H into pinned buffers while a host thread writes the previous chunk.
//   load: ckpt_filter_kernel checks every key (range, order, slab_keeps, read-only probe of the block hash) and
//         ckpt_kept_kernel compacts the kept ones; their records are read by a host thread and copied straight into
//         the pool slots they will get (n_blocks + j, beyond the pool counter, so the volume is unchanged), where
//         ckpt_verify_kernel checks checksums and record validity.  Only when every check passed are the keys
//         inserted (ckpt_insert_kernel) and the pool counter moved; otherwise the slots are zeroed again.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstring>
#include <thread>
#include <vector>

#include "volume.cuh"

namespace otslam {

constexpr char kCkptMagic[8] = {'O', 'T', 'S', 'L', 'A', 'M', 'C', 'K'};
constexpr uint32_t kCkptVersion = 1;
constexpr int64_t kCkptPage = 4096;
constexpr int64_t kBlockFileBytes = (int64_t)kVox * 16;
constexpr int kCkptChunk = 1024;                           // blocks per staging buffer: 64 MiB
constexpr uint64_t kGolden = 0x9E3779B97F4A7C15ull;

struct CkptHeader {
    char magic[8];
    uint32_t version, record_bytes, voxels_per_block;
    int32_t color_type;
    double voxel_length, sdf_trunc;
    int64_t frames, n_blocks;
    uint8_t reserved[4088 - 56];
    uint64_t checksum;          // over the 511 words before it
};
static_assert(sizeof(CkptHeader) == kCkptPage, "checkpoint header layout");

__host__ __device__ __forceinline__ uint64_t ckpt_word(uint64_t w, uint64_t i) { return splitmix64(w ^ (i * kGolden)); }

static inline int64_t page_pad(int64_t b) { return (b + kCkptPage - 1) & ~(kCkptPage - 1); }

struct CkptLayout {
    int64_t n, keys_off, cks_off, rec_off, total;
    explicit CkptLayout(int64_t n_blocks) : n(n_blocks) {
        keys_off = kCkptPage;
        cks_off = keys_off + page_pad(12 * n);
        rec_off = cks_off + page_pad(8 * n);
        total = rec_off + n * kBlockFileBytes;
    }
};

static uint64_t header_checksum(const CkptHeader& h) {
    uint64_t w[511], s = 0;
    memcpy(w, &h, sizeof(w));
    for (int i = 0; i < 511; ++i) s += ckpt_word(w[i], (uint64_t)i);
    return s;
}

// per-thread timings of the last save / load (otslam_checkpoint_profile)
thread_local double g_ckpt_prof[4] = {-1, -1, -1, -1};

using Clock = std::chrono::steady_clock;
static double ms_since(Clock::time_point t0) { return std::chrono::duration<double, std::milli>(Clock::now() - t0).count(); }

// full-length pread / pwrite; the time spent inside them is added to *ns
static bool pread_all(int fd, void* p, size_t n, int64_t off, std::atomic<int64_t>* ns) {
    const auto t0 = Clock::now();
    char* c = static_cast<char*>(p);
    while (n) {
        const ssize_t r = pread(fd, c, n, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) return false;
        c += r; n -= (size_t)r; off += r;
    }
    if (ns) *ns += std::chrono::duration_cast<std::chrono::nanoseconds>(Clock::now() - t0).count();
    return true;
}
static bool pwrite_all(int fd, const void* p, size_t n, int64_t off, std::atomic<int64_t>* ns) {
    const auto t0 = Clock::now();
    const char* c = static_cast<const char*>(p);
    while (n) {
        const ssize_t r = pwrite(fd, c, n, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) return false;
        c += r; n -= (size_t)r; off += r;
    }
    if (ns) *ns += std::chrono::duration_cast<std::chrono::nanoseconds>(Clock::now() - t0).count();
    return true;
}

// reads and validates the header of an open checkpoint (host only)
static int read_header(int fd, const char* path, CkptHeader& h) {
    struct stat st;
    if (fstat(fd, &st) != 0) return set_error(OTSLAM_ERR_INVALID, std::string("cannot stat ") + path);
    if (st.st_size < kCkptPage || !pread_all(fd, &h, sizeof(h), 0, nullptr))
        return set_error(OTSLAM_ERR_FORMAT, std::string("checkpoint too short for its header: ") + path);
    if (memcmp(h.magic, kCkptMagic, 8) != 0) return set_error(OTSLAM_ERR_FORMAT, std::string("not a volume checkpoint (bad magic): ") + path);
    if (h.version != kCkptVersion)
        return set_error(OTSLAM_ERR_FORMAT, "checkpoint format version " + std::to_string(h.version) + " (this library reads version 1)");
    if (header_checksum(h) != h.checksum) return set_error(OTSLAM_ERR_FORMAT, std::string("checkpoint header checksum mismatch: ") + path);
    if (h.record_bytes != 16 || h.voxels_per_block != (uint32_t)kVox || (h.color_type != OTSLAM_COLOR_NONE && h.color_type != OTSLAM_COLOR_RGB8) ||
        !(h.voxel_length > 0.0) || !(h.sdf_trunc > 0.0) || h.frames < 0 || h.frames > kMaxFramesPerVolume || h.n_blocks < 0 ||
        h.n_blocks > (int64_t)kMaxChunks * kChunkBlocks)
        return set_error(OTSLAM_ERR_FORMAT, std::string("checkpoint header fields out of range: ") + path);
    if (CkptLayout(h.n_blocks).total != (int64_t)st.st_size)
        return set_error(OTSLAM_ERR_FORMAT, "checkpoint size " + std::to_string((long long)st.st_size) + " does not match its " +
                                                std::to_string((long long)h.n_blocks) + " blocks (truncated or damaged)");
    return OTSLAM_OK;
}

struct Fd {
    int fd = -1;
    ~Fd() { if (fd >= 0) close(fd); }
};

// =============================================================================================
// kernels
// =============================================================================================
__device__ __forceinline__ uint64_t cta_sum_u64(uint64_t s, uint64_t* red /*[8]*/) {
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    uint64_t t = 0;
    if (threadIdx.x == 0)
        for (int w = 0; w < 8; ++w) t += red[w];
    return t;
}

// save: 1 for the blocks this volume is responsible for (slab ranks: owned blocks only)
__global__ void __launch_bounds__(256) ckpt_own_kernel(const uint64_t* __restrict__ keys, int n, SlabSpec slab, int* __restrict__ flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int x, y, z;
    unpack_key(keys[i], x, y, z);
    flag[i] = slab_owns(slab, x, y, z) ? 1 : 0;
}

// save: order-preserving compaction -> file keys (arena offset removed) and pool slots
__global__ void __launch_bounds__(256) ckpt_select_kernel(const int* __restrict__ flag, const int64_t* __restrict__ pos, int n,
                                                          const uint64_t* __restrict__ keys, const int32_t* __restrict__ slots, int x_off,
                                                          int32_t* __restrict__ out_keys, int32_t* __restrict__ out_slots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const int64_t p = pos[i];
    int x, y, z;
    unpack_key(keys[i], x, y, z);
    out_keys[3 * p] = x - x_off; out_keys[3 * p + 1] = y; out_keys[3 * p + 2] = z;
    out_slots[p] = slots[i];
}

// save: one CTA per block -- 64 KiB pool block -> staging, and its checksum
__global__ void __launch_bounds__(256) ckpt_gather_kernel(uint4* const* chunks, const int32_t* __restrict__ slots,
                                                          const int32_t* __restrict__ keys, uint4* __restrict__ out,
                                                          uint64_t* __restrict__ cks) {
    __shared__ uint64_t red[8];
    const int b = blockIdx.x;
    const uint4* src = block_ptr(chunks, slots[b]);
    uint4* dst = out + (size_t)b * kVox;
    uint64_t s = 0;
#pragma unroll 4
    for (int r = threadIdx.x; r < kVox; r += 256) {
        const uint4 q = src[r];
        __stcs(dst + r, q);
        s += ckpt_word((uint64_t)q.x | ((uint64_t)q.y << 32), 2 * r) + ckpt_word((uint64_t)q.z | ((uint64_t)q.w << 32), 2 * r + 1);
    }
    s = cta_sum_u64(s, red);
    if (threadIdx.x == 0) cks[b] = s + splitmix64(pack_key(keys[3 * b], keys[3 * b + 1], keys[3 * b + 2]));
}

// load: per file key -- range, strict ascending order, which blocks this volume keeps, and a read-only probe of the hash
enum LoadBad { kBadRange = 1, kBadOrder = 2, kBadPresent = 4, kBadChecksum = 8, kBadRecord = 16 };
struct FilterArgs {
    const int32_t* keys;        // [n][3] as in the file
    int n, x_off, arena;
    SlabSpec slab;
    HashTable table;
    int* flag;
    uint64_t* packed;
    int* bad;
};
__global__ void __launch_bounds__(256) ckpt_filter_kernel(FilterArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const int x = a.keys[3 * i], y = a.keys[3 * i + 1], z = a.keys[3 * i + 2];
    a.flag[i] = 0;
    if (i > 0) {
        const int px = a.keys[3 * i - 3], py = a.keys[3 * i - 2], pz = a.keys[3 * i - 1];
        if (!(px < x || (px == x && (py < y || (py == y && pz < z))))) atomicOr(a.bad, kBadOrder);
    }
    if (!key_in_range(x, y, z) || (a.arena && (x < -kObjHalf || x >= kObjHalf))) { atomicOr(a.bad, kBadRange); return; }
    const int sx = x + a.x_off;
    if (!slab_keeps(a.slab, sx, y, z)) return;
    const uint64_t k = pack_key(sx, y, z);
    if (hash_find(a.table, k) >= 0) atomicOr(a.bad, kBadPresent);
    a.flag[i] = 1;
    a.packed[i] = k;
}

// load: order-preserving compaction of the kept file indices
__global__ void __launch_bounds__(256) ckpt_kept_kernel(const int* __restrict__ flag, const int64_t* __restrict__ pos, int n,
                                                        const uint64_t* __restrict__ packed, int32_t* __restrict__ kept_idx,
                                                        uint64_t* __restrict__ kept_keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i]) return;
    kept_idx[pos[i]] = i;
    kept_keys[pos[i]] = packed[i];
}

// load: one CTA per block already copied into its future pool slot -- checksum and record validity
__global__ void __launch_bounds__(256) ckpt_verify_kernel(uint4* const* chunks, int first_slot, const int32_t* __restrict__ kept_idx,
                                                          const int32_t* __restrict__ keys, const uint64_t* __restrict__ cks,
                                                          uint32_t frames, int no_color, int* __restrict__ bad) {
    __shared__ uint64_t red[8];
    const int b = blockIdx.x;
    const uint4* blk = block_ptr(chunks, first_slot + b);
    uint64_t s = 0;
    bool ok = true;
#pragma unroll 4
    for (int r = threadIdx.x; r < kVox; r += 256) {
        const uint4 q = blk[r];
        s += ckpt_word((uint64_t)q.x | ((uint64_t)q.y << 32), 2 * r) + ckpt_word((uint64_t)q.z | ((uint64_t)q.w << 32), 2 * r + 1);
        const uint32_t w = rec_weight(q), cmax = no_color ? 0u : 255u * w;
        ok &= (w <= frames) & ((q.w >> 24) == 0u) & ((q.y & 0xFFFFFFu) <= cmax) & ((q.z & 0xFFFFFFu) <= cmax) & ((q.w & 0xFFFFFFu) <= cmax);
    }
    const int any_bad = __syncthreads_or(!ok);
    s = cta_sum_u64(s, red);
    if (threadIdx.x == 0) {
        const int i = kept_idx[b];
        if (s + splitmix64(pack_key(keys[3 * i], keys[3 * i + 1], keys[3 * i + 2])) != cks[i]) atomicOr(bad, kBadChecksum);
        if (any_bad) atomicOr(bad, kBadRecord);
    }
}

// load: keys known to be absent and distinct; kept block j gets pool slot first_slot + j (its records are already there)
__global__ void __launch_bounds__(256) ckpt_insert_kernel(const uint64_t* __restrict__ kept_keys, int m, int first_slot, HashTable t) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) hash_insert_absent(t, kept_keys[j], first_slot + j);
}

// =============================================================================================
// host side
// =============================================================================================
// page-locked staging pair, CUDA events per chunk (kernel / copy times); the I/O threads are joined on every return path
// before the buffers and events go
struct Staging {
    PinnedArray<char, cudaHostAllocPortable> host[2];
    std::vector<Event> ev;           // per chunk: kernel start / end, copy start / end
    std::thread io[2];
    ~Staging() {
        for (auto& t : io) if (t.joinable()) t.join();
    }
    int init(int n_chunks) {
        for (auto& p : host) OT_CUDA(p.reserve((size_t)kCkptChunk * kBlockFileBytes));
        ev.resize((size_t)n_chunks * 4);
        for (auto& e : ev) OT_CUDA(e.create());
        return OTSLAM_OK;
    }
    void join(int b) { if (io[b].joinable()) io[b].join(); }
    void times(double& kernel_ms, double& copy_ms) {      // after the stream has drained
        kernel_ms = copy_ms = 0;
        for (size_t c = 0; c + 3 < ev.size(); c += 4) {
            float a = 0, b = 0;
            if (cudaEventElapsedTime(&a, ev[c], ev[c + 1]) == cudaSuccess) kernel_ms += a;
            if (cudaEventElapsedTime(&b, ev[c + 2], ev[c + 3]) == cudaSuccess) copy_ms += b;
        }
    }
};

static bool same_bits(double a, double b) { return memcmp(&a, &b, sizeof(double)) == 0; }

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_checkpoint_info(const char* path, double* voxel_length, double* sdf_trunc, int32_t* color_type, int64_t* frames,
                           int64_t* n_blocks) {
    if (!path) return set_error(OTSLAM_ERR_INVALID, "null path");
    Fd f;
    f.fd = open(path, O_RDONLY | O_CLOEXEC);
    if (f.fd < 0) return set_error(OTSLAM_ERR_INVALID, std::string("cannot open ") + path + ": " + strerror(errno));
    CkptHeader h;
    OT_TRY(read_header(f.fd, path, h));
    if (voxel_length) *voxel_length = h.voxel_length;
    if (sdf_trunc) *sdf_trunc = h.sdf_trunc;
    if (color_type) *color_type = h.color_type;
    if (frames) *frames = h.frames;
    if (n_blocks) *n_blocks = h.n_blocks;
    return OTSLAM_OK;
}

int otslam_checkpoint_profile(double out[4]) {
    if (!out) return set_error(OTSLAM_ERR_INVALID, "null output");
    memcpy(out, g_ckpt_prof, sizeof(g_ckpt_prof));
    return OTSLAM_OK;
}

int otslam_volume_save(otslam_volume* v, const char* path) {
    if (!v || !path || !path[0]) return set_error(OTSLAM_ERR_INVALID, "null volume or path");
    const auto t_start = Clock::now();
    for (double& p : g_ckpt_prof) p = 0;
    OT_TRY(use_device(v->device));
    cudaStream_t s = v->stream;
    const uint64_t* dk = nullptr;
    const int32_t* ds = nullptr;
    int n_sorted = 0, x_off = 0;
    OT_TRY(volume_selected_blocks_device(v, &dk, &ds, &n_sorted, &x_off));   // arena: the selected object (error if none)

    // the blocks this volume is responsible for, in key order
    int m = 0;
    DevBuf<int> flag;
    DevBuf<int64_t> pos;
    DevBuf<int32_t> keys3, slots;
    if (n_sorted > 0) {
        OT_CUDA(flag.alloc(n_sorted)); OT_CUDA(pos.alloc((size_t)n_sorted + 1));
        OT_CUDA(keys3.alloc((size_t)n_sorted * 3)); OT_CUDA(slots.alloc(n_sorted));
        ckpt_own_kernel<<<(n_sorted + 255) / 256, 256, 0, s>>>(dk, n_sorted, v->slab, flag.p);
        OT_LAUNCHED();
        OT_TRY(device_exclusive_scan(flag.p, pos.p, n_sorted, s));
        ckpt_select_kernel<<<(n_sorted + 255) / 256, 256, 0, s>>>(flag.p, pos.p, n_sorted, dk, ds, x_off, keys3.p, slots.p);
        OT_LAUNCHED();
        int64_t total = 0;
        OT_CUDA(cudaMemcpyAsync(&total, pos.p + n_sorted, 8, cudaMemcpyDeviceToHost, s));
        OT_CUDA(cudaStreamSynchronize(s));
        m = (int)total;
    }
    CkptHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, kCkptMagic, 8);
    h.version = kCkptVersion; h.record_bytes = 16; h.voxels_per_block = kVox; h.color_type = v->color_type;
    h.voxel_length = v->voxel_length; h.sdf_trunc = v->sdf_trunc;
    h.frames = v->n_objects > 0 ? v->obj_frames[v->sel_obj] : v->frames_integrated;
    h.n_blocks = m;
    h.checksum = header_checksum(h);
    const CkptLayout L(m);
    std::vector<int32_t> hkeys((size_t)m * 3);
    std::vector<uint64_t> hcks((size_t)m);
    if (m) OT_CUDA(cudaMemcpyAsync(hkeys.data(), keys3.p, (size_t)m * 12, cudaMemcpyDeviceToHost, s));

    const std::string tmp = std::string(path) + ".tmp." + std::to_string((long long)getpid());
    Fd f;
    f.fd = open(tmp.c_str(), O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0644);
    if (f.fd < 0) return set_error(OTSLAM_ERR_INVALID, "cannot create " + tmp + ": " + strerror(errno));
    std::atomic<int64_t> file_ns{0};
    std::atomic<bool> io_ok{true};
    int rc = [&]() -> int {
        if (ftruncate(f.fd, (off_t)L.total) != 0) return set_error(OTSLAM_ERR_INVALID, "cannot size " + tmp + ": " + strerror(errno));
        const int n_chunks = (m + kCkptChunk - 1) / kCkptChunk;
        DevBuf<uint4> stage[2];
        DevBuf<uint64_t> cks;
        Staging st;
        if (m) {
            OT_CUDA(cks.alloc(m));
            for (auto& b : stage) OT_CUDA(b.alloc((size_t)std::min(m, kCkptChunk) * kVox));
            OT_TRY(st.init(n_chunks));
        }
        for (int c = 0; c < n_chunks; ++c) {
            const int b = c & 1, j0 = c * kCkptChunk, nb = std::min(kCkptChunk, m - j0);
            st.join(b);                                           // chunk c-2's write from host[b] is done
            if (!io_ok) break;
            const Event* e = &st.ev[(size_t)c * 4];
            OT_CUDA(cudaEventRecord(e[0], s));
            ckpt_gather_kernel<<<nb, 256, 0, s>>>(v->d_chunks.p, slots.p + j0, keys3.p + (size_t)j0 * 3, stage[b].p, cks.p + j0);
            OT_LAUNCHED();
            OT_CUDA(cudaEventRecord(e[1], s));
            OT_CUDA(cudaEventRecord(e[2], s));
            OT_CUDA(cudaMemcpyAsync(st.host[b].p, stage[b].p, (size_t)nb * kBlockFileBytes, cudaMemcpyDeviceToHost, s));
            OT_CUDA(cudaEventRecord(e[3], s));
            const int dev = v->device, fd = f.fd;
            void* src = st.host[b].p;
            const int64_t off = L.rec_off + (int64_t)j0 * kBlockFileBytes;
            st.io[b] = std::thread([=, &file_ns, &io_ok]() {      // overlaps the gather + copy of chunk c+1
                cudaSetDevice(dev);
                if (cudaEventSynchronize(e[3]) != cudaSuccess || !pwrite_all(fd, src, (size_t)nb * kBlockFileBytes, off, &file_ns)) io_ok = false;
            });
        }
        st.join(0); st.join(1);
        OT_CUDA(cudaStreamSynchronize(s));
        if (!io_ok) return set_error(OTSLAM_ERR_INVALID, "writing " + tmp + " failed: " + strerror(errno));
        if (m) OT_CUDA(cudaMemcpy(hcks.data(), cks.p, (size_t)m * 8, cudaMemcpyDeviceToHost));
        if (!pwrite_all(f.fd, &h, sizeof(h), 0, &file_ns) || !pwrite_all(f.fd, hkeys.data(), (size_t)m * 12, L.keys_off, &file_ns) ||
            !pwrite_all(f.fd, hcks.data(), (size_t)m * 8, L.cks_off, &file_ns))
            return set_error(OTSLAM_ERR_INVALID, "writing " + tmp + " failed: " + strerror(errno));
        const auto t_sync = Clock::now();
        if (fsync(f.fd) != 0) return set_error(OTSLAM_ERR_INVALID, "fsync of " + tmp + " failed: " + strerror(errno));
        file_ns += std::chrono::duration_cast<std::chrono::nanoseconds>(Clock::now() - t_sync).count();
        st.times(g_ckpt_prof[0], g_ckpt_prof[1]);
        return OTSLAM_OK;
    }();
    close(f.fd);
    f.fd = -1;
    if (rc == OTSLAM_OK && rename(tmp.c_str(), path) != 0) rc = set_error(OTSLAM_ERR_INVALID, std::string("cannot rename to ") + path + ": " + strerror(errno));
    if (rc != OTSLAM_OK) {
        unlink(tmp.c_str());
        return rc;
    }
    g_ckpt_prof[2] = file_ns.load() * 1e-6;
    g_ckpt_prof[3] = ms_since(t_start);
    return OTSLAM_OK;
}

int otslam_volume_load(otslam_volume* v, const char* path, int64_t* n_loaded) {
    if (!v || !path) return set_error(OTSLAM_ERR_INVALID, "null volume or path");
    if (n_loaded) *n_loaded = 0;
    const auto t_start = Clock::now();
    for (double& p : g_ckpt_prof) p = 0;
    Fd f;
    f.fd = open(path, O_RDONLY | O_CLOEXEC);
    if (f.fd < 0) return set_error(OTSLAM_ERR_INVALID, std::string("cannot open ") + path + ": " + strerror(errno));
    CkptHeader h;
    OT_TRY(read_header(f.fd, path, h));
    if (!same_bits(h.voxel_length, v->voxel_length) || !same_bits(h.sdf_trunc, v->sdf_trunc) || h.color_type != v->color_type)
        return set_error(OTSLAM_ERR_INVALID, "checkpoint voxel_length / sdf_trunc / color_type differ from the volume's");
    if (v->n_objects > 0 && v->sel_obj < 0) return set_error(OTSLAM_ERR_INVALID, "multi-object arena: otslam_volume_select_object first");
    OT_TRY(use_device(v->device));
    cudaStream_t s = v->stream;
    const int n = (int)h.n_blocks;
    const CkptLayout L(n);
    std::atomic<int64_t> file_ns{0};
    int m = 0, base = 0;
    if (n > 0) {
        std::vector<int32_t> fkeys((size_t)n * 3);
        if (!pread_all(f.fd, fkeys.data(), fkeys.size() * 4, L.keys_off, &file_ns))
            return set_error(OTSLAM_ERR_FORMAT, std::string("cannot read the key table of ") + path);
        DevBuf<int32_t> keys3, kept_idx;
        DevBuf<uint64_t> cks, packed, kept_keys;
        DevBuf<int> flag, bad;
        DevBuf<int64_t> pos;
        OT_CUDA(keys3.alloc((size_t)n * 3)); OT_CUDA(cks.alloc(n)); OT_CUDA(packed.alloc(n)); OT_CUDA(flag.alloc(n));
        OT_CUDA(pos.alloc((size_t)n + 1)); OT_CUDA(bad.alloc(1));
        OT_CUDA(cudaMemcpyAsync(keys3.p, fkeys.data(), (size_t)n * 12, cudaMemcpyHostToDevice, s));
        OT_CUDA(cudaMemsetAsync(bad.p, 0, 4, s));
        FilterArgs fa;
        fa.keys = keys3.p; fa.n = n; fa.x_off = v->n_objects > 0 ? obj_key_offset(v->sel_obj) : 0; fa.arena = v->n_objects > 0;
        fa.slab = v->slab; fa.table = volume_hash(v); fa.flag = flag.p; fa.packed = packed.p; fa.bad = bad.p;
        ckpt_filter_kernel<<<(n + 255) / 256, 256, 0, s>>>(fa);
        OT_LAUNCHED();
        OT_TRY(device_exclusive_scan(flag.p, pos.p, n, s));
        int hb = 0;
        int64_t total = 0;
        OT_CUDA(cudaMemcpyAsync(&hb, bad.p, 4, cudaMemcpyDeviceToHost, s));
        OT_CUDA(cudaMemcpyAsync(&total, pos.p + n, 8, cudaMemcpyDeviceToHost, s));
        OT_CUDA(cudaMemcpyAsync(&base, v->d_counters.p + kPoolCount, 4, cudaMemcpyDeviceToHost, s));   // first free pool slot
        OT_CUDA(cudaStreamSynchronize(s));
        if (hb & kBadRange) return set_error(OTSLAM_ERR_OVERFLOW, "checkpoint block key outside the volume's key range (arena objects: |kx| < 2^17)");
        if (hb & kBadOrder) return set_error(OTSLAM_ERR_FORMAT, "checkpoint keys are not strictly ascending (duplicate or unordered key)");
        if (hb & kBadPresent) return set_error(OTSLAM_ERR_INVALID, "checkpoint block already present in the volume");
        m = (int)total;
        if (m > 0) {
            std::vector<uint64_t> fcks((size_t)n);
            if (!pread_all(f.fd, fcks.data(), fcks.size() * 8, L.cks_off, &file_ns))
                return set_error(OTSLAM_ERR_FORMAT, std::string("cannot read the checksum table of ") + path);
            OT_CUDA(cudaMemcpyAsync(cks.p, fcks.data(), (size_t)n * 8, cudaMemcpyHostToDevice, s));
            OT_CUDA(kept_idx.alloc(m)); OT_CUDA(kept_keys.alloc(m));
            ckpt_kept_kernel<<<(n + 255) / 256, 256, 0, s>>>(flag.p, pos.p, n, packed.p, kept_idx.p, kept_keys.p);
            OT_LAUNCHED();
            std::vector<int32_t> hidx((size_t)m);
            OT_CUDA(cudaMemcpyAsync(hidx.data(), kept_idx.p, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
            OT_CUDA(cudaStreamSynchronize(s));
            // pool chunks for the new slots (zeroed; beyond the pool counter, so the volume's contents do not change)
            OT_TRY(ensure_pool(v, (int64_t)base + m));
            const int n_chunks = (m + kCkptChunk - 1) / kCkptChunk;
            Staging st;
            OT_TRY(st.init(n_chunks));
            std::atomic<bool> io_ok{true};
            auto read_chunk = [&, fd = f.fd](int c) {       // kept blocks of chunk c -> host[c & 1], runs of consecutive file blocks per pread
                const int b = c & 1, j0 = c * kCkptChunk, j1 = std::min(m, j0 + kCkptChunk);
                cudaSetDevice(v->device);
                if (c >= 2 && cudaEventSynchronize(st.ev[(size_t)(c - 2) * 4 + 3]) != cudaSuccess) { io_ok = false; return; }
                char* dst = st.host[b].p;
                for (int j = j0; j < j1;) {
                    int k = j + 1;
                    while (k < j1 && hidx[(size_t)k] == hidx[(size_t)k - 1] + 1) ++k;
                    if (!pread_all(fd, dst + (size_t)(j - j0) * kBlockFileBytes, (size_t)(k - j) * kBlockFileBytes,
                                   L.rec_off + (int64_t)hidx[(size_t)j] * kBlockFileBytes, &file_ns)) { io_ok = false; return; }
                    j = k;
                }
            };
            const uint32_t frames = (uint32_t)h.frames;
            const int no_color = v->color_type == OTSLAM_COLOR_NONE;
            int rc = [&]() -> int {
                st.io[0] = std::thread(read_chunk, 0);
                for (int c = 0; c < n_chunks; ++c) {
                    const int b = c & 1, j0 = c * kCkptChunk, nb = std::min(kCkptChunk, m - j0);
                    st.join(b);
                    if (!io_ok) return set_error(OTSLAM_ERR_FORMAT, std::string("cannot read the records of ") + path);
                    if (c + 1 < n_chunks) st.io[b ^ 1] = std::thread(read_chunk, c + 1);   // overlaps the copy + verify of chunk c
                    const Event* e = &st.ev[(size_t)c * 4];
                    OT_CUDA(cudaEventRecord(e[2], s));
                    for (int j = 0; j < nb;) {              // whole blocks into their slots, split at pool-chunk boundaries
                        const int slot = base + j0 + j, run = std::min(nb - j, kChunkBlocks - (slot & (kChunkBlocks - 1)));
                        OT_CUDA(cudaMemcpyAsync(v->chunks[(size_t)(slot >> kChunkBlocksLog2)].p + (size_t)(slot & (kChunkBlocks - 1)) * kVox,
                                                st.host[b].p + (size_t)j * kBlockFileBytes, (size_t)run * kBlockFileBytes,
                                                cudaMemcpyHostToDevice, s));
                        j += run;
                    }
                    OT_CUDA(cudaEventRecord(e[3], s));
                    OT_CUDA(cudaEventRecord(e[0], s));
                    ckpt_verify_kernel<<<nb, 256, 0, s>>>(v->d_chunks.p, base + j0, kept_idx.p + j0, keys3.p, cks.p, frames, no_color, bad.p);
                    OT_LAUNCHED();
                    OT_CUDA(cudaEventRecord(e[1], s));
                }
                OT_CUDA(cudaMemcpyAsync(&hb, bad.p, 4, cudaMemcpyDeviceToHost, s));
                OT_CUDA(cudaStreamSynchronize(s));
                if (hb & kBadChecksum) return set_error(OTSLAM_ERR_FORMAT, std::string("checkpoint block checksum mismatch (damaged file): ") + path);
                if (hb & kBadRecord)
                    return set_error(OTSLAM_ERR_FORMAT, "checkpoint records invalid (count > frames, colour sum > 255 * count, or colour in a NoColor file)");
                return OTSLAM_OK;
            }();
            st.join(0); st.join(1);
            if (rc != OTSLAM_OK) {                           // the slots beyond the pool counter must be zero again
                cudaStreamSynchronize(s);
                for (int j = 0; j < m;) {
                    const int slot = base + j, run = std::min(m - j, kChunkBlocks - (slot & (kChunkBlocks - 1)));
                    cudaMemsetAsync(v->chunks[(size_t)(slot >> kChunkBlocksLog2)].p + (size_t)(slot & (kChunkBlocks - 1)) * kVox, 0,
                                    (size_t)run * kBlockFileBytes, s);
                    j += run;
                }
                cudaStreamSynchronize(s);
                return rc;
            }
            // every check passed: insert
            OT_TRY(reserve_hash(v, (int64_t)base + m));
            Event ei[2];
            OT_CUDA(ei[0].create()); OT_CUDA(ei[1].create());
            OT_CUDA(cudaEventRecord(ei[0], s));
            ckpt_insert_kernel<<<(m + 255) / 256, 256, 0, s>>>(kept_keys.p, m, base, volume_hash(v));
            OT_LAUNCHED();
            OT_CUDA(cudaEventRecord(ei[1], s));
            const int pool = base + m;
            OT_CUDA(cudaMemcpyAsync(v->d_counters.p + kPoolCount, &pool, 4, cudaMemcpyHostToDevice, s));
            OT_CUDA(cudaStreamSynchronize(s));
            float ins_ms = 0.f;
            cudaEventElapsedTime(&ins_ms, ei[0], ei[1]);
            st.times(g_ckpt_prof[0], g_ckpt_prof[1]);
            g_ckpt_prof[0] += ins_ms;
            v->n_blocks = pool;
            ++v->epoch;
        }
    }
    if (v->n_objects > 0) v->obj_frames[v->sel_obj] = std::max<int64_t>(v->obj_frames[v->sel_obj], h.frames);
    else v->frames_integrated = std::max<int64_t>(v->frames_integrated, h.frames);
    if (n_loaded) *n_loaded = m;
    g_ckpt_prof[2] = file_ns.load() * 1e-6;
    g_ckpt_prof[3] = ms_since(t_start);
    return OTSLAM_OK;
}

}  // extern "C"
