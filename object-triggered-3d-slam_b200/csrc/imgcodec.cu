// imgcodec.cu -- capture files -> frames in HBM without the host touching a pixel (SURVEY 8f row 1, second half).
//
// The reference reads every frame pair with o3d.io.read_image (/root/reference/3d_model/reconstruct_rgbd.py:88-89): libjpeg
// and libpng on one CPU core, ~6 ms per pair -- 100x the GPU's integration time for the same frame.  Here a chunk of files is
// read by host threads (I/O only: chunk / marker walking, CRC), the COMPRESSED bytes cross PCIe (a 640x480 pair is ~130-400 KB
// instead of 1.5 MB raw), and the arithmetic of both decoders runs on the GPU:
//
//   depth PNG : png_inflate_kernel   one warp (lane 0) per file: RFC 1951 inflate, Huffman tables in shared memory
//               png_unfilter_kernel  one thread per band of scan lines (bands start at lines whose filter is None / Sub,
//                                    so they are independent; an all-Paeth file degenerates to one thread)
//               png_emit_kernel      one thread per pixel: big-endian samples -> u16 (RGB / RGBA PNG -> RGB8)
//   colour JPEG: jpeg_huff_kernel    one warp (lane 0) per file: the sequential entropy-coded scan -> int16 coefficients
//               jpeg_idct_kernel     8 lanes per 8x8 block: libjpeg's "islow" integer IDCT, column pass / row pass
//               jpeg_color_kernel    one thread per pixel: fancy chroma upsampling + YCbCr -> RGB
//
// A single file's entropy decoding is inherently sequential; the parallelism is across the files of a chunk (hundreds of
// independent bit streams, one per warp, latency-bound) -- which is the batch-of-frames shape the frame loop already has.
// All arithmetic lives in imgcodec_core.h as __host__ __device__ functions, checked bit for bit against OpenCV's
// libpng / libjpeg-turbo on the CPU (tests/test_imgcodec_model.py) and on the GPU (tests/test_gpu_zz_decode.py).
#include <fcntl.h>
#include <locale.h>
#include <sched.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "imgcodec_core.h"

using namespace otslam;
using namespace imgcodec;

namespace {

struct PngJob {
    PngFrame f;
    int64_t raw_off;              // the file's inflated scan lines inside d_raw
    int32_t slot, kind;           // kind 0 = depth (u16 out), 1 = colour (RGB8 out)
};

constexpr int kBandRows = 4;
constexpr int kMaxTableSets = 64;

// ---------------------------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------------------------
// One warp per file, all 32 lanes in lock step (imgcodec_core.h, "team"): every lane decodes the same symbols, the lanes
// share the copy of each match / stored block, lane 0 builds the Huffman tables in shared memory between two __syncwarp()s.
// (Round-2 first version: lane 0 alone, the match bytes copied one at a time through a store -> load dependency:
// 34.5 ms per 256 depth files of 640x480; the copy was 90 % of it.)
__global__ void __launch_bounds__(32) png_inflate_kernel(const PngJob* __restrict__ jobs, const uint8_t* __restrict__ blob,
                                                         uint8_t* __restrict__ raw, int32_t* __restrict__ status) {
    __shared__ InflateTables T;
    const PngJob j = jobs[blockIdx.x];
    if (j.f.status != IC_OK) return;
    const int64_t cap = (int64_t)(j.f.rowbytes + 1) * j.f.height;
    int64_t got = 0;
    // The tables are addressed through a generic pointer the compiler cannot see through: with the __shared__ object itself
    // it re-derived the shared-window base (S2R SR_CgaCtaId + LEA) for every symbol, 11 % of the kernel's stall samples.
    InflateTables* Tp = &T;
    asm volatile("" : "+l"(Tp));
    uint8_t* out = raw + j.raw_off;                               // likewise kept in registers instead of being re-derived from
    asm volatile("" : "+l"(out));                                 // the kernel parameters at every store
    int st = inflate_zlib(blob + j.f.z_off, j.f.z_len, out, cap, *Tp, &got, (int)threadIdx.x, 32);
    if (st == IC_OK && got != cap) st = IC_CORRUPT;              // libpng: "Not enough image data"
    if (threadIdx.x == 0) status[blockIdx.x] = st;
}

__global__ void __launch_bounds__(128) png_unfilter_kernel(const PngJob* __restrict__ jobs, uint8_t* __restrict__ raw,
                                                           int32_t* __restrict__ status) {
    const PngJob& j = jobs[blockIdx.y];
    if (j.f.status != IC_OK || status[blockIdx.y] != IC_OK) return;
    const int band = blockIdx.x * blockDim.x + threadIdx.x;
    const int H = j.f.height, stride = j.f.rowbytes + 1;
    if (band * kBandRows >= H) return;
    uint8_t* r = raw + j.raw_off;
    const int r0 = png_band_first(r, H, stride, band * kBandRows);
    if (r0 >= H) return;
    const int r1 = png_band_first(r, H, stride, (band + 1) * kBandRows);
    if (r0 >= r1) return;
    if (png_unfilter_band(r, H, j.f.rowbytes, j.f.bpp, r0, r1) != IC_OK) status[blockIdx.y] = IC_CORRUPT;
}

__global__ void __launch_bounds__(256) png_emit_kernel(const PngJob* __restrict__ jobs, const uint8_t* __restrict__ raw,
                                                       const int32_t* __restrict__ status, uint16_t* __restrict__ depth,
                                                       uint8_t* __restrict__ rgb) {
    const PngJob& j = jobs[blockIdx.y];
    if (j.f.status != IC_OK || status[blockIdx.y] != IC_OK) return;
    const int64_t px = (int64_t)j.f.width * j.f.height;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= px) return;
    const int y = (int)(i / j.f.width), x = (int)(i - (int64_t)y * j.f.width);
    uint8_t* out = j.kind == 0 ? reinterpret_cast<uint8_t*>(depth + (int64_t)j.slot * px) : rgb + (int64_t)j.slot * px * 3;
    png_emit_pixel(raw + j.raw_off, j.f, x, y, out);
}

// One warp per file; the scan is one sequential bit stream, so lane 0 decodes it (the other lanes help to stage the
// frame's Huffman tables in shared memory, then leave).
__global__ void __launch_bounds__(32) jpeg_huff_kernel(const JpegFrame* __restrict__ frames, const JpegTables* __restrict__ tables,
                                                       const uint8_t* __restrict__ blob, int16_t* __restrict__ coef,
                                                       int32_t* __restrict__ status) {
    __shared__ JpegFrame f;                                      // the per-component arrays are indexed at run time
    __shared__ JpegTables T;
    static_assert(sizeof(JpegTables) % 4 == 0 && sizeof(JpegFrame) % 4 == 0, "word copies");
    if (frames[blockIdx.x].status != IC_OK) return;
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(frames + blockIdx.x);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&f);
        for (int i = threadIdx.x; i < (int)(sizeof(JpegFrame) / 4); i += 32) dst[i] = src[i];
        src = reinterpret_cast<const uint32_t*>(tables + frames[blockIdx.x].tables);
        dst = reinterpret_cast<uint32_t*>(&T);
        for (int i = threadIdx.x; i < (int)(sizeof(JpegTables) / 4); i += 32) dst[i] = src[i];
    }
    __syncwarp();
    if (threadIdx.x != 0) return;
    status[blockIdx.x] = jpeg_decode_scan(f, T, blob + f.scan_off, coef + f.blk_off * 64);
}

// 256 threads = 32 blocks of 8x8 coefficients, 8 lanes per block: lane c runs column c (pass 1), then row c (pass 2)
__global__ void __launch_bounds__(256) jpeg_idct_kernel(const JpegFrame* __restrict__ frames, const JpegTables* __restrict__ tables,
                                                        const int16_t* __restrict__ coef, const int32_t* __restrict__ status,
                                                        uint8_t* __restrict__ samples) {
    __shared__ int32_t ws[32][8][9];
    const JpegFrame& f = frames[blockIdx.y];
    if (f.status != IC_OK || status[blockIdx.y] != IC_OK) return;
    const int lb = threadIdx.x >> 3, lane = threadIdx.x & 7;
    const int g = blockIdx.x * 32 + lb;
    const bool live = g < f.n_blocks;
    int c = 0;
    if (live) {
        c = g >= f.blk_base[2] ? 2 : (g >= f.blk_base[1] ? 1 : 0);
        int32_t col[8];
        idct_column(coef + (f.blk_off + g) * 64, tables[f.tables].q[f.tq[c]], lane, col);
#pragma unroll
        for (int r = 0; r < 8; ++r) ws[lb][lane][r] = col[r];
    }
    __syncthreads();
    if (!live) return;
    int32_t row[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) row[k] = ws[lb][k][lane];
    uint8_t o[8];
    idct_row(row, o);
    const int local = g - f.blk_base[c];
    const int by = local / f.wblk[c], bx = local - by * f.wblk[c];
    uint8_t* plane = samples + (f.blk_off + f.blk_base[c]) * 64;
    uint2 v;
    v.x = (uint32_t)o[0] | ((uint32_t)o[1] << 8) | ((uint32_t)o[2] << 16) | ((uint32_t)o[3] << 24);
    v.y = (uint32_t)o[4] | ((uint32_t)o[5] << 8) | ((uint32_t)o[6] << 16) | ((uint32_t)o[7] << 24);
    *reinterpret_cast<uint2*>(plane + ((int64_t)(by * 8 + lane) * f.wblk[c] + bx) * 8) = v;
}

__global__ void __launch_bounds__(256) jpeg_color_kernel(const JpegFrame* __restrict__ frames, const int32_t* __restrict__ status,
                                                         const uint8_t* __restrict__ samples, const int32_t* __restrict__ slots,
                                                         uint8_t* __restrict__ rgb) {
    const JpegFrame& f = frames[blockIdx.y];
    if (f.status != IC_OK || status[blockIdx.y] != IC_OK) return;
    const int64_t px = (int64_t)f.width * f.height;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= px) return;
    const int y = (int)(i / f.width), x = (int)(i - (int64_t)y * f.width);
    JpegPlanes P;
    const uint8_t* base = samples + f.blk_off * 64;
    P.y = base + (int64_t)f.blk_base[0] * 64;
    P.cb = base + (int64_t)f.blk_base[1] * 64;
    P.cr = base + (int64_t)f.blk_base[2] * 64;
    P.ys = f.wblk[0] * 8;
    P.cs = f.wblk[1] * 8;
    P.hmax = f.hmax;
    P.vmax = f.vmax;
    P.cw = (f.width + f.hmax - 1) / f.hmax;
    P.ch = (f.height + f.vmax - 1) / f.vmax;
    uint8_t c[3];
    jpeg_pixel_rgb(P, x, y, c);
    uint8_t* o = rgb + ((int64_t)slots[blockIdx.y] * px + i) * 3;
    o[0] = c[0];
    o[1] = c[1];
    o[2] = c[2];
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
// decoder buffers grow with head room (pinned n / 2, device n / 4) unless the call site asks for more
template <typename T>
cudaError_t grow(PinnedArray<T>& a, size_t n, size_t want = 0) { return a.reserve(n, std::max(want, n + n / 2)); }
template <typename T>
cudaError_t grow(DeviceArray<T>& a, size_t n, size_t want = 0) { return a.reserve(n, std::max(want, n + n / 4)); }

int host_threads() {
    const char* e = getenv("OTSLAM_DECODE_THREADS");
    int n = e ? atoi(e) : 0;
    if (n <= 0) {
        cpu_set_t set;
        n = (sched_getaffinity(0, sizeof(set), &set) == 0) ? CPU_COUNT(&set) : (int)std::thread::hardware_concurrency();
        n = std::min(n, 32);
    }
    return std::max(1, std::min(n, 64));
}

template <typename F>
void parallel_for(int n, F&& body) {
    const int nt = std::min(host_threads(), n);
    if (nt <= 1) {
        for (int i = 0; i < n; ++i) body(i);
        return;
    }
    std::atomic<int> next{0};
    std::vector<std::thread> pool;
    pool.reserve(nt);
    for (int t = 0; t < nt; ++t)
        pool.emplace_back([&] {
            for (int i; (i = next.fetch_add(1, std::memory_order_relaxed)) < n;) body(i);
        });
    for (auto& th : pool) th.join();
}

bool read_file(const char* path, std::vector<uint8_t>& out) {
    out.clear();
    if (!path) return false;
    const int fd = open(path, O_RDONLY | O_CLOEXEC);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) { close(fd); return false; }
    out.resize((size_t)st.st_size);
    size_t got = 0;
    while (got < out.size()) {
        const ssize_t r = read(fd, out.data() + got, out.size() - got);
        if (r <= 0) break;
        got += (size_t)r;
    }
    close(fd);
    if (got != out.size()) { out.clear(); return false; }
    return true;
}

}  // namespace

struct otslam_decoder {
    int device = 0, H = 0, W = 0, max_frames = 0;
    Stream s_png, s_jpg;
    Event ev[8];
    PinnedArray<uint8_t> h_zblob, h_jblob;
    DeviceArray<uint8_t> d_zblob, d_jblob, d_raw, d_samples, d_rgb;
    DeviceArray<uint16_t> d_depth;
    DeviceArray<int16_t> d_coef;
    PinnedArray<PngJob> h_jobs;
    DeviceArray<PngJob> d_jobs;
    PinnedArray<JpegFrame> h_frames;
    DeviceArray<JpegFrame> d_frames;
    PinnedArray<JpegTables> h_tables;
    DeviceArray<JpegTables> d_tables;
    PinnedArray<int32_t> h_status, h_slots;
    DeviceArray<int32_t> d_status, d_slots;
    int n_decoded = 0;
    double ms[6] = {};
};

namespace {

struct Source {                   // one compressed file in memory
    const uint8_t* p = nullptr;
    int64_t n = 0;
};

// The batch decoder behind both entry points.  color / depth: n sources each (p == nullptr: missing file), or null.
int decode_sources(otslam_decoder* d, int n, const Source* color, const Source* depth, int32_t* color_status, int32_t* depth_status) {
    static const Crc32 crc;
    const int H = d->H, W = d->W;
    const int64_t px = (int64_t)H * W;
    OT_TRY(use_device(d->device));
    d->n_decoded = 0;
    for (double& m : d->ms) m = 0.0;
    if (color_status) std::fill(color_status, color_status + n, (int32_t)IC_UNSUPPORTED);
    if (depth_status) std::fill(depth_status, depth_status + n, (int32_t)IC_UNSUPPORTED);
    if (n == 0) return OTSLAM_OK;

    // ---- classify, size the staging areas (every file's compressed payload is no larger than the file)
    std::vector<int64_t> zoff, joff;
    std::vector<int> png_src;     // job -> frame index * 2 + kind
    std::vector<int> jpg_src;     // jpeg frame -> frame index
    int64_t ztotal = 0, jtotal = 0;
    auto is_png = [](const Source& s) { return s.p && s.n >= 8 && s.p[0] == 0x89 && s.p[1] == 'P'; };
    auto is_jpg = [](const Source& s) { return s.p && s.n >= 4 && s.p[0] == 0xFF && s.p[1] == 0xD8; };
    for (int i = 0; i < n; ++i) {
        if (depth) {
            if (is_png(depth[i])) { png_src.push_back(i * 2); zoff.push_back(ztotal); ztotal += (depth[i].n + 15) & ~15ll; }
            else if (depth_status) depth_status[i] = depth[i].p ? IC_UNSUPPORTED : IC_CORRUPT;
        }
        if (color) {
            if (is_png(color[i])) { png_src.push_back(i * 2 + 1); zoff.push_back(ztotal); ztotal += (color[i].n + 15) & ~15ll; }
            else if (is_jpg(color[i])) { jpg_src.push_back(i); joff.push_back(jtotal); jtotal += (color[i].n + 15 + 8) & ~15ll; }
            else if (color_status) color_status[i] = color[i].p ? IC_UNSUPPORTED : IC_CORRUPT;
        }
    }
    const int n_png = (int)png_src.size(), n_jpg = (int)jpg_src.size();
    const size_t cap_jobs = (size_t)d->max_frames * 2;           // data-independent sizes: see the device buffers below
    OT_CUDA(grow(d->h_zblob, (size_t)ztotal + 16, (size_t)ztotal * 2 + 16));
    OT_CUDA(grow(d->h_jblob, (size_t)jtotal + 16, (size_t)jtotal * 2 + 16));
    OT_CUDA(grow(d->h_jobs, std::max(1, n_png), cap_jobs));
    OT_CUDA(grow(d->h_frames, std::max(1, n_jpg), (size_t)d->max_frames));
    OT_CUDA(grow(d->h_tables, kMaxTableSets));
    OT_CUDA(grow(d->h_status, (size_t)std::max(1, n_png + n_jpg), cap_jobs));
    OT_CUDA(grow(d->h_slots, (size_t)std::max(1, n_jpg), (size_t)d->max_frames));

    // ---- parse in parallel: PNG chunk walk + CRC + IDAT compaction; JPEG marker walk + scan copy
    std::vector<JpegHeader> jhdr((size_t)n_jpg);
    parallel_for(n_png + n_jpg, [&](int k) {
        if (k < n_png) {
            const int i = png_src[k] >> 1, kind = png_src[k] & 1;
            const Source& s = kind ? color[i] : depth[i];
            PngJob& j = d->h_jobs.p[k];
            png_parse(s.p, s.n, H, W, d->h_zblob.p + zoff[k], (s.n + 15) & ~15ll, &crc, j.f);
            j.f.z_off = zoff[k];
            j.slot = i;
            j.kind = kind;
            j.raw_off = 0;
            if (j.f.status == IC_OK && ((kind == 0) != (j.f.channels == 1))) j.f.status = IC_UNSUPPORTED;   // grey colour / RGB depth
        } else {
            const int q = k - n_png, i = jpg_src[q];
            JpegFrame& f = d->h_frames.p[q];
            jpeg_parse(color[i].p, color[i].n, H, W, f, jhdr[q]);
            if (f.status == IC_OK) {
                memcpy(d->h_jblob.p + joff[q], color[i].p + f.scan_off, (size_t)f.scan_len);
                memset(d->h_jblob.p + joff[q] + f.scan_len, 0, 8);
                f.scan_off = joff[q];
            }
            d->h_slots.p[q] = i;
        }
    });

    // ---- lay out the device buffers; de-duplicate the JPEG table sets
    int64_t raw_total = 0;
    for (int k = 0; k < n_png; ++k) {
        PngJob& j = d->h_jobs.p[k];
        if (j.f.status != IC_OK) continue;
        j.raw_off = raw_total;
        raw_total += (((int64_t)(j.f.rowbytes + 1) * j.f.height) + 15) & ~15ll;
    }
    int64_t blk_total = 0;
    int n_sets = 0;
    std::map<std::string, int> sets;
    for (int q = 0; q < n_jpg; ++q) {
        JpegFrame& f = d->h_frames.p[q];
        if (f.status != IC_OK) continue;
        const JpegHeader& hd = jhdr[q];
        std::string key;
        for (int c = 0; c < 3; ++c) {                              // only the tables the scan uses
            key.append(reinterpret_cast<const char*>(hd.q[f.tq[c]]), 64);
            const int sl[2] = {f.td[c], 2 + f.ta[c]};
            for (int s : sl) {
                key.append(reinterpret_cast<const char*>(hd.hbits[s]), 16);
                key.append(reinterpret_cast<const char*>(hd.hvals[s]), (size_t)hd.hn[s]);
            }
            key.push_back((char)f.tq[c]); key.push_back((char)f.td[c]); key.push_back((char)f.ta[c]);
        }
        auto it = sets.find(key);
        if (it == sets.end()) {
            if (n_sets == kMaxTableSets) { f.status = IC_UNSUPPORTED; continue; }
            JpegTables& T = d->h_tables.p[n_sets];
            memset(&T, 0, sizeof(T));
            bool ok = true;
            for (int s = 0; s < 4; ++s)
                if (hd.h_set[s]) ok = jpeg_build_huff(hd.hbits[s], hd.hvals[s], hd.hn[s], s < 2, T.h[s]) && ok;
            for (int t = 0; t < 4; ++t)
                for (int k = 0; k < 64; ++k) T.q[t][k] = hd.q[t][k];
            if (!ok) { f.status = IC_CORRUPT; continue; }           // libjpeg: "Bogus Huffman table definition"
            for (int a = 0; a < 2; ++a)
                if (hd.h_set[2 + a]) jpeg_build_acfast(T.h[2 + a], T.acfast[a]);
            it = sets.emplace(std::move(key), n_sets++).first;
        }
        f.tables = it->second;
        f.blk_off = blk_total;
        blk_total += f.n_blocks;
    }

    // Device buffers are sized by bounds that do not depend on the data -- (decoder's frame capacity) x (largest per-frame need
    // seen) -- and the two compressed-byte areas (host and device) with 2x head room: a decoder that served a chunk of small
    // files in one pass and a chunk of large ones in the next must not reallocate, because cudaFree / cudaFreeHost wait for
    // every kernel on the device, including the other decoders' long-running entropy kernels.
    int64_t raw_frame = 0, blk_frame = 0;
    for (int k = 0; k < n_png; ++k)
        if (d->h_jobs.p[k].f.status == IC_OK)
            raw_frame = std::max<int64_t>(raw_frame, (((int64_t)(d->h_jobs.p[k].f.rowbytes + 1) * d->h_jobs.p[k].f.height) + 15) & ~15ll);
    for (int q = 0; q < n_jpg; ++q)
        if (d->h_frames.p[q].status == IC_OK) blk_frame = std::max<int64_t>(blk_frame, d->h_frames.p[q].n_blocks);
    const size_t cap_frames = (size_t)d->max_frames * ((depth ? 1 : 0) + (color ? 1 : 0));      // >= n_png, >= n_jpg
    OT_CUDA(grow(d->d_zblob, (size_t)ztotal + 16, (size_t)ztotal * 2 + 16));
    OT_CUDA(grow(d->d_jblob, (size_t)jtotal + 16, (size_t)jtotal * 2 + 16));
    OT_CUDA(grow(d->d_raw, (size_t)raw_total + 16, cap_frames * (size_t)raw_frame + 16));
    OT_CUDA(grow(d->d_coef, (size_t)blk_total * 64 + 64, (size_t)d->max_frames * (size_t)blk_frame * 64 + 64));
    OT_CUDA(grow(d->d_samples, (size_t)blk_total * 64 + 64, (size_t)d->max_frames * (size_t)blk_frame * 64 + 64));
    OT_CUDA(grow(d->d_jobs, std::max(1, n_png), cap_frames));
    OT_CUDA(grow(d->d_frames, std::max(1, n_jpg), (size_t)d->max_frames));
    OT_CUDA(grow(d->d_tables, kMaxTableSets));
    OT_CUDA(grow(d->d_status, (size_t)std::max(1, n_png + n_jpg), cap_frames));
    OT_CUDA(grow(d->d_slots, (size_t)std::max(1, n_jpg), (size_t)d->max_frames));
    if (depth) OT_CUDA(grow(d->d_depth, (size_t)d->max_frames * px));
    if (color) OT_CUDA(grow(d->d_rgb, (size_t)d->max_frames * px * 3));

    // ---- PNG stream
    cudaStream_t sp = d->s_png, sj = d->s_jpg;
    if (n_png) {
        OT_CUDA(cudaMemcpyAsync(d->d_zblob.p, d->h_zblob.p, (size_t)ztotal, cudaMemcpyHostToDevice, sp));
        OT_CUDA(cudaMemcpyAsync(d->d_jobs.p, d->h_jobs.p, sizeof(PngJob) * n_png, cudaMemcpyHostToDevice, sp));
        OT_CUDA(cudaMemsetAsync(d->d_status.p, 0, sizeof(int32_t) * n_png, sp));
        OT_CUDA(cudaEventRecord(d->ev[0], sp));
        png_inflate_kernel<<<n_png, 32, 0, sp>>>(d->d_jobs.p, d->d_zblob.p, d->d_raw.p, d->d_status.p);
        OT_LAUNCHED();
        OT_CUDA(cudaEventRecord(d->ev[1], sp));
        const int bands = (H + kBandRows - 1) / kBandRows;
        png_unfilter_kernel<<<dim3((bands + 127) / 128, n_png), 128, 0, sp>>>(d->d_jobs.p, d->d_raw.p, d->d_status.p);
        OT_LAUNCHED();
        png_emit_kernel<<<dim3((unsigned)((px + 255) / 256), n_png), 256, 0, sp>>>(d->d_jobs.p, d->d_raw.p, d->d_status.p,
                                                                                   d->d_depth.p, d->d_rgb.p);
        OT_LAUNCHED();
        OT_CUDA(cudaEventRecord(d->ev[2], sp));
        OT_CUDA(cudaMemcpyAsync(d->h_status.p, d->d_status.p, sizeof(int32_t) * n_png, cudaMemcpyDeviceToHost, sp));
    }
    // ---- JPEG stream (runs beside the PNG stream: both are latency-bound single-lane decoders)
    if (n_jpg) {
        int32_t* st = d->d_status.p + n_png;
        OT_CUDA(cudaMemcpyAsync(d->d_jblob.p, d->h_jblob.p, (size_t)jtotal, cudaMemcpyHostToDevice, sj));
        OT_CUDA(cudaMemcpyAsync(d->d_frames.p, d->h_frames.p, sizeof(JpegFrame) * n_jpg, cudaMemcpyHostToDevice, sj));
        OT_CUDA(cudaMemcpyAsync(d->d_slots.p, d->h_slots.p, sizeof(int32_t) * n_jpg, cudaMemcpyHostToDevice, sj));
        if (n_sets) OT_CUDA(cudaMemcpyAsync(d->d_tables.p, d->h_tables.p, sizeof(JpegTables) * n_sets, cudaMemcpyHostToDevice, sj));
        OT_CUDA(cudaMemsetAsync(st, 0, sizeof(int32_t) * n_jpg, sj));
        OT_CUDA(cudaMemsetAsync(d->d_coef.p, 0, (size_t)blk_total * 128, sj));
        int max_blocks = 0;
        for (int q = 0; q < n_jpg; ++q)
            if (d->h_frames.p[q].status == IC_OK) max_blocks = std::max(max_blocks, d->h_frames.p[q].n_blocks);
        OT_CUDA(cudaEventRecord(d->ev[3], sj));
        if (max_blocks) {
            jpeg_huff_kernel<<<n_jpg, 32, 0, sj>>>(d->d_frames.p, d->d_tables.p, d->d_jblob.p, d->d_coef.p, st);
            OT_LAUNCHED();
            OT_CUDA(cudaEventRecord(d->ev[4], sj));
            jpeg_idct_kernel<<<dim3((max_blocks + 31) / 32, n_jpg), 256, 0, sj>>>(d->d_frames.p, d->d_tables.p, d->d_coef.p, st,
                                                                                  d->d_samples.p);
            OT_LAUNCHED();
            OT_CUDA(cudaEventRecord(d->ev[5], sj));
            jpeg_color_kernel<<<dim3((unsigned)((px + 255) / 256), n_jpg), 256, 0, sj>>>(d->d_frames.p, st, d->d_samples.p,
                                                                                         d->d_slots.p, d->d_rgb.p);
            OT_LAUNCHED();
        } else {
            OT_CUDA(cudaEventRecord(d->ev[4], sj));
            OT_CUDA(cudaEventRecord(d->ev[5], sj));
        }
        OT_CUDA(cudaEventRecord(d->ev[6], sj));
        OT_CUDA(cudaMemcpyAsync(d->h_status.p + n_png, st, sizeof(int32_t) * n_jpg, cudaMemcpyDeviceToHost, sj));
    }
    OT_CUDA(cudaStreamSynchronize(sp));
    OT_CUDA(cudaStreamSynchronize(sj));

    // ---- statuses back to frame order
    for (int k = 0; k < n_png; ++k) {
        const PngJob& j = d->h_jobs.p[k];
        int32_t* dst = j.kind ? color_status : depth_status;
        if (dst) dst[j.slot] = j.f.status != IC_OK ? j.f.status : d->h_status.p[k];
    }
    for (int q = 0; q < n_jpg; ++q)
        if (color_status) color_status[d->h_slots.p[q]] = d->h_frames.p[q].status != IC_OK ? d->h_frames.p[q].status : d->h_status.p[n_png + q];
    float t = 0.f;
    if (n_png) {
        if (cudaEventElapsedTime(&t, d->ev[0], d->ev[1]) == cudaSuccess) d->ms[0] = t;
        if (cudaEventElapsedTime(&t, d->ev[1], d->ev[2]) == cudaSuccess) d->ms[1] = t;
    }
    if (n_jpg) {
        if (cudaEventElapsedTime(&t, d->ev[3], d->ev[4]) == cudaSuccess) d->ms[2] = t;
        if (cudaEventElapsedTime(&t, d->ev[4], d->ev[5]) == cudaSuccess) d->ms[3] = t;
        if (cudaEventElapsedTime(&t, d->ev[5], d->ev[6]) == cudaSuccess) d->ms[4] = t;
    }
    d->ms[5] = (double)(ztotal + jtotal);
    d->n_decoded = n;
    return OTSLAM_OK;
}

}  // namespace

extern "C" {

int otslam_decoder_create(int device, int height, int width, int max_frames, otslam_decoder** out) {
    // (2 x max_frames is a grid dimension of the per-pixel kernels; an image's scan lines must stay below 2^31 bytes)
    if (!out || height <= 0 || width <= 0 || max_frames <= 0 || max_frames > 16384 || (int64_t)height * width > (1ll << 28))
        return set_error(OTSLAM_ERR_INVALID, "decoder_create: bad arguments (max_frames <= 16384, height x width <= 2^28)");
    *out = nullptr;
    OT_TRY(use_device(device));
    std::unique_ptr<otslam_decoder> d(new otslam_decoder());
    d->device = device;
    d->H = height;
    d->W = width;
    d->max_frames = max_frames;
    OT_CUDA(d->s_png.create(cudaStreamNonBlocking));
    OT_CUDA(d->s_jpg.create(cudaStreamNonBlocking));
    for (auto& ev : d->ev) OT_CUDA(ev.create());
    *out = d.release();
    return OTSLAM_OK;
}

int otslam_decoder_destroy(otslam_decoder* d) {
    if (!d) return OTSLAM_OK;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    delete d;
    return OTSLAM_OK;
}

int otslam_decoder_decode(otslam_decoder* d, int n, const uint8_t* color_blob, const int64_t* color_offsets, const uint8_t* depth_blob,
                          const int64_t* depth_offsets, int32_t* color_status, int32_t* depth_status) {
    if (!d || n < 0 || n > d->max_frames || (color_blob && !color_offsets) || (depth_blob && !depth_offsets))
        return set_error(OTSLAM_ERR_INVALID, "decoder_decode: bad arguments");
    std::vector<Source> cs, ds;
    if (color_blob) {
        cs.resize((size_t)n);
        for (int i = 0; i < n; ++i) {
            const int64_t len = color_offsets[i + 1] - color_offsets[i];
            if (len < 0) return set_error(OTSLAM_ERR_INVALID, "decoder_decode: offsets must not decrease");
            if (len > 0) cs[i] = Source{color_blob + color_offsets[i], len};
        }
    }
    if (depth_blob) {
        ds.resize((size_t)n);
        for (int i = 0; i < n; ++i) {
            const int64_t len = depth_offsets[i + 1] - depth_offsets[i];
            if (len < 0) return set_error(OTSLAM_ERR_INVALID, "decoder_decode: offsets must not decrease");
            if (len > 0) ds[i] = Source{depth_blob + depth_offsets[i], len};
        }
    }
    return decode_sources(d, n, color_blob ? cs.data() : nullptr, depth_blob ? ds.data() : nullptr, color_status, depth_status);
}

int otslam_decoder_decode_files(otslam_decoder* d, int n, const char* const* color_paths, const char* const* depth_paths,
                                int32_t* color_status, int32_t* depth_status) {
    if (!d || n < 0 || n > d->max_frames) return set_error(OTSLAM_ERR_INVALID, "decoder_decode_files: bad arguments");
    std::vector<std::vector<uint8_t>> cf(color_paths ? (size_t)n : 0), df(depth_paths ? (size_t)n : 0);
    parallel_for(n * 2, [&](int k) {
        const int i = k >> 1;
        if (k & 1) { if (color_paths) read_file(color_paths[i], cf[i]); }
        else if (depth_paths) read_file(depth_paths[i], df[i]);
    });
    std::vector<Source> cs(cf.size()), ds(df.size());
    for (size_t i = 0; i < cf.size(); ++i)
        if (!cf[i].empty()) cs[i] = Source{cf[i].data(), (int64_t)cf[i].size()};
    for (size_t i = 0; i < df.size(); ++i)
        if (!df[i].empty()) ds[i] = Source{df[i].data(), (int64_t)df[i].size()};
    return decode_sources(d, n, color_paths ? cs.data() : nullptr, depth_paths ? ds.data() : nullptr, color_status, depth_status);
}

int otslam_decoder_put(otslam_decoder* d, int slot, const uint16_t* depth, const uint8_t* rgb) {
    if (!d || slot < 0 || slot >= d->max_frames) return set_error(OTSLAM_ERR_INVALID, "decoder_put: bad slot");
    OT_TRY(use_device(d->device));
    const size_t px = (size_t)d->H * d->W;
    if (depth) {
        OT_CUDA(grow(d->d_depth, (size_t)d->max_frames * px));
        OT_CUDA(cudaMemcpy(d->d_depth.p + (size_t)slot * px, depth, px * 2, cudaMemcpyDefault));
    }
    if (rgb) {
        OT_CUDA(grow(d->d_rgb, (size_t)d->max_frames * px * 3));
        OT_CUDA(cudaMemcpy(d->d_rgb.p + (size_t)slot * px * 3, rgb, px * 3, cudaMemcpyDefault));
    }
    return OTSLAM_OK;
}

int otslam_decoder_fetch(otslam_decoder* d, int first, int count, uint16_t* depth, uint8_t* rgb) {
    if (!d || first < 0 || count < 0 || first + count > d->max_frames) return set_error(OTSLAM_ERR_INVALID, "decoder_fetch: bad range");
    OT_TRY(use_device(d->device));
    const size_t px = (size_t)d->H * d->W;
    if (depth) {
        if (!d->d_depth.p) return set_error(OTSLAM_ERR_INVALID, "decoder_fetch: no depth decoded");
        OT_CUDA(cudaMemcpy(depth, d->d_depth.p + (size_t)first * px, (size_t)count * px * 2, cudaMemcpyDefault));
    }
    if (rgb) {
        if (!d->d_rgb.p) return set_error(OTSLAM_ERR_INVALID, "decoder_fetch: no colour decoded");
        OT_CUDA(cudaMemcpy(rgb, d->d_rgb.p + (size_t)first * px * 3, (size_t)count * px * 3, cudaMemcpyDefault));
    }
    return OTSLAM_OK;
}

int otslam_decoder_integrate(otslam_decoder* d, otslam_volume* v, int n_keep, const int32_t* slots, const double intr[4],
                             const double* extrinsics, double depth_scale, double depth_trunc, const int32_t* object_ids) {
    if (!d || !v || n_keep < 0 || n_keep > d->max_frames || (n_keep && !slots))
        return set_error(OTSLAM_ERR_INVALID, "decoder_integrate: bad arguments");
    if (n_keep == 0) return OTSLAM_OK;
    OT_TRY(use_device(d->device));
    if (!d->d_depth.p) return set_error(OTSLAM_ERR_INVALID, "decoder_integrate: nothing decoded");
    const size_t px = (size_t)d->H * d->W;
    for (int i = 0; i < n_keep; ++i)
        if (slots[i] < i || slots[i] >= d->max_frames || (i && slots[i] <= slots[i - 1]))
            return set_error(OTSLAM_ERR_INVALID, "decoder_integrate: slots must ascend");
    // close the holes skipped frames left (moves whole frames downwards: source and destination never overlap)
    cudaStream_t s = d->s_png;
    for (int i = 0; i < n_keep; ++i) {
        if (slots[i] == i) continue;
        OT_CUDA(cudaMemcpyAsync(d->d_depth.p + (size_t)i * px, d->d_depth.p + (size_t)slots[i] * px, px * 2, cudaMemcpyDeviceToDevice, s));
        if (d->d_rgb.p)
            OT_CUDA(cudaMemcpyAsync(d->d_rgb.p + (size_t)i * px * 3, d->d_rgb.p + (size_t)slots[i] * px * 3, px * 3, cudaMemcpyDeviceToDevice, s));
    }
    OT_CUDA(cudaStreamSynchronize(s));
    if (object_ids)
        return otslam_volume_integrate_batch_objects(v, n_keep, d->d_depth.p, d->d_rgb.p, d->W, d->H, intr, extrinsics, object_ids,
                                                     depth_scale, depth_trunc, OTSLAM_MEM_DEVICE);
    return otslam_volume_integrate_batch(v, n_keep, d->d_depth.p, d->d_rgb.p, d->W, d->H, intr, extrinsics, depth_scale, depth_trunc,
                                         OTSLAM_MEM_DEVICE);
}

// np.loadtxt(pose_path) for the 4x4 text files of a capture tree.  Accepts exactly what the Python fast path accepts
// (pipeline.read_pose: 16 whitespace-separated plain decimal numbers, no comments, no commas) and converts with the C-locale
// strtod, which -- like Python's float() -- is correctly rounded, so the doubles are the same bits; everything else is left
// to np.loadtxt (status 1).  Host threads, no GPU involved: 16 interpreter threads parsing poses contended for the GIL and
// took 160 us per file, six times the single-threaded cost.
int otslam_read_pose_files(int n, const char* const* paths, double* poses, int32_t* status) {
    if (n < 0 || (n && (!paths || !poses || !status))) return set_error(OTSLAM_ERR_INVALID, "read_pose_files: bad arguments");
    static locale_t c_locale = newlocale(LC_ALL_MASK, "C", (locale_t)0);
    parallel_for(n, [&](int i) {
        status[i] = 2;
        for (int k = 0; k < 16; ++k) poses[(size_t)i * 16 + k] = 0.0;
        std::vector<uint8_t> buf;
        if (!read_file(paths[i], buf)) return;
        status[i] = 1;
        if (buf.size() > 16384) return;
        buf.push_back(0);
        const char* p = reinterpret_cast<const char*>(buf.data());
        const char* end = p + buf.size() - 1;
        double v[16];
        int cnt = 0;
        while (p < end) {
            const unsigned char c = (unsigned char)*p;
            if (c == ' ' || (c >= 9 && c <= 13)) { ++p; continue; }
            if (cnt == 16) return;                                           // a 17th token
            // [+-]? ( digits [. digits*] | . digits ) ( [eE] [+-]? digits )?
            const char* q = p;
            if (*q == '+' || *q == '-') ++q;
            int nd = 0;
            while (*q >= '0' && *q <= '9') { ++q; ++nd; }
            if (*q == '.') {
                ++q;
                while (*q >= '0' && *q <= '9') { ++q; ++nd; }
            }
            if (nd == 0) return;
            if (*q == 'e' || *q == 'E') {
                ++q;
                if (*q == '+' || *q == '-') ++q;
                int ne = 0;
                while (*q >= '0' && *q <= '9') { ++q; ++ne; }
                if (ne == 0) return;
            }
            const unsigned char t = (unsigned char)*q;
            if (!(q == end || t == ' ' || (t >= 9 && t <= 13))) return;      // anything else glued to the number (or a NUL inside the file)
            if (q - p > 1024) return;
            char* stop = nullptr;
            v[cnt] = c_locale ? strtod_l(p, &stop, c_locale) : strtod(p, &stop);
            if (stop != q) return;
            ++cnt;
            p = q;
        }
        if (cnt != 16) return;
        for (int k = 0; k < 16; ++k) poses[(size_t)i * 16 + k] = v[k];
        status[i] = 0;
    });
    return OTSLAM_OK;
}

int otslam_decoder_profile(otslam_decoder* d, double out_ms[6]) {
    if (!d || !out_ms) return set_error(OTSLAM_ERR_INVALID, "decoder_profile: null argument");
    for (int i = 0; i < 6; ++i) out_ms[i] = d->ms[i];
    return OTSLAM_OK;
}

}  // extern "C"
