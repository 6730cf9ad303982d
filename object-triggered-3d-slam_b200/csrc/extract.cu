// extract.cu -- surface extraction from the block-hashed TSDF volume on sm_100a.
//
// Replaces volume.extract_triangle_mesh() + mesh.compute_vertex_normals()
// (/root/reference/3d_model/reconstruct_rgbd.py:112-113; SURVEY A.5, A.9) and
// volume.extract_point_cloud() (north_star; SURVEY A.6).
//
// Marching cubes without a global edge->vertex hash map: every lattice edge is owned by the voxel
// at its lower end, so "vertex exists" is one bit per (voxel, axis).
//   mc_classify   per owned block: 17^3 tsdf tile in SMEM (neighbour planes through the block hash),
//                 cube index per voxel, triangle count, atomicOr of the used edge bits (possibly in
//                 the +x/+y/+z neighbour block, which exists whenever the cube is valid)
//   mc_count      per block: popcount of its edge bits -> vertex count + per-word prefix
//   scan          exclusive scans over blocks in sorted-key order (deterministic output order)
//   mc_vertices   per block: one vertex per set bit, FP64 arithmetic in the reference's order
//   mc_faces      per owned block: triangles, vertex ids by bit rank, winding swapped as in A.5
//   normals       area-weighted face normals accumulated per vertex, normalised
#include <algorithm>
#include <vector>

#include "cta_ops.cuh"
#include "volume_lookup.cuh"

#define MC_TABLE_QUAL static const
#include "mc_tables.h"

namespace otslam {

__device__ unsigned short d_edge_table[256];
__device__ signed char d_tri_table[256][16];
__device__ unsigned char d_ntri[256];
__device__ signed char d_edge_shift[12][4];

static int upload_tables() {
    static bool done[64] = {false};
    int dev = 0;
    OT_CUDA(cudaGetDevice(&dev));
    if (dev < 64 && done[dev]) return OTSLAM_OK;
    unsigned char ntri[256];
    for (int c = 0; c < 256; ++c) {
        int n = 0;
        while (n < 16 && MC_TRI_TABLE[c][n] != -1) ++n;
        ntri[c] = (unsigned char)(n / 3);
    }
    OT_CUDA(cudaMemcpyToSymbol(d_edge_table, MC_EDGE_TABLE, sizeof(MC_EDGE_TABLE)));
    OT_CUDA(cudaMemcpyToSymbol(d_tri_table, MC_TRI_TABLE, sizeof(MC_TRI_TABLE)));
    OT_CUDA(cudaMemcpyToSymbol(d_ntri, ntri, sizeof(ntri)));
    OT_CUDA(cudaMemcpyToSymbol(d_edge_shift, MC_EDGE_SHIFT, sizeof(MC_EDGE_SHIFT)));
    if (dev < 64) done[dev] = true;
    return OTSLAM_OK;
}

// neighbour table of a block: index = dx | dy<<1 | dz<<2
__device__ __forceinline__ void load_neighbours(const ExtractCtx& c, uint64_t key, int slot, int* nslot) {
    if (threadIdx.x < 8) {
        const int j = threadIdx.x;
        int kx, ky, kz;
        unpack_key(key, kx, ky, kz);                               // stored x: the arena offset included
        int s = slot;
        if (j) s = block_slot(c, kx - c.x_off + (j & 1), ky + ((j >> 1) & 1), kz + ((j >> 2) & 1));
        nslot[j] = s;
    }
}

constexpr int kFlagWords = 3 * (kVox / 32);   // 384 words: [axis][voxel bit], voxel bit = x*256+y*16+z

__global__ void __launch_bounds__(256) mc_classify_kernel(ExtractCtx c, uint32_t* flags, uint8_t* cube_idx, int* tri_count) {
    __shared__ float tile[17 * 17 * 17];
    __shared__ uint32_t s_flags[kFlagWords];      // edge bits of THIS block, merged into the global words once at the end
    __shared__ int nslot[8];
    __shared__ int s_tris;
    const int i = blockIdx.x;
    const int t = threadIdx.x;
    for (int w = t; w < kFlagWords; w += 256) s_flags[w] = 0;
    const uint64_t key = c.bkeys[i];
    const int slot = c.bslots[i];
    int kx, ky, kz;
    unpack_key(key, kx, ky, kz);
    if (!slab_owns(c.slab, kx, ky, kz)) {   // halo block: provides voxels, emits nothing
        if (t == 0) tri_count[i] = 0;
        return;
    }
    if (t == 0) s_tris = 0;
    load_neighbours(c, key, slot, nslot);
    __syncthreads();
    const float qnan = __int_as_float(0x7fc00000);       // NaN == unobserved (weight 0) or block missing
    auto tsdf_or_nan = [&](const uint4& r) { return rec_weight(r) != 0 ? __uint_as_float(r.x) : qnan; };
    // (1) the block itself, in MEMORY order (record index z*256 + x*16 + y): a warp reads 32 consecutive 16-byte
    //     records = 512 contiguous bytes per request, 8 requests of a thread in flight before the first use.
    //     (Round 1 walked the 17^3 tile in tile order, i.e. one record per 4 KiB stride per lane: 32 sectors per request,
    //     long-scoreboard 14.9 warps per issue slot, 339 us for 5844 blocks.)
    {
        const uint4* blk = block_ptr(c.chunks, slot);
#pragma unroll
        for (int h = 0; h < 16; h += 8) {
            uint4 r[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) r[k] = __ldg(blk + (h + k) * 256 + t);
#pragma unroll
            for (int k = 0; k < 8; ++k) tile[((t >> 4) * 17 + (t & 15)) * 17 + h + k] = tsdf_or_nan(r[k]);   // z = h + k, x = t >> 4, y = t & 15
        }
    }
    // (2) the +1 neighbour faces / edges / corner: 3 * 256 + 3 * 16 + 1 = 817 records from up to 7 other blocks
    for (int e = t; e < 817; e += 256) {
        int lx, ly, lz;
        if (e < 256)      { lx = 16; ly = e & 15; lz = e >> 4; }                 // +x face: 16 contiguous records per z
        else if (e < 512) { lx = (e - 256) >> 4; ly = 16; lz = e & 15; }         // +y face
        else if (e < 768) { lx = (e - 512) >> 4; ly = e & 15; lz = 16; }         // +z face: 256 contiguous records
        else if (e < 784) { lx = 16; ly = 16; lz = e - 768; }                    // edges
        else if (e < 800) { lx = 16; ly = e - 784; lz = 16; }
        else if (e < 816) { lx = e - 800; ly = 16; lz = 16; }
        else              { lx = 16; ly = 16; lz = 16; }                         // corner
        const int s = nslot[(lx >> 4) | ((ly >> 4) << 1) | ((lz >> 4) << 2)];
        float v = qnan;
        if (s >= 0) v = tsdf_or_nan(__ldg(block_ptr(c.chunks, s) + rec_index(lx & 15, ly & 15, lz & 15)));
        tile[(lx * 17 + ly) * 17 + lz] = v;
    }
    __syncthreads();
    int my_tris = 0;
    for (int k = 0; k < 16; ++k) {
        const int x = k, y = t >> 4, z = t & 15;
        int cube = 0;
        bool ok = true;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            // corner q of the cube: shift[q] = ((q ^ q>>1) & 1, q>>1 & 1, q>>2 & 1)  (SURVEY Appendix B)
            const float f = tile[((x + ((q ^ (q >> 1)) & 1)) * 17 + (y + ((q >> 1) & 1))) * 17 + (z + ((q >> 2) & 1))];
            if (f != f) ok = false;
            if (f < 0.f) cube |= 1 << q;
        }
        if (!ok || cube == 255) cube = 0;
        cube_idx[(size_t)slot * kVox + (x * 256 + y * 16 + z)] = (uint8_t)cube;
        if (cube) {
            my_tris += d_ntri[cube];
            const unsigned et = d_edge_table[cube];
            for (int e = 0; e < 12; ++e) {
                if (!(et & (1u << e))) continue;
                const int ox = x + d_edge_shift[e][0], oy = y + d_edge_shift[e][1], oz = z + d_edge_shift[e][2];
                const int axis = d_edge_shift[e][3];
                const int nb = (ox >> 4) | ((oy >> 4) << 1) | ((oz >> 4) << 2);
                const int bit = (ox & 15) * 256 + (oy & 15) * 16 + (oz & 15);
                const int word = axis * (kVox / 32) + (bit >> 5);
                if (nb == 0) {                // most edges belong to this block: shared-memory atomics (4 cubes share an edge)
                    if (!(s_flags[word] & (1u << (bit & 31)))) atomicOr(&s_flags[word], 1u << (bit & 31));
                } else {                      // the +x / +y / +z neighbour exists: the cube is valid, so that corner was observed
                    atomicOr(flags + (size_t)nslot[nb] * kFlagWords + word, 1u << (bit & 31));
                }
            }
        }
    }
    for (int o = 16; o; o >>= 1) my_tris += __shfl_xor_sync(0xffffffffu, my_tris, o);
    if ((t & 31) == 0 && my_tris) atomicAdd(&s_tris, my_tris);
    __syncthreads();
    if (t == 0) tri_count[i] = s_tris;
    for (int w = t; w < kFlagWords; w += 256)      // (the -x / -y / -z neighbours' cubes set bits of this block too: still an atomic)
        if (s_flags[w]) atomicOr(flags + (size_t)slot * kFlagWords + w, s_flags[w]);
}

// per block: vertex count and exclusive per-word prefix of its edge bits
__global__ void __launch_bounds__(128) mc_count_kernel(const int32_t* __restrict__ bslots, const uint32_t* __restrict__ flags,
                                                       uint16_t* __restrict__ word_prefix, int* __restrict__ vcount) {
    __shared__ int warp_sum[4];
    const int i = blockIdx.x, t = threadIdx.x;
    const int slot = bslots[i];
    const uint32_t* f = flags + (size_t)slot * kFlagWords;
    uint16_t* wp = word_prefix + (size_t)slot * kFlagWords;
    // thread t owns words 3t..3t+2
    const int c0 = __popc(f[3 * t]), c1 = __popc(f[3 * t + 1]), c2 = __popc(f[3 * t + 2]);
    const int v = c0 + c1 + c2;
    const int ex = cta_exclusive_scan<int, 4>(v, warp_sum, nullptr);
    wp[3 * t] = (uint16_t)ex;
    wp[3 * t + 1] = (uint16_t)(ex + c0);
    wp[3 * t + 2] = (uint16_t)(ex + c0 + c1);
    if (t == 127) vcount[i] = ex + v;
}

__global__ void scatter_base_kernel(const int32_t* __restrict__ bslots, const int64_t* __restrict__ vbase, int n,
                                    int64_t* __restrict__ vbase_by_slot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) vbase_by_slot[bslots[i]] = vbase[i];
}

__device__ __forceinline__ void rec_color01(const uint4& r, double* c) {
    const uint32_t w = rec_weight(r);
    const double dw = (double)w;
    // colour mean = exact integer sum / count (the reference keeps an FP64 running mean), then /255
    c[0] = __ddiv_rn(__ddiv_rn((double)(r.y & 0xFFFFFFu), dw), 255.0);
    c[1] = __ddiv_rn(__ddiv_rn((double)(r.z & 0xFFFFFFu), dw), 255.0);
    c[2] = __ddiv_rn(__ddiv_rn((double)(r.w & 0xFFFFFFu), dw), 255.0);
}

// One thread per VERTEX (round 1: one thread per 3 flag words, so the thread that owned a dense word produced up to 32
// vertices -- ~600 FP64-heavy instructions each -- while its neighbours idled: 122 us for 747 k vertices).  The block's flag
// words and their exclusive prefixes are staged in shared memory; vertex j of the block finds its word by binary search over
// the prefixes and its bit with __fns (n-th set bit).  Vertex ids are unchanged (rank of the bit), so are the faces.
__global__ void __launch_bounds__(128) mc_vertices_kernel(ExtractCtx c, const uint32_t* __restrict__ flags,
                                                          const uint16_t* __restrict__ word_prefix,
                                                          const int64_t* __restrict__ vbase, double* __restrict__ verts,
                                                          double* __restrict__ colors, int32_t* __restrict__ ekeys) {
    __shared__ int nslot[8];
    __shared__ uint32_t s_bits[kFlagWords];
    __shared__ uint16_t s_pre[kFlagWords];
    const int i = blockIdx.x, t = threadIdx.x;
    const uint64_t key = c.bkeys[i];
    const int slot = c.bslots[i];
    const int nvb = (int)(vbase[i + 1] - vbase[i]);
    if (nvb == 0) return;
    load_neighbours(c, key, slot, nslot);
    for (int w = t; w < kFlagWords; w += 128) {
        s_bits[w] = flags[(size_t)slot * kFlagWords + w];
        s_pre[w] = word_prefix[(size_t)slot * kFlagWords + w];
    }
    __syncthreads();
    int kx, ky, kz;
    unpack_key(key, kx, ky, kz);
    const uint4* blk = block_ptr(c.chunks, slot);
    for (int j = t; j < nvb; j += 128) {
        int lo = 0, hi = kFlagWords - 1;                  // last word whose exclusive prefix is <= j and that has a bit for j
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if ((int)s_pre[mid] <= j) lo = mid; else hi = mid - 1;
        }
        const int wi = lo;                                // (empty words share their successor's prefix: the search lands on the last
                                                          //  word with prefix <= j, which is the non-empty one that contains rank j)
        const uint32_t bits = s_bits[wi];
        const int bit = (int)__fns(bits, 0, j - (int)s_pre[wi] + 1);
        const int axis = wi / (kVox / 32);
        const int64_t vid = vbase[i] + j;
        {
            const int vox = (wi % (kVox / 32)) * 32 + bit;
            const int x = vox >> 8, y = (vox >> 4) & 15, z = vox & 15;
            int q[3] = {x, y, z};
            q[axis] += 1;
            const int nb = (q[0] >> 4) | ((q[1] >> 4) << 1) | ((q[2] >> 4) << 2);
            const uint4 r0 = blk[rec_index(x, y, z)];
            const uint4 r1 = block_ptr(c.chunks, nslot[nb])[rec_index(q[0] & 15, q[1] & 15, q[2] & 15)];
            const double f0 = fabs((double)__uint_as_float(r0.x)), f1 = fabs((double)__uint_as_float(r1.x));
            const int g[3] = {(kx - c.x_off) * kRes + x, ky * kRes + y, kz * kRes + z};
            double pt[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) pt[k] = __dadd_rn(c.half, __dmul_rn(c.vl, (double)g[k]));
            const double fs = __dadd_rn(f0, f1);
            pt[axis] = __dadd_rn(pt[axis], __ddiv_rn(__dmul_rn(f0, c.vl), fs));
            double c0[3], c1[3];
            rec_color01(r0, c0);
            rec_color01(r1, c1);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                verts[3 * vid + k] = pt[k];
                colors[3 * vid + k] = __ddiv_rn(__dadd_rn(__dmul_rn(f1, c0[k]), __dmul_rn(f0, c1[k])), fs);
            }
            if (ekeys) {
                ekeys[4 * vid] = g[0]; ekeys[4 * vid + 1] = g[1]; ekeys[4 * vid + 2] = g[2]; ekeys[4 * vid + 3] = axis;
            }
        }
    }
}

__global__ void __launch_bounds__(256) mc_faces_kernel(ExtractCtx c, const uint32_t* __restrict__ flags,
                                                       const uint16_t* __restrict__ word_prefix,
                                                       const int64_t* __restrict__ vbase_by_slot,
                                                       const uint8_t* __restrict__ cube_idx,
                                                       const int64_t* __restrict__ fbase, int32_t* __restrict__ faces) {
    __shared__ int nslot[8];
    __shared__ int warp_sum[8];
    const int i = blockIdx.x, t = threadIdx.x;
    if (fbase[i + 1] == fbase[i]) return;
    const uint64_t key = c.bkeys[i];
    const int slot = c.bslots[i];
    load_neighbours(c, key, slot, nslot);
    // thread t owns voxels 16t..16t+15 (reference order x*256+y*16+z)
    const uint8_t* ci = cube_idx + (size_t)slot * kVox + 16 * t;
    const uint4 packed = *reinterpret_cast<const uint4*>(ci);
    const uint32_t pw[4] = {packed.x, packed.y, packed.z, packed.w};
    int mine = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) mine += d_ntri[(pw[k >> 2] >> (8 * (k & 3))) & 0xFF];
    int64_t fo = fbase[i] + cta_exclusive_scan<int, 8>(mine, warp_sum, nullptr);
    for (int k = 0; k < 16; ++k) {
        const int cube = (pw[k >> 2] >> (8 * (k & 3))) & 0xFF;
        if (!cube) continue;
        const int vox = 16 * t + k;
        const int x = vox >> 8, y = (vox >> 4) & 15, z = vox & 15;
        const int nt = d_ntri[cube];
        for (int tr = 0; tr < nt; ++tr) {
            int vid[3];
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int e = d_tri_table[cube][3 * tr + j];
                const int ox = x + d_edge_shift[e][0], oy = y + d_edge_shift[e][1], oz = z + d_edge_shift[e][2];
                const int axis = d_edge_shift[e][3];
                const int os = nslot[(ox >> 4) | ((oy >> 4) << 1) | ((oz >> 4) << 2)];
                const int bit = (ox & 15) * 256 + (oy & 15) * 16 + (oz & 15);
                const int wi = axis * (kVox / 32) + (bit >> 5);
                const uint32_t wbits = flags[(size_t)os * kFlagWords + wi];
                vid[j] = (int)(vbase_by_slot[os] + word_prefix[(size_t)os * kFlagWords + wi] +
                               __popc(wbits & ((1u << (bit & 31)) - 1u)));
            }
            faces[3 * fo] = vid[0];
            faces[3 * fo + 1] = vid[2];   // winding swapped w.r.t. the table (SURVEY A.5)
            faces[3 * fo + 2] = vid[1];
            ++fo;
        }
    }
}

// ---- SURVEY A.9: compute_vertex_normals.  The reference adds each triangle's un-normalised normal to
// its three vertices in one sequential loop over the triangles, so a vertex's sum is taken in
// triangle-index order; FP64 atomics would make the low bits depend on the launch.  Here every vertex
// gets the list of its corners (corner id = 3 * triangle + k): degree count -> scan -> fill (integer
// atomics: the SET of a vertex's corners is deterministic, only its order in the list is not) -> one
// thread per vertex sorts its short list and adds the face normals in ascending corner order.
// Bit-identical to the scalar loop, and the same bits on every run.
__global__ void __launch_bounds__(256) face_normals_kernel(const double* __restrict__ verts, const int32_t* __restrict__ faces,
                                                           int64_t nf, int64_t nv, double* __restrict__ fnrm, int* __restrict__ deg) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nf) return;
    const int a = faces[3 * f], b = faces[3 * f + 1], cidx = faces[3 * f + 2];
    if ((unsigned)a >= (unsigned)nv || (unsigned)b >= (unsigned)nv || (unsigned)cidx >= (unsigned)nv) return;   // malformed face: ignored
    double e1[3], e2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        e1[k] = __dsub_rn(verts[3 * (size_t)b + k], verts[3 * (size_t)a + k]);
        e2[k] = __dsub_rn(verts[3 * (size_t)cidx + k], verts[3 * (size_t)a + k]);
    }
    fnrm[3 * f] = __dsub_rn(__dmul_rn(e1[1], e2[2]), __dmul_rn(e1[2], e2[1]));
    fnrm[3 * f + 1] = __dsub_rn(__dmul_rn(e1[2], e2[0]), __dmul_rn(e1[0], e2[2]));
    fnrm[3 * f + 2] = __dsub_rn(__dmul_rn(e1[0], e2[1]), __dmul_rn(e1[1], e2[0]));
    atomicAdd(deg + a, 1); atomicAdd(deg + b, 1); atomicAdd(deg + cidx, 1);
}

__global__ void __launch_bounds__(256) corner_fill_kernel(const int32_t* __restrict__ faces, int64_t n_corners,
                                                          int64_t nv, const int64_t* __restrict__ off, int* __restrict__ cursor,
                                                          int32_t* __restrict__ adj) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_corners) return;
    const int64_t f3 = c - c % 3;
    if ((unsigned)faces[f3] >= (unsigned)nv || (unsigned)faces[f3 + 1] >= (unsigned)nv || (unsigned)faces[f3 + 2] >= (unsigned)nv) return;
    const int v = faces[c];
    adj[off[v] + atomicAdd(cursor + v, 1)] = (int32_t)c;
}

__global__ void __launch_bounds__(128) vertex_normals_kernel(int64_t nv, const int64_t* __restrict__ off, int32_t* __restrict__ adj,
                                                             const double* __restrict__ fnrm, double* __restrict__ normals) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nv) return;
    int32_t* a = adj + off[i];
    const int d = (int)(off[i + 1] - off[i]);
    for (int p = 1; p < d; ++p) {                 // insertion sort: degrees are ~6 on marching-cubes meshes
        const int32_t x = a[p];
        int q = p - 1;
        for (; q >= 0 && a[q] > x; --q) a[q + 1] = a[q];
        a[q + 1] = x;
    }
    double n0 = 0.0, n1 = 0.0, n2 = 0.0;
    for (int p = 0; p < d; ++p) {
        const double* f = fnrm + 3 * (size_t)(a[p] / 3);
        n0 = __dadd_rn(n0, f[0]); n1 = __dadd_rn(n1, f[1]); n2 = __dadd_rn(n2, f[2]);
    }
    const double l = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(n0, n0), __dmul_rn(n1, n1)), __dmul_rn(n2, n2)));
    double* n = normals + 3 * i;
    if (l > 0.0) {
        n[0] = __ddiv_rn(n0, l); n[1] = __ddiv_rn(n1, l); n[2] = __ddiv_rn(n2, l);
    } else {
        n[0] = 0.0; n[1] = 0.0; n[2] = 1.0;
    }
}

int device_vertex_normals(const double* d_verts, int64_t nv, const int32_t* d_faces, int64_t nf, double* d_normals,
                          cudaStream_t s) {
    if (nv == 0) return OTSLAM_OK;
    if (nv > 0x7fffffffLL || 3 * nf > 0x7fffffffLL) return set_error(OTSLAM_ERR_OVERFLOW, "mesh exceeds int32 corner indices");
    DevBuf<double> fnrm;
    DevBuf<int> deg;                 // [2][nv]: degree, then the fill cursor
    DevBuf<int64_t> off;
    DevBuf<int32_t> adj;
    OT_CUDA(fnrm.alloc((size_t)std::max<int64_t>(nf, 1) * 3)); OT_CUDA(deg.alloc((size_t)nv * 2)); OT_CUDA(off.alloc(nv + 1));
    OT_CUDA(adj.alloc((size_t)std::max<int64_t>(nf, 1) * 3));
    OT_CUDA(cudaMemsetAsync(deg.p, 0, (size_t)nv * 2 * sizeof(int), s));
    if (nf > 0) {
        face_normals_kernel<<<(unsigned)((nf + 255) / 256), 256, 0, s>>>(d_verts, d_faces, nf, nv, fnrm.p, deg.p);
        OT_LAUNCHED();
    }
    OT_TRY(device_exclusive_scan(deg.p, off.p, (int)nv, s));
    if (nf > 0) {
        corner_fill_kernel<<<(unsigned)((3 * nf + 255) / 256), 256, 0, s>>>(d_faces, 3 * nf, nv, off.p, deg.p + nv, adj.p);
        OT_LAUNCHED();
    }
    vertex_normals_kernel<<<(unsigned)((nv + 127) / 128), 128, 0, s>>>(nv, off.p, adj.p, fnrm.p, d_normals);
    OT_LAUNCHED();
    return OTSLAM_OK;
}

// ---- SURVEY A.6: extract_point_cloud
__global__ void __launch_bounds__(256) pc_extract_kernel(ExtractCtx c, const int64_t* __restrict__ pbase, int* __restrict__ pcount,
                                                         double* __restrict__ pts, double* __restrict__ cols,
                                                         int32_t* __restrict__ ekeys) {
    __shared__ int nslot[8];
    __shared__ int warp_sum[8];
    const int i = blockIdx.x, t = threadIdx.x;
    const uint64_t key = c.bkeys[i];
    const int slot = c.bslots[i];
    int kx, ky, kz;
    unpack_key(key, kx, ky, kz);
    const bool count_only = (pbase == nullptr);
    if (!slab_owns(c.slab, kx, ky, kz)) {
        if (count_only && t == 0) pcount[i] = 0;
        return;
    }
    if (!count_only && pbase[i + 1] == pbase[i]) return;
    load_neighbours(c, key, slot, nslot);
    __syncthreads();
    const uint4* blk = block_ptr(c.chunks, slot);
    // thread t owns voxels 16t..16t+15 in reference order; pass 1 counts, pass 2 emits
    uint32_t hits[2] = {0, 0};   // 3 bits per voxel
    int mine = 0;
    for (int k = 0; k < 16; ++k) {
        const int vox = 16 * t + k;
        const int x = vox >> 8, y = (vox >> 4) & 15, z = vox & 15;
        const uint4 r0 = blk[rec_index(x, y, z)];
        const float f0 = __uint_as_float(r0.x);
        if (rec_weight(r0) == 0 || !(f0 < 0.98f && f0 >= -0.98f)) continue;
        for (int a = 0; a < 3; ++a) {
            int q[3] = {x, y, z};
            q[a] += 1;
            const int s = nslot[(q[0] >> 4) | ((q[1] >> 4) << 1) | ((q[2] >> 4) << 2)];
            if (s < 0) continue;
            const uint4 r1 = block_ptr(c.chunks, s)[rec_index(q[0] & 15, q[1] & 15, q[2] & 15)];
            const float f1 = __uint_as_float(r1.x);
            if (rec_weight(r1) == 0 || !(f1 < 0.98f && f1 >= -0.98f) || !(__fmul_rn(f0, f1) < 0.f)) continue;
            hits[k >> 3] |= 1u << (3 * (k & 7) + a);
            ++mine;
        }
    }
    const int rank = cta_exclusive_scan<int, 8>(mine, warp_sum, nullptr);
    if (count_only) {
        if (t == 255) pcount[i] = rank + mine;
        return;
    }
    int64_t o = pbase[i] + rank;
    for (int k = 0; k < 16; ++k) {
        const uint32_t h = (hits[k >> 3] >> (3 * (k & 7))) & 7u;
        if (!h) continue;
        const int vox = 16 * t + k;
        const int x = vox >> 8, y = (vox >> 4) & 15, z = vox & 15;
        const uint4 r0 = blk[rec_index(x, y, z)];
        const float r0a = fabsf(__uint_as_float(r0.x));                  // Open3D keeps r0, r1 and their sum in FP32
        const int g[3] = {(kx - c.x_off) * kRes + x, ky * kRes + y, kz * kRes + z};
        const int loc[3] = {x, y, z}, bk[3] = {kx - c.x_off, ky, kz};
        double p0[3];
#pragma unroll
        for (int j = 0; j < 3; ++j)     // (half + vl * x_local) + block_index * unit_length, as ExtractPointCloud forms it
            p0[j] = __dadd_rn(__dadd_rn(c.half, __dmul_rn(c.vl, (double)loc[j])), __dmul_rn((double)bk[j], c.unit));
        const uint32_t w0 = rec_weight(r0);
        for (int a = 0; a < 3; ++a) {
            if (!(h & (1u << a))) continue;
            int q[3] = {x, y, z};
            q[a] += 1;
            const int s = nslot[(q[0] >> 4) | ((q[1] >> 4) << 1) | ((q[2] >> 4) << 2)];
            const uint4 r1 = block_ptr(c.chunks, s)[rec_index(q[0] & 15, q[1] & 15, q[2] & 15)];
            const float r1a = fabsf(__uint_as_float(r1.x));
            const uint32_t w1 = rec_weight(r1);
            const float rs = __fadd_rn(r0a, r1a);
            double p[3] = {p0[0], p0[1], p0[2]};
            const double p1a = __dadd_rn(p0[a], c.vl);
            p[a] = __ddiv_rn(__dadd_rn(__dmul_rn(p0[a], (double)r1a), __dmul_rn(p1a, (double)r0a)), (double)rs);
            const uint32_t s0[3] = {r0.y & 0xFFFFFFu, r0.z & 0xFFFFFFu, r0.w & 0xFFFFFFu};
            const uint32_t s1[3] = {r1.y & 0xFFFFFFu, r1.z & 0xFFFFFFu, r1.w & 0xFFFFFFu};
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                pts[3 * o + j] = p[j];
                // voxel colour = exact sum / count in FP64 (the reference keeps an FP64 running mean), cast to float as
                // Open3D's c0, c1 are; interpolation and the division by 255.0f in FP32
                const float c0 = (float)__ddiv_rn((double)s0[j], (double)w0), c1 = (float)__ddiv_rn((double)s1[j], (double)w1);
                cols[3 * o + j] = (double)__fdiv_rn(__fdiv_rn(__fadd_rn(__fmul_rn(c0, r1a), __fmul_rn(c1, r0a)), rs), 255.0f);
            }
            if (ekeys) { ekeys[4 * o] = g[0]; ekeys[4 * o + 1] = g[1]; ekeys[4 * o + 2] = g[2]; ekeys[4 * o + 3] = a; }
            ++o;
        }
    }
}

// ---- ScalableTSDFVolume::GetNormalAt for extracted points (the normals ExtractPointCloud attaches): volume_lookup.cuh
__global__ void __launch_bounds__(128) pc_normals_kernel(ExtractCtx c, const double* __restrict__ pts, int64_t n, double gap,
                                                         double* __restrict__ normals) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double p[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    double nrm[3];
    normal_at(c, p, gap, nrm);
#pragma unroll
    for (int a = 0; a < 3; ++a) normals[3 * i + a] = nrm[a];
}

// the sorted block list lives in HBM (volume.cu: volume_sorted_blocks_device): no host round trip of the hash table
static int make_ctx(otslam_volume* v, ExtractCtx& c) {
    const uint64_t* dk = nullptr;
    const int32_t* ds = nullptr;
    int n = 0;
    int x_off = 0;
    OT_TRY(volume_selected_blocks_device(v, &dk, &ds, &n, &x_off));
    c.x_off = x_off;
    c.arena = v->n_objects > 0;
    c.table = volume_hash(v); c.chunks = v->d_chunks.p;
    c.bkeys = dk; c.bslots = ds; c.n = n; c.slab = v->slab;
    c.vl = v->voxel_length; c.half = 0.5 * v->voxel_length; c.unit = v->unit_length;
    return OTSLAM_OK;
}

}  // namespace otslam

using namespace otslam;

extern "C" {

int otslam_volume_extract_mesh(otslam_volume* v, int64_t* n_vertices, int64_t* n_faces) {
    if (!v || !n_vertices || !n_faces) return set_error(OTSLAM_ERR_INVALID, "null argument");
    OT_TRY(use_device(v->device));
    OT_TRY(upload_tables());
    v->mesh = {};
    *n_vertices = 0; *n_faces = 0;
    OpTimer timer(v->stream);
    ExtractCtx c;
    OT_TRY(make_ctx(v, c));
    const int n = c.n;
    if (n == 0) return OTSLAM_OK;
    cudaStream_t s = v->stream;
    DevBuf<uint32_t> flags;
    DevBuf<uint16_t> wprefix;
    DevBuf<uint8_t> cube;
    DevBuf<int> tri_count, vcount;
    DevBuf<int64_t> vbase, fbase, vbase_slot;
    const size_t n_slots = (size_t)v->n_blocks;      // per-slot arrays: an arena extracts a sub-list, slots range over the pool
    OT_CUDA(flags.alloc(n_slots * kFlagWords));
    OT_CUDA(wprefix.alloc(n_slots * kFlagWords));
    OT_CUDA(cube.alloc(n_slots * kVox));
    OT_CUDA(tri_count.alloc(n)); OT_CUDA(vcount.alloc(n));
    OT_CUDA(vbase.alloc(n + 1)); OT_CUDA(fbase.alloc(n + 1)); OT_CUDA(vbase_slot.alloc(n_slots));
    OT_CUDA(cudaMemsetAsync(flags.p, 0, n_slots * kFlagWords * 4, s));
    mc_classify_kernel<<<n, 256, 0, s>>>(c, flags.p, cube.p, tri_count.p);
    OT_LAUNCHED();
    mc_count_kernel<<<n, 128, 0, s>>>(c.bslots, flags.p, wprefix.p, vcount.p);
    OT_LAUNCHED();
    OT_TRY(device_exclusive_scan(vcount.p, vbase.p, n, s));
    OT_TRY(device_exclusive_scan(tri_count.p, fbase.p, n, s));
    scatter_base_kernel<<<(n + 255) / 256, 256, 0, s>>>(c.bslots, vbase.p, n, vbase_slot.p);
    OT_LAUNCHED();
    int64_t nv = 0, nf = 0;
    OT_CUDA(cudaMemcpyAsync(&nv, vbase.p + n, 8, cudaMemcpyDeviceToHost, s));
    OT_CUDA(cudaMemcpyAsync(&nf, fbase.p + n, 8, cudaMemcpyDeviceToHost, s));
    OT_CUDA(cudaStreamSynchronize(s));
    if (nv > 0x7fffffffLL || nf > 0x7fffffffLL) return set_error(OTSLAM_ERR_OVERFLOW, "mesh exceeds int32 indices");
    MeshResult m;
    m.nv = nv; m.nf = nf;
    if (nv > 0) {
        OT_CUDA(m.verts.alloc(nv * 3)); OT_CUDA(m.colors.alloc(nv * 3)); OT_CUDA(m.normals.alloc(nv * 3));
        OT_CUDA(m.ekeys.alloc(nv * 4)); OT_CUDA(m.faces.alloc(nf * 3));
        mc_vertices_kernel<<<n, 128, 0, s>>>(c, flags.p, wprefix.p, vbase.p, m.verts.p, m.colors.p, m.ekeys.p);
        OT_LAUNCHED();
        if (nf > 0) {
            mc_faces_kernel<<<n, 256, 0, s>>>(c, flags.p, wprefix.p, vbase_slot.p, cube.p, fbase.p, m.faces.p);
            OT_LAUNCHED();
        }
        OT_TRY(device_vertex_normals(m.verts.p, nv, m.faces.p, nf, m.normals.p, s));
    }
    OT_CUDA(cudaStreamSynchronize(s));
    v->mesh = std::move(m);
    *n_vertices = nv; *n_faces = nf;
    return OTSLAM_OK;
}

int otslam_volume_mesh_copy(otslam_volume* v, double* vertices, double* colors, double* normals, int32_t* faces,
                            int32_t* edge_keys) {
    if (!v) return set_error(OTSLAM_ERR_INVALID, "null volume");
    OT_TRY(use_device(v->device));
    const MeshResult& m = v->mesh;
    if (m.nv > 0) {
        if (vertices) OT_CUDA(cudaMemcpyAsync(vertices, m.verts.p, (size_t)m.nv * 24, cudaMemcpyDefault, v->stream));
        if (colors) OT_CUDA(cudaMemcpyAsync(colors, m.colors.p, (size_t)m.nv * 24, cudaMemcpyDefault, v->stream));
        if (normals) OT_CUDA(cudaMemcpyAsync(normals, m.normals.p, (size_t)m.nv * 24, cudaMemcpyDefault, v->stream));
        if (edge_keys) OT_CUDA(cudaMemcpyAsync(edge_keys, m.ekeys.p, (size_t)m.nv * 16, cudaMemcpyDefault, v->stream));
    }
    if (m.nf > 0 && faces) OT_CUDA(cudaMemcpyAsync(faces, m.faces.p, (size_t)m.nf * 12, cudaMemcpyDefault, v->stream));
    OT_CUDA(cudaStreamSynchronize(v->stream));     // destinations may be host or device pointers (unified addressing)
    return OTSLAM_OK;
}

int otslam_volume_extract_points(otslam_volume* v, int64_t* n_points) {
    if (!v || !n_points) return set_error(OTSLAM_ERR_INVALID, "null argument");
    OT_TRY(use_device(v->device));
    v->points = {};
    *n_points = 0;
    OpTimer timer(v->stream);
    ExtractCtx c;
    OT_TRY(make_ctx(v, c));
    const int n = c.n;
    if (n == 0) return OTSLAM_OK;
    cudaStream_t s = v->stream;
    DevBuf<int> pcount;
    DevBuf<int64_t> pbase;
    OT_CUDA(pcount.alloc(n)); OT_CUDA(pbase.alloc(n + 1));
    pc_extract_kernel<<<n, 256, 0, s>>>(c, nullptr, pcount.p, nullptr, nullptr, nullptr);
    OT_LAUNCHED();
    OT_TRY(device_exclusive_scan(pcount.p, pbase.p, n, s));
    int64_t np = 0;
    OT_CUDA(cudaMemcpyAsync(&np, pbase.p + n, 8, cudaMemcpyDeviceToHost, s));
    OT_CUDA(cudaStreamSynchronize(s));
    PointsResult p;
    p.n = np;
    if (np > 0) {
        OT_CUDA(p.pts.alloc(np * 3)); OT_CUDA(p.cols.alloc(np * 3)); OT_CUDA(p.ekeys.alloc(np * 4));
        pc_extract_kernel<<<n, 256, 0, s>>>(c, pbase.p, nullptr, p.pts.p, p.cols.p, p.ekeys.p);
        OT_LAUNCHED();
        OT_CUDA(cudaStreamSynchronize(s));
    }
    v->points = std::move(p);
    *n_points = np;
    return OTSLAM_OK;
}

int otslam_volume_points_normals(otslam_volume* v, double* normals) {
    if (!v || !normals) return set_error(OTSLAM_ERR_INVALID, "null argument");
    OT_TRY(use_device(v->device));
    const PointsResult& p = v->points;
    if (p.n == 0) return OTSLAM_OK;
    ExtractCtx c;
    OT_TRY(make_ctx(v, c));
    DevBuf<double> dn;
    OT_CUDA(dn.alloc((size_t)p.n * 3));
    pc_normals_kernel<<<(unsigned)((p.n + 127) / 128), 128, 0, v->stream>>>(c, p.pts.p, p.n, 0.99 * v->voxel_length, dn.p);
    OT_LAUNCHED();
    OT_CUDA(cudaMemcpyAsync(normals, dn.p, (size_t)p.n * 24, cudaMemcpyDefault, v->stream));
    OT_CUDA(cudaStreamSynchronize(v->stream));
    return OTSLAM_OK;
}

int otslam_volume_points_copy(otslam_volume* v, double* points, double* colors, int32_t* edge_keys) {
    if (!v) return set_error(OTSLAM_ERR_INVALID, "null volume");
    OT_TRY(use_device(v->device));
    const PointsResult& p = v->points;
    if (p.n > 0) {
        if (points) OT_CUDA(cudaMemcpyAsync(points, p.pts.p, (size_t)p.n * 24, cudaMemcpyDefault, v->stream));
        if (colors) OT_CUDA(cudaMemcpyAsync(colors, p.cols.p, (size_t)p.n * 24, cudaMemcpyDefault, v->stream));
        if (edge_keys) OT_CUDA(cudaMemcpyAsync(edge_keys, p.ekeys.p, (size_t)p.n * 16, cudaMemcpyDefault, v->stream));
        OT_CUDA(cudaStreamSynchronize(v->stream));
    }
    return OTSLAM_OK;
}

}  // extern "C"
