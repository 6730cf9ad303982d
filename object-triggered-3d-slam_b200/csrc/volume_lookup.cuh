// volume_lookup.cuh -- read-only voxel lookups through the block hash (hash_table.cuh), shared by extraction (extract.cu)
// and ray casting (raycast.cu): the range-checked block lookup, and Open3D's GetTSDFAt (trilinear TSDF at a world point,
// the basis of GetNormalAt).
#pragma once
#include "volume.cuh"

namespace otslam {

struct ExtractCtx {
    HashTable table;          // the volume's block hash
    uint4* const* chunks;
    const uint64_t* bkeys;    // [n] sorted block keys (extraction only)
    const int32_t* bslots;    // [n] their pool slots
    int n;
    SlabSpec slab;
    double vl, half, unit;    // voxel length, half of it, block edge length
    int x_off;                // multi-object arena: x-key offset of the selected object (stored key - x_off = true block x)
    bool arena;               // multi-object arena: a block whose true x lies outside [-2^17, 2^17) is absent
};

// pool slot of block (bx, by, bz) (true x: the arena offset is added here), -1 if absent, outside the key range or outside
// the selected arena object's window (the stored key one past an object's last block is the next object's first block)
__device__ __forceinline__ int block_slot(const ExtractCtx& c, int bx, int by, int bz) {
    if ((c.arena && (bx < -kObjHalf || bx >= kObjHalf)) || !key_in_range(bx + c.x_off, by, bz)) return -1;
    return hash_find(c.table, pack_key(bx + c.x_off, by, bz));
}

// ---- ScalableTSDFVolume::GetTSDFAt: trilinear interpolation of the TSDF at a world point (FP64).  Voxels of absent blocks
// read 0, observed or not does not matter (Open3D ignores the weight here); an absent base block gives 0.
__device__ inline double tsdf_at(const ExtractCtx& c, const double p[3]) {
    double pg[3], r[3];
    int index0[3], idx0[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double pl = __dsub_rn(p[i], c.half);
        index0[i] = (int)floor(__ddiv_rn(pl, c.unit));
        pg[i] = __ddiv_rn(__dsub_rn(pl, __dmul_rn((double)index0[i], c.unit)), c.vl);
    }
    if (block_slot(c, index0[0], index0[1], index0[2]) < 0) return 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        idx0[i] = min(max((int)floor(pg[i]), 0), kRes - 1);
        r[i] = __dsub_rn(pg[i], (double)idx0[i]);
    }
    double f[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        int v[3] = {idx0[0] + ((q ^ (q >> 1)) & 1), idx0[1] + ((q >> 1) & 1), idx0[2] + ((q >> 2) & 1)};
        int b[3] = {index0[0], index0[1], index0[2]};
#pragma unroll
        for (int j = 0; j < 3; ++j)
            if (v[j] >= kRes) { v[j] -= kRes; b[j] += 1; }
        const int s = block_slot(c, b[0], b[1], b[2]);
        f[q] = s >= 0 ? (double)__uint_as_float(block_ptr(c.chunks, s)[rec_index(v[0], v[1], v[2])].x) : 0.0;
    }
    const double o0 = __dsub_rn(1.0, r[0]), o1 = __dsub_rn(1.0, r[1]), o2 = __dsub_rn(1.0, r[2]);
    auto lerp2 = [&](double a, double b) { return __dadd_rn(__dmul_rn(o2, a), __dmul_rn(r[2], b)); };
    const double lo = __dadd_rn(__dmul_rn(o1, lerp2(f[0], f[4])), __dmul_rn(r[1], lerp2(f[3], f[7])));
    const double hi = __dadd_rn(__dmul_rn(o1, lerp2(f[1], f[5])), __dmul_rn(r[1], lerp2(f[2], f[6])));
    return __dadd_rn(__dmul_rn(o0, lo), __dmul_rn(r[0], hi));
}

// ---- ScalableTSDFVolume::GetNormalAt: central differences of tsdf_at at +-gap (0.99 voxel) on each axis, normalised
// (a zero gradient stays zero).  The normals extract_point_cloud attaches, and those of ray-cast hits.
__device__ inline void normal_at(const ExtractCtx& c, const double p[3], double gap, double n[3]) {
    double g[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double p0[3] = {p[0], p[1], p[2]}, p1[3] = {p[0], p[1], p[2]};
        p0[a] = __dsub_rn(p0[a], gap);
        p1[a] = __dadd_rn(p1[a], gap);
        g[a] = __dsub_rn(tsdf_at(c, p1), tsdf_at(c, p0));
    }
    const double l = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(g[0], g[0]), __dmul_rn(g[1], g[1])), __dmul_rn(g[2], g[2])));
#pragma unroll
    for (int a = 0; a < 3; ++a) n[a] = l > 0.0 ? __ddiv_rn(g[a], l) : g[a];
}

}  // namespace otslam
