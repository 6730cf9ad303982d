// oracle.cpp -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
//
// A CPU restatement of the algorithm that the reference's RGB-D reconstruction hot path runs.
// The reference scripts (/root/reference/3d_model/reconstruct_rgbd.py:79-118,
// reconstruct_rgbd_filter.py:81-140, multi_reconstruct_rgbd_filter.py:57-137,
// fusion/hybrid_map.py:25-121, check_one_frame.py:20-30) contain no arithmetic of their own: every
// heavy step is a call into the third-party `open3d` package (legacy CPU pipeline,
// ScalableTSDFVolume & friends).  open3d is NOT vendored in /root/reference, NOT version pinned by
// any manifest in it, and NOT installable here (no network).  This file therefore restates the
// published behaviour of Open3D's legacy pipeline (0.13-0.18; SURVEY.md Appendix A) from its
// documented semantics.
//
// **PARITY UNPINNED**: the reference holds no tests, golden vectors or fixtures for this path and
// the real backend cannot run here, so this oracle cannot be checked against the reference's own
// outputs.  It is pinned instead by closed-form self-tests (tests/test_oracle_*.py): analytic plane
// TSDF, weight == visible-frame count, marching-cubes table validation (sha1 + structural checks),
// scipy cKDTree cross-checks for k-NN, and byte-exact PLY round trips.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
// this library; the product (object-triggered-3d-slam_b200/) never does.
//
// Build: see oracle/Makefile (g++ -O2 -fopenmp -ffp-contract=off; x86-64 baseline = no FMA, which is
// what a manylinux Open3D wheel does numerically).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "mc_tables.h"

namespace {

thread_local std::string g_err;
int fail(const char* msg) { g_err = msg; return -1; }

constexpr int RES = 16;            // volume_unit_resolution default (SURVEY A.3)
constexpr int NVOX = RES * RES * RES;

struct Key {
    int x, y, z;
    bool operator==(const Key& o) const { return x == o.x && y == o.y && z == o.z; }
    bool operator<(const Key& o) const {
        if (x != o.x) return x < o.x;
        if (y != o.y) return y < o.y;
        return z < o.z;
    }
};
struct KeyHash {
    size_t operator()(const Key& k) const {
        uint64_t h = (uint64_t)(uint32_t)k.x * 0x9E3779B97F4A7C15ull;
        h ^= (uint64_t)(uint32_t)k.y * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2);
        h ^= (uint64_t)(uint32_t)k.z * 0x165667B19E3779F9ull + (h << 6) + (h >> 2);
        return (size_t)h;
    }
};

// One 16^3 volume unit.  Voxel index = x*256 + y*16 + z (SURVEY A.4).
struct Block {
    Key key;
    std::vector<float> tsdf, weight;
    std::vector<double> color;  // 3 per voxel, 0..255 scale, FP64 running mean (A.4)
    explicit Block(Key k) : key(k), tsdf(NVOX, 0.f), weight(NVOX, 0.f), color(3 * NVOX, 0.0) {}
};

struct Volume {
    double voxel_length, sdf_trunc, unit_length;
    int stride = 4;
    // slab sharding (SURVEY 8e); n_ranks==1 -> keep everything
    int slab_axis = 0, slab_thickness = 8, slab_ranks = 1, slab_rank = 0, slab_halo = 1;
    std::unordered_map<Key, Block*, KeyHash> blocks;
    ~Volume() { for (auto& kv : blocks) delete kv.second; }
};

inline int floordiv(int a, int b) { int q = a / b, r = a % b; return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q; }
inline int slab_owner(const Volume* v, int k) {
    int m = floordiv(k, v->slab_thickness) % v->slab_ranks;
    return m < 0 ? m + v->slab_ranks : m;
}
// ownership coordinate: a block axis, or kx + ky for axis 3 (diagonal slabs)
inline int key_axis(const Key& k, int axis) { return axis == 0 ? k.x : (axis == 1 ? k.y : (axis == 2 ? k.z : k.x + k.y)); }
// a rank keeps the blocks it owns plus a one-block halo on the +axis side (the +1 neighbours of
// owned blocks), so extraction never needs another rank's voxels.
inline bool slab_keeps(const Volume* v, const Key& k) {
    if (v->slab_ranks <= 1) return true;
    int a = key_axis(k, v->slab_axis);
    // slab_halo == 0: integrate owned blocks only; the boundary planes are exchanged before extraction
    return slab_owner(v, a) == v->slab_rank || (v->slab_halo && slab_owner(v, a - 1) == v->slab_rank);
}
inline bool slab_owns(const Volume* v, const Key& k) {
    if (v->slab_ranks <= 1) return true;
    return slab_owner(v, key_axis(k, v->slab_axis)) == v->slab_rank;
}

// General 4x4 inverse by cofactors (FP64, row-major).  Open3D inverts the extrinsic with Eigen; the
// exact Eigen instruction order is not reproducible here, so this routine DEFINES camera_pose for
// both the oracle and the product (SURVEY 7.2 "Allocation is FP64 and uses inv(extrinsic)").
bool inverse4(const double* m, double* o) {
    double a00 = m[0], a01 = m[1], a02 = m[2], a03 = m[3], a10 = m[4], a11 = m[5], a12 = m[6], a13 = m[7],
           a20 = m[8], a21 = m[9], a22 = m[10], a23 = m[11], a30 = m[12], a31 = m[13], a32 = m[14], a33 = m[15];
    double b00 = a00 * a11 - a01 * a10, b01 = a00 * a12 - a02 * a10, b02 = a00 * a13 - a03 * a10,
           b03 = a01 * a12 - a02 * a11, b04 = a01 * a13 - a03 * a11, b05 = a02 * a13 - a03 * a12,
           b06 = a20 * a31 - a21 * a30, b07 = a20 * a32 - a22 * a30, b08 = a20 * a33 - a23 * a30,
           b09 = a21 * a32 - a22 * a31, b10 = a21 * a33 - a23 * a31, b11 = a22 * a33 - a23 * a32;
    double det = b00 * b11 - b01 * b10 + b02 * b09 + b03 * b08 - b04 * b07 + b05 * b06;
    if (det == 0.0 || !std::isfinite(det)) return false;
    double id = 1.0 / det;
    o[0] = (a11 * b11 - a12 * b10 + a13 * b09) * id;
    o[1] = (a02 * b10 - a01 * b11 - a03 * b09) * id;
    o[2] = (a31 * b05 - a32 * b04 + a33 * b03) * id;
    o[3] = (a22 * b04 - a21 * b05 - a23 * b03) * id;
    o[4] = (a12 * b08 - a10 * b11 - a13 * b07) * id;
    o[5] = (a00 * b11 - a02 * b08 + a03 * b07) * id;
    o[6] = (a32 * b02 - a30 * b05 - a33 * b01) * id;
    o[7] = (a20 * b05 - a22 * b02 + a23 * b01) * id;
    o[8] = (a10 * b10 - a11 * b08 + a13 * b06) * id;
    o[9] = (a01 * b08 - a00 * b10 - a03 * b06) * id;
    o[10] = (a30 * b04 - a31 * b02 + a33 * b00) * id;
    o[11] = (a21 * b02 - a20 * b04 - a23 * b00) * id;
    o[12] = (a11 * b07 - a10 * b09 - a12 * b06) * id;
    o[13] = (a00 * b09 - a01 * b07 + a02 * b06) * id;
    o[14] = (a31 * b01 - a30 * b03 - a32 * b00) * id;
    o[15] = (a20 * b03 - a21 * b01 + a22 * b00) * id;
    return true;
}

// FP64 pinhole back-projection of pixel (i=row, j=col) at depth d followed by the camera->world
// transform (SURVEY A.3 / A.12).  Product order: ((c0*x + c1*y) + c2*z) + c3.
inline void backproject(const double* pose, double fx, double fy, double cx, double cy, int i, int j, float d,
                        double* P) {
    double z = (double)d;
    double x = ((double)j - cx) * z / fx;
    double y = ((double)i - cy) * z / fy;
    for (int r = 0; r < 3; ++r)
        P[r] = ((pose[4 * r + 0] * x + pose[4 * r + 1] * y) + pose[4 * r + 2] * z) + pose[4 * r + 3];
}

// SURVEY A.4: per-block projective integration (UniformTSDFVolume::IntegrateWithDepthToCamera-
// DistanceMultiplier as reached from volume.integrate, reconstruct_rgbd.py:107).  Returns the
// number of voxels whose weight increased.
int64_t integrate_block(Block* b, const Volume* v, const float* depth, const uint8_t* rgb, const float* mult, int W,
                        int H, const float* E /*row-major 4x4 f32*/, float fx, float fy, float cx, float cy) {
    const float vl = (float)v->voxel_length;
    const float half = vl * 0.5f;
    const float trunc = (float)v->sdf_trunc;
    const float trunc_inv = 1.0f / trunc;
    const float neg_trunc = -trunc;
    const float safe_w = (float)W - 0.0001f, safe_h = (float)H - 0.0001f;
    const double ox = (double)b->key.x * v->unit_length, oy = (double)b->key.y * v->unit_length,
                 oz = (double)b->key.z * v->unit_length;
    const float esx = E[2] * vl, esy = E[6] * vl, esz = E[10] * vl;  // (E*vl).col(2)
    int64_t nupd = 0;
    for (int x = 0; x < RES; ++x) {
        for (int y = 0; y < RES; ++y) {
            float px = (float)((double)(half + vl * (float)x) + ox);
            float py = (float)((double)(half + vl * (float)y) + oy);
            float pz = (float)((double)half + oz);
            float pcx = ((E[0] * px + E[1] * py) + E[2] * pz) + E[3];
            float pcy = ((E[4] * px + E[5] * py) + E[6] * pz) + E[7];
            float pcz = ((E[8] * px + E[9] * py) + E[10] * pz) + E[11];
            for (int z = 0; z < RES; ++z, pcx += esx, pcy += esy, pcz += esz) {
                if (pcz <= 0.f) continue;
                float u_f = pcx * fx / pcz + cx + 0.5f;
                float v_f = pcy * fy / pcz + cy + 0.5f;
                if (!(u_f >= 0.0001f && u_f < safe_w && v_f >= 0.0001f && v_f < safe_h)) continue;
                int u = (int)u_f, vv = (int)v_f;
                float d = depth[(size_t)vv * W + u];
                if (d <= 0.f) continue;
                float sdf = (d - pcz) * mult[(size_t)vv * W + u];
                if (sdf > neg_trunc) {
                    float t = std::min(1.0f, sdf * trunc_inv);
                    int idx = x * 256 + y * 16 + z;
                    float w = b->weight[idx];
                    float w1 = w + 1.0f;
                    b->tsdf[idx] = (b->tsdf[idx] * w + t) / w1;
                    const uint8_t* c = rgb + ((size_t)vv * W + u) * 3;
                    for (int k = 0; k < 3; ++k)
                        b->color[3 * idx + k] = (b->color[3 * idx + k] * (double)w + (double)c[k]) / (double)w1;
                    b->weight[idx] = w1;
                    ++nupd;
                }
            }
        }
    }
    return nupd;
}

// look up voxel at global voxel coordinate (gx,gy,gz); returns false if its block is absent
struct VoxRef { float tsdf, weight; const double* color; };
inline bool fetch(const Volume* v, int gx, int gy, int gz, VoxRef* out) {
    Key k{floordiv(gx, RES), floordiv(gy, RES), floordiv(gz, RES)};
    auto it = v->blocks.find(k);
    if (it == v->blocks.end()) return false;
    int lx = gx - k.x * RES, ly = gy - k.y * RES, lz = gz - k.z * RES;
    int idx = lx * 256 + ly * 16 + lz;
    out->tsdf = it->second->tsdf[idx];
    out->weight = it->second->weight[idx];
    out->color = &it->second->color[3 * idx];
    return true;
}

std::vector<Block*> sorted_blocks(const Volume* v) {
    std::vector<Block*> bl;
    bl.reserve(v->blocks.size());
    for (auto& kv : v->blocks) bl.push_back(kv.second);
    std::sort(bl.begin(), bl.end(), [](Block* a, Block* b) { return a->key < b->key; });
    return bl;
}

struct Key4 {
    int x, y, z, a;
    bool operator==(const Key4& o) const { return x == o.x && y == o.y && z == o.z && a == o.a; }
};
struct Key4Hash {
    size_t operator()(const Key4& k) const {
        uint64_t h = (uint64_t)(uint32_t)k.x * 0x9E3779B97F4A7C15ull;
        h ^= (uint64_t)(uint32_t)k.y * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2);
        h ^= (uint64_t)(uint32_t)k.z * 0x165667B19E3779F9ull + (h << 6) + (h >> 2);
        h ^= (uint64_t)(uint32_t)k.a * 0x27D4EB2F165667C5ull + (h << 6) + (h >> 2);
        return (size_t)h;
    }
};

struct Mesh {
    std::vector<double> verts, colors;  // 3 per vertex
    std::vector<int32_t> edge_keys;     // 4 per vertex: global voxel (X,Y,Z) + axis
    std::vector<int32_t> faces;         // 3 per face
};

// counter-based uniform RNG shared by oracle and product so that sampled clouds are comparable
// point by point (Open3D itself draws from an unseeded mt19937, SURVEY A.10).
inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
inline double u01(uint64_t seed, uint64_t ctr) {
    return (double)(splitmix64(seed * 0xD1342543DE82EF95ull + ctr) >> 11) * (1.0 / 9007199254740992.0);
}

}  // namespace

extern "C" {

const char* oracle_last_error() { return g_err.c_str(); }

int oracle_num_threads() {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

// bench.py's reference arm runs under torchrun, which exports OMP_NUM_THREADS=1 to every rank: the
// CPU baseline must use the host cores it was told to use, not the inherited setting.
int oracle_set_num_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
    return omp_get_max_threads();
#else
    return 1;
#endif
}

int oracle_inverse4(const double* m, double* out) { return inverse4(m, out) ? 0 : fail("singular matrix"); }

// SURVEY A.1: RGBDImage.create_from_color_and_depth(depth_scale, depth_trunc,
// convert_rgb_to_intensity=False) (reconstruct_rgbd.py:99-104): u16 -> f32, /scale, >= trunc -> 0.
int oracle_depth_convert(const uint16_t* depth, int64_t n, double depth_scale, double depth_trunc, float* out) {
    const float s = (float)depth_scale;
    for (int64_t i = 0; i < n; ++i) {
        float d = (float)depth[i];
        d /= s;
        if ((double)d >= depth_trunc) d = 0.f;
        out[i] = d;
    }
    return 0;
}

void* oracle_volume_create(double voxel_length, double sdf_trunc) {
    if (!(voxel_length > 0) || !(sdf_trunc > 0)) { fail("voxel_length and sdf_trunc must be > 0"); return nullptr; }
    Volume* v = new Volume();
    v->voxel_length = voxel_length;
    v->sdf_trunc = sdf_trunc;
    v->unit_length = voxel_length * RES;
    return v;
}
int oracle_volume_set_slab(void* h, int axis, int thickness, int n_ranks, int rank, int halo) {
    Volume* v = (Volume*)h;
    if (axis < 0 || axis > 3 || thickness < 1 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail("bad slab spec");
    if (axis == 3 && halo && n_ranks > 1) return fail("diagonal slabs need halo = 0");
    v->slab_axis = axis; v->slab_thickness = thickness; v->slab_ranks = n_ranks; v->slab_rank = rank; v->slab_halo = halo ? 1 : 0;
    return 0;
}

// Halo exchange for slab_halo == 0 (SURVEY 8e): the low-side boundary pieces (256 voxels each) of every owned
// block whose -axis neighbour belongs to another rank.  keys [n][4] = block key + piece kind: 0 / 1 / 2 = the
// plane x / y / z = 0 with voxel (u, w) = the two other axes in increasing order, 3 = the column x = y = 0
// (w = z; entries with u > 0 are zero).  Axis slabs send one plane; diagonal slabs (axis 3, coordinate
// kx + ky) send the x and y planes to the owner of coordinate a - 1 and the column to the owner of a - 2.
static void piece_coords(int kind, int u, int w, int c[3]) {
    if (kind == 3) { c[0] = 0; c[1] = 0; c[2] = w; return; }
    c[kind] = 0; c[(kind == 0) ? 1 : 0] = u; c[(kind == 2) ? 1 : 2] = w;
}
int64_t oracle_volume_halo_export(void* h, int32_t* keys, int32_t* dest, float* tsdf, float* weight, double* color) {
    Volume* v = (Volume*)h;
    int64_t n = 0;
    if (v->slab_ranks <= 1) return 0;
    auto emit = [&](Block* b, int kind, int d) {
        if (keys) {
            keys[4 * n] = b->key.x; keys[4 * n + 1] = b->key.y; keys[4 * n + 2] = b->key.z; keys[4 * n + 3] = kind;
            dest[n] = d;
            for (int u = 0; u < RES; ++u)
                for (int w = 0; w < RES; ++w) {
                    const int64_t o = n * 256 + u * 16 + w;
                    if (kind == 3 && u > 0) { tsdf[o] = 0.f; weight[o] = 0.f; color[3 * o] = color[3 * o + 1] = color[3 * o + 2] = 0.0; continue; }
                    int c[3];
                    piece_coords(kind, u, w, c);
                    const int idx = c[0] * 256 + c[1] * 16 + c[2];
                    tsdf[o] = b->tsdf[idx]; weight[o] = b->weight[idx];
                    for (int k = 0; k < 3; ++k) color[3 * o + k] = b->color[3 * idx + k];
                }
        }
        ++n;
    };
    for (Block* b : sorted_blocks(v)) {
        if (!slab_owns(v, b->key)) continue;
        const int a = key_axis(b->key, v->slab_axis);
        const int d1 = slab_owner(v, a - 1);
        if (v->slab_axis < 3) {
            if (d1 != v->slab_rank) emit(b, v->slab_axis, d1);
        } else {
            if (d1 != v->slab_rank) { emit(b, 0, d1); emit(b, 1, d1); }
            const int d2 = slab_owner(v, a - 2);
            if (d2 != v->slab_rank && d2 != d1) emit(b, 3, d2);
        }
    }
    return n;
}
int oracle_volume_halo_import(void* h, int64_t n, const int32_t* keys, const float* tsdf, const float* weight, const double* color) {
    Volume* v = (Volume*)h;
    for (int64_t i = 0; i < n; ++i) {
        Key k{keys[4 * i], keys[4 * i + 1], keys[4 * i + 2]};
        const int kind = keys[4 * i + 3];
        auto it = v->blocks.find(k);
        if (it == v->blocks.end()) it = v->blocks.emplace(k, new Block(k)).first;
        Block* b = it->second;
        for (int u = 0; u < (kind == 3 ? 1 : RES); ++u)
            for (int w = 0; w < RES; ++w) {
                int c[3];
                piece_coords(kind, u, w, c);
                const int idx = c[0] * 256 + c[1] * 16 + c[2];
                const int64_t o = i * 256 + u * 16 + w;
                b->tsdf[idx] = tsdf[o]; b->weight[idx] = weight[o];
                for (int kk = 0; kk < 3; ++kk) b->color[3 * idx + kk] = color[3 * o + kk];
            }
    }
    return 0;
}
// Whole blocks as export_blocks gives them (keys [n][3], tsdf / weight [n][4096], colour [n][4096][3] on the 0..255 scale;
// voxel index x*256 + y*16 + z): a block already present is overwritten.  Extraction, point normals and the ray-cast and
// tracking models then have a CPU reference for any block set, including keys no camera would reach.
int oracle_volume_import_blocks(void* h, int64_t n, const int32_t* keys, const float* tsdf, const float* weight, const double* color) {
    Volume* v = (Volume*)h;
    for (int64_t i = 0; i < n; ++i) {
        Key k{keys[3 * i], keys[3 * i + 1], keys[3 * i + 2]};
        auto it = v->blocks.find(k);
        if (it == v->blocks.end()) it = v->blocks.emplace(k, new Block(k)).first;
        Block* b = it->second;
        memcpy(b->tsdf.data(), tsdf + i * NVOX, NVOX * sizeof(float));
        memcpy(b->weight.data(), weight + i * NVOX, NVOX * sizeof(float));
        memcpy(b->color.data(), color + i * 3 * NVOX, 3 * NVOX * sizeof(double));
    }
    return 0;
}
void oracle_volume_destroy(void* h) { delete (Volume*)h; }
void oracle_volume_reset(void* h) {
    Volume* v = (Volume*)h;
    for (auto& kv : v->blocks) delete kv.second;
    v->blocks.clear();
}

// SURVEY A.2-A.4: ScalableTSDFVolume::Integrate (reconstruct_rgbd.py:107).  depth is the f32 metre
// image produced by A.1, rgb is RGB8, extrinsic is world->camera row-major FP64.
// n_touched / n_updated (nullable) receive the per-frame touched-block and updated-voxel counts.
int oracle_volume_integrate(void* h, const float* depth, const uint8_t* rgb, int W, int H, double fx, double fy,
                            double cx, double cy, const double* extrinsic, int64_t* n_touched, int64_t* n_updated) {
    Volume* v = (Volume*)h;
    if (!depth || !rgb || W <= 0 || H <= 0) return fail("[ScalableTSDFVolume::Integrate] Unsupported image format.");
    double pose[16];
    if (!inverse4(extrinsic, pose)) return fail("extrinsic is singular");
    // A.2 multiplier image, recomputed per call like the reference backend does
    std::vector<float> mult((size_t)W * H);
    {
        const float ix = 1.0f / (float)fx, iy = 1.0f / (float)fy, px = (float)cx, py = (float)cy;
        std::vector<float> xx(W), yy(H);
        for (int j = 0; j < W; ++j) xx[j] = ((float)j - px) * ix;
        for (int i = 0; i < H; ++i) yy[i] = ((float)i - py) * iy;
#pragma omp parallel for schedule(static)
        for (int i = 0; i < H; ++i)
            for (int j = 0; j < W; ++j) mult[(size_t)i * W + j] = sqrtf(xx[j] * xx[j] + yy[i] * yy[i] + 1.0f);
    }
    // A.3 allocation: stride-4 FP64 back-projection, +-trunc box -> unit keys
    std::vector<Block*> touched;
    {
        std::unordered_map<Key, char, KeyHash> seen;
        for (int i = 0; i < H; i += v->stride) {
            for (int j = 0; j < W; j += v->stride) {
                float d = depth[(size_t)i * W + j];
                if (!(d > 0.f)) continue;
                double P[3];
                backproject(pose, fx, fy, cx, cy, i, j, d, P);
                int lo[3], hi[3];
                for (int a = 0; a < 3; ++a) {
                    lo[a] = (int)std::floor((P[a] - v->sdf_trunc) / v->unit_length);
                    hi[a] = (int)std::floor((P[a] + v->sdf_trunc) / v->unit_length);
                }
                for (int kx = lo[0]; kx <= hi[0]; ++kx)
                    for (int ky = lo[1]; ky <= hi[1]; ++ky)
                        for (int kz = lo[2]; kz <= hi[2]; ++kz) {
                            Key k{kx, ky, kz};
                            if (!slab_keeps(v, k)) continue;
                            if (seen.emplace(k, 1).second) {
                                auto it = v->blocks.find(k);
                                if (it == v->blocks.end()) it = v->blocks.emplace(k, new Block(k)).first;
                                touched.push_back(it->second);
                            }
                        }
            }
        }
    }
    // A.4 per-block integration (blocks are independent, so parallelise across them)
    float E[16];
    for (int i = 0; i < 16; ++i) E[i] = (float)extrinsic[i];
    int64_t nupd = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : nupd)
    for (size_t t = 0; t < touched.size(); ++t)
        nupd += integrate_block(touched[t], v, depth, rgb, mult.data(), W, H, E, (float)fx, (float)fy, (float)cx,
                                (float)cy);
    if (n_touched) *n_touched = (int64_t)touched.size();
    if (n_updated) *n_updated = nupd;
    return 0;
}

int64_t oracle_volume_num_blocks(void* h) { return (int64_t)((Volume*)h)->blocks.size(); }

// blocks sorted lexicographically by key; voxel index x*256+y*16+z; colour on the 0..255 scale
int oracle_volume_export_blocks(void* h, int32_t* keys, float* tsdf, float* weight, double* color) {
    Volume* v = (Volume*)h;
    auto bl = sorted_blocks(v);
    for (size_t i = 0; i < bl.size(); ++i) {
        if (keys) { keys[3 * i] = bl[i]->key.x; keys[3 * i + 1] = bl[i]->key.y; keys[3 * i + 2] = bl[i]->key.z; }
        if (tsdf) memcpy(tsdf + i * NVOX, bl[i]->tsdf.data(), NVOX * sizeof(float));
        if (weight) memcpy(weight + i * NVOX, bl[i]->weight.data(), NVOX * sizeof(float));
        if (color) memcpy(color + i * 3 * NVOX, bl[i]->color.data(), 3 * NVOX * sizeof(double));
    }
    return 0;
}

// SURVEY A.5: ScalableTSDFVolume::ExtractTriangleMesh (reconstruct_rgbd.py:112).  Blocks are
// visited in sorted-key order (Open3D: hash order; callers canonicalise).  With slab sharding only
// cubes whose base voxel lies in an owned block are emitted.
void* oracle_volume_extract_mesh(void* h, int64_t* nv, int64_t* nf) {
    Volume* v = (Volume*)h;
    Mesh* m = new Mesh();
    std::unordered_map<Key4, int, Key4Hash> edge2vert;
    const double vl = v->voxel_length, half = 0.5 * vl;
    for (Block* b : sorted_blocks(v)) {
        if (!slab_owns(v, b->key)) continue;
        for (int x = 0; x < RES; ++x)
            for (int y = 0; y < RES; ++y)
                for (int z = 0; z < RES; ++z) {
                    int gx = b->key.x * RES + x, gy = b->key.y * RES + y, gz = b->key.z * RES + z;
                    float f[8];
                    double c[8][3];
                    int cube = 0;
                    bool ok = true;
                    for (int i = 0; i < 8 && ok; ++i) {
                        VoxRef r;
                        if (!fetch(v, gx + MC_SHIFT[i][0], gy + MC_SHIFT[i][1], gz + MC_SHIFT[i][2], &r) || r.weight == 0.f) {
                            ok = false;
                            break;
                        }
                        f[i] = r.tsdf;
                        if (f[i] < 0.f) cube |= 1 << i;
                        for (int k = 0; k < 3; ++k) c[i][k] = r.color[k] / 255.0;
                    }
                    if (!ok || cube == 0 || cube == 255) continue;
                    int ev[12];
                    for (int e = 0; e < 12; ++e) {
                        if (!(MC_EDGE_TABLE[cube] & (1 << e))) continue;
                        Key4 K{gx + MC_EDGE_SHIFT[e][0], gy + MC_EDGE_SHIFT[e][1], gz + MC_EDGE_SHIFT[e][2],
                               MC_EDGE_SHIFT[e][3]};
                        auto it = edge2vert.find(K);
                        if (it != edge2vert.end()) { ev[e] = it->second; continue; }
                        int a = MC_EDGE_TO_VERT[e][0], bb = MC_EDGE_TO_VERT[e][1];
                        double f0 = std::fabs((double)f[a]), f1 = std::fabs((double)f[bb]);
                        double pt[3] = {half + vl * (double)K.x, half + vl * (double)K.y, half + vl * (double)K.z};
                        pt[K.a] += f0 * vl / (f0 + f1);
                        int id = (int)(m->verts.size() / 3);
                        for (int k = 0; k < 3; ++k) {
                            m->verts.push_back(pt[k]);
                            m->colors.push_back((f1 * c[a][k] + f0 * c[bb][k]) / (f0 + f1));
                        }
                        m->edge_keys.insert(m->edge_keys.end(), {K.x, K.y, K.z, K.a});
                        edge2vert.emplace(K, id);
                        ev[e] = id;
                    }
                    for (int i = 0; MC_TRI_TABLE[cube][i] != -1; i += 3) {
                        m->faces.push_back(ev[MC_TRI_TABLE[cube][i]]);
                        m->faces.push_back(ev[MC_TRI_TABLE[cube][i + 2]]);  // winding swapped (A.5)
                        m->faces.push_back(ev[MC_TRI_TABLE[cube][i + 1]]);
                    }
                }
    }
    *nv = (int64_t)(m->verts.size() / 3);
    *nf = (int64_t)(m->faces.size() / 3);
    return m;
}
void oracle_mesh_copy(void* mh, double* verts, double* colors, int32_t* faces, int32_t* edge_keys) {
    Mesh* m = (Mesh*)mh;
    if (verts) memcpy(verts, m->verts.data(), m->verts.size() * sizeof(double));
    if (colors) memcpy(colors, m->colors.data(), m->colors.size() * sizeof(double));
    if (faces) memcpy(faces, m->faces.data(), m->faces.size() * sizeof(int32_t));
    if (edge_keys) memcpy(edge_keys, m->edge_keys.data(), m->edge_keys.size() * sizeof(int32_t));
}
void oracle_mesh_free(void* mh) { delete (Mesh*)mh; }

// SURVEY A.6: ScalableTSDFVolume::ExtractPointCloud (named by north_star; not called by the
// scripts).  Per voxel, +x/+y/+z zero crossings; missing neighbour block == unobserved.
// Output arrays sized by a first call with pts==nullptr.  Arithmetic as Open3D's ScalableTSDFVolume::ExtractPointCloud
// does it (ADVICE r1): r0 = |f0|, r1 = |f1| and their sum are FP32; the voxel centre is
// (half + vl * x_local) + block_index * unit_length in FP64; colours are interpolated in FP32 from the float-cast voxel
// colours and divided by 255.0f.  Normals: oracle_volume_point_normals.
int64_t oracle_volume_extract_points(void* h, double* pts, double* cols, int32_t* edge_keys) {
    Volume* v = (Volume*)h;
    const double vl = v->voxel_length, half = 0.5 * vl, unit = v->voxel_length * RES;
    int64_t n = 0;
    for (Block* b : sorted_blocks(v)) {
        if (!slab_owns(v, b->key)) continue;
        for (int x = 0; x < RES; ++x)
            for (int y = 0; y < RES; ++y)
                for (int z = 0; z < RES; ++z) {
                    int idx = x * 256 + y * 16 + z;
                    float w0 = b->weight[idx], f0 = b->tsdf[idx];
                    if (w0 == 0.f || !(f0 < 0.98f && f0 >= -0.98f)) continue;
                    int g[3] = {b->key.x * RES + x, b->key.y * RES + y, b->key.z * RES + z};
                    double p0[3] = {(half + vl * (double)x) + (double)b->key.x * unit, (half + vl * (double)y) + (double)b->key.y * unit,
                                    (half + vl * (double)z) + (double)b->key.z * unit};
                    for (int a = 0; a < 3; ++a) {
                        int q[3] = {g[0], g[1], g[2]};
                        q[a] += 1;
                        VoxRef r;
                        if (!fetch(v, q[0], q[1], q[2], &r)) continue;
                        float w1 = r.weight, f1 = r.tsdf;
                        if (w1 == 0.f || !(f1 < 0.98f && f1 >= -0.98f) || !(f0 * f1 < 0.f)) continue;
                        const float r0 = std::fabs(f0), r1 = std::fabs(f1);
                        const float rs = r0 + r1;
                        if (pts) {
                            double p[3] = {p0[0], p0[1], p0[2]};
                            double p1a = p0[a] + vl;
                            p[a] = (p0[a] * (double)r1 + p1a * (double)r0) / (double)rs;
                            for (int k = 0; k < 3; ++k) {
                                pts[3 * n + k] = p[k];
                                const float c0 = (float)b->color[3 * idx + k], c1 = (float)r.color[k];
                                cols[3 * n + k] = (double)(((c0 * r1 + c1 * r0) / rs) / 255.0f);
                            }
                            if (edge_keys) { edge_keys[4 * n] = g[0]; edge_keys[4 * n + 1] = g[1]; edge_keys[4 * n + 2] = g[2]; edge_keys[4 * n + 3] = a; }
                        }
                        ++n;
                    }
                }
    }
    return n;
}

// ScalableTSDFVolume::GetTSDFAt: trilinear interpolation of the TSDF at a world point; voxels of absent blocks read 0,
// observed or not does not matter (Open3D ignores the weight here).
static double tsdf_at(const Volume* v, const double p[3]) {
    const double vl = v->voxel_length, unit = v->voxel_length * RES;
    double pl[3], pg[3], r[3];
    int index0[3], idx0[3];
    for (int i = 0; i < 3; ++i) {
        pl[i] = p[i] - 0.5 * vl;
        index0[i] = (int)std::floor(pl[i] / unit);
    }
    if (v->blocks.find(Key{index0[0], index0[1], index0[2]}) == v->blocks.end()) return 0.0;
    for (int i = 0; i < 3; ++i) {
        pg[i] = (pl[i] - (double)index0[i] * unit) / vl;
        idx0[i] = (int)std::floor(pg[i]);
        if (idx0[i] < 0) idx0[i] = 0;
        if (idx0[i] >= RES) idx0[i] = RES - 1;
        r[i] = pg[i] - (double)idx0[i];
    }
    float f[8];
    for (int q = 0; q < 8; ++q) {
        const int sx = (q ^ (q >> 1)) & 1, sy = (q >> 1) & 1, sz = (q >> 2) & 1;     // SURVEY Appendix B corner order
        VoxRef ref;
        f[q] = fetch(v, index0[0] * RES + idx0[0] + sx, index0[1] * RES + idx0[1] + sy, index0[2] * RES + idx0[2] + sz, &ref) ? ref.tsdf : 0.f;
    }
    return (1 - r[0]) * ((1 - r[1]) * ((1 - r[2]) * f[0] + r[2] * f[4]) + r[1] * ((1 - r[2]) * f[3] + r[2] * f[7])) +
           r[0] * ((1 - r[1]) * ((1 - r[2]) * f[1] + r[2] * f[5]) + r[1] * ((1 - r[2]) * f[2] + r[2] * f[6]));
}

// ScalableTSDFVolume::GetNormalAt for n points: central TSDF differences at +-0.99 voxel, normalised (zero stays zero)
int oracle_volume_point_normals(void* h, const double* pts, int64_t n, double* normals) {
    Volume* v = (Volume*)h;
    const double gap = 0.99 * v->voxel_length;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; ++i) {
        double g[3];
        for (int a = 0; a < 3; ++a) {
            double p0[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]}, p1[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
            p0[a] -= gap;
            p1[a] += gap;
            g[a] = tsdf_at(v, p1) - tsdf_at(v, p0);
        }
        const double l = std::sqrt((g[0] * g[0] + g[1] * g[1]) + g[2] * g[2]);
        for (int a = 0; a < 3; ++a) normals[3 * i + a] = l > 0.0 ? g[a] / l : g[a];
    }
    return 0;
}

// SURVEY A.9: TriangleMesh.compute_vertex_normals (reconstruct_rgbd.py:113): un-normalised
// (area-weighted) face normals summed per vertex in face order, then normalised; zero -> (0,0,1).
int oracle_vertex_normals(const double* verts, int64_t nv, const int32_t* faces, int64_t nf, double* normals) {
    std::fill(normals, normals + 3 * nv, 0.0);
    for (int64_t t = 0; t < nf; ++t) {
        const int32_t* f = faces + 3 * t;
        const double *a = verts + 3 * f[0], *b = verts + 3 * f[1], *c = verts + 3 * f[2];
        double e1[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, e2[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
        double n[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        for (int k = 0; k < 3; ++k)
            for (int j = 0; j < 3; ++j) normals[3 * f[k] + j] += n[j];
    }
    for (int64_t i = 0; i < nv; ++i) {
        double* n = normals + 3 * i;
        double l = std::sqrt((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]);
        if (l > 0.0) { n[0] /= l; n[1] /= l; n[2] /= l; } else { n[0] = 0; n[1] = 0; n[2] = 1; }
    }
    return 0;
}

// SURVEY A.10: TriangleMesh.sample_points_uniformly (reconstruct_rgbd_filter.py:123).  Sequential
// area CDF; triangle t owns samples [round(cdf[t-1]*n), round(cdf[t]*n)); barycentric weights from
// the shared counter RNG.  tri_of (nullable) receives the triangle of each sample.
int oracle_sample_uniform(const double* verts, const double* colors, const double* normals, int64_t nv,
                          const int32_t* faces, int64_t nf, int64_t n, uint64_t seed, double* out_pts,
                          double* out_cols, double* out_normals, int32_t* tri_of) {
    (void)nv;
    if (n <= 0) return fail("number_of_points <= 0");
    if (nf <= 0) return fail("input mesh has no triangles");
    std::vector<double> cdf(nf);
    double total = 0.0;
    for (int64_t t = 0; t < nf; ++t) {
        const int32_t* f = faces + 3 * t;
        const double *a = verts + 3 * f[0], *b = verts + 3 * f[1], *c = verts + 3 * f[2];
        double e1[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, e2[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
        double x[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        double area = 0.5 * std::sqrt((x[0] * x[0] + x[1] * x[1]) + x[2] * x[2]);
        cdf[t] = area;
        total += area;
    }
    cdf[0] /= total;
    for (int64_t t = 1; t < nf; ++t) cdf[t] = cdf[t] / total + cdf[t - 1];
    int64_t idx = 0;
    for (int64_t t = 0; t < nf; ++t) {
        int64_t end = (int64_t)std::llround(cdf[t] * (double)n);
        if (t == nf - 1) end = n;
        const int32_t* f = faces + 3 * t;
        for (; idx < end && idx < n; ++idx) {
            double r1 = u01(seed, 2 * (uint64_t)idx), r2 = u01(seed, 2 * (uint64_t)idx + 1);
            double s = std::sqrt(r1);
            double a = 1.0 - s, b = s * (1.0 - r2), c = s * r2;
            for (int k = 0; k < 3; ++k) {
                out_pts[3 * idx + k] = (a * verts[3 * f[0] + k] + b * verts[3 * f[1] + k]) + c * verts[3 * f[2] + k];
                if (colors && out_cols)
                    out_cols[3 * idx + k] = (a * colors[3 * f[0] + k] + b * colors[3 * f[1] + k]) + c * colors[3 * f[2] + k];
                if (normals && out_normals)
                    out_normals[3 * idx + k] = (a * normals[3 * f[0] + k] + b * normals[3 * f[1] + k]) + c * normals[3 * f[2] + k];
            }
            if (tri_of) tri_of[idx] = (int32_t)t;
        }
    }
    return 0;
}

// reconstruct_rgbd_filter.py:126-132: mask = points[:,2] >= zmin, order-preserving rebuild.
int64_t oracle_zfilter(const double* pts, const double* cols, int64_t n, double zmin, double* out_pts, double* out_cols) {
    int64_t m = 0;
    for (int64_t i = 0; i < n; ++i)
        if (pts[3 * i + 2] >= zmin) {
            for (int k = 0; k < 3; ++k) { out_pts[3 * m + k] = pts[3 * i + k]; if (cols) out_cols[3 * m + k] = cols[3 * i + k]; }
            ++m;
        }
    return m;
}

// SURVEY 8(f) row 4 -- the rigid-body edits of fusion/hybrid_map_manual.py:86-119.
// PointCloud.transform(T) (:87): p' = (T * [p, 1]).head<3>() / w; normals rotate with T's 3x3 block.
// The FP64 product order is defined here as ((m0*x + m1*y) + m2*z) + m3 (Open3D leaves it to Eigen; same
// convention as the integration's extrinsic product).
void oracle_transform(const double* pts, const double* nrm, int64_t n, const double* T, double* out_pts, double* out_nrm) {
    for (int64_t i = 0; i < n; ++i) {
        const double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
        double h[4];
        for (int r = 0; r < 4; ++r) h[r] = ((T[4 * r] * x + T[4 * r + 1] * y) + T[4 * r + 2] * z) + T[4 * r + 3];
        for (int r = 0; r < 3; ++r) out_pts[3 * i + r] = h[r] / h[3];
        if (nrm && out_nrm) {
            const double a = nrm[3 * i], b = nrm[3 * i + 1], c = nrm[3 * i + 2];
            for (int r = 0; r < 3; ++r) out_nrm[3 * i + r] = (T[4 * r] * a + T[4 * r + 1] * b) + T[4 * r + 2] * c;
        }
    }
}
// PointCloud.get_center() (:110): the mean, coordinates summed in index order.
void oracle_center(const double* pts, int64_t n, double* c) {
    double s[3] = {0, 0, 0};
    for (int64_t i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) s[k] += pts[3 * i + k];
    for (int k = 0; k < 3; ++k) c[k] = n > 0 ? s[k] / (double)n : 0.0;
}
// PointCloud.rotate(R, center) (:112): p' = R * (p - center) + center, normals' = R * n.
void oracle_rotate(const double* pts, const double* nrm, int64_t n, const double* R, const double* c, double* out_pts, double* out_nrm) {
    for (int64_t i = 0; i < n; ++i) {
        const double d[3] = {pts[3 * i] - c[0], pts[3 * i + 1] - c[1], pts[3 * i + 2] - c[2]};
        for (int r = 0; r < 3; ++r) out_pts[3 * i + r] = ((R[3 * r] * d[0] + R[3 * r + 1] * d[1]) + R[3 * r + 2] * d[2]) + c[r];
        if (nrm && out_nrm) {
            const double a = nrm[3 * i], b = nrm[3 * i + 1], cc = nrm[3 * i + 2];
            for (int r = 0; r < 3; ++r) out_nrm[3 * i + r] = (R[3 * r] * a + R[3 * r + 1] * b) + R[3 * r + 2] * cc;
        }
    }
}

// SURVEY A.12: PointCloud.create_from_rgbd_image (check_one_frame.py:27): dense FP64
// back-projection in row-major pixel order, colour/255.
int64_t oracle_backproject_rgbd(const float* depth, const uint8_t* rgb, int W, int H, double fx, double fy, double cx,
                                double cy, const double* extrinsic, double* pts, double* cols) {
    double pose[16];
    if (!inverse4(extrinsic, pose)) return fail("extrinsic is singular");
    int64_t n = 0;
    for (int i = 0; i < H; ++i)
        for (int j = 0; j < W; ++j) {
            float d = depth[(size_t)i * W + j];
            if (!(d > 0.f)) continue;
            backproject(pose, fx, fy, cx, cy, i, j, d, pts + 3 * n);
            if (rgb && cols)
                for (int k = 0; k < 3; ++k) cols[3 * n + k] = (double)rgb[((size_t)i * W + j) * 3 + k] / 255.0;
            ++n;
        }
    return n;
}

// SURVEY A.7: PointCloud.voxel_down_sample (check_one_frame.py:28).  Output sorted by voxel key
// (Open3D: hash order).  counts (nullable) = points per voxel, keys (nullable) = int32 xyz.
int64_t oracle_voxel_down_sample(const double* pts, const double* cols, int64_t n, double voxel, double* out_pts,
                                 double* out_cols, int32_t* out_keys, int32_t* out_counts) {
    if (!(voxel > 0.0)) return fail("voxel_size <= 0");
    if (n == 0) return 0;
    double mn[3] = {pts[0], pts[1], pts[2]}, mx[3] = {pts[0], pts[1], pts[2]};
    for (int64_t i = 1; i < n; ++i)
        for (int k = 0; k < 3; ++k) { mn[k] = std::min(mn[k], pts[3 * i + k]); mx[k] = std::max(mx[k], pts[3 * i + k]); }
    double vmin[3], vmaxv[3];
    for (int k = 0; k < 3; ++k) { vmin[k] = mn[k] - voxel * 0.5; vmaxv[k] = mx[k] + voxel * 0.5; }
    for (int k = 0; k < 3; ++k)
        if (voxel * 2147483647.0 < vmaxv[k] - vmin[k]) return fail("voxel_size is too small");
    struct Acc { double p[3], c[3]; int cnt; };
    std::unordered_map<Key, Acc, KeyHash> acc;
    for (int64_t i = 0; i < n; ++i) {
        Key k{(int)std::floor((pts[3 * i] - vmin[0]) / voxel), (int)std::floor((pts[3 * i + 1] - vmin[1]) / voxel),
              (int)std::floor((pts[3 * i + 2] - vmin[2]) / voxel)};
        auto it = acc.find(k);
        if (it == acc.end()) it = acc.emplace(k, Acc{{0, 0, 0}, {0, 0, 0}, 0}).first;
        for (int j = 0; j < 3; ++j) { it->second.p[j] += pts[3 * i + j]; if (cols) it->second.c[j] += cols[3 * i + j]; }
        it->second.cnt++;
    }
    std::vector<Key> keys;
    keys.reserve(acc.size());
    for (auto& kv : acc) keys.push_back(kv.first);
    std::sort(keys.begin(), keys.end());
    if (out_pts)
        for (size_t m = 0; m < keys.size(); ++m) {
            const Acc& a = acc[keys[m]];
            for (int j = 0; j < 3; ++j) { out_pts[3 * m + j] = a.p[j] / (double)a.cnt; if (cols && out_cols) out_cols[3 * m + j] = a.c[j] / (double)a.cnt; }
            if (out_keys) { out_keys[3 * m] = keys[m].x; out_keys[3 * m + 1] = keys[m].y; out_keys[3 * m + 2] = keys[m].z; }
            if (out_counts) out_counts[m] = a.cnt;
        }
    return (int64_t)keys.size();
}

// SURVEY A.8: PointCloud.remove_statistical_outlier (north_star; no reference call site).
// Exact FP64 k-NN (query point included), neighbours ascending, sequential mean / Bessel sigma.
// Uses a uniform-grid accelerated exact search (ring expansion); mean_dist (nullable) gets d-bar_i.
int64_t oracle_remove_statistical_outlier(const double* pts, int64_t n, int nb_neighbors, double std_ratio,
                                          int64_t* out_indices, double* mean_dist_out) {
    if (nb_neighbors < 1 || !(std_ratio > 0.0)) return fail("Illegal input parameters, the number of neighbors and standard deviation ratio must be positive.");
    if (n == 0) return 0;
    const int k = (int)std::min<int64_t>(nb_neighbors, n);
    double mn[3] = {pts[0], pts[1], pts[2]}, mx[3] = {pts[0], pts[1], pts[2]};
    for (int64_t i = 1; i < n; ++i)
        for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], pts[3 * i + a]); mx[a] = std::max(mx[a], pts[3 * i + a]); }
    // cell size: ~2 points per cell on average over the bounding box's occupied extent
    double ext[3] = {mx[0] - mn[0], mx[1] - mn[1], mx[2] - mn[2]};
    double vol = std::max(ext[0], 1e-9) * std::max(ext[1], 1e-9) * std::max(ext[2], 1e-9);
    double cell = std::cbrt(vol / std::max<double>(1.0, (double)n / 2.0));
    double maxext = std::max(ext[0], std::max(ext[1], ext[2]));
    cell = std::max(cell, maxext / 512.0);
    if (!(cell > 0.0)) cell = 1.0;
    int dim[3];
    for (int a = 0; a < 3; ++a) dim[a] = std::max(1, (int)std::floor(ext[a] / cell) + 1);
    auto cell_of = [&](const double* p, int* c) {
        for (int a = 0; a < 3; ++a) { int v = (int)std::floor((p[a] - mn[a]) / cell); c[a] = std::min(std::max(v, 0), dim[a] - 1); }
    };
    std::vector<int64_t> start((size_t)dim[0] * dim[1] * dim[2] + 1, 0);
    std::vector<int64_t> cid(n);
    for (int64_t i = 0; i < n; ++i) { int c[3]; cell_of(pts + 3 * i, c); cid[i] = ((int64_t)c[0] * dim[1] + c[1]) * dim[2] + c[2]; start[cid[i] + 1]++; }
    for (size_t c = 1; c < start.size(); ++c) start[c] += start[c - 1];
    std::vector<int64_t> order(n), fill(start.begin(), start.end() - 1);
    for (int64_t i = 0; i < n; ++i) order[fill[cid[i]]++] = i;
    std::vector<double> dbar(n);
#pragma omp parallel
    {
        std::vector<double> best;
#pragma omp for schedule(dynamic, 256)
        for (int64_t i = 0; i < n; ++i) {
            const double* q = pts + 3 * i;
            int c[3];
            cell_of(q, c);
            best.assign(k, INFINITY);  // max-heap of the k smallest squared distances
            int found = 0;
            int maxring = std::max(dim[0], std::max(dim[1], dim[2]));
            for (int ring = 0; ring <= maxring; ++ring) {
                // once k candidates are known and the ring's inner boundary is farther than the k-th, stop
                if (found >= k && ring >= 1) {
                    double reach = INFINITY;  // min distance from q to anything outside the (ring-1) shell box
                    for (int a = 0; a < 3; ++a) {
                        double lo = mn[a] + (double)(c[a] - (ring - 1)) * cell, hi = mn[a] + (double)(c[a] + ring) * cell;
                        if (c[a] - (ring - 1) > 0) reach = std::min(reach, q[a] - lo);
                        if (c[a] + ring < dim[a]) reach = std::min(reach, hi - q[a]);
                    }
                    if (reach == INFINITY) break;  // box covers the whole grid
                    if (reach > 0 && reach * reach > best[0]) break;
                }
                for (int x = c[0] - ring; x <= c[0] + ring; ++x) {
                    if (x < 0 || x >= dim[0]) continue;
                    for (int y = c[1] - ring; y <= c[1] + ring; ++y) {
                        if (y < 0 || y >= dim[1]) continue;
                        bool edge_xy = (x == c[0] - ring || x == c[0] + ring || y == c[1] - ring || y == c[1] + ring);
                        for (int z = c[2] - ring; z <= c[2] + ring; ++z) {
                            if (z < 0 || z >= dim[2]) continue;
                            if (!edge_xy && z != c[2] - ring && z != c[2] + ring) continue;  // shell only
                            int64_t cc = ((int64_t)x * dim[1] + y) * dim[2] + z;
                            for (int64_t s = start[cc]; s < start[cc + 1]; ++s) {
                                const double* p = pts + 3 * order[s];
                                double dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
                                double d2 = (dx * dx + dy * dy) + dz * dz;
                                if (found < k) {
                                    best[found++] = d2;
                                    if (found == k) std::make_heap(best.begin(), best.end());
                                } else if (d2 < best[0]) {
                                    std::pop_heap(best.begin(), best.end());
                                    best[k - 1] = d2;
                                    std::push_heap(best.begin(), best.end());
                                }
                            }
                        }
                    }
                }
            }
            std::sort(best.begin(), best.begin() + found);
            double s = 0.0;
            for (int j = 0; j < found; ++j) s += std::sqrt(best[j]);
            dbar[i] = found > 0 ? s / (double)found : -1.0;
        }
    }
    // sequential global statistics (index order)
    int64_t valid = 0;
    double sum = 0.0;
    for (int64_t i = 0; i < n; ++i) { if (dbar[i] > 0.0) { sum += dbar[i]; } if (dbar[i] >= 0.0) ++valid; }
    if (mean_dist_out) memcpy(mean_dist_out, dbar.data(), n * sizeof(double));
    if (valid == 0) return 0;
    double mean = sum / (double)valid, sq = 0.0;
    for (int64_t i = 0; i < n; ++i) if (dbar[i] > 0.0) sq += (dbar[i] - mean) * (dbar[i] - mean);
    double sd = valid > 1 ? std::sqrt(sq / (double)(valid - 1)) : 0.0;
    double thr = mean + std_ratio * sd;
    int64_t m = 0;
    for (int64_t i = 0; i < n; ++i) if (dbar[i] > 0.0 && dbar[i] < thr) out_indices[m++] = i;
    return m;
}

// fusion/hybrid_map.py:45-55: occupied pixels (< thresh) in row-major order ->
// (ox + c*res, oy + (h-1-r)*res, 0.0).
int64_t oracle_grid_to_points(const uint8_t* img, int w, int h, double res, double ox, double oy, int thresh, double* out) {
    int64_t n = 0;
    for (int r = 0; r < h; ++r)
        for (int c = 0; c < w; ++c)
            if ((int)img[(size_t)r * w + c] < thresh) {
                if (out) { out[3 * n] = ox + ((double)c * res); out[3 * n + 1] = oy + ((double)(h - 1 - r) * res); out[3 * n + 2] = 0.0; }
                ++n;
            }
    return n;
}

// SURVEY Appendix C: 27-byte binary PLY vertex records (3 x f64 + 3 x u8), colour byte =
// round(clamp(c,0,1)*255); used for fusion/hybrid_map.py:88-91,115,121 (paint + concat + write).
int oracle_pack_ply_cloud(const double* pts, const double* cols, int64_t n, uint8_t* out) {
    for (int64_t i = 0; i < n; ++i) {
        memcpy(out + 27 * i, pts + 3 * i, 24);
        for (int k = 0; k < 3; ++k) {
            double c = cols ? cols[3 * i + k] : 0.0;
            c = std::min(1.0, std::max(0.0, c));
            out[27 * i + 24 + k] = (uint8_t)std::floor(c * 255.0 + 0.5);
        }
    }
    return 0;
}

}  // extern "C"
