// raycast_model.cpp -- CPU restatement of the ray caster (DESIGN.md §4 "Ray casting"), the reference the CUDA kernel
// (object-triggered-3d-slam_b200/csrc/raycast.cu) is compared with bit for bit (colour: within one level).
//
// It reads a volume as the CPU oracle exports it (oracle.Volume.export_blocks: block keys, f32 TSDF, f32 weights, FP64
// running-mean colours on the 0..255 scale, voxel index x*256 + y*16 + z) and the camera poses as oracle.inverse4 gives
// them, so the voxels and poses are the oracle's own.  GetTSDFAt (tsdf_at) is restated with the oracle's arithmetic
// (oracle/oracle.cpp).  Compiled by tests/test_raycast_oracle.py with g++ -O2 -fopenmp -ffp-contract=off (no FMA).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <unordered_map>
#include <vector>

namespace {

constexpr int RES = 16;
constexpr int NVOX = RES * RES * RES;

inline int floordiv(int a, int b) { int q = a / b, r = a % b; return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q; }

struct Blocks {
    const int32_t* keys;
    const float *tsdf, *weight;
    const double* color;       // nullable
    double vl, unit;
    std::unordered_map<uint64_t, int64_t> index;
    static uint64_t pack(int x, int y, int z) {
        return ((uint64_t)(uint32_t)(x + (1 << 20)) << 42) | ((uint64_t)(uint32_t)(y + (1 << 20)) << 21) | (uint64_t)(uint32_t)(z + (1 << 20));
    }
    bool has(int bx, int by, int bz) const { return index.count(pack(bx, by, bz)) != 0; }
    // voxel at global voxel coordinate: false if its block is absent
    bool fetch(int gx, int gy, int gz, float* f, float* w, const double** c) const {
        const int bx = floordiv(gx, RES), by = floordiv(gy, RES), bz = floordiv(gz, RES);
        auto it = index.find(pack(bx, by, bz));
        if (it == index.end()) return false;
        const int64_t i = it->second * NVOX + (gx - bx * RES) * 256 + (gy - by * RES) * 16 + (gz - bz * RES);
        *f = tsdf[i]; *w = weight[i];
        if (c) *c = color ? color + 3 * i : nullptr;
        return true;
    }
};

// ScalableTSDFVolume::GetTSDFAt as oracle/oracle.cpp states it
double tsdf_at(const Blocks& v, const double p[3]) {
    const double vl = v.vl, unit = v.vl * RES;
    double pl[3], pg[3], r[3];
    int index0[3], idx0[3];
    for (int i = 0; i < 3; ++i) {
        pl[i] = p[i] - 0.5 * vl;
        index0[i] = (int)std::floor(pl[i] / unit);
    }
    if (!v.has(index0[0], index0[1], index0[2])) return 0.0;
    for (int i = 0; i < 3; ++i) {
        pg[i] = (pl[i] - (double)index0[i] * unit) / vl;
        idx0[i] = (int)std::floor(pg[i]);
        if (idx0[i] < 0) idx0[i] = 0;
        if (idx0[i] >= RES) idx0[i] = RES - 1;
        r[i] = pg[i] - (double)idx0[i];
    }
    float f[8];
    for (int q = 0; q < 8; ++q) {
        const int sx = (q ^ (q >> 1)) & 1, sy = (q >> 1) & 1, sz = (q >> 2) & 1;
        float t, w;
        f[q] = v.fetch(index0[0] * RES + idx0[0] + sx, index0[1] * RES + idx0[1] + sy, index0[2] * RES + idx0[2] + sz, &t, &w, nullptr)
                   ? t : 0.f;
    }
    return (1 - r[0]) * ((1 - r[1]) * ((1 - r[2]) * f[0] + r[2] * f[4]) + r[1] * ((1 - r[2]) * f[3] + r[2] * f[7])) +
           r[0] * ((1 - r[1]) * ((1 - r[2]) * f[1] + r[2] * f[5]) + r[1] * ((1 - r[2]) * f[2] + r[2] * f[6]));
}

}  // namespace

extern "C" {

// n_blocks blocks (keys [n][3], tsdf / weight [n][4096], color [n][4096][3] or null); poses [n_views][16] = camera_pose =
// inverse4(extrinsic) row-major; intr = (fx, fy, cx, cy).  Outputs nullable: depth [n][H][W] f32, vertex / normal
// [n][H][W][3] f32, color [n][H][W][3] u8; 0 where a ray hits nothing.  Returns the number of hits, -1 on a bad argument.
int64_t raycast_model(int64_t n_blocks, const int32_t* keys, const float* tsdf, const float* weight, const double* vcolor,
                      double voxel_length, double sdf_trunc, int n_views, int W, int H, const double* intr, const double* poses,
                      double depth_min, double depth_max, float* depth, float* vertex, float* normal, uint8_t* color) {
    if (n_views < 0 || W <= 0 || H <= 0 || !(intr[0] > 0.0) || !(intr[1] > 0.0) || !(depth_min > 0.0) || !(depth_min < depth_max))
        return -1;
    Blocks v{keys, tsdf, weight, vcolor, voxel_length, voxel_length * RES, {}};
    for (int64_t i = 0; i < n_blocks; ++i) v.index.emplace(Blocks::pack(keys[3 * i], keys[3 * i + 1], keys[3 * i + 2]), i);
    const float cx = (float)intr[2], cy = (float)intr[3], ifx = 1.0f / (float)intr[0], ify = 1.0f / (float)intr[1];
    const float vl = (float)voxel_length, ktr = (float)(0.5 * sdf_trunc);   // k = 0.5
    const float dmin = (float)depth_min, dmax = (float)depth_max;
    const double vld = voxel_length, half = 0.5 * vld, gap = 0.99 * vld;
    float max_len = 0.f;
    for (int u : {0, W - 1})
        for (int vv : {0, H - 1}) {
            const float xc = ((float)u - cx) * ifx, yc = ((float)vv - cy) * ify;
            max_len = std::max(max_len, std::sqrt((xc * xc + yc * yc) + 1.0f));
        }
    if (!(depth_max * max_len / vld <= 4194304.0)) return -1;
    const int64_t cap = (int64_t)std::ceil(2.0 * (depth_max - depth_min) * max_len / vld) + 5;
    int64_t hits = 0;
    for (int view = 0; view < n_views; ++view) {
        const double* pose = poses + 16 * (size_t)view;
        float R[9], o[3];
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) R[3 * r + c] = (float)pose[4 * r + c];
            o[r] = (float)pose[4 * r + 3];
        }
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : hits)
        for (int vv = 0; vv < H; ++vv) {
            for (int u = 0; u < W; ++u) {
                const float xc = ((float)u - cx) * ifx, yc = ((float)vv - cy) * ify;
                const float len = std::sqrt((xc * xc + yc * yc) + 1.0f);
                float d[3];
                for (int r = 0; r < 3; ++r) d[r] = (R[3 * r] * xc + R[3 * r + 1] * yc) + R[3 * r + 2];
                const float dt_vox = vl / len;
                float t = dmin, t_prev = 0.f, f_prev = 0.f, t_hit = 0.f;
                bool have_prev = false, hit = false;
                for (int64_t it = 0; it < cap && t < dmax; ++it) {
                    float q[3];
                    for (int r = 0; r < 3; ++r) q[r] = std::floor((o[r] + t * d[r]) / vl);
                    float tn;
                    if (!(std::fabs(q[0]) < 16777216.f && std::fabs(q[1]) < 16777216.f && std::fabs(q[2]) < 16777216.f)) {
                        have_prev = false;                    // beyond the key range: one voxel
                        tn = t + dt_vox;
                    } else {
                        const int g[3] = {(int)q[0], (int)q[1], (int)q[2]};
                        float f, w;
                        if (!v.fetch(g[0], g[1], g[2], &f, &w, nullptr)) {
                            have_prev = false;                // absent block: to its exit plane, at least one voxel
                            float t_exit = INFINITY;
                            for (int r = 0; r < 3; ++r) {
                                if (d[r] == 0.f) continue;
                                const int b = floordiv(g[r], RES);
                                const float plane = (float)(16 * (d[r] > 0.f ? b + 1 : b)) * vl;
                                t_exit = std::min(t_exit, (plane - o[r]) / d[r]);
                            }
                            tn = std::max(t_exit, t + dt_vox);
                        } else if (w == 0.f) {                // unobserved: one voxel, forget the previous sample
                            have_prev = false;
                            tn = t + dt_vox;
                        } else {
                            if (have_prev && f_prev > 0.f && f <= 0.f) {
                                // refinement: zero of the trilinear TSDF on [t_prev, t], or on the one-voxel segment before
                                // t_prev / after t when the trilinear values put it there; else the detecting samples
                                auto F = [&](float tt) {
                                    double p[3];
                                    for (int r = 0; r < 3; ++r) p[r] = (double)(o[r] + tt * d[r]);
                                    return tsdf_at(v, p);
                                };
                                float ta = t_prev, tb = t;
                                double Fa = F(ta), Fb = F(tb);
                                bool ok = Fa > 0.0 && Fb <= 0.0;
                                if (Fa <= 0.0) {
                                    const float tz = t_prev - dt_vox;
                                    if (tz >= dmin) {
                                        const double Fz = F(tz);
                                        if (Fz > 0.0) { tb = ta; Fb = Fa; ta = tz; Fa = Fz; ok = true; }
                                    }
                                } else if (Fb > 0.0) {
                                    const float tz = t + dt_vox;
                                    if (tz < dmax) {
                                        const double Fz = F(tz);
                                        if (Fz <= 0.0) { ta = tb; Fa = Fb; tb = tz; Fb = Fz; ok = true; }
                                    }
                                }
                                if (ok) {
                                    t_hit = (float)((double)ta + ((double)tb - (double)ta) * (Fa / (Fa - Fb)));
                                } else {
                                    ta = t_prev; tb = t;
                                    t_hit = t_prev + ((t - t_prev) * f_prev) / (f_prev - f);
                                }
                                t_hit = std::min(std::max(t_hit, ta), tb);
                                hit = true;
                                break;
                            }
                            have_prev = true; f_prev = f; t_prev = t;
                            tn = f > 0.f ? t + std::max(f * ktr, vl) / len : t + dt_vox;
                        }
                    }
                    t = tn > t ? tn : std::nextafter(t, INFINITY);
                }
                const size_t idx = ((size_t)view * H + vv) * W + u;
                float P[3] = {0.f, 0.f, 0.f}, N[3] = {0.f, 0.f, 0.f};
                uint8_t C[3] = {0, 0, 0};
                if (hit) {
                    ++hits;
                    for (int r = 0; r < 3; ++r) P[r] = o[r] + t_hit * d[r];
                    const double Pd[3] = {(double)P[0], (double)P[1], (double)P[2]};
                    if (normal) {                             // GetNormalAt, as oracle_volume_point_normals
                        double g[3];
                        for (int a = 0; a < 3; ++a) {
                            double p0[3] = {Pd[0], Pd[1], Pd[2]}, p1[3] = {Pd[0], Pd[1], Pd[2]};
                            p0[a] -= gap;
                            p1[a] += gap;
                            g[a] = tsdf_at(v, p1) - tsdf_at(v, p0);
                        }
                        const double l = std::sqrt((g[0] * g[0] + g[1] * g[1]) + g[2] * g[2]);
                        for (int a = 0; a < 3; ++a) N[a] = (float)(l > 0.0 ? g[a] / l : g[a]);
                    }
                    if (color && vcolor) {                    // trilinear over the observed corners, renormalised
                        int g0[3];
                        double rr[3];
                        for (int a = 0; a < 3; ++a) {
                            const double pv = (Pd[a] - half) / vld;
                            const double fl = std::floor(pv);
                            g0[a] = (int)fl;
                            rr[a] = pv - fl;
                        }
                        double acc[3] = {0.0, 0.0, 0.0}, wsum = 0.0;
                        for (int qc = 0; qc < 8; ++qc) {
                            const int sx = qc & 1, sy = (qc >> 1) & 1, sz = qc >> 2;
                            float cf, cw;
                            const double* cc = nullptr;
                            if (!v.fetch(g0[0] + sx, g0[1] + sy, g0[2] + sz, &cf, &cw, &cc) || cw == 0.f) continue;
                            const double wq = ((sx ? rr[0] : 1.0 - rr[0]) * (sy ? rr[1] : 1.0 - rr[1])) * (sz ? rr[2] : 1.0 - rr[2]);
                            for (int k = 0; k < 3; ++k) acc[k] += wq * cc[k];
                            wsum += wq;
                        }
                        for (int k = 0; k < 3; ++k) {
                            const double c = wsum > 0.0 ? std::floor(acc[k] / wsum + 0.5) : 0.0;
                            C[k] = (uint8_t)std::min(std::max(c, 0.0), 255.0);
                        }
                    }
                }
                if (depth) depth[idx] = hit ? t_hit : 0.f;
                for (int k = 0; k < 3; ++k) {
                    if (vertex) vertex[3 * idx + k] = P[k];
                    if (normal) normal[3 * idx + k] = N[k];
                    if (color) color[3 * idx + k] = C[k];
                }
            }
        }
    }
    return hits;
}

}  // extern "C"
