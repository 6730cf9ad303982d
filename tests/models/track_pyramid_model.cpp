// track_pyramid_model.cpp -- CPU restatement of coarse-to-fine frame-to-model tracking (DESIGN.md §4 "Frame-to-model
// tracking", "Coarse to fine"), the reference the CUDA kernels (object-triggered-3d-slam_b200/csrc/track.cu) are compared
// with bit for bit at more than one level: the depth pyramid, the level intrinsics and the level loop.
//
// It includes track_model.cpp (the single-scale model, unchanged) for its shared pieces -- the cofactor inverse, the affine
// product and the Cholesky solve -- and restates the per-pixel terms and the association for a depth source that is either
// the u16 frame (level 0) or a level's float depth.  With one level it gives track_model's bits, which
// tests/test_track_pyramid_oracle.py checks.  Compiled with g++ -O2 -ffp-contract=off (no FMA) together with
// raycast_model.cpp; track_model.cpp is not compiled separately.
#include "track_model.cpp"

namespace {

struct Level {
    const uint16_t* depth;          // level 0: the u16 frame
    const float* fdepth;            // levels >= 1: the level's depth (metres)
    const float *vertex, *normal;   // model maps at E0, rendered at this level
    int W, H;
    float scale;
    double dmax, ddiff2, fx, fy, cx, cy;
    const double* E0;
};

// the 30 terms of pixel (u, v) at camera pose T (track_model.cpp's pixel_terms, with the level's depth source)
void level_terms(const Level& F, const double* T, int u, int v, double t[NT]) {
    for (int k = 0; k < NT; ++k) t[k] = 0.0;
    const size_t i = (size_t)v * F.W + u;
    const float d = F.fdepth ? F.fdepth[i] : (float)F.depth[i] / F.scale;
    if (!(d > 0.f && (double)d < F.dmax)) return;
    t[29] = 1.0;
    const double z = (double)d;
    const double pc[3] = {(((double)u - F.cx) / F.fx) * z, (((double)v - F.cy) / F.fy) * z, z};
    double p[3], q[3];
    affine(T, pc, p);
    affine(F.E0, p, q);
    if (!(q[2] > 0.0)) return;
    const double uf = std::floor((F.fx * q[0]) / q[2] + F.cx + 0.5), vf = std::floor((F.fy * q[1]) / q[2] + F.cy + 0.5);
    if (!(uf >= 0.0 && uf < (double)F.W && vf >= 0.0 && vf < (double)F.H)) return;
    const size_t m = 3 * ((size_t)vf * F.W + (size_t)uf);
    const double N[3] = {(double)F.normal[m], (double)F.normal[m + 1], (double)F.normal[m + 2]};
    if (N[0] == 0.0 && N[1] == 0.0 && N[2] == 0.0) return;
    const double e[3] = {p[0] - (double)F.vertex[m], p[1] - (double)F.vertex[m + 1], p[2] - (double)F.vertex[m + 2]};
    if (!((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2] <= F.ddiff2)) return;
    const double r = (N[0] * e[0] + N[1] * e[1]) + N[2] * e[2];
    const double J[6] = {p[1] * N[2] - p[2] * N[1], p[2] * N[0] - p[0] * N[2], p[0] * N[1] - p[1] * N[0], N[0], N[1], N[2]};
    int k = 0;
    for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b) t[k++] = J[a] * J[b];
    for (int a = 0; a < 6; ++a) t[21 + a] = J[a] * r;
    t[27] = r * r;
    t[28] = 1.0;
}

// one association pass at a level: the 30 sums by the kernels' two fixed trees
void level_associate(const Level& F, const double* T, double S[NT]) {
    const int tx = (F.W + TW - 1) / TW, ty = (F.H + TH - 1) / TH, nt = tx * ty;
    int P = 1;
    while (P < nt) P *= 2;
    std::vector<double> part((size_t)NT * P, 0.0);
    std::vector<double> sm((size_t)NT * TPX);
    for (int by = 0; by < ty; ++by)
        for (int bx = 0; bx < tx; ++bx) {
            for (int lane = 0; lane < TPX; ++lane) {
                const int u = bx * TW + lane % TW, v = by * TH + lane / TW;
                double t[NT];
                if (u < F.W && v < F.H) level_terms(F, T, u, v, t);
                else for (int k = 0; k < NT; ++k) t[k] = 0.0;
                for (int k = 0; k < NT; ++k) sm[(size_t)k * TPX + lane] = t[k];
            }
            for (int s = TPX / 2; s > 0; s >>= 1)
                for (int k = 0; k < NT; ++k)
                    for (int i = 0; i < s; ++i) sm[(size_t)k * TPX + i] = sm[(size_t)k * TPX + i] + sm[(size_t)k * TPX + i + s];
            for (int k = 0; k < NT; ++k) part[(size_t)k * P + by * tx + bx] = sm[(size_t)k * TPX];
        }
    for (int h = P / 2; h > 0; h >>= 1)
        for (int k = 0; k < NT; ++k)
            for (int i = 0; i < h; ++i) {
                const double x = i < nt ? part[(size_t)k * P + i] : 0.0, y = i + h < nt ? part[(size_t)k * P + i + h] : 0.0;
                part[(size_t)k * P + i] = x + y;
            }
    for (int k = 0; k < NT; ++k) S[k] = part[(size_t)k * P];
}

// level l + 1 (Wd x Hd) of the depth pyramid from level l (Ws wide): the valid depths of each 2x2 block within `band` of the
// block's smallest, summed in FP64 in raster order, over their count, rounded to FP32; 0 when none is valid.  Level 0 is
// src16 / scale (valid iff > 0 and < dmax), the others srcf (valid iff > 0).
void pyr_down(const uint16_t* src16, const float* srcf, int Ws, int Wd, int Hd, float scale, double dmax, double band, float* dst) {
    for (int v = 0; v < Hd; ++v)
        for (int u = 0; u < Wd; ++u) {
            const size_t b = (size_t)(2 * v) * Ws + 2 * u;
            const size_t at[4] = {b, b + 1, b + Ws, b + Ws + 1};
            float d[4], lo = INFINITY;
            bool ok[4];
            for (int k = 0; k < 4; ++k) {
                d[k] = src16 ? (float)src16[at[k]] / scale : srcf[at[k]];
                ok[k] = src16 ? d[k] > 0.f && (double)d[k] < dmax : d[k] > 0.f;
                if (ok[k] && d[k] < lo) lo = d[k];
            }
            double sum = 0.0;
            int n = 0;
            for (int k = 0; k < 4; ++k)
                if (ok[k] && (double)d[k] - (double)lo <= band) { sum = sum + (double)d[k]; ++n; }
            dst[(size_t)v * Wd + u] = n ? (float)(sum / (double)n) : 0.f;
        }
}

// levels 1 .. n_levels - 1 of one frame's pyramid, back to back
void pyramid(const uint16_t* depth, int W, int H, float scale, double dmax, double band, int n_levels, float* out) {
    const float* prev = nullptr;
    for (int l = 1; l < n_levels; ++l) {
        const int Ws = W >> (l - 1), Wd = W >> l, Hd = H >> l;
        pyr_down(l == 1 ? depth : nullptr, prev, Ws, Wd, Hd, scale, dmax, band, out);
        prev = out;
        out += (size_t)Wd * Hd;
    }
}

// the intrinsics of level l: fx / 2, fy / 2, (cx - 0.5) / 2, (cy - 0.5) / 2 per level, in FP64
void level_intr(const double* intr, int l, double* out) {
    for (int k = 0; k < 4; ++k) out[k] = intr[k];
    for (int i = 0; i < l; ++i) out[0] = out[0] / 2.0, out[1] = out[1] / 2.0, out[2] = (out[2] - 0.5) / 2.0, out[3] = (out[3] - 0.5) / 2.0;
}

}  // namespace

extern "C" {

// The pyramid of n frames depth [n][H][W] u16: levels 1 .. n_levels - 1 of each frame back to back in `out` (frame-major),
// band = 4 voxel lengths.  Returns the floats written per frame, or -1 on a bad argument.
int64_t track_model_levels(int n, const uint16_t* depth, int W, int H, double depth_scale, double depth_max, double voxel_length,
                           int n_levels, float* out) {
    if (n < 0 || W <= 0 || H <= 0 || n_levels < 1 || n_levels > 4) return -1;
    int64_t per = 0;
    for (int l = 1; l < n_levels; ++l) per += (int64_t)(W >> l) * (H >> l);
    for (int f = 0; f < n; ++f)
        pyramid(depth + (size_t)W * H * f, W, H, (float)depth_scale, depth_max, 4.0 * voxel_length, n_levels, out + per * f);
    return per;
}

// The intrinsics of pyramid level l as the tracker uses them (out[4]).
void track_model_level_intr(const double* intr, int l, double* out) { level_intr(intr, l, out); }

// Tracks n frames (depth [n][H][W] u16) of the oracle volume given by its exported blocks (keys [nb][3], tsdf / weight
// [nb][4096]) from init_ext [n][16], coarse to fine over n_levels pyramid levels with depth_diff[l] and max_it[l] (index =
// level, 0 = full resolution).  Outputs ext_out [n][16], status / iters [n] i32 (level 0's status, iterations summed over
// the levels), fitness / rmse [n] (level 0).  Returns 0, or -1 on a bad argument (the ray-cast model refuses a level's
// window, or an initial extrinsic is singular).
int track_model_pyramid(int64_t n_blocks, const int32_t* keys, const float* tsdf, const float* weight, double voxel_length,
                        double sdf_trunc, int n, const uint16_t* depth, int W, int H, const double* intr, const double* init_ext,
                        double depth_scale, double depth_min, double depth_max, int n_levels, const double* depth_diff,
                        const int32_t* max_it, double* ext_out, int32_t* status, int32_t* iters, double* fitness, double* rmse) {
    if (n < 0 || W <= 0 || H <= 0 || !(depth_scale > 0.0) || n_levels < 1 || n_levels > 4) return -1;
    for (int l = 0; l < n_levels; ++l)
        if (!(depth_diff[l] > 0.0) || max_it[l] < 1 || max_it[l] > 100) return -1;
    if (n_levels > 1 && ((W >> (n_levels - 1)) < TW || (H >> (n_levels - 1)) < TH)) return -1;
    std::vector<float> vtx[4], nrm[4], pyr;
    double li[4][4];
    size_t pyr_n = 0;
    for (int l = 0; l < n_levels; ++l) {
        const size_t px = (size_t)(W >> l) * (H >> l);
        vtx[l].resize(3 * px);
        nrm[l].resize(3 * px);
        if (l) pyr_n += px;
        level_intr(intr, l, li[l]);
    }
    pyr.resize(pyr_n);
    for (int f = 0; f < n; ++f) {
        const double* E0 = init_ext + 16 * (size_t)f;
        const uint16_t* d0 = depth + (size_t)W * H * f;
        double T[16], E[16];
        if (!inverse4(E0, T)) return -1;
        pyramid(d0, W, H, (float)depth_scale, depth_max, 4.0 * voxel_length, n_levels, pyr.data());
        Level F[4];
        const float* lev = pyr.data();
        for (int l = 0; l < n_levels; ++l) {
            const int Wl = W >> l, Hl = H >> l;
            if (raycast_model(n_blocks, keys, tsdf, weight, nullptr, voxel_length, sdf_trunc, 1, Wl, Hl, li[l], T, depth_min,
                              depth_max, nullptr, vtx[l].data(), nrm[l].data(), nullptr) < 0)
                return -1;
            F[l] = Level{d0, l ? lev : nullptr, vtx[l].data(), nrm[l].data(), Wl, Hl, (float)depth_scale, depth_max,
                         depth_diff[l] * depth_diff[l], li[l][0], li[l][1], li[l][2], li[l][3], E0};
            if (l) lev += (size_t)Wl * Hl;
        }
        std::memcpy(E, E0, sizeof E);
        int st = 1, it_done = 0;
        for (int l = n_levels - 1; l >= 0; --l) {      // each level from the pose the coarser one returned, whatever its status
            st = 1;
            double last_step = INFINITY;
            for (int it = 0; it < max_it[l]; ++it) {
                double S[NT];
                level_associate(F[l], T, S);
                ++it_done;
                if (S[28] < 64.0) { st = 2; break; }
                double xi[6];
                if (!solve6(S, xi)) { st = 3; break; }
                const double h[3] = {0.5 * xi[0], 0.5 * xi[1], 0.5 * xi[2]};
                const double n2 = (h[0] * h[0] + h[1] * h[1]) + h[2] * h[2];
                const double c = 2.0 / (1.0 + n2);
                const double K[9] = {0.0, -h[2], h[1], h[2], 0.0, -h[0], -h[1], h[0], 0.0};
                double D[16];
                for (int i = 0; i < 3; ++i) {
                    for (int j = 0; j < 3; ++j) {
                        double k2 = h[i] * h[j];
                        if (i == j) k2 = k2 - n2;
                        D[4 * i + j] = (i == j ? 1.0 : 0.0) + c * (K[3 * i + j] + k2);
                    }
                    D[4 * i + 3] = xi[3 + i];
                }
                D[12] = 0.0; D[13] = 0.0; D[14] = 0.0; D[15] = 1.0;
                double Tn[16], En[16];
                for (int r = 0; r < 4; ++r)
                    for (int cc = 0; cc < 4; ++cc)
                        Tn[4 * r + cc] = ((D[4 * r] * T[cc] + D[4 * r + 1] * T[4 + cc]) + D[4 * r + 2] * T[8 + cc]) + D[4 * r + 3] * T[12 + cc];
                if (!inverse4(Tn, En)) { st = 3; break; }
                std::memcpy(T, Tn, sizeof T);
                std::memcpy(E, En, sizeof E);
                double step = 0.0;
                for (int k = 0; k < 6; ++k)
                    if (std::fabs(xi[k]) > step) step = std::fabs(xi[k]);
                const bool stalled = step <= 1e-5 && step >= last_step;   // a 2-cycle of flipping associations
                last_step = step;
                if (step <= 1e-6 || stalled) { st = 0; break; }
            }
        }
        double S[NT];
        level_associate(F[0], T, S);
        std::memcpy(ext_out + 16 * (size_t)f, E, sizeof E);
        status[f] = st;
        iters[f] = it_done;
        fitness[f] = S[29] > 0.0 ? S[28] / S[29] : 0.0;
        rmse[f] = S[28] > 0.0 ? std::sqrt(S[27] / S[28]) : 0.0;
    }
    return 0;
}

}  // extern "C"
