// track_model.cpp -- CPU restatement of frame-to-model tracking (DESIGN.md §4 "Frame-to-model tracking"), the reference
// the CUDA kernels (object-triggered-3d-slam_b200/csrc/track.cu) are compared with bit for bit: poses, status, iterations,
// fitness and RMSE.
//
// The model maps come from raycast_model.cpp (compiled into the same library), on an oracle volume's exported voxels, at
// the poses inverse4 (the shared cofactor inverse, restated below as oracle/oracle.cpp states it) gives.  Steps 2-7 of
// the design are restated in plain C++ compiled with g++ -O2 -ffp-contract=off (no FMA), including the two fixed
// pairwise summation trees: over the 128 pixels of a 16x8 tile, then over the tiles padded to a power of two.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

extern "C" int64_t raycast_model(int64_t n_blocks, const int32_t* keys, const float* tsdf, const float* weight,
                                 const double* vcolor, double voxel_length, double sdf_trunc, int n_views, int W, int H,
                                 const double* intr, const double* poses, double depth_min, double depth_max, float* depth,
                                 float* vertex, float* normal, uint8_t* color);

namespace {

constexpr int TW = 16, TH = 8, TPX = TW * TH, NT = 30;

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

void affine(const double* M, const double p[3], double out[3]) {
    for (int r = 0; r < 3; ++r) out[r] = ((M[4 * r] * p[0] + M[4 * r + 1] * p[1]) + M[4 * r + 2] * p[2]) + M[4 * r + 3];
}

struct Frame {
    const uint16_t* depth;
    const float *vertex, *normal;   // model maps at E0
    int W, H;
    float scale;
    double dmax, ddiff2, fx, fy, cx, cy;
    double E0[16];
};

// the 30 terms of pixel (u, v) at camera pose T
void pixel_terms(const Frame& F, const double* T, int u, int v, double t[NT]) {
    for (int k = 0; k < NT; ++k) t[k] = 0.0;
    const float d = (float)F.depth[(size_t)v * F.W + u] / F.scale;
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
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) t[k++] = J[i] * J[j];
    for (int i = 0; i < 6; ++i) t[21 + i] = J[i] * r;
    t[27] = r * r;
    t[28] = 1.0;
}

// one association pass: the 30 sums by the kernels' two fixed trees
void associate(const Frame& F, const double* T, double S[NT]) {
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
                if (u < F.W && v < F.H) pixel_terms(F, T, u, v, t);
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

bool solve6(const double* S, double xi[6]) {
    double A[6][6], L[6][6], y[6];
    int k = 0;
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) { A[i][j] = S[k]; A[j][i] = S[k]; ++k; }
    double maxd = A[0][0];
    for (int i = 1; i < 6; ++i)
        if (A[i][i] > maxd) maxd = A[i][i];
    const double thr = 1e-10 * maxd;
    for (int j = 0; j < 6; ++j) {
        double s = A[j][j];
        for (int c = 0; c < j; ++c) s = s - L[j][c] * L[j][c];
        if (!(s > thr)) return false;
        L[j][j] = std::sqrt(s);
        for (int i = j + 1; i < 6; ++i) {
            double w = A[i][j];
            for (int c = 0; c < j; ++c) w = w - L[i][c] * L[j][c];
            L[i][j] = w / L[j][j];
        }
    }
    for (int i = 0; i < 6; ++i) {
        double w = S[21 + i];
        for (int c = 0; c < i; ++c) w = w - L[i][c] * y[c];
        y[i] = w / L[i][i];
    }
    for (int i = 5; i >= 0; --i) {
        double w = y[i];
        for (int c = i + 1; c < 6; ++c) w = w - L[c][i] * xi[c];
        xi[i] = w / L[i][i];
    }
    for (int i = 0; i < 6; ++i) xi[i] = -xi[i];
    return true;
}

}  // namespace

extern "C" {

// Tracks n frames (depth [n][H][W] u16) of the oracle volume given by its exported blocks (keys [nb][3], tsdf / weight
// [nb][4096]) from init_ext [n][16].  Outputs ext_out [n][16], status / iters [n] i32, fitness / rmse [n].  Returns 0, or
// -1 on a bad argument (the ray-cast model refuses the window, or an initial extrinsic is singular).
int track_model(int64_t n_blocks, const int32_t* keys, const float* tsdf, const float* weight, double voxel_length,
                double sdf_trunc, int n, const uint16_t* depth, int W, int H, const double* intr, const double* init_ext,
                double depth_scale, double depth_min, double depth_max, double depth_diff, int max_it, double* ext_out,
                int32_t* status, int32_t* iters, double* fitness, double* rmse) {
    if (n < 0 || W <= 0 || H <= 0 || !(depth_scale > 0.0) || !(depth_diff > 0.0) || max_it < 1 || max_it > 100) return -1;
    const size_t px = (size_t)W * H;
    std::vector<float> vtx(3 * px), nrm(3 * px);
    for (int f = 0; f < n; ++f) {
        const double* E0 = init_ext + 16 * (size_t)f;
        double T[16], E[16];
        if (!inverse4(E0, T)) return -1;
        if (raycast_model(n_blocks, keys, tsdf, weight, nullptr, voxel_length, sdf_trunc, 1, W, H, intr, T, depth_min, depth_max,
                          nullptr, vtx.data(), nrm.data(), nullptr) < 0)
            return -1;
        Frame F{depth + px * f, vtx.data(), nrm.data(), W, H, (float)depth_scale, depth_max, depth_diff * depth_diff,
                intr[0], intr[1], intr[2], intr[3], {}};
        std::memcpy(F.E0, E0, sizeof F.E0);
        std::memcpy(E, E0, sizeof E);
        int st = 1, it_done = 0;
        double last_step = INFINITY;
        for (int it = 0; it < max_it; ++it) {
            double S[NT];
            associate(F, T, S);
            it_done = it + 1;
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
        double S[NT];
        associate(F, T, S);
        std::memcpy(ext_out + 16 * (size_t)f, E, sizeof E);
        status[f] = st;
        iters[f] = it_done;
        fitness[f] = S[29] > 0.0 ? S[28] / S[29] : 0.0;
        rmse[f] = S[28] > 0.0 ? std::sqrt(S[27] / S[28]) : 0.0;
    }
    return 0;
}

}  // extern "C"
