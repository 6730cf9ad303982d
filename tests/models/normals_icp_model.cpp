// normals_icp_model.cpp -- CPU restatement of normal estimation and point-to-plane ICP (DESIGN.md §4 "Normals and
// point-to-plane registration"), the reference the CUDA kernels (object-triggered-3d-slam_b200/csrc/knn.cu:
// otslam_cloud_estimate_normals, otslam_cloud_icp_point_to_plane) are compared with bit for bit.
//
// The neighbour search is an exact search of its own (a uniform grid, ring by ring): the (d2, index) order fixes the
// neighbour list, so the result does not depend on the search structure.  Covariance, the Jacobi eigenvector, the sign
// rules, the ICP terms and the two fixed summation trees (over the 128 source points of a CTA, then over the CTAs padded
// to a power of two) are restated in plain C++ compiled with g++ -O2 -ffp-contract=off (no FMA).  The 6x6 solve and the
// Euler update are the library's own host code (icp_solve.h), as the issue of this feature asks of the reference.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../object-triggered-3d-slam_b200/csrc/icp_solve.h"

namespace {

typedef std::pair<double, int32_t> Nb;       // (d2, index); std::pair's < is the (d2, index) order

struct Grid {
    double mn[3], cell;
    int dim[3];
    std::vector<int64_t> start, order;
};

Grid make_grid(const double* pts, int64_t n) {
    Grid g;
    double mx[3];
    for (int a = 0; a < 3; ++a) g.mn[a] = mx[a] = pts[a];
    for (int64_t i = 1; i < n; ++i)
        for (int a = 0; a < 3; ++a) { g.mn[a] = std::min(g.mn[a], pts[3 * i + a]); mx[a] = std::max(mx[a], pts[3 * i + a]); }
    const double ext[3] = {mx[0] - g.mn[0], mx[1] - g.mn[1], mx[2] - g.mn[2]};
    const double vol = std::max(ext[0], 1e-9) * std::max(ext[1], 1e-9) * std::max(ext[2], 1e-9);
    double cell = std::cbrt(vol / std::max<double>(1.0, (double)n / 2.0));
    cell = std::max(cell, std::max(ext[0], std::max(ext[1], ext[2])) / 256.0);
    if (!(cell > 0.0)) cell = 1.0;
    g.cell = cell;
    for (int a = 0; a < 3; ++a) g.dim[a] = std::max(1, (int)std::floor(ext[a] / cell) + 1);
    g.start.assign((size_t)g.dim[0] * g.dim[1] * g.dim[2] + 1, 0);
    std::vector<int64_t> cid(n);
    for (int64_t i = 0; i < n; ++i) {
        int c[3];
        for (int a = 0; a < 3; ++a) c[a] = std::min(std::max((int)std::floor((pts[3 * i + a] - g.mn[a]) / cell), 0), g.dim[a] - 1);
        cid[i] = ((int64_t)c[0] * g.dim[1] + c[1]) * g.dim[2] + c[2];
        g.start[cid[i] + 1]++;
    }
    for (size_t c = 1; c < g.start.size(); ++c) g.start[c] += g.start[c - 1];
    g.order.resize(n);
    std::vector<int64_t> fill(g.start.begin(), g.start.end() - 1);
    for (int64_t i = 0; i < n; ++i) g.order[fill[cid[i]]++] = i;
    return g;
}

// the min(k, m) smallest (d2, index) pairs among the m points with d2 < r2, ascending
void neighbours(const Grid& g, const double* pts, const double* q, int k, double r2, std::vector<Nb>& heap) {
    heap.clear();
    int c[3];
    for (int a = 0; a < 3; ++a) c[a] = std::min(std::max((int)std::floor((q[a] - g.mn[a]) / g.cell), 0), g.dim[a] - 1);
    const int maxring = std::max(g.dim[0], std::max(g.dim[1], g.dim[2]));
    for (int ring = 0; ring <= maxring; ++ring) {
        if (ring >= 1) {
            double reach = INFINITY;   // distance from q to the nearest face of the scanned box with grid behind it
            for (int a = 0; a < 3; ++a) {
                if (c[a] - (ring - 1) > 0) reach = std::min(reach, q[a] - (g.mn[a] + (double)(c[a] - (ring - 1)) * g.cell));
                if (c[a] + ring < g.dim[a]) reach = std::min(reach, (g.mn[a] + (double)(c[a] + ring) * g.cell) - q[a]);
            }
            if (reach == INFINITY) break;
            reach -= 1e-9 * g.cell;
            if (reach > 0.0 && (int)heap.size() == k && reach * reach > heap.front().first) break;
            if (reach > 0.0 && reach * reach >= r2) break;
        }
        for (int x = c[0] - ring; x <= c[0] + ring; ++x) {
            if (x < 0 || x >= g.dim[0]) continue;
            for (int y = c[1] - ring; y <= c[1] + ring; ++y) {
                if (y < 0 || y >= g.dim[1]) continue;
                const bool edge = x == c[0] - ring || x == c[0] + ring || y == c[1] - ring || y == c[1] + ring;
                for (int z = c[2] - ring; z <= c[2] + ring; ++z) {
                    if (z < 0 || z >= g.dim[2]) continue;
                    if (!edge && z != c[2] - ring && z != c[2] + ring) continue;
                    const int64_t cc = ((int64_t)x * g.dim[1] + y) * g.dim[2] + z;
                    for (int64_t s = g.start[cc]; s < g.start[cc + 1]; ++s) {
                        const int32_t j = (int32_t)g.order[s];
                        const double* p = pts + 3 * (size_t)j;
                        const double dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
                        const Nb e((dx * dx + dy * dy) + dz * dz, j);
                        if (!(e.first < r2)) continue;
                        if ((int)heap.size() < k) {
                            heap.push_back(e);
                            std::push_heap(heap.begin(), heap.end());
                        } else if (e < heap.front()) {
                            std::pop_heap(heap.begin(), heap.end());
                            heap.back() = e;
                            std::push_heap(heap.begin(), heap.end());
                        }
                    }
                }
            }
        }
    }
    std::sort(heap.begin(), heap.end());
}

void jacobi_rotate(double (&A)[3][3], double (&V)[3][3], int p, int q) {
    const double apq = A[p][q];
    if (apq == 0.0) return;
    const int r = 3 - p - q;
    const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
    double t;
    if (std::fabs(theta) > 1e150) t = 0.5 / theta;
    else {
        t = 1.0 / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        if (theta < 0.0) t = -t;
    }
    const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
    const double app = A[p][p] - t * apq, aqq = A[q][q] + t * apq;
    const double arp = A[r][p], arq = A[r][q];
    A[r][p] = A[p][r] = c * arp - s * arq;
    A[r][q] = A[q][r] = s * arp + c * arq;
    A[p][p] = app; A[q][q] = aqq; A[p][q] = A[q][p] = 0.0;
    for (int i = 0; i < 3; ++i) {
        const double vp = V[i][p], vq = V[i][q];
        V[i][p] = c * vp - s * vq;
        V[i][q] = s * vp + c * vq;
    }
}

void smallest_eigenvector(const double (&C)[6], double (&n)[3]) {
    double s = 0.0;
    for (int i = 0; i < 6; ++i) s = std::fmax(s, std::fabs(C[i]));
    if (!(s > 0.0)) { n[0] = n[1] = n[2] = 0.0; return; }
    const double a00 = C[0] / s, a01 = C[1] / s, a02 = C[2] / s, a11 = C[3] / s, a12 = C[4] / s, a22 = C[5] / s;
    double A[3][3] = {{a00, a01, a02}, {a01, a11, a12}, {a02, a12, a22}};
    double V[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
    for (int sweep = 0; sweep < 16; ++sweep) {
        if (A[0][1] == 0.0 && A[0][2] == 0.0 && A[1][2] == 0.0) break;
        jacobi_rotate(A, V, 0, 1);
        jacobi_rotate(A, V, 0, 2);
        jacobi_rotate(A, V, 1, 2);
    }
    int m = 0;
    if (A[1][1] <= A[m][m]) m = 1;
    if (A[2][2] <= A[m][m]) m = 2;
    const double x = V[0][m], y = V[1][m], z = V[2][m];
    const double len = std::sqrt((x * x + y * y) + z * z);
    n[0] = x / len; n[1] = y / len; n[2] = z / len;
}

void normal_of(const double* pts, const std::vector<Nb>& nb, const double* prior, double (&n)[3]) {
    const int found = (int)nb.size();
    double C[6] = {1.0, 0.0, 0.0, 1.0, 0.0, 1.0};
    if (found >= 3) {
        double m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (const Nb& e : nb) {
            const double* p = pts + 3 * (size_t)e.second;
            m[0] += p[0]; m[1] += p[1]; m[2] += p[2];
            m[3] += p[0] * p[0]; m[4] += p[0] * p[1]; m[5] += p[0] * p[2];
            m[6] += p[1] * p[1]; m[7] += p[1] * p[2]; m[8] += p[2] * p[2];
        }
        for (int c = 0; c < 9; ++c) m[c] /= (double)found;
        C[0] = m[3] - m[0] * m[0]; C[1] = m[4] - m[0] * m[1]; C[2] = m[5] - m[0] * m[2];
        C[3] = m[6] - m[1] * m[1]; C[4] = m[7] - m[1] * m[2]; C[5] = m[8] - m[2] * m[2];
    }
    smallest_eigenvector(C, n);
    if (n[0] == 0.0 && n[1] == 0.0 && n[2] == 0.0) {
        if (prior) { n[0] = prior[0]; n[1] = prior[1]; n[2] = prior[2]; }
        else n[2] = 1.0;
    } else if (prior) {
        if ((n[0] * prior[0] + n[1] * prior[1]) + n[2] * prior[2] < 0.0) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }
    } else {
        int b = 0;
        if (std::fabs(n[1]) > std::fabs(n[b])) b = 1;
        if (std::fabs(n[2]) > std::fabs(n[b])) b = 2;
        if (n[b] < 0.0) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }
    }
}

constexpr int kCta = 128, kTerms = 30;

// nearest target strictly within the radius, ties to the lower index: a hash grid of cell = radius, 27 cells
struct CellGrid {
    double mn[3], cell;
    std::unordered_map<uint64_t, std::vector<int32_t>> cells;
    void key(const double* p, int c[3]) const {   // clamped: cells 2^20 away from the target hold nothing in range anyway
        for (int a = 0; a < 3; ++a) c[a] = (int)std::fmin(std::fmax(std::floor((p[a] - mn[a]) / cell), -1048575.0), 1048574.0);
    }
    static uint64_t pack(int x, int y, int z) {
        return ((uint64_t)(uint32_t)(x + 1048576) << 42) | ((uint64_t)(uint32_t)(y + 1048576) << 21) | (uint64_t)(uint32_t)(z + 1048576);
    }
};

void transform(double* pts, int64_t n, const double* T) {
    for (int64_t i = 0; i < n; ++i) {
        const double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
        double h[4];
        for (int r = 0; r < 4; ++r) h[r] = ((T[4 * r] * x + T[4 * r + 1] * y) + T[4 * r + 2] * z) + T[4 * r + 3];
        for (int r = 0; r < 3; ++r) pts[3 * i + r] = h[r] / h[3];
    }
}

}  // namespace

extern "C" {

// neighbour lists: idx [n][max_nn] (-1 beyond count[i]), count [n]
int model_neighbours(const double* pts, int64_t n, double radius, int max_nn, int32_t* idx, int32_t* count) {
    if (n <= 0) return 0;
    const Grid g = make_grid(pts, n);
    const int k = (int)std::min<int64_t>(max_nn, n);
    const double r2 = radius * radius;
#pragma omp parallel
    {
        std::vector<Nb> nb;
#pragma omp for schedule(dynamic, 256)
        for (int64_t i = 0; i < n; ++i) {
            neighbours(g, pts, pts + 3 * i, k, r2, nb);
            count[i] = (int32_t)nb.size();
            for (int j = 0; j < max_nn; ++j) idx[(size_t)i * max_nn + j] = j < (int)nb.size() ? nb[j].second : -1;
        }
    }
    return 0;
}

int model_estimate_normals(const double* pts, int64_t n, const double* prior, double radius, int max_nn, double* out) {
    if (n < 0 || max_nn < 1 || max_nn > 128 || !(radius > 0.0)) return -1;
    if (n == 0) return 0;
    const Grid g = make_grid(pts, n);
    const int k = (int)std::min<int64_t>(max_nn, n);
    const double r2 = radius * radius;
#pragma omp parallel
    {
        std::vector<Nb> nb;
#pragma omp for schedule(dynamic, 256)
        for (int64_t i = 0; i < n; ++i) {
            neighbours(g, pts, pts + 3 * i, k, r2, nb);
            double v[3];
            normal_of(pts, nb, prior ? prior + 3 * i : nullptr, v);
            for (int a = 0; a < 3; ++a) out[3 * i + a] = v[a];
        }
    }
    return 0;
}

int model_icp_point_to_plane(const double* source, int64_t ns, const double* target, const double* tn, int64_t nt, double max_distance,
                             const double* init, double relative_fitness, double relative_rmse, int max_iteration, double* T_out,
                             double* fitness, double* rmse_out, int32_t* iterations, int32_t* corr) {
    if (ns < 0 || nt < 0 || !(max_distance > 0.0) || max_iteration < 0) return -1;
    double T[16];
    for (int k = 0; k < 16; ++k) T[k] = init[k];
    if (ns == 0) {
        std::memcpy(T_out, T, sizeof(T));
        *fitness = 0.0; *rmse_out = 0.0; *iterations = 0;
        return 0;
    }
    CellGrid g;
    g.cell = max_distance;
    for (int a = 0; a < 3; ++a) g.mn[a] = nt ? target[a] : 0.0;
    for (int64_t j = 1; j < nt; ++j)
        for (int a = 0; a < 3; ++a) g.mn[a] = std::min(g.mn[a], target[3 * j + a]);
    for (int64_t j = 0; j < nt; ++j) {
        int c[3];
        g.key(target + 3 * j, c);
        g.cells[CellGrid::pack(c[0], c[1], c[2])].push_back((int32_t)j);
    }
    const double r2 = max_distance * max_distance;
    std::vector<double> src(source, source + 3 * ns);
    transform(src.data(), ns, T);
    const int64_t n_cta = (ns + kCta - 1) / kCta;
    int64_t P = 1;
    while (P < n_cta) P *= 2;
    std::vector<double> part((size_t)kTerms * P);
    double S[kTerms];
    auto evaluate = [&](double& fit, double& rmse) {
#pragma omp parallel for schedule(dynamic, 16)
        for (int64_t b = 0; b < n_cta; ++b) {
            double v[kTerms][kCta];
            for (int l = 0; l < kCta; ++l) {
                double t[kTerms] = {};
                const int64_t i = b * kCta + l;
                if (i < ns) {
                    const double* p = &src[3 * i];
                    int c[3];
                    g.key(p, c);
                    int bi = -1;
                    double best = r2;
                    for (int dz = -1; dz <= 1; ++dz)
                        for (int dy = -1; dy <= 1; ++dy)
                            for (int dx = -1; dx <= 1; ++dx) {
                                auto it = g.cells.find(CellGrid::pack(c[0] + dx, c[1] + dy, c[2] + dz));
                                if (it == g.cells.end()) continue;
                                for (int32_t j : it->second) {
                                    const double ex = p[0] - target[3 * (size_t)j], ey = p[1] - target[3 * (size_t)j + 1],
                                                 ez = p[2] - target[3 * (size_t)j + 2];
                                    const double d2 = (ex * ex + ey * ey) + ez * ez;
                                    if (d2 < best || (d2 == best && bi >= 0 && j < bi)) { best = d2; bi = j; }
                                }
                            }
                    corr[i] = bi;
                    if (bi >= 0) {
                        const double* q = target + 3 * (size_t)bi;
                        const double* N = tn + 3 * (size_t)bi;
                        const double r = ((p[0] - q[0]) * N[0] + (p[1] - q[1]) * N[1]) + (p[2] - q[2]) * N[2];
                        const double J[6] = {p[1] * N[2] - p[2] * N[1], p[2] * N[0] - p[0] * N[2], p[0] * N[1] - p[1] * N[0], N[0], N[1], N[2]};
                        int k = 0;
                        for (int a = 0; a < 6; ++a)
                            for (int e = a; e < 6; ++e) t[k++] = J[a] * J[e];
                        for (int a = 0; a < 6; ++a) t[21 + a] = J[a] * r;
                        t[27] = r * r;
                        t[28] = 1.0;
                        t[29] = best;
                    }
                }
                for (int k = 0; k < kTerms; ++k) v[k][l] = t[k];
            }
            for (int s = kCta / 2; s > 0; s >>= 1)
                for (int k = 0; k < kTerms; ++k)
                    for (int e = 0; e < s; ++e) v[k][e] = v[k][e] + v[k][e + s];
            for (int k = 0; k < kTerms; ++k) part[(size_t)k * P + b] = v[k][0];
        }
        for (int k = 0; k < kTerms; ++k) {
            double* w = &part[(size_t)k * P];
            for (int64_t b = n_cta; b < P; ++b) w[b] = 0.0;
            for (int64_t h = P / 2; h > 0; h >>= 1)
                for (int64_t i = 0; i < h; ++i) w[i] = w[i] + w[i + h];
            S[k] = w[0];
        }
        fit = S[28] / (double)ns;
        rmse = S[28] > 0.0 ? std::sqrt(S[29] / S[28]) : 0.0;
    };
    double fit = 0.0, rmse = 0.0;
    evaluate(fit, rmse);
    int it = 0;
    while (it < max_iteration) {
        double U[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1}, xi[6], Tn[16];
        if (S[28] > 0.0 && otslam::solve6(S, xi)) otslam::euler_update(xi, U);
        otslam::matmul4(U, T, Tn);
        std::memcpy(T, Tn, sizeof(T));
        transform(src.data(), ns, U);
        const double fit0 = fit, rmse0 = rmse;
        evaluate(fit, rmse);
        ++it;
        if (std::fabs(fit0 - fit) < relative_fitness && std::fabs(rmse0 - rmse) < relative_rmse) break;
    }
    std::memcpy(T_out, T, sizeof(T));
    *fitness = fit; *rmse_out = rmse; *iterations = it;
    return 0;
}

}  // extern "C"
