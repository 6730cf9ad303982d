// CPU restatement of otslam_cloud_cluster_dbscan and otslam_cloud_segment_plane (DESIGN.md §4 "Plane segmentation and
// DBSCAN clustering"), the definition the CUDA kernels of csrc/segment.cu are compared with bit for bit.
//
//   DBSCAN   Open3D's ClusterDBSCAN loop, literally: labels start undefined (-2); the points are visited in index order; an
//            undefined point with fewer than min_points neighbours becomes noise (-1); otherwise it seeds a new cluster, which
//            grows breadth-first: a reached noise point joins it, a reached undefined point joins it and, when it is core,
//            queues its neighbours.  Neighbours (d2 < eps^2, d2 = (dx^2 + dy^2) + dz^2) are listed on demand from a grid
//            (cell = eps enlarged by 2^-20, the 27 cells around the point) instead of all at once; the set is the same.
//   RANSAC   hypotheses h = 0, 1, ... in order: Floyd's sample on u01(seed, h * r + k), the triangle plane (r = 3) or
//            GetPlaneFromPoints over the sample (r > 3), evaluation with the distance sum in the tree order below, and
//            Open3D's selection and break rule; the best plane's inliers and GetPlaneFromPoints over them by the same trees.
//
// The tree of a sum over positions 0 .. m-1 (values v, 0.0 beyond m): tiles of 2048 positions; thread t of tile c adds
// v[c * 2048 + k * 256 + t] for k = 0 .. 7 to 0.0 in k order; inside each warp of 32 threads lane l += lane l + 16, then + 8,
// + 4, + 2, + 1; the 8 warp sums w += w + 4, + 2, + 1; the tile sums, padded with 0.0 to a power of two P, i += i + P/2,
// then + P/4, ..., + 1.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <unordered_map>
#include <vector>

namespace {

uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
double u01(uint64_t seed, uint64_t ctr) {
    return (double)(splitmix64(seed * 0xD1342543DE82EF95ull + ctr) >> 11) * (1.0 / 9007199254740992.0);
}

double d2_of(const double* a, const double* b) {
    const double ex = a[0] - b[0], ey = a[1] - b[1], ez = a[2] - b[2];
    return (ex * ex + ey * ey) + ez * ez;
}

// ---- DBSCAN
struct Grid {
    const double* p;
    int64_t n;
    double mn[3], cell;
    std::unordered_map<uint64_t, std::vector<int>> cells;
    int64_t key_of(const double* q, int64_t c[3]) const {
        for (int a = 0; a < 3; ++a) c[a] = (int64_t)std::floor((q[a] - mn[a]) / cell);
        return 0;
    }
    static uint64_t pack(int64_t x, int64_t y, int64_t z) {
        return ((uint64_t)(x & 0x1FFFFF) << 42) | ((uint64_t)(y & 0x1FFFFF) << 21) | (uint64_t)(z & 0x1FFFFF);
    }
    Grid(const double* pts, int64_t n_, double eps) : p(pts), n(n_) {
        for (int a = 0; a < 3; ++a) mn[a] = n ? pts[a] : 0.0;
        double mx[3] = {mn[0], mn[1], mn[2]};
        for (int64_t i = 0; i < n; ++i)
            for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], pts[3 * i + a]); mx[a] = std::max(mx[a], pts[3 * i + a]); }
        // at most 2^20 cells per axis (the cell may grow, never shrink: 27 cells still cover the ball)
        double ext = std::max(mx[0] - mn[0], std::max(mx[1] - mn[1], mx[2] - mn[2]));
        cell = std::max(eps * (1.0 + 1.0 / 1048576.0), ext / 1048576.0);
        for (int64_t i = 0; i < n; ++i) {
            int64_t c[3];
            key_of(pts + 3 * i, c);
            cells[pack(c[0], c[1], c[2])].push_back((int)i);
        }
    }
    void neighbours(int64_t i, double r2, std::vector<int>& out) const {
        out.clear();
        int64_t c[3];
        key_of(p + 3 * i, c);
        for (int dz = -1; dz <= 1; ++dz)
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    auto it = cells.find(pack(c[0] + dx, c[1] + dy, c[2] + dz));
                    if (it == cells.end()) continue;
                    for (int j : it->second)
                        if (d2_of(p + 3 * i, p + 3 * (int64_t)j) < r2) out.push_back(j);
                }
    }
};

// ---- RANSAC
constexpr int kTile = 2048, kThreads = 256, kItems = 8;

template <typename F>
double tree_sum(int64_t m, F v) {
    const int64_t n_cta = (m + kTile - 1) / kTile;
    int64_t P = 1;
    while (P < n_cta) P *= 2;
    std::vector<double> part(P, 0.0);
    for (int64_t c = 0; c < n_cta; ++c) {
        double w[8];
        for (int wp = 0; wp < 8; ++wp) {
            double u[32];
            for (int l = 0; l < 32; ++l) {
                double acc = 0.0;
                for (int k = 0; k < kItems; ++k) {
                    const int64_t pos = c * kTile + (int64_t)k * kThreads + wp * 32 + l;
                    acc = acc + (pos < m ? v(pos) : 0.0);
                }
                u[l] = acc;
            }
            for (int o = 16; o; o >>= 1)
                for (int l = 0; l < o; ++l) u[l] = u[l] + u[l + o];
            w[wp] = u[0];
        }
        for (int o = 4; o; o >>= 1)
            for (int k = 0; k < o; ++k) w[k] = w[k] + w[k + o];
        part[c] = w[0];
    }
    for (int64_t h = P / 2; h > 0; h >>= 1)
        for (int64_t i = 0; i < h; ++i) part[i] = part[i] + part[i + h];
    return part[0];
}

bool plane_from_moments(const double c[3], const double m[6], double out[4]) {
    const double xx = m[0], xy = m[1], xz = m[2], yy = m[3], yz = m[4], zz = m[5];
    const double det_x = yy * zz - yz * yz, det_y = xx * zz - xz * xz, det_z = xx * yy - xy * xy;
    double a, b, cc;
    if (det_x > det_y && det_x > det_z) { a = det_x; b = xz * yz - xy * zz; cc = xy * yz - xz * yy; }
    else if (det_y > det_z) { a = xz * yz - xy * zz; b = det_y; cc = xy * xz - yz * xx; }
    else { a = xy * yz - xz * yy; b = xy * xz - yz * xx; cc = det_z; }
    const double norm = std::sqrt((a * a + b * b) + cc * cc);
    if (norm == 0.0) { out[0] = out[1] = out[2] = out[3] = 0.0; return false; }
    a = a / norm; b = b / norm; cc = cc / norm;
    out[0] = a; out[1] = b; out[2] = cc;
    out[3] = -((a * c[0] + b * c[1]) + cc * c[2]);
    return true;
}

void sample(int64_t n, int r, uint64_t seed, int64_t h, int64_t* s) {
    for (int k = 0; k < r; ++k) {
        const int64_t j = n - r + k;
        int64_t t = (int64_t)std::floor(u01(seed, (uint64_t)h * (uint64_t)r + (uint64_t)k) * (double)(j + 1));
        if (t > j) t = j;
        for (int e = 0; e < k; ++e)
            if (s[e] == t) { t = j; break; }
        s[k] = t;
    }
}

// hypothesis h's plane (all zero = invalid)
void hypothesis(const double* p, int64_t n, int r, uint64_t seed, int64_t h, double pl[4]) {
    int64_t s[16];
    sample(n, r, seed, h, s);
    if (r == 3) {
        const double *p0 = p + 3 * s[0], *p1 = p + 3 * s[1], *p2 = p + 3 * s[2];
        const double e0[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]}, e1[3] = {p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2]};
        double a = e0[1] * e1[2] - e0[2] * e1[1], b = e0[2] * e1[0] - e0[0] * e1[2], c = e0[0] * e1[1] - e0[1] * e1[0];
        const double norm = std::sqrt((a * a + b * b) + c * c);
        if (norm == 0.0) { pl[0] = pl[1] = pl[2] = pl[3] = 0.0; return; }
        a = a / norm; b = b / norm; c = c / norm;
        pl[0] = a; pl[1] = b; pl[2] = c;
        pl[3] = -((a * p0[0] + b * p0[1]) + c * p0[2]);
        return;
    }
    double cen[3] = {0.0, 0.0, 0.0}, m[6] = {0, 0, 0, 0, 0, 0};
    for (int k = 0; k < r; ++k)
        for (int a = 0; a < 3; ++a) cen[a] = cen[a] + p[3 * s[k] + a];
    for (int a = 0; a < 3; ++a) cen[a] = cen[a] / (double)r;
    for (int k = 0; k < r; ++k) {
        const double x = p[3 * s[k]] - cen[0], y = p[3 * s[k] + 1] - cen[1], z = p[3 * s[k] + 2] - cen[2];
        m[0] = m[0] + x * x; m[1] = m[1] + x * y; m[2] = m[2] + x * z;
        m[3] = m[3] + y * y; m[4] = m[4] + y * z; m[5] = m[5] + z * z;
    }
    plane_from_moments(cen, m, pl);
}

double plane_dist(const double pl[4], const double* q) { return std::fabs(((pl[0] * q[0] + pl[1] * q[1]) + pl[2] * q[2]) + pl[3]); }

}  // namespace

extern "C" {

int model_dbscan(const double* p, int64_t n, double eps, int64_t min_points, int32_t* labels, int32_t* n_clusters) {
    if (!(eps > 0.0) || !std::isfinite(eps) || min_points < 0 || n < 0) return -1;
    Grid g(p, n, eps);
    const double r2 = eps * eps;
    std::vector<int> lab(n, -2), nb, qnb, queue;
    std::vector<int64_t> visited(n, -1);        // nbs_visited of the cluster being grown: its label
    int cluster = 0;
    for (int64_t idx = 0; idx < n; ++idx) {
        if (lab[idx] != -2) continue;
        g.neighbours(idx, r2, nb);
        if ((int64_t)nb.size() < min_points) { lab[idx] = -1; continue; }
        queue.clear();
        visited[idx] = cluster;
        for (int j : nb)
            if (visited[j] != cluster) { visited[j] = cluster; queue.push_back(j); }
        lab[idx] = cluster;
        for (size_t qi = 0; qi < queue.size(); ++qi) {
            const int q = queue[qi];
            if (lab[q] == -1) lab[q] = cluster;
            if (lab[q] != -2) continue;
            lab[q] = cluster;
            g.neighbours(q, r2, qnb);
            if ((int64_t)qnb.size() >= min_points)
                for (int j : qnb)
                    if (visited[j] != cluster) { visited[j] = cluster; queue.push_back(j); }
        }
        ++cluster;
    }
    for (int64_t i = 0; i < n; ++i) labels[i] = lab[i];
    if (n_clusters) *n_clusters = cluster;
    return 0;
}

// planes [count][4] of hypotheses h0 .. h0 + count - 1
int model_hypothesis_planes(const double* p, int64_t n, int r, uint64_t seed, int64_t h0, int64_t count, double* planes) {
    if (r < 3 || r > 16 || n < r) return -1;
    for (int64_t k = 0; k < count; ++k) hypothesis(p, n, r, seed, h0 + k, planes + 4 * k);
    return 0;
}

// the break bound B after a replacement with this fitness
int64_t model_ransac_bound(double fitness, int r, double probability, int num_iterations) {
    if (fitness < 1.0) {
        const double q = std::log(1.0 - probability) / std::log(1.0 - std::pow(fitness, (double)r));
        return (q >= 0.0 && q < (double)num_iterations) ? (int64_t)std::floor(q) : (int64_t)num_iterations;
    }
    return 0;
}

// (count, tree sum of the inlier distances) of one plane
void model_evaluate(const double* p, int64_t n, const double pl[4], double thr, int64_t* count, double* sum) {
    int64_t c = 0;
    for (int64_t i = 0; i < n; ++i) c += plane_dist(pl, p + 3 * i) < thr;
    *count = c;
    *sum = tree_sum(n, [&](int64_t i) { const double d = plane_dist(pl, p + 3 * i); return d < thr ? d : 0.0; });
}

int model_segment_plane(const double* p, int64_t n, double thr, int r, int num_iterations, double probability, uint64_t seed,
                        double* plane_out, int64_t* inliers, int64_t* n_inliers, int32_t* n_evaluated) {
    if (!(thr >= 0.0) || !std::isfinite(thr) || r < 3 || r > 16 || num_iterations < 0 || !(probability > 0.0 && probability <= 1.0) ||
        n < r)
        return -1;
    for (int k = 0; k < 4; ++k) plane_out[k] = 0.0;
    *n_inliers = 0;
    int64_t B = INT64_MAX;
    bool have = false;
    double best_fit = 0.0, best_rmse = 0.0, best_pl[4] = {0, 0, 0, 0};
    int32_t evaluated = 0;
    constexpr int64_t kBlock = 64;               // hypotheses evaluated in parallel; the selection stays sequential
    for (int64_t h0 = 0; h0 < num_iterations && h0 <= B; h0 += kBlock) {
        const int64_t cnt = std::min<int64_t>(kBlock, num_iterations - h0);
        std::vector<double> pl(4 * cnt), sum(cnt);
        std::vector<int64_t> count(cnt);
#pragma omp parallel for schedule(dynamic, 1)
        for (int64_t w = 0; w < cnt; ++w) {
            if (h0 + w > B) continue;
            hypothesis(p, n, r, seed, h0 + w, &pl[4 * w]);
            model_evaluate(p, n, &pl[4 * w], thr, &count[w], &sum[w]);
        }
        for (int64_t w = 0; w < cnt; ++w) {
            const int64_t h = h0 + w;
            if (h > B) break;
            ++evaluated;
            const double* q = &pl[4 * w];
            if (q[0] == 0.0 && q[1] == 0.0 && q[2] == 0.0 && q[3] == 0.0) continue;
            const double fit = (double)count[w] / (double)n;
            const double rmse = count[w] > 0 ? sum[w] / std::sqrt((double)count[w]) : 0.0;
            if (fit > best_fit || (fit == best_fit && rmse < best_rmse)) {
                best_fit = fit;
                best_rmse = rmse;
                have = true;
                std::memcpy(best_pl, q, sizeof(best_pl));
                B = model_ransac_bound(fit, r, probability, num_iterations);
            }
        }
    }
    if (n_evaluated) *n_evaluated = evaluated;
    if (!have) return 0;
    int64_t m = 0;
    for (int64_t i = 0; i < n; ++i)
        if (plane_dist(best_pl, p + 3 * i) < thr) inliers[m++] = i;
    double cen[3], mom[6];
    for (int a = 0; a < 3; ++a) cen[a] = tree_sum(m, [&](int64_t k) { return p[3 * inliers[k] + a]; }) / (double)m;
    const int ta[6] = {0, 0, 0, 1, 1, 2}, tb[6] = {0, 1, 2, 1, 2, 2};
    for (int t = 0; t < 6; ++t)
        mom[t] = tree_sum(m, [&](int64_t k) {
            const double* q = p + 3 * inliers[k];
            return (q[ta[t]] - cen[ta[t]]) * (q[tb[t]] - cen[tb[t]]);
        });
    plane_from_moments(cen, mom, plane_out);
    *n_inliers = m;
    return 0;
}

}  // extern "C"
