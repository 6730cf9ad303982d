// icp_solve.h -- the point-to-plane terms and the 6x6 Gauss-Newton solve shared by the point-to-plane solvers: frame-to-model
// tracking (track.cu, all on the device) and cloud-to-cloud ICP (knn.cu, terms on the device, solve on the host), plus the
// Euler-angle update of the cloud ICP.  Every FP64 operation
// is explicit round-to-nearest with no FMA, so the device and the host (compiled with -ffp-contract=off) give the same bits.
// Plain C++ too: the CPU model of the cloud ICP (tests/models/normals_icp_model.cpp) includes this file rather than
// restating it.
#ifndef OTSLAM_ICP_SOLVE_H
#define OTSLAM_ICP_SOLVE_H
#include <cmath>

#ifdef __CUDACC__
#define OT_HD __host__ __device__
#else
#define OT_HD
#endif

namespace otslam {

constexpr double kPivotRel = 1e-10;                 // a Cholesky pivot <= kPivotRel * max diag(A) is degenerate

OT_HD inline double rn_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
OT_HD inline double rn_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
OT_HD inline double rn_sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
OT_HD inline double rn_div(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
OT_HD inline double rn_sqrt(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return std::sqrt(a);
#endif
}

// The point-to-plane terms of one correspondence, in the layout solve6 reads: p the source point at the current pose, n the
// model's normal, e = p - the model's point; r = (n0 e0 + n1 e1) + n2 e2 and J = [p x n, n].  t[stride * k] = term k:
// 0..20 J_a J_b for a <= b (row-major), 21..26 J_a r, 27 r^2, 28 1.0 (one inlier).  Terms after 28 are the caller's.
OT_HD inline void point_to_plane_terms(const double p[3], const double n[3], const double e[3], double* t, int stride) {
    const double r = rn_add(rn_add(rn_mul(n[0], e[0]), rn_mul(n[1], e[1])), rn_mul(n[2], e[2]));
    const double J[6] = {rn_sub(rn_mul(p[1], n[2]), rn_mul(p[2], n[1])), rn_sub(rn_mul(p[2], n[0]), rn_mul(p[0], n[2])),
                         rn_sub(rn_mul(p[0], n[1]), rn_mul(p[1], n[0])), n[0], n[1], n[2]};
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = a; b < 6; ++b) t[stride * k++] = rn_mul(J[a], J[b]);
#pragma unroll
    for (int a = 0; a < 6; ++a) t[stride * (21 + a)] = rn_mul(J[a], r);
    t[stride * 27] = rn_mul(r, r);
    t[stride * 28] = 1.0;
}

// Cholesky solve of A xi = -b, A from S[0..20] (upper triangle, row-major) and b = S[21..26]; false when a pivot is
// <= kPivotRel * max diag(A)
OT_HD inline bool solve6(const double* S, double xi[6]) {
    double A[6][6], L[6][6], y[6];
    int k = 0;
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) { A[i][j] = S[k]; A[j][i] = S[k]; ++k; }
    double maxd = A[0][0];
    for (int i = 1; i < 6; ++i)
        if (A[i][i] > maxd) maxd = A[i][i];
    const double thr = rn_mul(kPivotRel, maxd);
    for (int j = 0; j < 6; ++j) {
        double s = A[j][j];
        for (int c = 0; c < j; ++c) s = rn_sub(s, rn_mul(L[j][c], L[j][c]));
        if (!(s > thr)) return false;
        L[j][j] = rn_sqrt(s);
        for (int i = j + 1; i < 6; ++i) {
            double w = A[i][j];
            for (int c = 0; c < j; ++c) w = rn_sub(w, rn_mul(L[i][c], L[j][c]));
            L[i][j] = rn_div(w, L[j][j]);
        }
    }
    for (int i = 0; i < 6; ++i) {
        double w = S[21 + i];
        for (int c = 0; c < i; ++c) w = rn_sub(w, rn_mul(L[i][c], y[c]));
        y[i] = rn_div(w, L[i][i]);
    }
    for (int i = 5; i >= 0; --i) {
        double w = y[i];
        for (int c = i + 1; c < 6; ++c) w = rn_sub(w, rn_mul(L[c][i], xi[c]));
        xi[i] = rn_div(w, L[i][i]);
    }
    for (int i = 0; i < 6; ++i) xi[i] = -xi[i];
    return true;
}

// Open3D's TransformVector6dToMatrix4d on the host: R = (Rz(x2) Ry(x1)) Rx(x0) from the plain axis matrices, each 3x3
// product in index order, t = x[3..5]
inline void euler_update(const double x[6], double U[16]) {
    const double ca = std::cos(x[0]), sa = std::sin(x[0]), cb = std::cos(x[1]), sb = std::sin(x[1]), cg = std::cos(x[2]),
                 sg = std::sin(x[2]);
    const double Rz[9] = {cg, -sg, 0.0, sg, cg, 0.0, 0.0, 0.0, 1.0};
    const double Ry[9] = {cb, 0.0, sb, 0.0, 1.0, 0.0, -sb, 0.0, cb};
    const double Rx[9] = {1.0, 0.0, 0.0, 0.0, ca, -sa, 0.0, sa, ca};
    double ZY[9], R[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            ZY[3 * i + j] = rn_add(rn_add(rn_mul(Rz[3 * i], Ry[j]), rn_mul(Rz[3 * i + 1], Ry[3 + j])), rn_mul(Rz[3 * i + 2], Ry[6 + j]));
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            R[3 * i + j] = rn_add(rn_add(rn_mul(ZY[3 * i], Rx[j]), rn_mul(ZY[3 * i + 1], Rx[3 + j])), rn_mul(ZY[3 * i + 2], Rx[6 + j]));
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) U[4 * i + j] = R[3 * i + j];
        U[4 * i + 3] = x[3 + i];
    }
    U[12] = 0.0; U[13] = 0.0; U[14] = 0.0; U[15] = 1.0;
}

// C = A B for 4x4 row-major matrices, each entry ((a0 b0 + a1 b1) + a2 b2) + a3 b3
inline void matmul4(const double* A, const double* B, double* C) {
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c)
            C[4 * r + c] = rn_add(rn_add(rn_add(rn_mul(A[4 * r], B[c]), rn_mul(A[4 * r + 1], B[4 + c])), rn_mul(A[4 * r + 2], B[8 + c])),
                                  rn_mul(A[4 * r + 3], B[12 + c]));
}

}  // namespace otslam

#endif
