// Per-thread arithmetic used by the kernels: every function restates one OpenCV primitive the reference
// calls on its hot path (SURVEY.md 2.2 / Appendix A).  All f64 code here must not be contracted into FMAs
// (the library is compiled with -fmad=false) so that results match the x86 evaluation order.
#pragma once
#include <math.h>
#include <float.h>
#include <stdint.h>
#include "ab_trace.cuh"
#include "../../include/aruco_b200.h"

namespace ab {

// ---------------------------------------------------------------------------------------------------
// approxPolyDP pieces (reference call: src/markerdetector.cpp:522; OpenCV 4.13 semantics, SURVEY A.3)
// ---------------------------------------------------------------------------------------------------
// squared distance of p to the SEGMENT s-e, f64 on integer coordinates
AB_HD double seg_dist2(int px, int py, int sx, int sy, int ex, int ey) {
    double dx = (double)(ex - sx), dy = (double)(ey - sy);
    double qx = (double)(px - sx), qy = (double)(py - sy);
    double dd = dx * dx + dy * dy;
    double t = qx * dx + qy * dy;
    if (t < 0) return qx * qx + qy * qy;
    if (t > dd) {
        double fx = (double)(px - ex), fy = (double)(py - ey);
        return fx * fx + fy * fy;
    }
    double c = qx * dy - qy * dx;
    return c * c / dd;
}

// final clean-up pass of approxPolyDP over the emitted closed polygon (in place). E = eps^2.
AB_HD int dp_cleanup(int* px, int* py, int count, double E) {
    int new_count = count;
    if (count == 0) return 0;
    int pos = count - 1;
    int sx = px[pos], sy = py[pos];
    if (++pos >= count) pos = 0;
    int wpos = pos;
    int tx = px[pos], ty = py[pos];
    if (++pos >= count) pos = 0;
    for (int i = 0; i < count && new_count > 2; i++) {
        int ex = px[pos], ey = py[pos];
        if (++pos >= count) pos = 0;
        double dx = (double)(ex - sx), dy = (double)(ey - sy);
        double dist = fabs((double)(tx - sx) * dy - (double)(ty - sy) * dx);
        double sip = (double)((tx - sx) * (ex - tx) + (ty - sy) * (ey - ty));
        if (dist * dist <= 0.5 * E * (dx * dx + dy * dy) && dx != 0 && dy != 0 && sip >= 0) {
            new_count--;
            px[wpos] = sx = ex;
            py[wpos] = sy = ey;
            if (++wpos >= count) wpos = 0;
            tx = px[pos];
            ty = py[pos];
            if (++pos >= count) pos = 0;
            i++;
            continue;
        }
        px[wpos] = sx = tx;
        py[wpos] = sy = ty;
        if (++wpos >= count) wpos = 0;
        tx = ex;
        ty = ey;
    }
    return new_count;
}

// cv::isContourConvex on 4 integer points (src/markerdetector.cpp:535, SURVEY A.4)
AB_HD bool is_convex4(const int* x, const int* y) {
    int px = x[2], py = y[2], cx = x[3], cy = y[3];
    int dx0 = cx - px, dy0 = cy - py;
    int orientation = 0;
    for (int i = 0; i < 4; i++) {
        px = cx;
        py = cy;
        cx = x[i];
        cy = y[i];
        int dx = cx - px, dy = cy - py;
        long long dxdy0 = (long long)dx * dy0, dydx0 = (long long)dy * dx0;
        orientation |= (dydx0 > dxdy0) ? 1 : ((dydx0 < dxdy0) ? 2 : 3);
        if (orientation == 3) return false;
        dx0 = dx;
        dy0 = dy;
    }
    return true;
}

// aruco::perimeter (src/utils.h:37-44): f64 norms of f32 differences summed into an f32
AB_HD float perimeter4(const float* c) {
    float sum = 0.f;
    for (int i = 0; i < 4; i++) {
        int j = (i + 1) & 3;
        float dx = c[2 * i] - c[2 * j], dy = c[2 * i + 1] - c[2 * j + 1];
        sum = (float)((double)sum + sqrt((double)dx * (double)dx + (double)dy * (double)dy));
    }
    return sum;
}

// ---------------------------------------------------------------------------------------------------
// getPerspectiveTransform + warpPerspective(INTER_NEAREST) (src/markerdetector.cpp:684-697, A.5/A.6)
// ---------------------------------------------------------------------------------------------------
// Gaussian elimination with partial pivoting in the operation order of OpenCV's LUImpl<double>.
AB_HD bool lu_solve8(double A[8][8], double b[8]) {
    for (int i = 0; i < 8; i++) {
        int k = i;
        for (int j = i + 1; j < 8; j++)
            if (fabs(A[j][i]) > fabs(A[k][i])) k = j;
        if (fabs(A[k][i]) < DBL_EPSILON * 100) return false;
        if (k != i) {
            for (int j = i; j < 8; j++) {
                double t = A[i][j];
                A[i][j] = A[k][j];
                A[k][j] = t;
            }
            double t = b[i];
            b[i] = b[k];
            b[k] = t;
        }
        double d = -1 / A[i][i];
        for (int j = i + 1; j < 8; j++) {
            double alpha = A[j][i] * d;
            for (int c = i + 1; c < 8; c++) A[j][c] += alpha * A[i][c];
            b[j] += alpha * b[i];
        }
    }
    for (int i = 7; i >= 0; i--) {
        double s = b[i];
        for (int c = i + 1; c < 8; c++) s -= A[i][c] * b[c];
        b[i] = s / A[i][i];
    }
    return true;
}

// M maps src quad -> dst quad (both 4x(x,y)); row-major 3x3 with M[8] = 1
AB_HD bool perspective_transform(const float* src, const float* dst, double* M) {
    double a[8][8], b[8];
    for (int i = 0; i < 4; i++) {
        float sx = src[2 * i], sy = src[2 * i + 1], dx = dst[2 * i], dy = dst[2 * i + 1];
        a[i][0] = a[i + 4][3] = sx;
        a[i][1] = a[i + 4][4] = sy;
        a[i][2] = a[i + 4][5] = 1;
        a[i][3] = a[i][4] = a[i][5] = a[i + 4][0] = a[i + 4][1] = a[i + 4][2] = 0;
        a[i][6] = (double)(-sx * dx);
        a[i][7] = (double)(-sy * dx);
        a[i + 4][6] = (double)(-sx * dy);
        a[i + 4][7] = (double)(-sy * dy);
        b[i] = dx;
        b[i + 4] = dy;
    }
    if (!lu_solve8(a, b)) return false;
    for (int i = 0; i < 8; i++) M[i] = b[i];
    M[8] = 1.0;
    return true;
}

// closed-form 3x3 inverse as cv::invert does for 3x3 (adjugate * 1/det)
AB_HD bool invert3(const double* m, double* t) {
    double d = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
    if (d == 0.) return false;
    d = 1. / d;
    t[0] = (m[4] * m[8] - m[5] * m[7]) * d;
    t[1] = (m[2] * m[7] - m[1] * m[8]) * d;
    t[2] = (m[1] * m[5] - m[2] * m[4]) * d;
    t[3] = (m[5] * m[6] - m[3] * m[8]) * d;
    t[4] = (m[0] * m[8] - m[2] * m[6]) * d;
    t[5] = (m[2] * m[3] - m[0] * m[5]) * d;
    t[6] = (m[3] * m[7] - m[4] * m[6]) * d;
    t[7] = (m[1] * m[6] - m[0] * m[7]) * d;
    t[8] = (m[0] * m[4] - m[1] * m[3]) * d;
    return true;
}

AB_HD double clamp_int_range(double v) { return v < -2147483648.0 ? -2147483648.0 : (v > 2147483647.0 ? 2147483647.0 : v); }

// source pixel of destination pixel (x,y) under inverse map Mi; OpenCV processes the row in blocks of
// `bw` columns whose origin bx enters the affine part first (block size rule of WarpPerspectiveInvoker).
AB_HD void warp_src_coord(const double* Mi, int x, int y, int bw, int* sx, int* sy) {
    int bx = (x / bw) * bw, x1 = x - bx;
    double X0 = Mi[0] * bx + Mi[1] * y + Mi[2];
    double Y0 = Mi[3] * bx + Mi[4] * y + Mi[5];
    double W0 = Mi[6] * bx + Mi[7] * y + Mi[8];
    double W = W0 + Mi[6] * x1;
    W = W ? 1. / W : 0;
    double fX = clamp_int_range((X0 + Mi[0] * x1) * W);
    double fY = clamp_int_range((Y0 + Mi[3] * x1) * W);
    *sx = (int)rint(fX);
    *sy = (int)rint(fY);
}

AB_HD int warp_block_width(int S) {
    int bh0 = 16 < S ? 16 : S;
    int bw0 = (1024 / bh0) < S ? (1024 / bh0) : S;
    return bw0;
}

// ---------------------------------------------------------------------------------------------------
// threshold(BINARY|OTSU) threshold value from a 256-bin histogram of N samples (SURVEY A.7)
// ---------------------------------------------------------------------------------------------------
AB_HD int otsu_threshold(const int* h, int N) {
    double mu = 0, scale = 1. / N;
    for (int i = 0; i < 256; i++) mu += i * (double)h[i];
    mu *= scale;
    double mu1 = 0, q1 = 0, max_sigma = 0, max_val = 0;
    for (int i = 0; i < 256; i++) {
        double p_i = h[i] * scale;
        mu1 *= q1;
        q1 += p_i;
        double q2 = 1. - q1;
        double mn = q1 < q2 ? q1 : q2, mx = q1 < q2 ? q2 : q1;
        if (mn < FLT_EPSILON || mx > 1. - FLT_EPSILON) continue;
        mu1 = (mu1 + i * p_i) / q1;
        double mu2 = (mu - q1 * mu1) / q2;
        double sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2);
        if (sigma > max_sigma) {
            max_sigma = sigma;
            max_val = i;
        }
    }
    return (int)max_val;
}

// ---------------------------------------------------------------------------------------------------
// FiducidalMarkers decode from the 7x7 cell majority bits (src/arucofidmarkers.cpp:100-137, 168-184)
// cells[y*7+x] = 1 when the cell is white.  Returns id or -1; *nrot in 0..3.
// ---------------------------------------------------------------------------------------------------
AB_HD int fid_row_dist(int bits5) {
    // words 10000 10111 01001 01110 (bit 4 = column 0)
    const int w[4] = {0x10, 0x17, 0x09, 0x0E};
    int best = 100000;
    for (int p = 0; p < 4; p++) {
#if defined(__CUDA_ARCH__)
        int d = __popc((unsigned)(bits5 ^ w[p]));
#else
        int d = __builtin_popcount((unsigned)(bits5 ^ w[p]));
#endif
        if (d < best) best = d;
    }
    return best;
}

AB_HD int fid_decode(const uint8_t* cells, int* nrot) {
    *nrot = 0;  // SURVEY B.1
    for (int y = 0; y < 7; y++) {
        int inc = (y == 0 || y == 6) ? 1 : 6;
        for (int x = 0; x < 7; x += inc)
            if (cells[y * 7 + x]) return -1;
    }
    uint8_t cur[25], nxt[25];
    for (int y = 0; y < 5; y++)
        for (int x = 0; x < 5; x++) cur[y * 5 + x] = cells[(y + 1) * 7 + x + 1];
    int minDist = 1 << 30, bestRot = 0;
    uint8_t best[25];
    for (int r = 0; r < 4; r++) {
        if (r > 0) {
            for (int i = 0; i < 5; i++)
                for (int j = 0; j < 5; j++) nxt[i * 5 + j] = cur[(5 - j - 1) * 5 + i];
            for (int i = 0; i < 25; i++) cur[i] = nxt[i];
        }
        int dist = 0;
        for (int y = 0; y < 5; y++) {
            int v = 0;
            for (int x = 0; x < 5; x++) v = (v << 1) | cur[y * 5 + x];
            dist += fid_row_dist(v);
        }
        if (dist < minDist) {
            minDist = dist;
            bestRot = r;
            for (int i = 0; i < 25; i++) best[i] = cur[i];
        }
    }
    *nrot = bestRot;
    if (minDist != 0) return -1;
    int id = 0;
    for (int y = 0; y < 5; y++) id |= ((best[y * 5 + 1] << 1) | best[y * 5 + 3]) << (2 * (4 - y));
    return id;
}

// ---------------------------------------------------------------------------------------------------
// HRM: bit strings / folded ids of the 4 rotations (src/highlyreliablemarkers.cpp:149-180, SURVEY B.4)
// code[y*n+x] in {0,1}; bits[r] has bit pos set for rotation r; ids[r] = OR-fold with x86 shift semantics
// ---------------------------------------------------------------------------------------------------
AB_HD void hrm_rotations(const uint8_t* code, int n, uint64_t bits[4], uint32_t ids[4]) {
    for (int r = 0; r < 4; r++) {
        bits[r] = 0;
        ids[r] = 0;
    }
    for (int y = 0; y < n; y++)
        for (int x = 0; x < n; x++) {
            if (!code[y * n + x]) continue;
            for (int r = 0; r < 4; r++) {
                int _x = x, _y = y;
                if (r == 1) {
                    _y = x;
                    _x = n - y - 1;
                } else if (r == 2) {
                    _y = n - y - 1;
                    _x = n - x - 1;
                } else if (r == 3) {
                    _y = n - x - 1;
                    _x = y;
                }
                int pos = _y * n + _x;
                bits[r] |= (uint64_t)1 << pos;
                int sh = pos & 31;
                ids[r] |= (sh == 31) ? 0u : (2u << sh);
            }
        }
}

// ---------------------------------------------------------------------------------------------------
// Camera model helpers (K, D arrive as f32 and are widened; SURVEY A.12)
// ---------------------------------------------------------------------------------------------------
struct Camera {
    double fx, fy, cx, cy;
    double k1, k2, p1, p2, k3;
    float fxf, fyf, cxf, cyf;
    int has_K, has_D;
    int zero_D;  // all distortion coefficients are 0: cv::undistortPoints is then the identity on pixel coordinates
                 // after its f32 rounding ((u - cx) / fx * fx + cx is within 1e-12 of u, f32 spacing is >= 6e-5)
};

// cv::undistortPoints(src, K, D, R=I, P=K): 5 fixed-point iterations, result rounded to f32
AB_HD void undistort_point_px(const Camera& c, float u, float v, float* ou, float* ov) {
    double x0 = ((double)u - c.cx) / c.fx, y0 = ((double)v - c.cy) / c.fy;
    double x = x0, y = y0;
    for (int j = 0; j < 5; j++) {
        double r2 = x * x + y * y;
        double icdist = 1. / (1 + ((c.k3 * r2 + c.k2) * r2 + c.k1) * r2);
        double deltaX = 2 * c.p1 * x * y + c.p2 * (r2 + 2 * x * x);
        double deltaY = c.p1 * (r2 + 2 * y * y) + 2 * c.p2 * x * y;
        x = (x0 - deltaX) * icdist;
        y = (y0 - deltaY) * icdist;
    }
    *ou = (float)(x * c.fx + c.cx);
    *ov = (float)(y * c.fy + c.cy);
}

// same iteration but returning normalised coordinates in f64 (used by the pose initialisation)
AB_HD void undistort_point_norm(const Camera& c, double u, double v, double* ox, double* oy) {
    double x0 = (u - c.cx) / c.fx, y0 = (v - c.cy) / c.fy;
    double x = x0, y = y0;
    for (int j = 0; j < (c.zero_D ? 0 : 20); j++) {  // zero coefficients: every iteration returns (x0, y0) exactly
        double r2 = x * x + y * y;
        double icdist = 1. / (1 + ((c.k3 * r2 + c.k2) * r2 + c.k1) * r2);
        double deltaX = 2 * c.p1 * x * y + c.p2 * (r2 + 2 * x * x);
        double deltaY = c.p1 * (r2 + 2 * y * y) + 2 * c.p2 * x * y;
        x = (x0 - deltaX) * icdist;
        y = (y0 - deltaY) * icdist;
    }
    *ox = x;
    *oy = y;
}

// forward distortion of a normalised point, pixel output in f64
AB_HD void distort_norm_to_px(const Camera& c, double x, double y, double* u, double* v) {
    double r2 = x * x + y * y, r4 = r2 * r2, r6 = r4 * r2;
    double a1 = 2 * x * y, a2 = r2 + 2 * x * x, a3 = r2 + 2 * y * y;
    double cdist = 1 + c.k1 * r2 + c.k2 * r4 + c.k3 * r6;
    double xd = x * cdist + c.p1 * a1 + c.p2 * a2;
    double yd = y * cdist + c.p1 * a3 + c.p2 * a1;
    *u = xd * c.fx + c.cx;
    *v = yd * c.fy + c.cy;
}

// ---------------------------------------------------------------------------------------------------
// cv::solve(A, B, X, DECOMP_SVD) in CV_32F as the LINES refinement uses it (src/markerdetector.cpp:112,124,138):
// OpenCV's one-sided Jacobi SVD on the two columns of A (f32 rotations, f64 dot products, eps = 2*FLT_EPSILON)
// followed by its back substitution (f32 products accumulated in f64).  The pieces below are shared by the scalar
// 2x2 solve of getCrossPoint and by the warp-parallel m x 2 fit in k_refine_lines.

// Jacobi rotation (c, s) that orthogonalises two columns with squared norms a, b and dot product p
AB_HD void jacobi_rotation_f32(double a, double b, double p, float* c, float* s) {
    p *= 2;
    double beta = a - b, gamma = hypot(p, beta);
    if (beta < 0) {
        double delta = (gamma - beta) * 0.5;
        *s = (float)sqrt(delta / gamma);
        *c = (float)(p / (gamma * (double)*s * 2));
    } else {
        *c = (float)sqrt((gamma + beta) / (gamma * 2));
        *s = (float)(p / (gamma * (double)*c * 2));
    }
}

// X = V * diag(1/w) * U^T b from the two singular triplets (SVBkSb): W2 = squared column norms after the last sweep,
// ub[i] = sum_j (u_i[j] * b[j]) with u_i = column i scaled by sc[i] (see jacobi_scales_f32), Vt rows = right vectors
// returns the index of the larger singular value (they are used in descending order)
AB_HD int jacobi_scales_f32(const double W2[2], float w[2], float sc[2]) {
    double sd[2];
    for (int i = 0; i < 2; i++) {
        sd[i] = sqrt(W2[i]);
        w[i] = (float)sd[i];
        sc[i] = (float)(sd[i] > (double)FLT_MIN ? 1 / sd[i] : 0.);
    }
    return sd[0] < sd[1] ? 1 : 0;
}
AB_HD void jacobi_backsubst_f32(int o0, const float w[2], const double ub[2], const float Vt[2][2], float X[2]) {
    const int ord[2] = {o0, 1 - o0};
    const double threshold = ((double)w[0] + (double)w[1]) * (double)(float)(DBL_EPSILON * 2);
    X[0] = X[1] = 0.f;
    for (int k = 0; k < 2; k++) {
        const int i = ord[k];
        double wi = w[i];
        if (fabs(wi) <= threshold) continue;
        double sv = ub[i] * (1 / wi);
        for (int j = 0; j < 2; j++) X[j] = (float)((double)X[j] + sv * (double)Vt[i][j]);
    }
}

// getCrossPoint (src/markerdetector.cpp:132-139): Matx22f(l1.x, l1.y; l2.x, l2.y).solve(Vec2f(-l1.z, -l2.z), DECOMP_SVD)
AB_HD void cross_point_f32(const float* l1, const float* l2, float* x, float* y) {
    float A0[2] = {l1[0], l2[0]}, A1[2] = {l1[1], l2[1]};
    const float rhs[2] = {-l1[2], -l2[2]};
    float Vt[2][2] = {{1.f, 0.f}, {0.f, 1.f}};
    double W2[2] = {(double)A0[0] * A0[0] + (double)A0[1] * A0[1], (double)A1[0] * A1[0] + (double)A1[1] * A1[1]};
    for (int iter = 0; iter < 30; iter++) {
        double p = (double)A0[0] * A1[0] + (double)A0[1] * A1[1];
        if (fabs(p) <= (double)(FLT_EPSILON * 2) * sqrt(W2[0] * W2[1])) break;
        float c, s;
        jacobi_rotation_f32(W2[0], W2[1], p, &c, &s);
        double a = 0, b = 0;
        for (int k = 0; k < 2; k++) {
            float t0 = c * A0[k] + s * A1[k], t1 = -s * A0[k] + c * A1[k];
            A0[k] = t0;
            A1[k] = t1;
            a += (double)t0 * t0;
            b += (double)t1 * t1;
            float v0 = c * Vt[0][k] + s * Vt[1][k], v1 = -s * Vt[0][k] + c * Vt[1][k];
            Vt[0][k] = v0;
            Vt[1][k] = v1;
        }
        W2[0] = a;
        W2[1] = b;
    }
    float w[2], sc[2], X[2];
    const int o0 = jacobi_scales_f32(W2, w, sc);
    double ub[2] = {0, 0};
    for (int k = 0; k < 2; k++) {
        ub[0] += (double)((A0[k] * sc[0]) * rhs[k]);
        ub[1] += (double)((A1[k] * sc[1]) * rhs[k]);
    }
    jacobi_backsubst_f32(o0, w, ub, Vt, X);
    *x = X[0];
    *y = X[1];
}

// ---------------------------------------------------------------------------------------------------
// Pose: cv::solvePnP(SOLVEPNP_ITERATIVE) for 4 coplanar points (src/markerdetector.cpp:458, marker.cpp:118)
// planar homography initialisation + Levenberg-Marquardt on the pixel reprojection error (SURVEY A.9)
// ---------------------------------------------------------------------------------------------------
AB_HD void rodrigues_to_mat(const double* r, double* R) {
    double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    if (theta < DBL_EPSILON) {
        R[0] = R[4] = R[8] = 1;
        R[1] = R[2] = R[3] = R[5] = R[6] = R[7] = 0;
        return;
    }
    double c = cos(theta), s = sin(theta), c1 = 1. - c, it = 1. / theta;
    double x = r[0] * it, y = r[1] * it, z = r[2] * it;
    R[0] = c + c1 * x * x;
    R[1] = c1 * x * y - s * z;
    R[2] = c1 * x * z + s * y;
    R[3] = c1 * x * y + s * z;
    R[4] = c + c1 * y * y;
    R[5] = c1 * y * z - s * x;
    R[6] = c1 * x * z - s * y;
    R[7] = c1 * y * z + s * x;
    R[8] = c + c1 * z * z;
}

// rotation matrix (already orthonormal) -> Rodrigues vector, cv::Rodrigues conventions incl. theta ~ pi
AB_HD void mat_to_rodrigues(const double* R, double* r) {
    double rx = R[7] - R[5], ry = R[2] - R[6], rz = R[3] - R[1];
    double s = sqrt((rx * rx + ry * ry + rz * rz) * 0.25);
    double c = (R[0] + R[4] + R[8] - 1) * 0.5;
    c = c > 1. ? 1. : (c < -1. ? -1. : c);
    double theta = acos(c);
    if (s < 1e-5) {
        if (c > 0) {
            r[0] = r[1] = r[2] = 0;
        } else {
            double t = (R[0] + 1) * 0.5;
            rx = sqrt(t > 0 ? t : 0);
            t = (R[4] + 1) * 0.5;
            ry = sqrt(t > 0 ? t : 0) * (R[1] < 0 ? -1. : 1.);
            t = (R[8] + 1) * 0.5;
            rz = sqrt(t > 0 ? t : 0) * (R[2] < 0 ? -1. : 1.);
            if (fabs(rx) < fabs(ry) && fabs(rx) < fabs(rz) && (R[5] > 0) != (ry * rz > 0)) rz = -rz;
            theta /= sqrt(rx * rx + ry * ry + rz * rz);
            r[0] = rx * theta;
            r[1] = ry * theta;
            r[2] = rz * theta;
        }
    } else {
        double vth = 1 / (2 * s);
        vth *= theta;
        r[0] = rx * vth;
        r[1] = ry * vth;
        r[2] = rz * vth;
    }
}

AB_HD void mat3_inv_transpose(const double* m, double* o) {
    // o = (m^-1)^T = cofactor(m) / det
    double c0 = m[4] * m[8] - m[5] * m[7], c1 = m[5] * m[6] - m[3] * m[8], c2 = m[3] * m[7] - m[4] * m[6];
    double det = m[0] * c0 + m[1] * c1 + m[2] * c2;
    double id = 1. / det;
    o[0] = c0 * id;
    o[1] = c1 * id;
    o[2] = c2 * id;
    o[3] = (m[2] * m[7] - m[1] * m[8]) * id;
    o[4] = (m[0] * m[8] - m[2] * m[6]) * id;
    o[5] = (m[1] * m[6] - m[0] * m[7]) * id;
    o[6] = (m[1] * m[5] - m[2] * m[4]) * id;
    o[7] = (m[2] * m[3] - m[0] * m[5]) * id;
    o[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// nearest rotation (polar factor U*V^T of the SVD) by Newton iteration R <- (R + R^-T)/2
AB_HD void orthonormalize3(double* R) {
    for (int it = 0; it < 30; it++) {
        double T[9], diff = 0;
        mat3_inv_transpose(R, T);
        for (int i = 0; i < 9; i++) {
            double n = 0.5 * (R[i] + T[i]);
            diff += fabs(n - R[i]);
            R[i] = n;
        }
        if (diff < 1e-15) break;
    }
}

AB_HD void project_marker(const Camera& cam, const double* p, const float* obj, double* uv) {
    double R[9];
    rodrigues_to_mat(p, R);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        double X = obj[3 * i], Y = obj[3 * i + 1], Z = obj[3 * i + 2];
        double x = R[0] * X + R[1] * Y + R[2] * Z + p[3];
        double y = R[3] * X + R[4] * Y + R[5] * Z + p[4];
        double z = R[6] * X + R[7] * Y + R[8] * Z + p[5];
        z = z ? 1. / z : 1.;
        x *= z;
        y *= z;
        distort_norm_to_px(cam, x, y, &uv[2 * i], &uv[2 * i + 1]);
    }
}

// residual (projection - measurement) of the 4 marker corners for pose p = (rvec, tvec)
AB_HD void pnp_residual(const Camera& cam, const double* p, const float* obj, const double* m, double* err) {
    double uv[8];
    project_marker(cam, p, obj, uv);
    for (int i = 0; i < 8; i++) err[i] = uv[i] - m[i];
}

// d(rotation matrix)/d(rvec): dR[k][i] = dR_i/dr_k (cvRodrigues2 jacobian), analytic
AB_HD void rodrigues_jacobian(const double* r, double* R, double dR[3][9]) {
    double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    if (theta < DBL_EPSILON) {
        for (int i = 0; i < 9; i++) R[i] = (i % 4 == 0) ? 1. : 0.;
        for (int k = 0; k < 3; k++)
            for (int i = 0; i < 9; i++) dR[k][i] = 0;
        dR[0][5] = -1; dR[0][7] = 1;
        dR[1][2] = 1;  dR[1][6] = -1;
        dR[2][1] = -1; dR[2][3] = 1;
        return;
    }
    double c = cos(theta), s = sin(theta), c1 = 1. - c, it = 1. / theta;
    double rv[3] = {r[0] * it, r[1] * it, r[2] * it};
    double rrt[9], rx[9] = {0, -rv[2], rv[1], rv[2], 0, -rv[0], -rv[1], rv[0], 0};
    const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) rrt[i * 3 + j] = rv[i] * rv[j];
#pragma unroll
    for (int i = 0; i < 9; i++) R[i] = c * I[i] + c1 * rrt[i] + s * rx[i];
    // R = c I + (1-c) n n^T + s [n]x with n = r/theta
#pragma unroll
    for (int k = 0; k < 3; k++) {
        // dtheta/dr_k = n_k ; dn_i/dr_k = (delta_ik - n_i n_k)/theta
        double dn[3];
#pragma unroll
        for (int i = 0; i < 3; i++) dn[i] = ((i == k ? 1. : 0.) - rv[i] * rv[k]) * it;
        double drrt[9], drx[9] = {0, -dn[2], dn[1], dn[2], 0, -dn[0], -dn[1], dn[0], 0};
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
            for (int j = 0; j < 3; j++) drrt[i * 3 + j] = dn[i] * rv[j] + rv[i] * dn[j];
#pragma unroll
        for (int i = 0; i < 9; i++)
            dR[k][i] = rv[k] * (-s * I[i] + s * rrt[i] + c * rx[i]) + c1 * drrt[i] + s * drx[i];
    }
}

// residual and analytic Jacobian d(u,v)/d(rvec,tvec) (cvProjectPoints2 with dpdr, dpdt)
AB_HD void pnp_residual_jacobian(const Camera& cam, const double* p, const float* obj, const double* m, double* err,
                                 double J[8][6]) {
    double R[9], dR[3][9];
    rodrigues_jacobian(p, R, dR);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        double X = obj[3 * i], Y = obj[3 * i + 1], Z = obj[3 * i + 2];
        double x = R[0] * X + R[1] * Y + R[2] * Z + p[3];
        double y = R[3] * X + R[4] * Y + R[5] * Z + p[4];
        double z = R[6] * X + R[7] * Y + R[8] * Z + p[5];
        double iz = z ? 1. / z : 1.;
        double xn = x * iz, yn = y * iz;
        double r2 = xn * xn + yn * yn, r4 = r2 * r2, r6 = r4 * r2;
        double a1 = 2 * xn * yn, a2 = r2 + 2 * xn * xn, a3 = r2 + 2 * yn * yn;
        double cdist = 1 + cam.k1 * r2 + cam.k2 * r4 + cam.k3 * r6;
        double dc = cam.k1 + 2 * cam.k2 * r2 + 3 * cam.k3 * r4;  // d cdist / d r2
        double xd = xn * cdist + cam.p1 * a1 + cam.p2 * a2, yd = yn * cdist + cam.p1 * a3 + cam.p2 * a1;
        err[2 * i] = xd * cam.fx + cam.cx - m[2 * i];
        err[2 * i + 1] = yd * cam.fy + cam.cy - m[2 * i + 1];
        // d(xd,yd)/d(xn,yn)
        double dxdx = cdist + 2 * xn * xn * dc + 2 * cam.p1 * yn + 6 * cam.p2 * xn;
        double dxdy = 2 * xn * yn * dc + 2 * cam.p1 * xn + 2 * cam.p2 * yn;
        double dydx = 2 * xn * yn * dc + 2 * cam.p1 * xn + 2 * cam.p2 * yn;
        double dydy = cdist + 2 * yn * yn * dc + 6 * cam.p1 * yn + 2 * cam.p2 * xn;
        // d(xn,yn)/d(x,y,z)
        double dxn[3] = {iz, 0, -xn * iz}, dyn[3] = {0, iz, -yn * iz};
        double du[3], dv[3];  // d(u,v)/d(camera point)
#pragma unroll
        for (int c = 0; c < 3; c++) {
            du[c] = cam.fx * (dxdx * dxn[c] + dxdy * dyn[c]);
            dv[c] = cam.fy * (dydx * dxn[c] + dydy * dyn[c]);
        }
#pragma unroll
        for (int k = 0; k < 3; k++) {
            double dX[3] = {dR[k][0] * X + dR[k][1] * Y + dR[k][2] * Z, dR[k][3] * X + dR[k][4] * Y + dR[k][5] * Z,
                            dR[k][6] * X + dR[k][7] * Y + dR[k][8] * Z};
            J[2 * i][k] = du[0] * dX[0] + du[1] * dX[1] + du[2] * dX[2];
            J[2 * i + 1][k] = dv[0] * dX[0] + dv[1] * dX[1] + dv[2] * dX[2];
            J[2 * i][3 + k] = du[k];
            J[2 * i + 1][3 + k] = dv[k];
        }
    }
}

AB_HD bool solve6(double A[6][6], double* b) {
    for (int i = 0; i < 6; i++) {
        int k = i;
        for (int j = i + 1; j < 6; j++)
            if (fabs(A[j][i]) > fabs(A[k][i])) k = j;
        if (fabs(A[k][i]) < 1e-300) return false;
        if (k != i) {
            for (int j = 0; j < 6; j++) {
                double t = A[i][j];
                A[i][j] = A[k][j];
                A[k][j] = t;
            }
            double t = b[i];
            b[i] = b[k];
            b[k] = t;
        }
        for (int j = i + 1; j < 6; j++) {
            double f = A[j][i] / A[i][i];
            for (int c = i; c < 6; c++) A[j][c] -= f * A[i][c];
            b[j] -= f * b[i];
        }
    }
    for (int i = 5; i >= 0; i--) {
        double s = b[i];
        for (int c = i + 1; c < 6; c++) s -= A[i][c] * b[c];
        b[i] = s / A[i][i];
    }
    return true;
}

// A x = b for the symmetric positive definite 6x6 system of a damped Gauss-Newton step (J^T J with its diagonal scaled by
// 1 + lambda): Cholesky with every index known at compile time, so the factor lives in registers (the pivoting LU above
// indexes its rows dynamically, which puts the matrix into local memory: one L1 round trip per access in the middle of the
// dependent chain of a Levenberg-Marquardt iteration).  Only the upper triangle of A is read.  Returns false when a pivot
// is not positive (degenerate geometry); the caller then falls back to the pivoting solver.
AB_HD bool solve6_spd(const double A[6][6], double* b) {
    double L[6][6];
#pragma unroll
    for (int j = 0; j < 6; j++) {
        double d = A[j][j];
#pragma unroll
        for (int k = 0; k < j; k++) d -= L[j][k] * L[j][k];
        if (!(d > 0.0)) return false;
        const double inv = 1.0 / sqrt(d);
        L[j][j] = inv;  // the reciprocal of the diagonal entry
#pragma unroll
        for (int i = j + 1; i < 6; i++) {
            double v = A[j][i];
#pragma unroll
            for (int k = 0; k < j; k++) v -= L[i][k] * L[j][k];
            L[i][j] = v * inv;
        }
    }
#pragma unroll
    for (int i = 0; i < 6; i++) {  // L y = b
        double v = b[i];
#pragma unroll
        for (int k = 0; k < i; k++) v -= L[i][k] * b[k];
        b[i] = v * L[i][i];
    }
#pragma unroll
    for (int i = 5; i >= 0; i--) {  // L^T x = y
        double v = b[i];
#pragma unroll
        for (int k = i + 1; k < 6; k++) v -= L[k][i] * b[k];
        b[i] = v * L[i][i];
    }
    return true;
}

// corners: 4 x (u,v) f32 in the reference's order; size = marker side; out rvec/tvec f64.
AB_HD bool solve_pnp_marker(const Camera& cam, const float* corners, float size, double* rvec, double* tvec) {
    float h = size / 2.f;  // getObjectPoints, src/marker.cpp:91-108
    float obj[12] = {-h, -h, 0, -h, h, 0, h, h, 0, h, -h, 0};
    // 1. normalised image points
    float nsrc[8], ndst[8];
    double xn[8];
    for (int i = 0; i < 4; i++) {
        undistort_point_norm(cam, corners[2 * i], corners[2 * i + 1], &xn[2 * i], &xn[2 * i + 1]);
        nsrc[2 * i] = obj[3 * i];
        nsrc[2 * i + 1] = obj[3 * i + 1];
    }
    // 2. exact 4-point homography object plane -> normalised image (f64 system)
    double a[8][8], b[8];
    for (int i = 0; i < 4; i++) {
        double sx = nsrc[2 * i], sy = nsrc[2 * i + 1], dx = xn[2 * i], dy = xn[2 * i + 1];
        for (int c = 0; c < 8; c++) a[i][c] = a[i + 4][c] = 0;
        a[i][0] = a[i + 4][3] = sx;
        a[i][1] = a[i + 4][4] = sy;
        a[i][2] = a[i + 4][5] = 1;
        a[i][6] = -sx * dx;
        a[i][7] = -sy * dx;
        a[i + 4][6] = -sx * dy;
        a[i + 4][7] = -sy * dy;
        b[i] = dx;
        b[i + 4] = dy;
    }
    (void)ndst;
    if (!lu_solve8(a, b)) return false;
    double h1[3] = {b[0], b[3], b[6]}, h2[3] = {b[1], b[4], b[7]}, h3[3] = {b[2], b[5], 1.0};
    double n1 = sqrt(h1[0] * h1[0] + h1[1] * h1[1] + h1[2] * h1[2]);
    double n2 = sqrt(h2[0] * h2[0] + h2[1] * h2[1] + h2[2] * h2[2]);
    if (!(n1 > DBL_EPSILON) || !(n2 > DBL_EPSILON)) return false;
    for (int i = 0; i < 3; i++) {
        h1[i] /= n1;
        h2[i] /= n2;
    }
    double sc = 2. / (n1 + n2);
    double p[6];
    p[3] = h3[0] * sc;
    p[4] = h3[1] * sc;
    p[5] = h3[2] * sc;
    double c3[3] = {h1[1] * h2[2] - h1[2] * h2[1], h1[2] * h2[0] - h1[0] * h2[2], h1[0] * h2[1] - h1[1] * h2[0]};
    double R[9] = {h1[0], h2[0], c3[0], h1[1], h2[1], c3[1], h1[2], h2[2], c3[2]};
    orthonormalize3(R);
    mat_to_rodrigues(R, p);
    // 3. Levenberg-Marquardt exactly as OpenCV's CvLevMarq drives it inside cvFindExtrinsicCameraParams2:
    //    lambda = 10^k (k starts at -3), diag(JtJ) *= 1 + lambda, step = param - solve(JtJN, Jt err); a step
    //    that raises |err| is retried with k+1 (up to 16), an accepted one lowers k; stop after 20 accepted
    //    steps or when |param - prev| / |prev| < FLT_EPSILON.  Matching the trajectory (not just the
    //    minimum) matters: near-frontal markers have two pose minima and 20 iterations may not converge.
    double m[8];
    for (int i = 0; i < 8; i++) m[i] = corners[i];
    double J[8][6], err[8], JtJ[6][6], JtErr[6], prev[6];
    int lambdaLg10 = -3, iters = 0;
    double prevErrNorm = 0;
    pnp_residual_jacobian(cam, p, obj, m, err, J);
    for (;;) {
        // state CALC_J (J^T J is symmetric: the upper triangle is computed, the lower mirrored)
#pragma unroll
        for (int i = 0; i < 6; i++) {
            double s = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) s += J[k][i] * err[k];
            JtErr[i] = s;
#pragma unroll
            for (int j = i; j < 6; j++) {
                double q = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) q += J[k][i] * J[k][j];
                JtJ[i][j] = q;
                JtJ[j][i] = q;
            }
            prev[i] = p[i];
        }
        if (iters == 0) {
            double s = 0;
            for (int k = 0; k < 8; k++) s += err[k] * err[k];
            prevErrNorm = sqrt(s);
        }
        double errNorm = 0;
        for (;;) {
            double lambda = exp(lambdaLg10 * 2.302585092994046);
            double A[6][6], d[6];
#pragma unroll
            for (int i = 0; i < 6; i++) {
#pragma unroll
                for (int j = 0; j < 6; j++) A[i][j] = JtJ[i][j];
                A[i][i] *= 1. + lambda;
                d[i] = JtErr[i];
            }
            if (!solve6_spd(A, d)) {  // cold path: its dynamically indexed copy keeps `A` itself in registers
                double A2[6][6];
                for (int i = 0; i < 6; i++) {
                    for (int j = 0; j < 6; j++) A2[i][j] = JtJ[i][j];
                    A2[i][i] *= 1. + lambda;
                    d[i] = JtErr[i];
                }
                if (!solve6(A2, d))
                    for (int i = 0; i < 6; i++) d[i] = 0;
            }
            for (int i = 0; i < 6; i++) p[i] = prev[i] - d[i];
            // state CHECK_ERR
            pnp_residual(cam, p, obj, m, err);
            double s = 0;
            for (int k = 0; k < 8; k++) s += err[k] * err[k];
            errNorm = sqrt(s);
            if (errNorm > prevErrNorm && ++lambdaLg10 <= 16) continue;
            break;
        }
        lambdaLg10 = lambdaLg10 - 1 > -16 ? lambdaLg10 - 1 : -16;
        double dn = 0, pn = 0;
        for (int i = 0; i < 6; i++) {
            dn += (p[i] - prev[i]) * (p[i] - prev[i]);
            pn += prev[i] * prev[i];
        }
        if (++iters >= 20 || sqrt(dn) / sqrt(pn) < FLT_EPSILON) break;
        prevErrNorm = errNorm;
        pnp_residual_jacobian(cam, p, obj, m, err, J);
    }
    for (int i = 0; i < 3; i++) {
        rvec[i] = p[i];
        tvec[i] = p[3 + i];
    }
    return true;
}

// aruco::rotateXAxis (src/utils.cpp:16-30): R(f32) = Rodrigues(rvec) * RX(90 deg) (f32), back to a vector
AB_HD void rotate_x_axis(double* rvec) {
    double Rd[9];
    rodrigues_to_mat(rvec, Rd);
    float R[9], RX[9] = {1, 0, 0, 0, 0, 0, 0, 0, 0}, O[9];
    for (int i = 0; i < 9; i++) R[i] = (float)Rd[i];
    float ang = (float)(3.14159265358979323846 / 2);
    RX[4] = (float)cos((double)ang);
    RX[5] = -(float)sin((double)ang);
    RX[7] = (float)sin((double)ang);
    RX[8] = (float)cos((double)ang);
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            float s = 0;
            for (int k = 0; k < 3; k++) s += R[i * 3 + k] * RX[k * 3 + j];
            O[i * 3 + j] = s;
        }
    for (int i = 0; i < 9; i++) Rd[i] = O[i];
    orthonormalize3(Rd);
    mat_to_rodrigues(Rd, rvec);
}

// ---------------------------------------------------------------------------------------------------
// N-point planar pose (BoardDetector::detect -> cv::solvePnP on 4*M stacked marker corners,
// src/boarddetector.cpp:132-157, and its outlier re-solve :172-194).  Same structure as
// cvFindExtrinsicCameraParams2's planar branch: centre the object points, homography to the normalised image
// points (normalised DLT, least squares for N > 4), decomposition, then the CvLevMarq schedule over all points.
// ---------------------------------------------------------------------------------------------------
AB_HD void jacobi_eigen9(double A[9][9], double V[9][9]) {
    for (int i = 0; i < 9; i++)
        for (int j = 0; j < 9; j++) V[i][j] = (i == j) ? 1. : 0.;
    for (int sweep = 0; sweep < 30; sweep++) {
        double off = 0;
        for (int i = 0; i < 9; i++)
            for (int j = i + 1; j < 9; j++) off += A[i][j] * A[i][j];
        if (off < 1e-300) break;
        for (int p = 0; p < 8; p++)
            for (int q = p + 1; q < 9; q++) {
                if (fabs(A[p][q]) < 1e-300) continue;
                double th = (A[q][q] - A[p][p]) / (2 * A[p][q]);
                double t = (th >= 0 ? 1. : -1.) / (fabs(th) + sqrt(th * th + 1));
                double c = 1 / sqrt(t * t + 1), sn = t * c;
                for (int k = 0; k < 9; k++) {
                    double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - sn * akq;
                    A[k][q] = sn * akp + c * akq;
                }
                for (int k = 0; k < 9; k++) {
                    double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - sn * aqk;
                    A[q][k] = sn * apk + c * aqk;
                }
                for (int k = 0; k < 9; k++) {
                    double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - sn * vkq;
                    V[k][q] = sn * vkp + c * vkq;
                }
            }
    }
}

// How the loops over the N stacked points run: one thread over all of them (the host check, and any single-thread caller),
// or the 32 lanes of a warp over every 32nd point with butterfly sums that leave the same value in every lane (k_board_pose:
// 96 points of a 24-marker board took 1.4 ms per solve in one thread).  Everything between the loops -- eigen decomposition,
// Cholesky, the CvLevMarq control flow -- runs redundantly and identically in all lanes.
struct PnpSerial {
    AB_HD static int first() { return 0; }
    AB_HD static int step() { return 1; }
    AB_HD static double sum(double v) { return v; }
};
#if defined(__CUDACC__)
struct PnpWarp {
    __device__ static int first() { return (int)(threadIdx.x & 31u); }
    __device__ static int step() { return 32; }
    __device__ static double sum(double v) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
        return v;
    }
};
#endif

// residual (and J^T J, J^T e) of all N points for pose p; returns |e|^2
template <class PAR>
AB_HD double pnp_accumulate(const Camera& cam, const double* p, const float* obj, const float* img, int N, bool with_jac,
                            double JtJ[6][6], double* JtErr) {
    double R[9], dR[3][9];
    if (with_jac) {
        rodrigues_jacobian(p, R, dR);
        for (int i = 0; i < 6; i++) {
            JtErr[i] = 0;
            for (int j = 0; j < 6; j++) JtJ[i][j] = 0;
        }
    } else {
        rodrigues_to_mat(p, R);
    }
    double e2 = 0;
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        double X = obj[3 * n], Y = obj[3 * n + 1], Z = obj[3 * n + 2];
        double x = R[0] * X + R[1] * Y + R[2] * Z + p[3];
        double y = R[3] * X + R[4] * Y + R[5] * Z + p[4];
        double z = R[6] * X + R[7] * Y + R[8] * Z + p[5];
        double iz = z ? 1. / z : 1.;
        double xn = x * iz, yn = y * iz;
        double r2 = xn * xn + yn * yn, r4 = r2 * r2, r6 = r4 * r2;
        double a1 = 2 * xn * yn, a2 = r2 + 2 * xn * xn, a3 = r2 + 2 * yn * yn;
        double cdist = 1 + cam.k1 * r2 + cam.k2 * r4 + cam.k3 * r6;
        double xd = xn * cdist + cam.p1 * a1 + cam.p2 * a2, yd = yn * cdist + cam.p1 * a3 + cam.p2 * a1;
        double eu = xd * cam.fx + cam.cx - (double)img[2 * n], ev = yd * cam.fy + cam.cy - (double)img[2 * n + 1];
        e2 += eu * eu + ev * ev;
        if (!with_jac) continue;
        double dc = cam.k1 + 2 * cam.k2 * r2 + 3 * cam.k3 * r4;
        double dxdx = cdist + 2 * xn * xn * dc + 2 * cam.p1 * yn + 6 * cam.p2 * xn;
        double dxdy = 2 * xn * yn * dc + 2 * cam.p1 * xn + 2 * cam.p2 * yn;
        double dydx = dxdy;
        double dydy = cdist + 2 * yn * yn * dc + 6 * cam.p1 * yn + 2 * cam.p2 * xn;
        double dxn[3] = {iz, 0, -xn * iz}, dyn[3] = {0, iz, -yn * iz};
        double du[3], dv[3], Ju[6], Jv[6];
        for (int c = 0; c < 3; c++) {
            du[c] = cam.fx * (dxdx * dxn[c] + dxdy * dyn[c]);
            dv[c] = cam.fy * (dydx * dxn[c] + dydy * dyn[c]);
        }
        for (int k = 0; k < 3; k++) {
            double dX[3] = {dR[k][0] * X + dR[k][1] * Y + dR[k][2] * Z, dR[k][3] * X + dR[k][4] * Y + dR[k][5] * Z,
                            dR[k][6] * X + dR[k][7] * Y + dR[k][8] * Z};
            Ju[k] = du[0] * dX[0] + du[1] * dX[1] + du[2] * dX[2];
            Jv[k] = dv[0] * dX[0] + dv[1] * dX[1] + dv[2] * dX[2];
            Ju[3 + k] = du[k];
            Jv[3 + k] = dv[k];
        }
        for (int i = 0; i < 6; i++) {
            JtErr[i] += Ju[i] * eu + Jv[i] * ev;
            for (int j = i; j < 6; j++) JtJ[i][j] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
        }
    }
    if (with_jac) {
        for (int i = 0; i < 6; i++) {
            JtErr[i] = PAR::sum(JtErr[i]);
            for (int j = i; j < 6; j++) {
                JtJ[i][j] = PAR::sum(JtJ[i][j]);
                JtJ[j][i] = JtJ[i][j];
            }
        }
    }
    return PAR::sum(e2);
}

// Normalised DLT (cv::findHomography, method 0, without its refinement): Hm maps object (X, Y) to the undistorted
// normalised image point of `cam` (with fx = fy = 1, cx = cy = 0 and zero_D: to the pixel itself), scaled so that
// Hm[8] = 1.  Mc = the object centroid.  Returns false for degenerate input.
template <class PAR>
AB_HD bool planar_homography_t(const Camera& cam, const float* obj, const float* img, int N, const double* Mc, double* Hm) {
    double cM[2] = {Mc[0], Mc[1]}, cm[2] = {0, 0}, sM[2] = {0, 0}, sm[2] = {0, 0};
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        double xn, yn;
        undistort_point_norm(cam, img[2 * n], img[2 * n + 1], &xn, &yn);
        cm[0] += xn;
        cm[1] += yn;
    }
    cm[0] = PAR::sum(cm[0]) / N;
    cm[1] = PAR::sum(cm[1]) / N;
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        double xn, yn;
        undistort_point_norm(cam, img[2 * n], img[2 * n + 1], &xn, &yn);
        sm[0] += fabs(xn - cm[0]);
        sm[1] += fabs(yn - cm[1]);
        sM[0] += fabs(obj[3 * n] - cM[0]);
        sM[1] += fabs(obj[3 * n + 1] - cM[1]);
    }
    for (int c = 0; c < 2; c++) {
        sm[c] = PAR::sum(sm[c]);
        sM[c] = PAR::sum(sM[c]);
    }
    if (fabs(sM[0]) < DBL_EPSILON || fabs(sM[1]) < DBL_EPSILON || fabs(sm[0]) < DBL_EPSILON || fabs(sm[1]) < DBL_EPSILON) return false;
    sm[0] = N / sm[0];
    sm[1] = N / sm[1];
    sM[0] = N / sM[0];
    sM[1] = N / sM[1];
    double LtL[9][9], V[9][9];
    for (int i = 0; i < 9; i++)
        for (int j = 0; j < 9; j++) LtL[i][j] = 0;
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        double xn, yn;
        undistort_point_norm(cam, img[2 * n], img[2 * n + 1], &xn, &yn);
        double x = (xn - cm[0]) * sm[0], y = (yn - cm[1]) * sm[1];
        double X = (obj[3 * n] - cM[0]) * sM[0], Y = (obj[3 * n + 1] - cM[1]) * sM[1];
        double Lx[9] = {X, Y, 1, 0, 0, 0, -x * X, -x * Y, -x}, Ly[9] = {0, 0, 0, X, Y, 1, -y * X, -y * Y, -y};
        for (int j = 0; j < 9; j++)
            for (int k = j; k < 9; k++) LtL[j][k] += Lx[j] * Lx[k] + Ly[j] * Ly[k];
    }
    for (int j = 0; j < 9; j++)
        for (int k = j; k < 9; k++) LtL[j][k] = PAR::sum(LtL[j][k]);
    for (int j = 0; j < 9; j++)
        for (int k = 0; k < j; k++) LtL[j][k] = LtL[k][j];
    jacobi_eigen9(LtL, V);
    int best = 0;
    for (int j = 1; j < 9; j++)
        if (LtL[j][j] < LtL[best][best]) best = j;
    double H0[9];
    for (int j = 0; j < 9; j++) H0[j] = V[j][best];
    // H = invHnorm * H0 * Hnorm2
    double iH[9] = {1. / sm[0], 0, cm[0], 0, 1. / sm[1], cm[1], 0, 0, 1};
    double H2[9] = {sM[0], 0, -cM[0] * sM[0], 0, sM[1], -cM[1] * sM[1], 0, 0, 1};
    double T[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double q = 0;
            for (int k = 0; k < 3; k++) q += iH[i * 3 + k] * H0[k * 3 + j];
            T[i * 3 + j] = q;
        }
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double q = 0;
            for (int k = 0; k < 3; k++) q += T[i * 3 + k] * H2[k * 3 + j];
            Hm[i * 3 + j] = q;
        }
    if (fabs(Hm[8]) < 1e-300) return false;
    for (int j = 0; j < 9; j++) Hm[j] /= Hm[8];
    return true;
}

// obj: N x 3 (a z = const plane), img: N x 2 pixels.  Returns false for degenerate input.
template <class PAR>
AB_HD bool solve_pnp_planar_t(const Camera& cam, const float* obj, const float* img, int N, double* rvec, double* tvec) {
    if (N < 4) return false;
    // object centroid; the board must lie in a z = const plane (every reference board configuration does)
    double Mc[3] = {0, 0, 0};
    for (int n = PAR::first(); n < N; n += PAR::step())
        for (int c = 0; c < 3; c++) Mc[c] += obj[3 * n + c];
    for (int c = 0; c < 3; c++) Mc[c] = PAR::sum(Mc[c]) / N;
    double spread = 0, zdev = 0;
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        spread += fabs(obj[3 * n] - Mc[0]) + fabs(obj[3 * n + 1] - Mc[1]);
        zdev += fabs(obj[3 * n + 2] - Mc[2]);
    }
    spread = PAR::sum(spread);
    zdev = PAR::sum(zdev);
    if (!(spread > 0) || zdev > 1e-6 * spread) return false;
    // Hm maps ABSOLUTE object (X,Y) (Hnorm2 removes the centroid); the reference maps centred coordinates and
    // adds R*T_transform afterwards -- identical pose
    double Hm[9];
    if (!planar_homography_t<PAR>(cam, obj, img, N, Mc, Hm)) return false;
    double h1[3] = {Hm[0], Hm[3], Hm[6]}, h2[3] = {Hm[1], Hm[4], Hm[7]}, h3[3] = {Hm[2], Hm[5], Hm[8]};
    double n1 = sqrt(h1[0] * h1[0] + h1[1] * h1[1] + h1[2] * h1[2]);
    double n2 = sqrt(h2[0] * h2[0] + h2[1] * h2[1] + h2[2] * h2[2]);
    if (!(n1 > DBL_EPSILON) || !(n2 > DBL_EPSILON)) return false;
    for (int i = 0; i < 3; i++) {
        h1[i] /= n1;
        h2[i] /= n2;
    }
    double sc = 2. / (n1 + n2);
    double p[6];
    double c3[3] = {h1[1] * h2[2] - h1[2] * h2[1], h1[2] * h2[0] - h1[0] * h2[2], h1[0] * h2[1] - h1[1] * h2[0]};
    double R[9] = {h1[0], h2[0], c3[0], h1[1], h2[1], c3[1], h1[2], h2[2], c3[2]};
    orthonormalize3(R);
    mat_to_rodrigues(R, p);
    // translation of the plane origin (z = Mc[2] offset folded in: t = h3*sc - R*(0,0,Mc_z) ... the homography was
    // fitted on (X,Y) only, so the plane's constant z enters through R's third column)
    p[3] = h3[0] * sc - R[2] * Mc[2];
    p[4] = h3[1] * sc - R[5] * Mc[2];
    p[5] = h3[2] * sc - R[8] * Mc[2];
    if (p[5] < 0) {  // the plane must be in front of the camera: take the mirrored decomposition
        for (int i = 0; i < 3; i++) {
            h1[i] = -h1[i];
            h2[i] = -h2[i];
        }
        double R2[9] = {h1[0], h2[0], c3[0], h1[1], h2[1], c3[1], h1[2], h2[2], c3[2]};
        orthonormalize3(R2);
        mat_to_rodrigues(R2, p);
        p[3] = -h3[0] * sc - R2[2] * Mc[2];
        p[4] = -h3[1] * sc - R2[5] * Mc[2];
        p[5] = -h3[2] * sc - R2[8] * Mc[2];
    }
    // CvLevMarq schedule (see solve_pnp_marker)
    double JtJ[6][6], JtErr[6], prev[6];
    int lambdaLg10 = -3, iters = 0;
    double prevErrNorm = sqrt(pnp_accumulate<PAR>(cam, p, obj, img, N, true, JtJ, JtErr));
    for (;;) {
        for (int i = 0; i < 6; i++) prev[i] = p[i];
        double errNorm = 0;
        for (;;) {
            double lambda = exp(lambdaLg10 * 2.302585092994046);
            double A[6][6], d[6];
#pragma unroll
            for (int i = 0; i < 6; i++) {
#pragma unroll
                for (int j = 0; j < 6; j++) A[i][j] = JtJ[i][j];
                A[i][i] *= 1. + lambda;
                d[i] = JtErr[i];
            }
            if (!solve6_spd(A, d)) {
#pragma unroll
                for (int i = 0; i < 6; i++) d[i] = JtErr[i];
                if (!solve6(A, d))
                    for (int i = 0; i < 6; i++) d[i] = 0;
            }
            for (int i = 0; i < 6; i++) p[i] = prev[i] - d[i];
            errNorm = sqrt(pnp_accumulate<PAR>(cam, p, obj, img, N, false, nullptr, nullptr));
            if (errNorm > prevErrNorm && ++lambdaLg10 <= 16) continue;
            break;
        }
        lambdaLg10 = lambdaLg10 - 1 > -16 ? lambdaLg10 - 1 : -16;
        double dn = 0, pn = 0;
        for (int i = 0; i < 6; i++) {
            dn += (p[i] - prev[i]) * (p[i] - prev[i]);
            pn += prev[i] * prev[i];
        }
        if (++iters >= 20 || sqrt(dn) / sqrt(pn) < FLT_EPSILON) break;
        prevErrNorm = errNorm;
        pnp_accumulate<PAR>(cam, p, obj, img, N, true, JtJ, JtErr);
    }
    for (int i = 0; i < 3; i++) {
        rvec[i] = p[i];
        tvec[i] = p[3 + i];
    }
    return true;
}
AB_HD bool solve_pnp_planar(const Camera& cam, const float* obj, const float* img, int N, double* rvec, double* tvec) {
    return solve_pnp_planar_t<PnpSerial>(cam, obj, img, N, rvec, tvec);
}


// BoardDetector::detect's selection (src/boarddetector.cpp:104-111, 132-150): the markers whose id is in the configuration, in
// detection order (the first configuration entry with that id wins), stacked as 4 object / image correspondences each.
// obj: 12 * cap floats, img: 8 * cap floats, slots: cap marker indices.  mpp is the configuration's metres per pixel (1 for
// a configuration in metres), computed once on the host.  Returns the number of matched markers.
AB_HD int board_select_stack(const ab_marker* ms, int nm, const int32_t* ids, const float* corners, int n_cfg, double mpp, int cap,
                             float* obj, float* img, int32_t* slots) {
    int nb = 0;
    for (int i = 0; i < nm; i++) {
        int k = -1;
        for (int j = 0; j < n_cfg; j++)
            if (ids[j] == ms[i].id) {
                k = j;
                break;
            }
        if (k < 0) continue;
        AB_BOUND(nb < cap);
        slots[nb] = i;
        for (int p = 0; p < 4; p++) {
            img[8 * nb + 2 * p] = ms[i].corners[2 * p];
            img[8 * nb + 2 * p + 1] = ms[i].corners[2 * p + 1];
            for (int c = 0; c < 3; c++) obj[12 * nb + 3 * p + c] = (float)((double)corners[(size_t)k * 12 + 3 * p + c] * mpp);  // Point3f * double
        }
        nb++;
    }
    return nb;
}

}  // namespace ab
