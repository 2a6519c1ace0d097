// cv::calibrateCamera (flags 0) for planar targets: the arithmetic of k_calibrate (k_calib.cuh) as AB_HD functions, so that a
// host build runs exactly the same code (tests/hostcheck/hostcheck_calib.cpp).
//
// Free parameters: fx, fy, cx, cy, k1, k2, p1, p2, k3 (skew 0, k4..k6 / thin prism / tilt fixed at 0) and 6 per view.
//   1. initIntrinsicParams2D: one homography per view (normalised DLT), principal point ((w-1)/2, (h-1)/2), focal lengths
//      from the vanishing-point constraints by least squares.
//   2. cvFindExtrinsicCameraParams2 per view with D = 0 (solve_pnp_planar_t).
//   3. CvLevMarq over all parameters, TermCriteria(COUNT + EPS, 30, DBL_EPSILON).  The normal equations have an arrow shape
//      (9 x 9 intrinsic block, one 6 x 6 block per view, 9 x 6 couplings); each damped step is solved by the Schur complement
//      of the view blocks instead of a dense solve of the (9 + 6N)^2 system.
// Every sum over views runs in view order (never by atomics), so a camera's result does not depend on the launch it is in.
#pragma once
#include <string.h>
#include "ab_math.cuh"

namespace ab {

constexpr int CALIB_NI = 9;          // fx fy cx cy k1 k2 p1 p2 k3
constexpr int CALIB_MAX_ITERS = 30;  // TermCriteria(COUNT + EPS, 30, DBL_EPSILON)
constexpr int CALIB_NU = CALIB_NI * (CALIB_NI + 1) / 2;  // upper triangle of the intrinsic block

// One camera's input: views v = 0..n_views-1 hold n_points[v] points starting at point offset[v] of obj (x, y, z) / img (u, v).
struct CalibCamera {
    int width, height, n_views;
    const int32_t* n_points;
    const int32_t* offset;
    const float* obj;
    const float* img;
};

// Per-view workspace (global memory on the device).
struct CalibView {
    double p[6], prev[6];        // rvec, tvec
    double V[6][6];              // Je^T Je
    double W[CALIB_NI][6];       // Ji^T Je
    double g[6];                 // Je^T e
    double U[CALIB_NU];          // Ji^T Ji (upper triangle, row-major)
    double gI[CALIB_NI];         // Ji^T e
    double C[CALIB_NI][CALIB_NI + 1];  // W Vd^-1 [W^T | g]: this view's share of the Schur complement and its right-hand side
    double e2, dn, pn;
    double rows[6];              // focal-length constraints: A (2 x 2, row-major), b (2)
    double zs[2];                // sum z, sum z^2
    int ok;
};

// Per-camera state (shared memory on the device).
struct CalibShared {
    double k[CALIB_NI], kprev[CALIB_NI], dI[CALIB_NI];
    double U[CALIB_NU], gI[CALIB_NI];
    double e2, dn, pn;
    int status;
};

// Who runs what: the host build is one thread over all views and points; the kernel is one CTA per camera with warps over
// views (PnpWarp over a view's points) and the threads of the CTA over the entries of per-view sums.
struct CalibSerialExec {
    typedef PnpSerial PAR;
    AB_HD static int warp() { return 0; }
    AB_HD static int n_warps() { return 1; }
    AB_HD static int tid() { return 0; }
    AB_HD static int n_threads() { return 1; }
    AB_HD static bool lane0() { return true; }
    AB_HD static void sync() {}
};
#if defined(__CUDACC__)
struct CalibCtaExec {
    typedef PnpWarp PAR;
    __device__ static int warp() { return (int)(threadIdx.x >> 5); }
    __device__ static int n_warps() { return (int)(blockDim.x >> 5); }
    __device__ static int tid() { return (int)threadIdx.x; }
    __device__ static int n_threads() { return (int)blockDim.x; }
    __device__ static bool lane0() { return (threadIdx.x & 31u) == 0; }
    __device__ static void sync() { __syncthreads(); }
};
#endif

// Cholesky factor of the upper triangle of the N x N SPD matrix A (row-major, full storage): L lower, diagonal holds 1/L_jj.
template <int N>
AB_HD bool chol_factor(const double* A, double* L) {
    for (int j = 0; j < N; j++) {
        double d = A[j * N + j];
        for (int k = 0; k < j; k++) d -= L[j * N + k] * L[j * N + k];
        if (!(d > 0.0)) return false;
        const double inv = 1.0 / sqrt(d);
        L[j * N + j] = inv;
        for (int i = j + 1; i < N; i++) {
            double v = A[j * N + i];
            for (int k = 0; k < j; k++) v -= L[i * N + k] * L[j * N + k];
            L[i * N + j] = v * inv;
        }
    }
    return true;
}
template <int N>
AB_HD void chol_solve(const double* L, double* b) {
    for (int i = 0; i < N; i++) {
        double v = b[i];
        for (int k = 0; k < i; k++) v -= L[i * N + k] * b[k];
        b[i] = v * L[i * N + i];
    }
    for (int i = N - 1; i >= 0; i--) {
        double v = b[i];
        for (int k = i + 1; k < N; k++) v -= L[k * N + i] * b[k];
        b[i] = v * L[i * N + i];
    }
}

// Projection of the plane point (X, Y, 0) under intrinsics k and pose (R, t) (cvProjectPoints2 with k1 k2 p1 p2 k3), residual
// e = projection - (u, v) and, with jac, its derivatives ju / jv with respect to (fx fy cx cy k1 k2 p1 p2 k3 | rvec tvec).
AB_HD void calib_project(const double* k, const double* R, const double dR[3][9], const double* t, double X, double Y, double u,
                         double v, bool jac, double* e, double* ju, double* jv) {
    const double fx = k[0], fy = k[1], cx = k[2], cy = k[3], k1 = k[4], k2 = k[5], p1 = k[6], p2 = k[7], k3 = k[8];
    double x = R[0] * X + R[1] * Y + t[0];
    double y = R[3] * X + R[4] * Y + t[1];
    double z = R[6] * X + R[7] * Y + t[2];
    double iz = z ? 1. / z : 1.;
    double xn = x * iz, yn = y * iz;
    double r2 = xn * xn + yn * yn, r4 = r2 * r2, r6 = r4 * r2;
    double a1 = 2 * xn * yn, a2 = r2 + 2 * xn * xn, a3 = r2 + 2 * yn * yn;
    double cdist = 1 + k1 * r2 + k2 * r4 + k3 * r6;
    double xd = xn * cdist + p1 * a1 + p2 * a2, yd = yn * cdist + p1 * a3 + p2 * a1;
    e[0] = xd * fx + cx - u;
    e[1] = yd * fy + cy - v;
    if (!jac) return;
    ju[0] = xd; ju[1] = 0; ju[2] = 1; ju[3] = 0;
    jv[0] = 0; jv[1] = yd; jv[2] = 0; jv[3] = 1;
    ju[4] = fx * xn * r2; ju[5] = fx * xn * r4; ju[6] = fx * a1; ju[7] = fx * a2; ju[8] = fx * xn * r6;
    jv[4] = fy * yn * r2; jv[5] = fy * yn * r4; jv[6] = fy * a3; jv[7] = fy * a1; jv[8] = fy * yn * r6;
    double dc = k1 + 2 * k2 * r2 + 3 * k3 * r4;
    double dxdx = cdist + 2 * xn * xn * dc + 2 * p1 * yn + 6 * p2 * xn;
    double dxdy = 2 * xn * yn * dc + 2 * p1 * xn + 2 * p2 * yn;
    double dydy = cdist + 2 * yn * yn * dc + 6 * p1 * yn + 2 * p2 * xn;
    double dxn[3] = {iz, 0, -xn * iz}, dyn[3] = {0, iz, -yn * iz};
    double du[3], dv[3];
    for (int c = 0; c < 3; c++) {
        du[c] = fx * (dxdx * dxn[c] + dxdy * dyn[c]);
        dv[c] = fy * (dxdy * dxn[c] + dydy * dyn[c]);
    }
    for (int q = 0; q < 3; q++) {
        double dX[3] = {dR[q][0] * X + dR[q][1] * Y, dR[q][3] * X + dR[q][4] * Y, dR[q][6] * X + dR[q][7] * Y};
        ju[CALIB_NI + q] = du[0] * dX[0] + du[1] * dX[1] + du[2] * dX[2];
        jv[CALIB_NI + q] = dv[0] * dX[0] + dv[1] * dX[1] + dv[2] * dX[2];
        ju[CALIB_NI + 3 + q] = du[q];
        jv[CALIB_NI + 3 + q] = dv[q];
    }
}

// The sums of one view at intrinsics k and pose p.  PART 0: |e|^2 only; PART 1: |e|^2, Ji^T Ji, Ji^T e; PART 2: Je^T Je,
// Ji^T Je, Je^T e.  (Two Jacobian passes instead of one halve the per-lane accumulators: 54 and 81 instead of 136.)
template <class PAR, int PART>
AB_HD void calib_view_sums(const double* k, const double* p, const float* obj, const float* img, int N, CalibView& out, bool write) {
    double R[9], dR[3][9];
    if (PART == 0) rodrigues_to_mat(p, R);
    else rodrigues_jacobian(p, R, dR);
    constexpr int NA = PART == 1 ? CALIB_NU + CALIB_NI : (PART == 2 ? 21 + 6 * CALIB_NI + 6 : 0);
    double acc[NA > 0 ? NA : 1], e2 = 0;
    for (int i = 0; i < NA; i++) acc[i] = 0;
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        double e[2], ju[CALIB_NI + 6], jv[CALIB_NI + 6];
        calib_project(k, R, dR, p + 3, obj[3 * n], obj[3 * n + 1], img[2 * n], img[2 * n + 1], PART != 0, e, ju, jv);
        e2 += e[0] * e[0] + e[1] * e[1];
        if (PART == 1) {
            int a = 0;
            for (int i = 0; i < CALIB_NI; i++)
                for (int j = i; j < CALIB_NI; j++) acc[a++] += ju[i] * ju[j] + jv[i] * jv[j];
            for (int i = 0; i < CALIB_NI; i++) acc[a++] += ju[i] * e[0] + jv[i] * e[1];
        } else if (PART == 2) {
            int a = 0;
            for (int i = 0; i < 6; i++)
                for (int j = i; j < 6; j++) acc[a++] += ju[CALIB_NI + i] * ju[CALIB_NI + j] + jv[CALIB_NI + i] * jv[CALIB_NI + j];
            for (int i = 0; i < CALIB_NI; i++)
                for (int j = 0; j < 6; j++) acc[a++] += ju[i] * ju[CALIB_NI + j] + jv[i] * jv[CALIB_NI + j];
            for (int i = 0; i < 6; i++) acc[a++] += ju[CALIB_NI + i] * e[0] + jv[CALIB_NI + i] * e[1];
        }
    }
    for (int i = 0; i < NA; i++) acc[i] = PAR::sum(acc[i]);
    e2 = PAR::sum(e2);
    if (!write) return;
    if (PART != 2) out.e2 = e2;
    int a = 0;
    if (PART == 1) {
        for (int i = 0; i < CALIB_NU; i++) out.U[i] = acc[a++];
        for (int i = 0; i < CALIB_NI; i++) out.gI[i] = acc[a++];
    } else if (PART == 2) {
        for (int i = 0; i < 6; i++)
            for (int j = i; j < 6; j++) out.V[i][j] = out.V[j][i] = acc[a++];
        for (int i = 0; i < CALIB_NI; i++)
            for (int j = 0; j < 6; j++) out.W[i][j] = acc[a++];
        for (int i = 0; i < 6; i++) out.g[i] = acc[a++];
    }
}

// The view's damped pose block Vd = V with its diagonal scaled by 1 + lambda, factored.
AB_HD bool calib_view_factor(const CalibView& w, double lambda, double L[36]) {
    double A[36];
    for (int i = 0; i < 6; i++)
        for (int j = 0; j < 6; j++) A[i * 6 + j] = w.V[i][j];
    for (int i = 0; i < 6; i++) A[i * 6 + i] *= 1. + lambda;
    return chol_factor<6>(A, L);
}

// initIntrinsicParams2D's two constraints of one view from its homography H (object plane -> pixels, H[8] = 1) and the
// principal point (a2, a5): rows = {A00, A01, A10, A11, b0, b1}
AB_HD void calib_focal_rows(double* H, double a2, double a5, double* rows) {
    H[0] -= H[6] * a2; H[1] -= H[7] * a2; H[2] -= H[8] * a2;
    H[3] -= H[6] * a5; H[4] -= H[7] * a5; H[5] -= H[8] * a5;
    double h[3], v[3], d1[3], d2[3], n[4] = {0, 0, 0, 0};
    for (int j = 0; j < 3; j++) {
        double t0 = H[j * 3], t1 = H[j * 3 + 1];
        h[j] = t0;
        v[j] = t1;
        d1[j] = (t0 + t1) * 0.5;
        d2[j] = (t0 - t1) * 0.5;
        n[0] += t0 * t0;
        n[1] += t1 * t1;
        n[2] += d1[j] * d1[j];
        n[3] += d2[j] * d2[j];
    }
    for (int j = 0; j < 4; j++) n[j] = 1. / sqrt(n[j]);
    for (int j = 0; j < 3; j++) {
        h[j] *= n[0];
        v[j] *= n[1];
        d1[j] *= n[2];
        d2[j] *= n[3];
    }
    rows[0] = h[0] * v[0];
    rows[1] = h[1] * v[1];
    rows[2] = d1[0] * d2[0];
    rows[3] = d1[1] * d2[1];
    rows[4] = -h[2] * v[2];
    rows[5] = -d1[2] * d2[2];
}

AB_HD bool calib_finite(double x) { return x == x && x - x == 0; }

// Smallest ratio of a focal-length constraint system's eigenvalues (A^T A, 2 x 2) below which the views do not determine the
// focal lengths (every view parallel to the image plane, or all views tilted about one axis).
constexpr double CALIB_MIN_FOCAL_CONDITION = 1e-10;
// Largest focal length, in units of the image's larger side, taken as determined by the views (a field of view under 0.6
// degrees).  Views parallel to the image plane leave the focal length free: with noise the estimate wanders to 1e2..1e3 times
// the image size (cv::calibrateCamera returns such values without complaint); such a camera is reported as degenerate.
constexpr double CALIB_MAX_FOCAL_RATIO = 100.0;

// cv::calibrateCamera of one camera.  ws: n_views CalibView records; sh: the camera's shared state.  On return (every thread):
// sh.status = 0 and sh.k, ws[v].p, sh.e2 hold the result, or sh.status = AB_E_INVALID for degenerate input.  *iters: the
// CvLevMarq iterations run.
template <class EX>
AB_HD void calibrate_camera_t(const CalibCamera& cam, CalibView* ws, CalibShared& sh, int* iters_out) {
    typedef typename EX::PAR PAR;
    const int nv = cam.n_views;
    // ---- 1. planarity, per-view homographies and the focal-length constraints ----------------------------------------
    const double a2 = cam.width ? (cam.width - 1) * 0.5 : 0.5, a5 = cam.height ? (cam.height - 1) * 0.5 : 0.5;
    Camera ident;
    memset(&ident, 0, sizeof(ident));
    ident.fx = ident.fy = 1.;
    ident.has_K = 1;
    ident.zero_D = 1;
    for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
        const int N = cam.n_points[v];
        const float* obj = cam.obj + 3 * (size_t)cam.offset[v];
        const float* img = cam.img + 2 * (size_t)cam.offset[v];
        double zs = 0, zq = 0, Mc[3] = {0, 0, 0};
        for (int n = PAR::first(); n < N; n += PAR::step()) {
            double z = obj[3 * n + 2];
            zs += z;
            zq += z * z;
            Mc[0] += obj[3 * n];
            Mc[1] += obj[3 * n + 1];
        }
        zs = PAR::sum(zs);
        zq = PAR::sum(zq);
        for (int c = 0; c < 2; c++) Mc[c] = PAR::sum(Mc[c]) / (N > 0 ? N : 1);
        double H[9], rows[6] = {0, 0, 0, 0, 0, 0};
        bool ok = N >= 4 && planar_homography_t<PAR>(ident, obj, img, N, Mc, H);
        if (ok) {
            calib_focal_rows(H, a2, a5, rows);
            for (int i = 0; i < 6; i++) ok = ok && calib_finite(rows[i]);
        }
        if (EX::lane0()) {
            ws[v].zs[0] = zs;
            ws[v].zs[1] = zq;
            for (int i = 0; i < 6; i++) ws[v].rows[i] = rows[i];
            ws[v].ok = ok;
        }
    }
    EX::sync();
    if (EX::tid() == 0) {
        // cv::calibrateCamera: meanStdDev of z over all points, |mean| and sdv at most 1e-5, else "non-planar calibration rig"
        double zs = 0, zq = 0, AtA[3] = {0, 0, 0}, Atb[2] = {0, 0};
        long long total = 0;
        bool ok = nv >= 2;
        for (int v = 0; v < nv; v++) {
            const CalibView& w = ws[v];
            ok = ok && w.ok;
            zs += w.zs[0];
            zq += w.zs[1];
            total += cam.n_points[v];
            for (int r = 0; r < 2; r++) {
                const double x0 = w.rows[2 * r], x1 = w.rows[2 * r + 1], b = w.rows[4 + r];
                AtA[0] += x0 * x0;
                AtA[1] += x0 * x1;
                AtA[2] += x1 * x1;
                Atb[0] += x0 * b;
                Atb[1] += x1 * b;
            }
        }
        if (ok) {
            const double mean = zs / (double)total, var = zq / (double)total - mean * mean;
            ok = fabs(mean) <= 1e-5 && sqrt(var > 0 ? var : 0.) <= 1e-5;
        }
        // least squares A f = b through the normal equations (solve(DECOMP_NORMAL | DECOMP_SVD)), f = (1/fx^2, 1/fy^2)
        const double det = AtA[0] * AtA[2] - AtA[1] * AtA[1], tr = AtA[0] + AtA[2];
        ok = ok && det > CALIB_MIN_FOCAL_CONDITION * tr * tr;
        double f0 = 0, f1 = 0;
        const double fmax = CALIB_MAX_FOCAL_RATIO * (cam.width > cam.height ? cam.width : cam.height);
        if (ok) {
            f0 = (AtA[2] * Atb[0] - AtA[1] * Atb[1]) / det;
            f1 = (AtA[0] * Atb[1] - AtA[1] * Atb[0]) / det;
            ok = f0 > 0 && f1 > 0;  // 1 / f^2 of a real camera
        }
        for (int i = 0; i < CALIB_NI; i++) sh.k[i] = 0;
        if (ok) {
            sh.k[0] = sqrt(fabs(1. / f0));
            sh.k[1] = sqrt(fabs(1. / f1));
            sh.k[2] = a2;
            sh.k[3] = a5;
            ok = calib_finite(sh.k[0]) && calib_finite(sh.k[1]) && sh.k[0] <= fmax && sh.k[1] <= fmax;
        }
        sh.status = ok ? 0 : AB_E_INVALID;
    }
    EX::sync();
    *iters_out = 0;
    if (sh.status) return;
    // ---- 2. each view's pose with the initial intrinsics and D = 0 (cvFindExtrinsicCameraParams2) -----------------------
    Camera c0;
    memset(&c0, 0, sizeof(c0));
    c0.fx = sh.k[0];
    c0.fy = sh.k[1];
    c0.cx = sh.k[2];
    c0.cy = sh.k[3];
    c0.has_K = 1;
    c0.zero_D = 1;
    for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
        double r[3] = {0, 0, 0}, t[3] = {0, 0, 0};
        const bool ok = solve_pnp_planar_t<PAR>(c0, cam.obj + 3 * (size_t)cam.offset[v], cam.img + 2 * (size_t)cam.offset[v], cam.n_points[v], r, t);
        if (EX::lane0()) {
            for (int i = 0; i < 3; i++) {
                ws[v].p[i] = r[i];
                ws[v].p[3 + i] = t[i];
            }
            ws[v].ok = ok;
        }
    }
    EX::sync();
    if (EX::tid() == 0) {
        for (int v = 0; v < nv; v++)
            if (!ws[v].ok) sh.status = AB_E_INVALID;
    }
    EX::sync();
    if (sh.status) return;
    // ---- 3. CvLevMarq (updateAlt) over all 9 + 6 n_views parameters ------------------------------------------------------
    // J^T J, J^T e and |e|^2 at the current parameters; per-view parts stay in ws, the intrinsic sums go to sh in view order
    auto calc_j = [&]() {
        for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
            const float* obj = cam.obj + 3 * (size_t)cam.offset[v];
            const float* img = cam.img + 2 * (size_t)cam.offset[v];
            calib_view_sums<PAR, 1>(sh.k, ws[v].p, obj, img, cam.n_points[v], ws[v], EX::lane0());
            calib_view_sums<PAR, 2>(sh.k, ws[v].p, obj, img, cam.n_points[v], ws[v], EX::lane0());
        }
        EX::sync();
        for (int i = EX::tid(); i < CALIB_NU + CALIB_NI + 1; i += EX::n_threads()) {
            double s = 0;
            for (int v = 0; v < nv; v++) s += i < CALIB_NU ? ws[v].U[i] : (i < CALIB_NU + CALIB_NI ? ws[v].gI[i - CALIB_NU] : ws[v].e2);
            if (i < CALIB_NU) sh.U[i] = s;
            else if (i < CALIB_NU + CALIB_NI) sh.gI[i - CALIB_NU] = s;
            else sh.e2 = s;
        }
        EX::sync();
    };
    // CvLevMarq::step(): params = prev - solve(JtJ with diag *= 1 + lambda, JtErr), then |e|^2 at the new parameters
    auto step = [&](double lambda) {
        for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
            CalibView& w = ws[v];
            double L[36], y[6];
            const bool ok = calib_view_factor(w, lambda, L);
            for (int i = 0; i < CALIB_NI + 1; i++) {  // Vd^-1 [W^T | g], column by column, then W times it
                for (int j = 0; j < 6; j++) y[j] = i < CALIB_NI ? w.W[i][j] : w.g[j];
                if (ok) chol_solve<6>(L, y);
                for (int r = 0; r < CALIB_NI; r++) {
                    double s = 0;
                    for (int j = 0; j < 6; j++) s += w.W[r][j] * y[j];
                    if (EX::lane0()) w.C[r][i] = ok ? s : 0.;
                }
            }
        }
        EX::sync();
        if (EX::tid() == 0) {  // Schur complement S = Ud - sum W Vd^-1 W^T, rhs = gI - sum W Vd^-1 g, in view order
            double S[CALIB_NI * CALIB_NI], rhs[CALIB_NI], Ls[CALIB_NI * CALIB_NI];
            int a = 0;
            for (int i = 0; i < CALIB_NI; i++)
                for (int j = i; j < CALIB_NI; j++) S[i * CALIB_NI + j] = sh.U[a++] * (i == j ? 1. + lambda : 1.);
            for (int i = 0; i < CALIB_NI; i++) rhs[i] = sh.gI[i];
            for (int v = 0; v < nv; v++)
                for (int i = 0; i < CALIB_NI; i++) {
                    for (int j = i; j < CALIB_NI; j++) S[i * CALIB_NI + j] -= ws[v].C[i][j];
                    rhs[i] -= ws[v].C[i][CALIB_NI];
                }
            if (chol_factor<CALIB_NI>(S, Ls)) chol_solve<CALIB_NI>(Ls, rhs);
            else
                for (int i = 0; i < CALIB_NI; i++) rhs[i] = 0;  // not positive definite: no step
            for (int i = 0; i < CALIB_NI; i++) {
                sh.dI[i] = rhs[i];
                sh.k[i] = sh.kprev[i] - rhs[i];
            }
        }
        EX::sync();
        for (int v = EX::warp(); v < nv; v += EX::n_warps()) {  // back substitution: dv = Vd^-1 (g - W^T dI)
            CalibView& w = ws[v];
            double L[36], d[6];
            const bool ok = calib_view_factor(w, lambda, L);
            for (int j = 0; j < 6; j++) {
                double s = w.g[j];
                for (int i = 0; i < CALIB_NI; i++) s -= w.W[i][j] * sh.dI[i];
                d[j] = s;
            }
            if (ok) chol_solve<6>(L, d);
            else
                for (int j = 0; j < 6; j++) d[j] = 0;
            double p[6];
            for (int j = 0; j < 6; j++) p[j] = w.prev[j] - d[j];
            const int N = cam.n_points[v];
            calib_view_sums<PAR, 0>(sh.k, p, cam.obj + 3 * (size_t)cam.offset[v], cam.img + 2 * (size_t)cam.offset[v], N, w, EX::lane0());
            if (EX::lane0())
                for (int j = 0; j < 6; j++) w.p[j] = p[j];
        }
        EX::sync();
        if (EX::tid() == 0) {
            double s = 0;
            for (int v = 0; v < nv; v++) s += ws[v].e2;
            sh.e2 = s;
        }
        EX::sync();
    };
    int lambdaLg10 = -3, iters = 0;
    calc_j();
    for (;;) {
        // CALC_J -> step
        for (int v = EX::warp(); v < nv; v += EX::n_warps())
            if (EX::lane0())
                for (int j = 0; j < 6; j++) ws[v].prev[j] = ws[v].p[j];
        if (EX::tid() == 0)
            for (int i = 0; i < CALIB_NI; i++) sh.kprev[i] = sh.k[i];
        const double prevErrNorm = sh.e2;
        EX::sync();
        double errNorm;
        for (;;) {
            step(exp(lambdaLg10 * 2.302585092994046));
            errNorm = sh.e2;
            if (errNorm > prevErrNorm && ++lambdaLg10 <= 16) continue;  // CHECK_ERR: worse, raise lambda and step again
            break;
        }
        lambdaLg10 = lambdaLg10 - 1 > -16 ? lambdaLg10 - 1 : -16;
        // cvNorm(param, prevParam, CV_RELATIVE_L2) over all parameters
        for (int v = EX::warp(); v < nv; v += EX::n_warps())
            if (EX::lane0()) {
                double dn = 0, pn = 0;
                for (int j = 0; j < 6; j++) {
                    dn += (ws[v].p[j] - ws[v].prev[j]) * (ws[v].p[j] - ws[v].prev[j]);
                    pn += ws[v].prev[j] * ws[v].prev[j];
                }
                ws[v].dn = dn;
                ws[v].pn = pn;
            }
        EX::sync();
        if (EX::tid() == 0) {
            double dn = 0, pn = 0;
            for (int i = 0; i < CALIB_NI; i++) {
                dn += (sh.k[i] - sh.kprev[i]) * (sh.k[i] - sh.kprev[i]);
                pn += sh.kprev[i] * sh.kprev[i];
            }
            for (int v = 0; v < nv; v++) {
                dn += ws[v].dn;
                pn += ws[v].pn;
            }
            sh.dn = dn;
            sh.pn = pn;
        }
        EX::sync();
        if (++iters >= CALIB_MAX_ITERS || sqrt(sh.dn) / sqrt(sh.pn) < DBL_EPSILON) break;
        calc_j();
    }
    *iters_out = iters;
    if (EX::tid() == 0) {
        const double fmax = CALIB_MAX_FOCAL_RATIO * (cam.width > cam.height ? cam.width : cam.height);
        bool ok = calib_finite(sh.e2) && sh.k[0] > 0 && sh.k[1] > 0 && sh.k[0] <= fmax && sh.k[1] <= fmax;
        for (int i = 0; i < CALIB_NI; i++) ok = ok && calib_finite(sh.k[i]);
        for (int v = 0; v < nv; v++)
            for (int j = 0; j < 6; j++) ok = ok && calib_finite(ws[v].p[j]);
        if (!ok) sh.status = AB_E_INVALID;
    }
    EX::sync();
}

}  // namespace ab
