// cv::stereoCalibrate with CALIB_FIX_INTRINSIC for planar targets: the arithmetic of k_stereo_calibrate (k_calib.cuh) as AB_HD
// functions, so that a host build runs exactly the same code (tests/hostcheck/hostcheck_stereo.cpp).
//
// Free parameters: the relative pose (omL, TL) of camera 2 with respect to camera 1 and camera 1's pose (om_i, t_i) of every
// view; camera 2 sees view i under R_L R_i, R_L t_i + T_L.  K and D of both cameras are fixed.
//   1. cvFindExtrinsicCameraParams2 per view and camera with that camera's K and D (solve_pnp_planar_t); the relative pose of
//      each view is R2 R1^T, t2 - R2 R1^T t1, and (omL, TL) starts at the component-wise median over the views
//      (std::nth_element at n / 2).  Camera 1's poses start the views.
//   2. CvLevMarq (levmarq_schedule) over all 6 + 6 N parameters with the caller's TermCriteria(COUNT + EPS, max_iter, eps).
//      The Jacobian of camera 2 is the chain rule on x2 = R_L (R_i X + t_i) + T_L.  The normal equations have an arrow shape
//      (6 x 6 relative-pose block, one 6 x 6 block per view, 6 x 6 couplings); each damped step is solved by the Schur
//      complement of the view blocks.
// Every sum over views runs in view order (never by atomics), so a pair's result does not depend on the launch it is in.
#pragma once
#include "ab_calib.cuh"

namespace ab {

// One pair's input: views v = 0..n_views-1 hold n_points[v] points starting at point offset[v] of obj (x, y, z) and of the
// two cameras' image points img1 / img2 (u, v).  kk1 / kk2: fx fy cx cy k1 k2 p1 p2 k3 of each camera.
struct StereoPair {
    int n_views;
    const int32_t* n_points;
    const int32_t* offset;
    const float* obj;
    const float* img1;
    const float* img2;
    double kk1[CALIB_NI], kk2[CALIB_NI];
};

// Per-view workspace (global memory on the device).
struct StereoView {
    double p[6], prev[6];  // camera 1's rvec, tvec
    double V[6][6];        // Jv^T Jv (both cameras)
    double W[6][6];        // Jg^T Jv (camera 2): g = (omL, TL)
    double g[6];           // Jv^T e
    double U[21];          // Jg^T Jg (upper triangle, row-major)
    double gG[6];          // Jg^T e
    double C[6][7];        // W Vd^-1 [W^T | g]: this view's share of the Schur complement and its right-hand side
    double e2[2];          // |e|^2 of camera 1 and camera 2
    double dn, pn;
    double rel[6];         // the view's initial relative pose: om, T
    double zs[2];          // sum z, sum z^2
    int ok;
};

// Per-pair state (shared memory on the device).
struct StereoShared {
    double G[6], Gprev[6], dG[6];  // omL, TL
    double U[21], gG[6];
    double e2, dn, pn;
    int status;
};

// Smallest ratio det / trace^2 of a view's object-point scatter matrix (2 x 2, about the centroid) below which its points are
// taken as collinear: the view does not determine a pose.
constexpr double STEREO_MIN_SPREAD_CONDITION = 1e-10;

// Derivatives of one residual with respect to a pose (rvec, tvec) whose rotation moves the plane point (X, Y, 0): a = d e / d
// (the rotated and translated point), dR = d R / d rvec.
AB_HD void stereo_pose_jac(const double* a, const double dR[3][9], double X, double Y, double* J) {
    for (int q = 0; q < 3; q++) {
        double dX[3] = {dR[q][0] * X + dR[q][1] * Y, dR[q][3] * X + dR[q][4] * Y, dR[q][6] * X + dR[q][7] * Y};
        J[q] = a[0] * dX[0] + a[1] * dX[1] + a[2] * dX[2];
        J[3 + q] = a[q];
    }
}

// The sums of one view at relative pose G and camera-1 pose p.  PART 0: |e|^2 of each camera only; PART 1: |e|^2, Jv^T Jv,
// Jv^T e; PART 2: Jg^T Jg, Jg^T e, Jg^T Jv (camera 2 only).
template <class PAR, int PART>
AB_HD void stereo_view_sums(const StereoPair& pr, const double* G, const double* p, int v, StereoView& out, bool write) {
    const int N = pr.n_points[v];
    const float* obj = pr.obj + 3 * (size_t)pr.offset[v];
    const float* img1 = pr.img1 + 2 * (size_t)pr.offset[v];
    const float* img2 = pr.img2 + 2 * (size_t)pr.offset[v];
    // the rotations of every part come from rodrigues_jacobian: |e|^2 of the Jacobian pass and of the step must round alike, or
    // near the minimum CvLevMarq rejects steps over rounding differences (rodrigues_to_mat rounds differently)
    double R[9], dR[3][9], RL[9], dRL[3][9];
    rodrigues_jacobian(p, R, dR);
    rodrigues_jacobian(G, RL, dRL);
    constexpr int NA = PART == 1 ? 21 + 6 : (PART == 2 ? 21 + 6 + 36 : 0);
    double acc[NA > 0 ? NA : 1], e2[2] = {0, 0};
    for (int i = 0; i < NA; i++) acc[i] = 0;
    for (int n = PAR::first(); n < N; n += PAR::step()) {
        const double X = obj[3 * n], Y = obj[3 * n + 1];
        const double y[3] = {R[0] * X + R[1] * Y + p[3], R[3] * X + R[4] * Y + p[4], R[6] * X + R[7] * Y + p[5]};
        double e[2], ju[CALIB_NI], jv[CALIB_NI], du[3], dv[3], Ju[6], Jv[6];
        if (PART != 2) {  // camera 1
            calib_distort(pr.kk1, y[0], y[1], y[2], img1[2 * n], img1[2 * n + 1], PART == 1, e, ju, jv, du, dv);
            e2[0] += e[0] * e[0] + e[1] * e[1];
            if (PART == 1) {
                stereo_pose_jac(du, dR, X, Y, Ju);
                stereo_pose_jac(dv, dR, X, Y, Jv);
                int a = 0;
                for (int i = 0; i < 6; i++)
                    for (int j = i; j < 6; j++) acc[a++] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
                for (int i = 0; i < 6; i++) acc[a++] += Ju[i] * e[0] + Jv[i] * e[1];
            }
        }
        // camera 2: x2 = RL y + TL
        const double x2[3] = {RL[0] * y[0] + RL[1] * y[1] + RL[2] * y[2] + G[3], RL[3] * y[0] + RL[4] * y[1] + RL[5] * y[2] + G[4],
                              RL[6] * y[0] + RL[7] * y[1] + RL[8] * y[2] + G[5]};
        calib_distort(pr.kk2, x2[0], x2[1], x2[2], img2[2 * n], img2[2 * n + 1], PART != 0, e, ju, jv, du, dv);
        if (PART != 2) e2[1] += e[0] * e[0] + e[1] * e[1];
        if (PART == 0) continue;
        // d e / d y = d e / d x2 RL: the view's derivatives, as for camera 1
        double au[3], av[3];
        for (int c = 0; c < 3; c++) {
            au[c] = du[0] * RL[c] + du[1] * RL[3 + c] + du[2] * RL[6 + c];
            av[c] = dv[0] * RL[c] + dv[1] * RL[3 + c] + dv[2] * RL[6 + c];
        }
        stereo_pose_jac(au, dR, X, Y, Ju);
        stereo_pose_jac(av, dR, X, Y, Jv);
        if (PART == 1) {
            int a = 0;
            for (int i = 0; i < 6; i++)
                for (int j = i; j < 6; j++) acc[a++] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
            for (int i = 0; i < 6; i++) acc[a++] += Ju[i] * e[0] + Jv[i] * e[1];
        } else {
            // d x2 / d omL = dRL y, d x2 / d TL = I
            double Gu[6], Gv[6];
            for (int q = 0; q < 3; q++) {
                double dX[3] = {dRL[q][0] * y[0] + dRL[q][1] * y[1] + dRL[q][2] * y[2], dRL[q][3] * y[0] + dRL[q][4] * y[1] + dRL[q][5] * y[2],
                                dRL[q][6] * y[0] + dRL[q][7] * y[1] + dRL[q][8] * y[2]};
                Gu[q] = du[0] * dX[0] + du[1] * dX[1] + du[2] * dX[2];
                Gv[q] = dv[0] * dX[0] + dv[1] * dX[1] + dv[2] * dX[2];
                Gu[3 + q] = du[q];
                Gv[3 + q] = dv[q];
            }
            int a = 0;
            for (int i = 0; i < 6; i++)
                for (int j = i; j < 6; j++) acc[a++] += Gu[i] * Gu[j] + Gv[i] * Gv[j];
            for (int i = 0; i < 6; i++) acc[a++] += Gu[i] * e[0] + Gv[i] * e[1];
            for (int i = 0; i < 6; i++)
                for (int j = 0; j < 6; j++) acc[a++] += Gu[i] * Ju[j] + Gv[i] * Jv[j];
        }
    }
    for (int i = 0; i < NA; i++) acc[i] = PAR::sum(acc[i]);
    e2[0] = PAR::sum(e2[0]);
    e2[1] = PAR::sum(e2[1]);
    if (!write) return;
    if (PART != 2) {
        out.e2[0] = e2[0];
        out.e2[1] = e2[1];
    }
    int a = 0;
    if (PART == 1) {
        for (int i = 0; i < 6; i++)
            for (int j = i; j < 6; j++) out.V[i][j] = out.V[j][i] = acc[a++];
        for (int i = 0; i < 6; i++) out.g[i] = acc[a++];
    } else if (PART == 2) {
        for (int i = 0; i < 21; i++) out.U[i] = acc[a++];
        for (int i = 0; i < 6; i++) out.gG[i] = acc[a++];
        for (int i = 0; i < 6; i++)
            for (int j = 0; j < 6; j++) out.W[i][j] = acc[a++];
    }
}

AB_HD void stereo_camera(const double* kk, Camera& c) {
    memset(&c, 0, sizeof(c));
    c.fx = kk[0];
    c.fy = kk[1];
    c.cx = kk[2];
    c.cy = kk[3];
    c.k1 = kk[4];
    c.k2 = kk[5];
    c.p1 = kk[6];
    c.p2 = kk[7];
    c.k3 = kk[8];
    c.has_K = c.has_D = 1;
    c.zero_D = kk[4] == 0 && kk[5] == 0 && kk[6] == 0 && kk[7] == 0 && kk[8] == 0;
}

// cv::stereoCalibrate of one pair.  ws: n_views StereoView records; sh: the pair's shared state.  On return (every thread):
// sh.status = 0 and sh.G, ws[v].p, ws[v].e2, sh.e2 hold the result, or sh.status = AB_E_INVALID for degenerate input.  *iters:
// the CvLevMarq iterations run.
template <class EX>
AB_HD void stereo_calibrate_t(const StereoPair& pr, StereoView* ws, StereoShared& sh, int max_iter, double eps, int* iters_out) {
    typedef typename EX::PAR PAR;
    const int nv = pr.n_views;
    *iters_out = 0;
    // ---- 1. planarity, each view's pose in both cameras, and its relative pose -----------------------------------------
    Camera c1, c2;
    stereo_camera(pr.kk1, c1);
    stereo_camera(pr.kk2, c2);
    for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
        const int N = pr.n_points[v];
        const float* obj = pr.obj + 3 * (size_t)pr.offset[v];
        double zs = 0, zq = 0, Mc[2] = {0, 0}, s[3] = {0, 0, 0};
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
        for (int n = PAR::first(); n < N; n += PAR::step()) {
            const double dx = obj[3 * n] - Mc[0], dy = obj[3 * n + 1] - Mc[1];
            s[0] += dx * dx;
            s[1] += dx * dy;
            s[2] += dy * dy;
        }
        for (int c = 0; c < 3; c++) s[c] = PAR::sum(s[c]);
        const double tr = s[0] + s[2];
        bool ok = N >= 4 && s[0] * s[2] - s[1] * s[1] > STEREO_MIN_SPREAD_CONDITION * tr * tr;
        double r1[3] = {0, 0, 0}, t1[3] = {0, 0, 0}, r2[3] = {0, 0, 0}, t2[3] = {0, 0, 0};
        if (ok) ok = solve_pnp_planar_t<PAR>(c1, obj, pr.img1 + 2 * (size_t)pr.offset[v], N, r1, t1);
        if (ok) ok = solve_pnp_planar_t<PAR>(c2, obj, pr.img2 + 2 * (size_t)pr.offset[v], N, r2, t2);
        double rel[6] = {0, 0, 0, 0, 0, 0};
        if (ok) {  // R = R2 R1^T, T = t2 - R t1
            double R1[9], R2[9], R[9];
            rodrigues_to_mat(r1, R1);
            rodrigues_to_mat(r2, R2);
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) R[i * 3 + j] = R2[i * 3] * R1[j * 3] + R2[i * 3 + 1] * R1[j * 3 + 1] + R2[i * 3 + 2] * R1[j * 3 + 2];
            for (int i = 0; i < 3; i++) rel[3 + i] = t2[i] - (R[i * 3] * t1[0] + R[i * 3 + 1] * t1[1] + R[i * 3 + 2] * t1[2]);
            orthonormalize3(R);
            mat_to_rodrigues(R, rel);
            for (int i = 0; i < 6; i++) ok = ok && calib_finite(rel[i]);
        }
        if (EX::lane0()) {
            ws[v].zs[0] = zs;
            ws[v].zs[1] = zq;
            for (int i = 0; i < 3; i++) {
                ws[v].p[i] = r1[i];
                ws[v].p[3 + i] = t1[i];
            }
            for (int i = 0; i < 6; i++) ws[v].rel[i] = rel[i];
            ws[v].ok = ok;
        }
    }
    EX::sync();
    if (EX::tid() == 0) {
        // the planarity test of calibrate_camera_t: |mean z| and its standard deviation at most 1e-5
        double zs = 0, zq = 0;
        long long total = 0;
        bool ok = nv >= 1;
        for (int v = 0; v < nv; v++) {
            ok = ok && ws[v].ok;
            zs += ws[v].zs[0];
            zq += ws[v].zs[1];
            total += pr.n_points[v];
        }
        if (ok) {
            const double mean = zs / (double)total, var = zq / (double)total - mean * mean;
            ok = fabs(mean) <= 1e-5 && sqrt(var > 0 ? var : 0.) <= 1e-5;
        }
        for (int i = 0; i < 6; i++) sh.G[i] = 0;
        sh.status = ok ? 0 : AB_E_INVALID;
    }
    EX::sync();
    if (sh.status) return;
    // the median of each component: the value of rank n / 2 under (value, view index) order, which is std::nth_element's
    for (int c = 0; c < 6; c++)
        for (int i = EX::tid(); i < nv; i += EX::n_threads()) {
            const double x = ws[i].rel[c];
            int rank = 0;
            for (int j = 0; j < nv; j++) {
                const double y = ws[j].rel[c];
                rank += y < x || (y == x && j < i);
            }
            if (rank == nv / 2) sh.G[c] = x;
        }
    EX::sync();
    // ---- 2. CvLevMarq over all 6 + 6 n_views parameters ---------------------------------------------------------------------
    auto calc_j = [&]() {
        for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
            stereo_view_sums<PAR, 1>(pr, sh.G, ws[v].p, v, ws[v], EX::lane0());
            stereo_view_sums<PAR, 2>(pr, sh.G, ws[v].p, v, ws[v], EX::lane0());
        }
        EX::sync();
        for (int i = EX::tid(); i < 21 + 6 + 1; i += EX::n_threads()) {
            double s = 0;
            for (int v = 0; v < nv; v++) s += i < 21 ? ws[v].U[i] : (i < 27 ? ws[v].gG[i - 21] : ws[v].e2[0] + ws[v].e2[1]);
            if (i < 21) sh.U[i] = s;
            else if (i < 27) sh.gG[i - 21] = s;
            else sh.e2 = s;
        }
        EX::sync();
    };
    auto save = [&]() {
        for (int v = EX::warp(); v < nv; v += EX::n_warps())
            if (EX::lane0())
                for (int j = 0; j < 6; j++) ws[v].prev[j] = ws[v].p[j];
        if (EX::tid() == 0)
            for (int i = 0; i < 6; i++) sh.Gprev[i] = sh.G[i];
    };
    // CvLevMarq::step(): params = prev - solve(JtJ with diag *= 1 + lambda, JtErr), then |e|^2 at the new parameters
    auto step = [&](double lambda) {
        for (int v = EX::warp(); v < nv; v += EX::n_warps()) {
            StereoView& w = ws[v];
            double L[36], y[6];
            const bool ok = chol_damped(w.V, lambda, L);
            for (int i = 0; i < 7; i++) {  // Vd^-1 [W^T | g], column by column, then W times it
                for (int j = 0; j < 6; j++) y[j] = i < 6 ? w.W[i][j] : w.g[j];
                if (ok) chol_solve<6>(L, y);
                for (int r = 0; r < 6; r++) {
                    double s = 0;
                    for (int j = 0; j < 6; j++) s += w.W[r][j] * y[j];
                    if (EX::lane0()) w.C[r][i] = ok ? s : 0.;
                }
            }
        }
        EX::sync();
        if (EX::tid() == 0) {  // Schur complement S = Ud - sum W Vd^-1 W^T, rhs = gG - sum W Vd^-1 g, in view order
            double S[36], rhs[6], Ls[36];
            int a = 0;
            for (int i = 0; i < 6; i++)
                for (int j = i; j < 6; j++) S[i * 6 + j] = sh.U[a++] * (i == j ? 1. + lambda : 1.);
            for (int i = 0; i < 6; i++) rhs[i] = sh.gG[i];
            for (int v = 0; v < nv; v++)
                for (int i = 0; i < 6; i++) {
                    for (int j = i; j < 6; j++) S[i * 6 + j] -= ws[v].C[i][j];
                    rhs[i] -= ws[v].C[i][6];
                }
            if (chol_factor<6>(S, Ls)) chol_solve<6>(Ls, rhs);
            else
                for (int i = 0; i < 6; i++) rhs[i] = 0;  // not positive definite: no step
            for (int i = 0; i < 6; i++) {
                sh.dG[i] = rhs[i];
                sh.G[i] = sh.Gprev[i] - rhs[i];
            }
        }
        EX::sync();
        for (int v = EX::warp(); v < nv; v += EX::n_warps()) {  // back substitution: dv = Vd^-1 (g - W^T dG)
            StereoView& w = ws[v];
            double L[36], d[6];
            const bool ok = chol_damped(w.V, lambda, L);
            for (int j = 0; j < 6; j++) {
                double s = w.g[j];
                for (int i = 0; i < 6; i++) s -= w.W[i][j] * sh.dG[i];
                d[j] = s;
            }
            if (ok) chol_solve<6>(L, d);
            else
                for (int j = 0; j < 6; j++) d[j] = 0;
            double p[6];
            for (int j = 0; j < 6; j++) p[j] = w.prev[j] - d[j];
            stereo_view_sums<PAR, 0>(pr, sh.G, p, v, w, EX::lane0());
            if (EX::lane0())
                for (int j = 0; j < 6; j++) w.p[j] = p[j];
        }
        EX::sync();
        if (EX::tid() == 0) {
            double s = 0;
            for (int v = 0; v < nv; v++) s += ws[v].e2[0] + ws[v].e2[1];
            sh.e2 = s;
        }
        EX::sync();
    };
    // cvNorm(param, prevParam, CV_RELATIVE_L2) over all parameters
    auto rel_change = [&]() {
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
            for (int i = 0; i < 6; i++) {
                dn += (sh.G[i] - sh.Gprev[i]) * (sh.G[i] - sh.Gprev[i]);
                pn += sh.Gprev[i] * sh.Gprev[i];
            }
            for (int v = 0; v < nv; v++) {
                dn += ws[v].dn;
                pn += ws[v].pn;
            }
            sh.dn = dn;
            sh.pn = pn;
        }
        EX::sync();
        return sqrt(sh.dn) / sqrt(sh.pn);
    };
    *iters_out = levmarq_schedule<EX>(sh.e2, calc_j, save, step, rel_change, max_iter, eps);
    // The reported errors: cv::stereoCalibrate (4.13, pinned as a black box) returns the rms and per-view errors of the last
    // views' poses under the relative pose of the last Jacobian pass (Gprev), not under the relative pose it returns.  Its
    // accept / reject decisions follow the errors of the current parameters, as the schedule above does.
    for (int v = EX::warp(); v < nv; v += EX::n_warps()) stereo_view_sums<PAR, 0>(pr, sh.Gprev, ws[v].p, v, ws[v], EX::lane0());
    EX::sync();
    if (EX::tid() == 0) {
        double s = 0;
        for (int v = 0; v < nv; v++) s += ws[v].e2[0] + ws[v].e2[1];
        sh.e2 = s;
    }
    EX::sync();
    if (EX::tid() == 0) {
        bool ok = calib_finite(sh.e2);
        for (int i = 0; i < 6; i++) ok = ok && calib_finite(sh.G[i]);
        for (int v = 0; v < nv; v++)
            for (int j = 0; j < 6; j++) ok = ok && calib_finite(ws[v].p[j]);
        if (!ok) sh.status = AB_E_INVALID;
    }
    EX::sync();
}

// StereoPair's intrinsics from a camera matrix K (row-major) and k1 k2 p1 p2 k3
AB_HD void stereo_intrinsics(const double* K, const double* D, double* kk) {
    kk[0] = K[0];
    kk[1] = K[4];
    kk[2] = K[2];
    kk[3] = K[5];
    for (int i = 0; i < 5; i++) kk[4 + i] = D[i];
}

// cv::stereoCalibrate's outputs from the relative pose G = (omL, TL): R, T, E = [T]x R and F = K2^-T E K1^-1 scaled to
// F[8] = 1.  K1 / K2: camera matrices, row-major.
AB_HD void stereo_outputs(const double* G, const double* K1, const double* K2, double* R, double* T, double* E, double* F) {
    rodrigues_to_mat(G, R);
    for (int i = 0; i < 3; i++) T[i] = G[3 + i];
    const double tx[9] = {0, -T[2], T[1], T[2], 0, -T[0], -T[1], T[0], 0};
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) E[i * 3 + j] = tx[i * 3] * R[j] + tx[i * 3 + 1] * R[3 + j] + tx[i * 3 + 2] * R[6 + j];
    double iK2t[9], iK1t[9], M[9];  // K^-T
    mat3_inv_transpose(K2, iK2t);
    mat3_inv_transpose(K1, iK1t);
    for (int i = 0; i < 3; i++)  // M = K2^-T E
        for (int j = 0; j < 3; j++) M[i * 3 + j] = iK2t[i * 3] * E[j] + iK2t[i * 3 + 1] * E[3 + j] + iK2t[i * 3 + 2] * E[6 + j];
    for (int i = 0; i < 3; i++)  // F = M K1^-1 = M (K1^-T)^T
        for (int j = 0; j < 3; j++) F[i * 3 + j] = M[i * 3] * iK1t[j * 3] + M[i * 3 + 1] * iK1t[j * 3 + 1] + M[i * 3 + 2] * iK1t[j * 3 + 2];
    const double s = fabs(F[8]) > 0 ? 1. / F[8] : 1.;
    for (int i = 0; i < 9; i++) F[i] *= s;
}

// One pair's result after stereo_calibrate_t (all zeros but the status for a degenerate pair).  K1 / K2: its camera matrices.
AB_HD void stereo_result(const StereoPair& pr, const StereoShared& sh, const double* K1, const double* K2, int iters, ab_stereo_result& r) {
    memset(&r, 0, sizeof(r));
    r.iterations = iters;
    r.status = sh.status;
    if (sh.status) return;
    stereo_outputs(sh.G, K1, K2, r.R, r.T, r.E, r.F);
    long long total = 0;
    for (int v = 0; v < pr.n_views; v++) total += pr.n_points[v];
    r.rms = sqrt(sh.e2 / (2. * (double)total));
}

// View v's outputs: camera 1's pose (rvec, tvec) and the per-view errors sqrt(|e|^2 / n_points) of both cameras.
AB_HD void stereo_view_result(const StereoPair& pr, const StereoView* ws, const StereoShared& sh, int v, double* pose, double* err) {
    const bool ok = sh.status == 0;
    for (int j = 0; j < 6; j++) pose[j] = ok ? ws[v].p[j] : 0.;
    for (int k = 0; k < 2; k++) err[k] = ok ? sqrt(ws[v].e2[k] / (double)pr.n_points[v]) : 0.;
}

}  // namespace ab
