// Host-compiled harness around stereo_calibrate_t (ab_stereo.cuh): the arithmetic every CTA of k_stereo_calibrate runs, here in
// one thread over all views.  TEST INFRASTRUCTURE, like hostcheck.cpp: never linked into libaruco_b200.so and not a CPU fallback.
#include <stdint.h>
#include <vector>
#include "../../aruco_b200/csrc/ab_stereo.cuh"

// the same outputs as one pair of ab_stereo_calibrate; returns the pair's status
extern "C" int hc_stereo_calibrate(int n_views, const int32_t* n_points, const float* obj, const float* img1, const float* img2,
                                   const double* K1, const double* D1, const double* K2, const double* D2, int max_iter, double eps,
                                   ab_stereo_result* out, double* rvecs, double* tvecs, double* per_view_errors) {
    std::vector<int32_t> offset(n_views > 0 ? n_views : 1);
    long long total = 0;
    for (int v = 0; v < n_views; v++) {
        offset[v] = (int32_t)total;
        total += n_points[v];
    }
    ab::StereoPair pr;
    pr.n_views = n_views;
    pr.n_points = n_points;
    pr.offset = offset.data();
    pr.obj = obj;
    pr.img1 = img1;
    pr.img2 = img2;
    ab::stereo_intrinsics(K1, D1, pr.kk1);
    ab::stereo_intrinsics(K2, D2, pr.kk2);
    std::vector<ab::StereoView> ws(n_views > 0 ? n_views : 1);
    ab::StereoShared sh;
    int iters = 0;
    ab::stereo_calibrate_t<ab::CalibSerialExec>(pr, ws.data(), sh, max_iter, eps, &iters);
    ab::stereo_result(pr, sh, K1, K2, iters, *out);
    for (int v = 0; v < n_views; v++) {
        double pose[6];
        ab::stereo_view_result(pr, ws.data(), sh, v, pose, per_view_errors + 2 * v);
        for (int i = 0; i < 3; i++) {
            rvecs[3 * v + i] = pose[i];
            tvecs[3 * v + i] = pose[3 + i];
        }
    }
    return sh.status;
}
