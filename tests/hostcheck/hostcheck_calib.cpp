// Host-compiled harness around calibrate_camera_t (ab_calib.cuh): the arithmetic every CTA of k_calibrate runs, here in one
// thread over all views.  TEST INFRASTRUCTURE, like hostcheck.cpp: never linked into libaruco_b200.so and not a CPU fallback.
#include <stdint.h>
#include <vector>
#include "../../aruco_b200/csrc/ab_calib.cuh"

// the same outputs as one camera of ab_calibrate_cameras; returns the camera's status
extern "C" int hc_calibrate(int width, int height, int n_views, const int32_t* n_points, const float* obj, const float* img, double* K,
                            double* D, double* rms, int32_t* iterations, double* rvecs, double* tvecs) {
    std::vector<int32_t> offset(n_views > 0 ? n_views : 1);
    long long total = 0;
    for (int v = 0; v < n_views; v++) {
        offset[v] = (int32_t)total;
        total += n_points[v];
    }
    ab::CalibCamera cam{width, height, n_views, n_points, offset.data(), obj, img};
    std::vector<ab::CalibView> ws(n_views > 0 ? n_views : 1);
    ab::CalibShared sh;
    int iters = 0;
    ab::calibrate_camera_t<ab::CalibSerialExec>(cam, ws.data(), sh, &iters);
    const bool ok = sh.status == 0;
    for (int i = 0; i < 9; i++) K[i] = 0;
    for (int i = 0; i < 5; i++) D[i] = ok ? sh.k[4 + i] : 0.;
    if (ok) {
        K[0] = sh.k[0];
        K[2] = sh.k[2];
        K[4] = sh.k[1];
        K[5] = sh.k[3];
        K[8] = 1;
    }
    *rms = ok ? sqrt(sh.e2 / (double)total) : 0.;
    *iterations = iters;
    for (int v = 0; v < n_views; v++)
        for (int i = 0; i < 3; i++) {
            rvecs[3 * v + i] = ok ? ws[v].p[i] : 0.;
            tvecs[3 * v + i] = ok ? ws[v].p[3 + i] : 0.;
        }
    return sh.status;
}
