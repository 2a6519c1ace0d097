// k_calibrate: cv::calibrateCamera (flags 0) for many cameras in one launch -- one CTA per camera, warps striding over its
// views, one warp reducing one view's points with shuffles (PnpWarp).  The arithmetic is calibrate_camera_t (ab_calib.cuh);
// per-view partial sums go to the view's CalibView record and are combined in view order, so a camera's result is
// bit-identical from run to run and whichever cameras share the launch.
#pragma once
#include "ab_calib.cuh"

namespace ab {

constexpr int CALIB_THREADS = 128;

struct CalibCamRec {    // one camera of the launch
    int width, height, n_views;
    int view0;          // index of its first view in the launch's view arrays
};

struct CalibArgs {
    const CalibCamRec* cams;
    const int32_t* n_points;  // [views]
    const int32_t* offset;    // [views]: first point of the view in obj / img
    const float* obj;         // [points][3]
    const float* img;         // [points][2]
    CalibView* ws;            // [views]
    ab_calib_result* out;     // [cameras]
    double* poses;            // [views][6]: rvec, tvec
};

__global__ void __launch_bounds__(CALIB_THREADS) k_calibrate(CalibArgs a) {
    __shared__ CalibShared sh;
    const CalibCamRec rec = a.cams[blockIdx.x];
    CalibCamera cam;
    cam.width = rec.width;
    cam.height = rec.height;
    cam.n_views = rec.n_views;
    cam.n_points = a.n_points + rec.view0;
    cam.offset = a.offset + rec.view0;
    cam.obj = a.obj;
    cam.img = a.img;
    CalibView* ws = a.ws + rec.view0;
    int iters = 0;
    calibrate_camera_t<CalibCtaExec>(cam, ws, sh, &iters);
    const bool ok = sh.status == 0;
    for (int i = threadIdx.x; i < 6 * rec.n_views; i += blockDim.x) a.poses[6 * (size_t)rec.view0 + i] = ok ? ws[i / 6].p[i % 6] : 0.;
    if (threadIdx.x != 0) return;
    ab_calib_result& r = a.out[blockIdx.x];
    for (int i = 0; i < 9; i++) r.K[i] = 0;
    for (int i = 0; i < 5; i++) r.D[i] = 0;
    r.rms = 0;
    r.iterations = iters;
    r.status = sh.status;
    if (!ok) return;
    r.K[0] = sh.k[0];
    r.K[2] = sh.k[2];
    r.K[4] = sh.k[1];
    r.K[5] = sh.k[3];
    r.K[8] = 1;
    for (int i = 0; i < 5; i++) r.D[i] = sh.k[4 + i];
    long long total = 0;
    for (int v = 0; v < rec.n_views; v++) total += cam.n_points[v];
    r.rms = sqrt(sh.e2 / (double)total);
}

}  // namespace ab
