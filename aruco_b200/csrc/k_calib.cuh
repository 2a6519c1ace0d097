// k_calibrate: cv::calibrateCamera (flags 0) for many cameras in one launch -- one CTA per camera, warps striding over its
// views, one warp reducing one view's points with shuffles (PnpWarp).  The arithmetic is calibrate_camera_t (ab_calib.cuh);
// per-view partial sums go to the view's CalibView record and are combined in view order, so a camera's result is
// bit-identical from run to run and whichever cameras share the launch.
#pragma once
#include "ab_calib.cuh"
#include "ab_stereo.cuh"

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

// k_stereo_calibrate: cv::stereoCalibrate (CALIB_FIX_INTRINSIC) for many camera pairs in one launch, laid out as k_calibrate.
// The arithmetic is stereo_calibrate_t (ab_stereo.cuh).
struct StereoPairRec {  // one pair of the launch
    int n_views;
    int view0;          // index of its first view in the launch's view arrays
    double K1[9], K2[9];
    double kk1[CALIB_NI], kk2[CALIB_NI];
};

struct StereoArgs {
    const StereoPairRec* pairs;
    const int32_t* n_points;  // [views]
    const int32_t* offset;    // [views]: first point of the view in obj / img1 / img2
    const float* obj;         // [points][3]
    const float* img1;        // [points][2]
    const float* img2;        // [points][2]
    int max_iter;
    double eps;
    StereoView* ws;           // [views]
    ab_stereo_result* out;    // [pairs]
    double* poses;            // [views][6]: camera 1's rvec, tvec
    double* errs;             // [views][2]: per-view errors of camera 1 and camera 2
};

__global__ void __launch_bounds__(CALIB_THREADS) k_stereo_calibrate(StereoArgs a) {
    __shared__ StereoShared sh;
    const StereoPairRec& rec = a.pairs[blockIdx.x];
    StereoPair pr;
    pr.n_views = rec.n_views;
    pr.n_points = a.n_points + rec.view0;
    pr.offset = a.offset + rec.view0;
    pr.obj = a.obj;
    pr.img1 = a.img1;
    pr.img2 = a.img2;
    for (int i = 0; i < CALIB_NI; i++) {
        pr.kk1[i] = rec.kk1[i];
        pr.kk2[i] = rec.kk2[i];
    }
    StereoView* ws = a.ws + rec.view0;
    int iters = 0;
    stereo_calibrate_t<CalibCtaExec>(pr, ws, sh, a.max_iter, a.eps, &iters);
    for (int v = threadIdx.x; v < rec.n_views; v += blockDim.x)
        stereo_view_result(pr, ws, sh, v, a.poses + 6 * ((size_t)rec.view0 + v), a.errs + 2 * ((size_t)rec.view0 + v));
    if (threadIdx.x == 0) stereo_result(pr, sh, rec.K1, rec.K2, iters, a.out[blockIdx.x]);
}

}  // namespace ab
