// Headless stereo calibration on the C++ facade: batched board detection over the frames of two cameras, the views both cameras
// saw, stereo calibration with the cameras' intrinsics fixed on the device, and R, T, E, F saved for cv::FileStorage:
//   aruco_stereo_calibration <frames1.raw> <frames2.raw> <width> <height> <n_frames> <boardConfig.yml> <markerSizeMeters>
//                            <cam1.yml> <cam2.yml> <out.yml>
// reads n_frames packed 8-bit grey frames per camera (frame f of camera 1 and of camera 2 taken together); frames with fewer
// than 4 common board markers are skipped.  Prints the number of views used and the rms reprojection error.  Corners are
// refined with SUBPIX, as aruco_calibration refines them.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "../../include/aruco/serialization.hpp"

static bool read_frames(const char* path, std::vector<uint8_t>& img) {
    FILE* f = std::fopen(path, "rb");
    const bool ok = f && std::fread(img.data(), 1, img.size(), f) == img.size();
    if (f) std::fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc < 11) {
        std::fprintf(stderr, "usage: aruco_stereo_calibration frames1.raw frames2.raw W H N board.yml marker_size cam1.yml cam2.yml out.yml\n");
        return 2;
    }
    const int W = std::atoi(argv[3]), H = std::atoi(argv[4]), N = std::atoi(argv[5]);
    if (W < 1 || H < 1 || N < 1) { std::fprintf(stderr, "bad geometry\n"); return 2; }
    std::vector<uint8_t> img1((size_t)W * H * N), img2(img1.size());
    if (!read_frames(argv[1], img1) || !read_frames(argv[2], img2)) { std::fprintf(stderr, "cannot read frames\n"); return 2; }
    try {
        aruco::BoardConfiguration TheBoardConfig;
        TheBoardConfig.readFromFile(argv[6]);
        const aruco::CameraParameters cam1 = aruco::readCameraParameters(argv[8]), cam2 = aruco::readCameraParameters(argv[9]);
        aruco::MarkerDetector MDetector;
        MDetector.setCornerRefinementMethod(aruco::MarkerDetector::SUBPIX);
        aruco::BoardDetector BD(MDetector);
        BD.setParams(TheBoardConfig, aruco::CameraParameters(), (float)std::atof(argv[7]));
        std::vector<std::vector<aruco::Marker>> Markers;
        const std::vector<aruco::Board> boards1 = BD.detectBatch(aruco::ImageView(img1.data(), H, W), N, 0, Markers);
        const std::vector<aruco::Board> boards2 = BD.detectBatch(aruco::ImageView(img2.data(), H, W), N, 0, Markers);
        std::vector<std::vector<std::array<float, 3>>> objPoints;
        std::vector<std::vector<aruco::Point2f>> imgPoints1, imgPoints2;
        BD.stackStereoViews(boards1, boards2, objPoints, imgPoints1, imgPoints2);
        aruco::StereoParameters sp;
        const double rms = aruco::stereoCalibrate(MDetector, objPoints, imgPoints1, imgPoints2, cam1, cam2, sp);
        aruco::saveStereoParameters(sp, argv[10]);
        std::printf("%zu %.17g\n", objPoints.size(), rms);
    } catch (const aruco::Exception& e) {
        std::fprintf(stderr, "aruco::Exception %d: %s\n", e.code, e.what());
        return 1;
    }
    return 0;
}
