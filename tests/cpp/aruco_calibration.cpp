// Headless counterpart of the reference's utils/aruco_calibration on the C++ facade: batched board detection over n frames,
// camera calibration from the detected boards on the device, intrinsics saved as CameraParameters::saveToFile does:
//   aruco_calibration <frames.raw> <width> <height> <n_frames> <boardConfig.yml> <markerSizeMeters> <out_intrinsics.yml>
// reads n_frames packed 8-bit grey frames; frames with fewer than 4 board markers are skipped.  Prints the number of views
// used and the rms reprojection error.  Corners are refined with SUBPIX: LINES corners of rendered views leave 0.7 px rms
// (2.2 px with erosion) and bias the focal length by 0.6 %, SUBPIX corners 0.3 px and 0.3 %.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "../../include/aruco/serialization.hpp"

int main(int argc, char** argv) {
    if (argc < 8) { std::fprintf(stderr, "usage: aruco_calibration frames.raw W H N board.yml marker_size out_intrinsics.yml\n"); return 2; }
    const int W = std::atoi(argv[2]), H = std::atoi(argv[3]), N = std::atoi(argv[4]);
    if (W < 1 || H < 1 || N < 1) { std::fprintf(stderr, "bad geometry\n"); return 2; }
    std::vector<uint8_t> img((size_t)W * H * N);
    FILE* f = std::fopen(argv[1], "rb");
    if (!f || std::fread(img.data(), 1, img.size(), f) != img.size()) { std::fprintf(stderr, "cannot read frames\n"); return 2; }
    std::fclose(f);
    try {
        aruco::BoardConfiguration TheBoardConfig;
        TheBoardConfig.readFromFile(argv[5]);
        aruco::MarkerDetector MDetector;
        MDetector.setCornerRefinementMethod(aruco::MarkerDetector::SUBPIX);
        aruco::BoardDetector BD(MDetector);
        BD.setParams(TheBoardConfig, aruco::CameraParameters(), (float)std::atof(argv[6]));
        std::vector<std::vector<aruco::Marker>> Markers;
        std::vector<aruco::Board> boards = BD.detectBatch(aruco::ImageView(img.data(), H, W), N, 0, Markers);
        std::vector<std::vector<std::array<float, 3>>> objPoints;
        std::vector<std::vector<aruco::Point2f>> imgPoints;
        BD.stackViews(boards, objPoints, imgPoints);
        aruco::CameraParameters CamParam;
        const double rms = aruco::calibrateCamera(MDetector, objPoints, imgPoints, aruco::Size(W, H), CamParam);
        aruco::saveCameraParameters(CamParam, argv[7]);
        std::printf("%zu %.17g\n", objPoints.size(), rms);
    } catch (const aruco::Exception& e) {
        std::fprintf(stderr, "aruco::Exception %d: %s\n", e.code, e.what());
        return 1;
    }
    return 0;
}
