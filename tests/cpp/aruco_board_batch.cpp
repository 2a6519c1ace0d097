// Headless batch counterpart of aruco_simple_board on the C++ facade: BoardDetector::detect(const cv::Mat&) over a batch of
// frames in one call (BoardDetector::detectBatch):
//   aruco_board_batch <frames.raw> <width> <height> <n_frames> <boardConfig.yml> <intrinsics.yml> <markerSizeMeters> <out_prefix>
// reads n_frames packed 8-bit grey frames and saves the Board of frame f to <out_prefix><f>.yml in the format of the
// reference's golden files; prints one line per frame: markers found, board probability, board markers.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "../../include/aruco/serialization.hpp"

int main(int argc, char** argv) {
    if (argc < 9) { std::fprintf(stderr, "usage: aruco_board_batch frames.raw W H N board.yml intrinsics.yml size out_prefix\n"); return 2; }
    const int W = std::atoi(argv[2]), H = std::atoi(argv[3]), N = std::atoi(argv[4]);
    if (W < 1 || H < 1 || N < 1) { std::fprintf(stderr, "bad geometry\n"); return 2; }
    std::vector<uint8_t> img((size_t)W * H * N);
    FILE* f = std::fopen(argv[1], "rb");
    if (!f || std::fread(img.data(), 1, img.size(), f) != img.size()) { std::fprintf(stderr, "cannot read frames\n"); return 2; }
    std::fclose(f);
    try {
        aruco::BoardConfiguration TheBoardConfig;
        TheBoardConfig.readFromFile(argv[5]);
        aruco::CameraParameters CamParam = aruco::readCameraParameters(argv[6]);
        CamParam.resize(aruco::Size(W, H));
        aruco::MarkerDetector MDetector;
        aruco::BoardDetector BD(MDetector);
        BD.setParams(TheBoardConfig, CamParam, (float)std::atof(argv[7]));
        std::vector<std::vector<aruco::Marker>> Markers;
        std::vector<float> prob;
        std::vector<aruco::Board> boards = BD.detectBatch(aruco::ImageView(img.data(), H, W), N, 0, Markers, &prob);
        for (int i = 0; i < N; i++) {
            std::printf("%zu %.6f %zu\n", Markers[i].size(), prob[i], boards[i].size());
            aruco::saveBoard(boards[i], std::string(argv[8]) + std::to_string(i) + ".yml");
        }
    } catch (const aruco::Exception& e) {
        std::fprintf(stderr, "aruco::Exception %d: %s\n", e.code, e.what());
        return 1;
    }
    return 0;
}
