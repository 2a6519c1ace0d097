// Host-compiled harness around the board stage's per-frame selection (board_select_stack, ab_math.cuh): lane 0 of every
// frame's warp in k_board_batch runs exactly this function.  TEST INFRASTRUCTURE, like hostcheck.cpp: never linked into
// libaruco_b200.so and not a CPU fallback.
#include <stdint.h>
#include "../../aruco_b200/csrc/ab_math.cuh"

extern "C" int hc_board_select(const ab_marker* ms, int nm, const int32_t* ids, const float* corners, int n_cfg, double mpp, float* obj,
                               float* img, int32_t* slots) {
    return ab::board_select_stack(ms, nm, ids, corners, n_cfg, mpp, nm, obj, img, slots);
}
