// Device-side data layout of one batch (fixed-capacity SoA buffers, see DESIGN.md "Data layout in HBM").
#pragma once
#include <stdint.h>
#include "../../include/aruco_b200.h"
#include "ab_math.cuh"

namespace ab {

enum : unsigned {
    ERR_STARTS_OVERFLOW = 1u,
    ERR_CONTOURS_OVERFLOW = 2u,
    ERR_POOL_OVERFLOW = 4u,
    ERR_QUADS_OVERFLOW = 8u,
    ERR_CANDS_OVERFLOW = 16u,
    ERR_LINE_FIT = 32u,  // LINES: the Jacobi SVD of a side needed more sweeps than the kernel replays
};

constexpr int MAX_QUADS = 1024;  // hard upper bound of quads per frame handled by the per-frame filter
constexpr int MAX_CANDS = 1024;   // hard upper bound of candidates per frame

// frame: bit 31 = border type (outer/hole), bit 30 = long contour (closed by k_trace<true>, which copied the points it
// recorded while walking into the pool; k_emit only adds the TRACE_PARK_N steps walked before the walk was parked)
constexpr uint32_t CONTOUR_LONG = 0x40000000u, CONTOUR_FRAME_MASK = 0x3FFFFFFFu;
struct ContourRec {
    uint32_t frame;
    uint32_t off;  // first point in the pool
    uint32_t n;    // number of points
    uint32_t key;  // raster scan position of the Suzuki start (ordering = reverse discovery)
};

// a border walk parked by k_trace<false> for k_trace<true> (full walker state)
struct LongRec {
    uint32_t frame;  // bit 31 = border type
    uint32_t key;
    uint32_t sxy, fxy, bxy;  // start / forward walker / backward walker pixel (x | y << 16)
    uint32_t dirs;           // fw.b | bw.b << 4 | start.b << 8
    uint32_t nf, ng;
};

struct QuadRec {
    short x[4], y[4];
    uint32_t key;
    uint32_t contour;
};

struct CandRec {
    float c[8];        // corners entering warp (after the orientation swap), integer valued
    float refined[8];  // corners after LINES / SUBPIX / HARRIS (== c when NONE)
    uint32_t contour;
    int32_t swapped;
    int32_t id;
    int32_t nrot;
};

// per-candidate scratch of the identification stage (k_decode.cuh)
struct CandAux {
    double Mi[9];  // canonical -> image homography (inverse of getPerspectiveTransform)
    int32_t ok;    // 0: degenerate quad
    int32_t thr;   // Otsu threshold of the canonical image
};

// counters zeroed at the start of every batch
struct Counters {
    unsigned long long n_starts;
    unsigned long long pool_used;
    unsigned int n_contours;
    unsigned int trace_work;
    unsigned int err;
    unsigned int emit_work;
    unsigned int n_long, long_work;
    unsigned int canny_changed, pad3;
    unsigned long long n_quads_total, n_cands_total, n_markers_total;
};

struct HrmDict {
    const uint64_t* bits;  // count rotation-0 bit strings
    const uint32_t* ids;   // sorted folded ids (tree order) .. see k_decode
    const uint32_t* ord_ids;
    const int32_t* ord_pos;
    const int32_t* tree;  // 2*count children
    int root;
    int count;
    int n;
    int correction;
};

// floats of board-stage scratch per marker slot: 4 object points (12) + 4 image points (8), twice (the outlier re-solve)
constexpr int BOARD_PTS_PER_MARKER = 40;

// an armed BoardConfiguration with its camera (BoardDetector::setParams); d01, mpp and ssize are computed on the host
struct BoardArgs {
    const int32_t* ids;    // [n_cfg], device
    const float* corners;  // [n_cfg][12], device
    int n_cfg;
    int pose;              // a camera was given and the configuration has enough information (boarddetector.cpp:117-130)
    double mpp;            // marker_meter_per_pix (:132-136)
    float ssize;
    float repj_err_thres;
    int set_y_perp;
    Camera cam;
};

struct Batch {
    int W, H, B, wpr;
    int n_t;  // threshold images per frame (2*range+1, setThresholdParamRange); bits/thres hold B*n_t virtual frames
    size_t bits_words;  // per frame
    const uint8_t* grey;
    size_t grey_row, grey_frame;
    uint8_t* thres;   // [B][H][W]
    uint32_t* bits;   // [B][bits_words]
    uint32_t* bits2;  // scratch for erosion
    uint2* starts;
    unsigned long long cap_starts;
    ContourRec* contours;
    unsigned int cap_contours;
    uint32_t* pool;
    unsigned long long cap_pool;
    LongRec* longq;
    unsigned int cap_long;
    const uint8_t* walk_lut;  // WALK_LUT_FW then WALK_LUT_BW (ab_trace.cuh)
    uint2* trace_rec;       // k_trace<true>: per-lane record of the pixels visited (forward, backward) since the walk was resumed
    unsigned int rec_half;  // entries per lane (max_len / 2 + 2)
    QuadRec* quads;  // [B][cap_q]
    int cap_q;
    CandRec* cands;  // [B][cap_c]
    int cap_c;
    uint8_t* canon;  // [B][cap_c][S*S]
    CandAux* aux;    // [B][cap_c]
    unsigned short* hist;  // [B][cap_c][256] histogram of the canonical image
    ab_marker* markers;  // [B][cap_c]
    Counters* cnt;
    unsigned int* n_quads;    // [B]
    unsigned int* n_cands;    // [B]
    unsigned int* n_markers;  // [B]
    // board stage (k_board_batch), only when a board configuration is armed (boards == nullptr otherwise)
    ab_board* boards;      // [B]
    int32_t* board_slots;  // [B][cap_c] marker indices of the matched markers
    float* board_pts;      // [B][cap_c * BOARD_PTS_PER_MARKER] obj | img | obj2 | img2 of the stacked correspondences
    // parameters
    int min_len, max_len;  // contour length limits (exclusive)
    int S;                 // warp size
    int decoder;
    int corner_method;
    int subpix_win;
    int locked;
    int set_y_perp;
    int vx0, vy0, vx1, vy1;  // valid region of the border filter
    float marker_size;
    Camera cam;
    HrmDict dict;
    AB_HD BitImage bit_image(int f) const { return BitImage{bits + (size_t)f * bits_words, wpr, W, H}; }
};

}  // namespace ab
