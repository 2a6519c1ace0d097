/* aruco_b200 -- C ABI of the B200-native marker-detection hot path.
 *
 * Drop-in boundary for paroj/aruco's aruco::MarkerDetector (src/markerdetector.h:43-311 of the reference).
 * Every entry point names the reference interface it replaces.  Plain pointers and sizes only; no C++ or
 * torch types; every call returns 0 on success or a negative ab_status, with a message retrievable through
 * ab_last_error().  Capacity overflows are reported (AB_E_CAPACITY), never truncated.  There is no CPU
 * fallback: ab_create fails when no CUDA device is available.
 *
 * One ab_context per host thread (the reference's MarkerDetector instance is not re-entrant either:
 * it mutates `thres` and `_candidates`, markerdetector.h:306-308).
 */
#ifndef ARUCO_B200_H
#define ARUCO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define AB_API __declspec(dllexport)
#else
#define AB_API __attribute__((visibility("default")))
#endif

typedef struct ab_context ab_context;

typedef enum ab_status {
    AB_OK = 0,
    AB_E_INVALID = -1,   /* bad argument (the reference would CV_Assert, e.g. markerdetector.cpp:644,1032,1048) */
    AB_E_CUDA = -2,      /* CUDA runtime error                                                     */
    AB_E_CAPACITY = -3,  /* a fixed-capacity device buffer overflowed; call ab_reserve with more    */
    AB_E_NO_DEVICE = -4, /* no usable CUDA device (this library has no CPU path)                   */
    AB_E_STATE = -5      /* call order error (e.g. HRM decoder selected without a dictionary)      */
} ab_status;

/* enum ThresholdMethods, markerdetector.h:125 */
enum { AB_THRES_FIXED = 0, AB_THRES_ADAPTIVE = 1, AB_THRES_CANNY = 2 };
/* enum CornerRefinementMethod, markerdetector.h:186 */
enum { AB_CORNER_NONE = 0, AB_CORNER_HARRIS = 1, AB_CORNER_SUBPIX = 2, AB_CORNER_LINES = 3 };
/* which decoder sits behind setMakerDetectorFunction (markerdetector.h:243): the two built-ins run on the
 * device, anything else is called back on the host with the canonical images */
enum { AB_DECODER_FIDUCIDAL = 0, AB_DECODER_HRM = 1, AB_DECODER_HOST_CALLBACK = 2 };

/* Private state of MarkerDetector (markerdetector.h:288-311); defaults = ctor (markerdetector.cpp:235-249).
 * Limits of this implementation that the reference does not have (ab_set_params / the detect calls return AB_E_INVALID):
 * thres_param1_range <= 7 (2r+1 <= 15 threshold images per frame), adaptive block size (thres_param1 made odd, >= 3) <= 63,
 * SUBPIX / locked-corner window (int)thres_param1 in 1..24, warp_size <= 128, frames 8..16384 pixels per side.            */
typedef struct ab_params {
    int32_t thres_method;        /* _thresMethod      (setThresholdMethod, h:129)            */
    double thres_param1;         /* _thresParam1      (setThresholdParams, h:140)            */
    double thres_param2;         /* _thresParam2                                             */
    int32_t corner_method;       /* _cornerMethod     (setCornerRefinementMethod, h:189)     */
    float min_size;              /* _minSize          (setMinMaxSize, h:200)                 */
    float max_size;              /* _maxSize                                                 */
    int32_t warp_size;           /* _markerWarpSize   (setWarpSize, h:232)                   */
    float border_dist;           /* _borderDistThres  (cpp:248)                              */
    int32_t locked_corners;      /* _useLockedCorners (enableLockedCornersMethod, h:165)     */
    int32_t erosion;             /* enableErosion (API-compat extension, default 0)          */
    int32_t decoder;             /* AB_DECODER_*      (setMakerDetectorFunction, h:243)      */
    int32_t set_y_perpendicular; /* detect(..., setYPerpendicular) h:102                     */
    int32_t thres_param1_range;  /* _thresParam1_range (setThresholdParamRange, h:152): 2r+1 threshold images */
} ab_params;

/* aruco::Marker (marker.h:46-141): 4 corners, id, ssize, Rvec/Tvec (f64). has_pose=0 => Rvec/Tvec empty. */
typedef struct ab_marker {
    int32_t id;
    int32_t has_pose;
    float corners[8];
    float ssize;
    float pad_;
    double rvec[3];
    double tvec[3];
} ab_marker;

/* MarkerdetectorFunc (markerdetector.h:78): `int f(const cv::Mat& in, int& nRotations)`; `canonical` is a
 * writable S x S 8UC1 image (the built-ins threshold it in place, arucofidmarkers.cpp:441-446). */
typedef int (*ab_decoder_fn)(uint8_t* canonical, int size, int* n_rotations, void* user);

/* ---- lifetime ------------------------------------------------------------------------------------ */
AB_API int ab_create(int device, ab_context** out);            /* MarkerDetector::MarkerDetector, cpp:235 */
AB_API void ab_destroy(ab_context* ctx);                       /* ~MarkerDetector, cpp:257               */
AB_API const char* ab_last_error(const ab_context* ctx);
AB_API const char* ab_version(void);

/* ---- configuration ------------------------------------------------------------------------------- */
AB_API int ab_default_params(ab_params* p);                    /* ctor defaults, cpp:235-249             */
AB_API int ab_set_params(ab_context* ctx, const ab_params* p); /* the set* methods, h:129-245            */
AB_API int ab_get_params(const ab_context* ctx, ab_params* p);
/* HighlyReliableMarkers::loadDictionary (highlyreliablemarkers.h:198-199, cpp:312-328):
 * bits = count*n*n bytes (row-major, 0/1), correction radius = rate*((tau0-1)/2).                        */
AB_API int ab_load_hrm_dictionary(ab_context* ctx, int n, int count, const uint8_t* bits, int tau0, float rate);
AB_API int ab_set_decoder_callback(ab_context* ctx, ab_decoder_fn fn, void* user); /* h:243 (custom fn)  */
/* Sizes device buffers. max_start_candidates / max_contour_points are per frame; <=0 picks defaults.  The capacities
 * are remembered: later automatic re-reservations (a larger batch, another warp size) keep them.  On failure the
 * context holds no buffers and the next call reserves again.
 * One buffer is sized at the first batch instead, because it depends on the maximum contour size in force then: the
 * strips in which the border walkers record their pixels (4 * (max contour length + 4) bytes per walker lane; 4.7 GB per
 * in-flight batch for 4K frames with the default sizes).  It never exceeds 6 GB unless the environment variable
 * ARUCO_B200_TRACE_REC_MB says otherwise -- a smaller budget only means fewer walker lanes.                            */
AB_API int ab_reserve(ab_context* ctx, int width, int height, int max_batch, int max_quads_per_frame,
                      int max_candidates_per_frame, int64_t max_start_candidates_per_frame,
                      int64_t max_contour_points_per_frame);
/* Names the caller's CUDA stream: every ab_enqueue_batch_device is ordered after the work already submitted to it (an
 * event is recorded there and the library's own stream waits for it), so frames produced on that stream need no host
 * synchronisation.  The handle is used as given: NULL is the legacy default stream (handle 0), which is what
 * torch.cuda.current_stream().cuda_stream reports for the default stream.  The library launches on private streams (one
 * per in-flight batch); results are ordered by ab_fetch_results.  Without this call nothing is ordered: the frames must be
 * complete on the device when they are enqueued.                                                                  */
AB_API int ab_set_stream(ab_context* ctx, void* cuda_stream);

/* ---- detect: MarkerDetector::detect (markerdetector.h:102-120, cpp:302-478) ----------------------- */
/* Host frames (8UC1, row stride `row_stride`, consecutive frames `frame_stride` bytes apart). Copies in,
 * runs the whole path for the batch, copies the markers out.  K: 9 floats row-major or NULL; D: 5 floats
 * or NULL (CameraParameters holds f32, cameraparameters.cpp:204-219).  out: n_frames*cap_per_frame.       */
AB_API int ab_detect_batch(ab_context* ctx, const uint8_t* frames, int width, int height, size_t row_stride,
                           size_t frame_stride, int n_frames, const float* K, const float* D, float marker_size,
                           ab_marker* out, int cap_per_frame, int32_t* counts);
/* Same with frames already resident in device memory: enqueue is asynchronous, fetch copies the markers to the host
 * and reports device-side errors.  TWO batches may be in flight: a second enqueue before the first fetch runs on a
 * second, library-owned set of buffers and a second internal stream, so its kernels overlap the tail of the first batch; a third enqueue returns AB_E_STATE.  ab_fetch_results returns the
 * batches in enqueue order.  The frames of a batch must stay untouched until that batch has been fetched.  The state
 * getters below read the batch last enqueued or fetched.                                                           */
AB_API int ab_enqueue_batch_device(ab_context* ctx, const uint8_t* dev_frames, int width, int height,
                                   size_t row_stride, size_t frame_stride, int n_frames, const float* K,
                                   const float* D, float marker_size);
AB_API int ab_fetch_results(ab_context* ctx, ab_marker* out, int cap_per_frame, int32_t* counts);
/* 8UC3 BGR front step (cvtColor BGR2GRAY, cpp:307-310) for host frames.                                   */
AB_API int ab_detect_batch_bgr(ab_context* ctx, const uint8_t* frames_bgr, int width, int height, size_t row_stride,
                               size_t frame_stride, int n_frames, const float* K, const float* D, float marker_size,
                               ab_marker* out, int cap_per_frame, int32_t* counts);

/* ---- state left by the last detect ----------------------------------------------------------------- */
AB_API int ab_get_thresholded(ab_context* ctx, int frame, uint8_t* dst, size_t dst_stride); /* getThresholdedImage h:183 */
AB_API int ab_get_grey(ab_context* ctx, int frame, uint8_t* dst, size_t dst_stride);
/* every candidate that reached the decoder, in the reference's order (cpp:350): quads = n*8 floats (the
 * corners entering warp), ids (-1 = rejected -> getCandidates h:266), n_rot.                              */
AB_API int ab_get_candidates(ab_context* ctx, int frame, float* quads, int32_t* ids, int32_t* n_rot, int cap, int32_t* n);
/* canonical image of a candidate: S*S bytes, S = the warp size the batch ran with (ab_get_canonical_size), which
 * differs from the current parameters when the warp size was changed after that batch was enqueued            */
AB_API int ab_get_canonical(ab_context* ctx, int frame, int candidate, uint8_t* dst /* S*S */);
AB_API int ab_get_canonical_size(ab_context* ctx, int32_t* size);
AB_API int ab_get_contour(ab_context* ctx, int frame, int candidate, int32_t* xy, int cap_points, int32_t* n);
/* counters[0]=start candidates [1]=contours kept (min<n<max) [2]=contour points [3]=quads before the
 * too-near filter [4]=candidates [5]=markers (summed over the batch)                                      */
AB_API int ab_get_counters(ab_context* ctx, int64_t* counters, int n);
/* per-stage device milliseconds of the last ab_detect_batch/ab_enqueue (needs ab_enable_timing):
 * [0]=threshold [1]=candidates [2]=decode [3]=refine [4]=filter+pose  (the reference's 5 phases, cpp:469-477) */
AB_API int ab_enable_timing(ab_context* ctx, int enable);
AB_API int ab_get_stage_ms(ab_context* ctx, float* ms, int n);
/* per-kernel device milliseconds of the last batch: [0]=threshold(+erosion) [1]=scan_starts [2]=trace (short walks)
 * [3]=trace (parked long walks) [4]=emit [5]=polygon [6]=frame_filter [7]=homography + sample (the warp stage)
 * [8]=otsu + identify [9]=refine [10]=finalize(+pose) [11]=board (k_board_batch; ~0 when no board is armed)     */
AB_API int ab_get_kernel_ms(ab_context* ctx, float* ms, int n);

/* ---- public workers of MarkerDetector ---------------------------------------------------------------- */
/* thresHold (h:255, cpp:643-677) */
AB_API int ab_threshold(ab_context* ctx, const uint8_t* grey, int width, int height, size_t row_stride, int method,
                        double param1, double param2, uint8_t* out, size_t out_stride);
/* detectRectangles (h:261, cpp:486-494): quads = cap*8 floats */
AB_API int ab_detect_rectangles(ab_context* ctx, const uint8_t* thres, int width, int height, size_t row_stride,
                                float* quads, int cap, int32_t* n);
/* warp (h:275, cpp:684-697) */
AB_API int ab_warp(ab_context* ctx, const uint8_t* grey, int width, int height, size_t row_stride, const float* quad,
                   int size, uint8_t* out);
/* refineCandidateLines (h:280, cpp:931-997): LINES refinement of one candidate.  contour_xy = n_points (x, y) pairs in
 * the order MarkerCandidate::contour holds them (h:45-62), corners = the 4 (integer valued) corners, which must be
 * points of the contour; replaced by the intersections of the fitted side lines.  The contour is undistorted first
 * only when BOTH K and D are given (cpp:957-959).                                                                   */
AB_API int ab_refine_candidate_lines(ab_context* ctx, const int32_t* contour_xy, int n_points, float* corners /* 8, in/out */,
                                     const float* K, const float* D);
/* Marker::calculateExtrinsics (marker.h / marker.cpp:112-125) for n markers */
AB_API int ab_calculate_extrinsics(ab_context* ctx, ab_marker* markers, int n, const float* K, const float* D,
                                   float marker_size, int set_y_perpendicular);

/* ---- next row: BoardDetector::detect (src/boarddetector.cpp:90-204) ------------------------------------ */
/* BoardConfiguration (src/board.h:56-97): ids + 4 object corners per marker, in pixels (info_type 0) or meters (1) */
typedef struct ab_board_config {
    int32_t n_markers;
    int32_t info_type;      /* BoardConfiguration::PIX = 0, METERS = 1 */
    const int32_t* ids;     /* n_markers */
    const float* corners;   /* n_markers * 4 * 3 */
} ab_board_config;
/* Board (src/board.h:103-140): the matched markers are returned separately; pose as in ab_marker */
typedef struct ab_board {
    int32_t n_markers;      /* detected markers that belong to the configuration */
    int32_t has_pose;
    float prob;             /* return value of BoardDetector::detect: n_markers / config size */
    float ssize;
    double rvec[3];
    double tvec[3];
} ab_board;
/* id filter, stacked 4*M-point solvePnP, optional reprojection-outlier re-solve (repj_err_thres > 0, cpp:172-194),
 * optional rotateXAxis.  board_markers (cap n) receives the matched markers in input order.  Runs the board kernel of the
 * batch path (ab_set_board) on these markers as a one-frame batch.                                                   */
AB_API int ab_detect_board(ab_context* ctx, const ab_marker* markers, int n, const ab_board_config* cfg, const float* K,
                           const float* D, float marker_size, float repj_err_thres, int set_y_perpendicular,
                           ab_marker* board_markers, ab_board* out);
/* largest configuration ab_set_board accepts (a 32 x 32 board) */
#define AB_BOARD_MAX_MARKERS 1024
/* BoardDetector::setParams (boarddetector.h) for the batch path: every later ab_enqueue_batch_device / ab_detect_batch /
 * ab_detect_batch_bgr of this context also runs BoardDetector::detect (boarddetector.cpp:90-204) on each frame's markers, in
 * one more kernel of the batch whose results come back with the markers.
 * The configuration is copied (the caller's arrays may be freed on return); K/D/marker_size are the BOARD's camera, independent
 * of the K/D given to the enqueue (those still govern the marker stage: LINES undistortion, per-marker pose).
 * cfg == NULL disarms.  AB_E_STATE while a batch is in flight; AB_E_INVALID for an empty configuration, NULL ids / corners
 * or more than AB_BOARD_MAX_MARKERS markers.                                                                         */
AB_API int ab_set_board(ab_context* ctx, const ab_board_config* cfg, const float* K, const float* D, float marker_size,
                        float repj_err_thres, int set_y_perpendicular);
/* The boards of the batch most recently returned by ab_fetch_results / ab_detect_batch(_bgr): boards[n_frames]; board_markers
 * (n_frames * cap_per_frame, may be NULL) receives each frame's matched markers in detection order with ssize set -- exactly what
 * ab_detect_board returns for that frame's markers.  AB_E_STATE if that batch ran without a board armed, n_frames differs, or
 * board_markers is requested but the markers were not fetched (out == NULL); AB_E_CAPACITY if a frame matched more markers
 * than cap_per_frame.                                                                                                 */
AB_API int ab_get_boards(ab_context* ctx, int n_frames, ab_board* boards, ab_marker* board_markers, int cap_per_frame);

/* ---- camera calibration from board views: cv::calibrateCamera (flags 0), planar targets ----------------------------------- */
/* the views of one camera: view v holds n_points[v] correspondences, the views' points stored one after another */
typedef struct ab_calib_camera {
    int32_t width, height;         /* imageSize                                 */
    int32_t n_views;
    const int32_t* n_points;       /* [n_views]                                 */
    const float* obj;              /* [sum n_points][3], the z = 0 plane        */
    const float* img;              /* [sum n_points][2] pixels                  */
} ab_calib_camera;
typedef struct ab_calib_result {
    double K[9];                   /* camera matrix, row-major                  */
    double D[5];                   /* k1 k2 p1 p2 k3                            */
    double rms;                    /* sqrt(sum |e|^2 / total points), as cv::calibrateCamera returns it */
    int32_t iterations;            /* Levenberg-Marquardt iterations (at most 30) */
    int32_t status;                /* 0, or AB_E_INVALID for a degenerate camera (K, D, rms, poses are then 0) */
} ab_calib_result;
/* limits of this implementation (larger inputs return AB_E_INVALID) */
#define AB_CALIB_MAX_CAMERAS 65536
#define AB_CALIB_MAX_VIEWS 1024           /* per camera   */
#define AB_CALIB_MAX_VIEW_POINTS 4096     /* per view     */
/* Calibrates n_cams cameras in one launch: free parameters fx, fy, cx, cy, k1, k2, p1, p2, k3 and a pose per view; skew, k4..k6,
 * the thin-prism and tilt terms are 0; termination TermCriteria(COUNT + EPS, 30, DBL_EPSILON).  A camera whose object points
 * are not in the z = 0 plane (|mean z| or its standard deviation above 1e-5), that has fewer than 2 views, a view with fewer
 * than 4 points, or views that do not determine the focal lengths (e.g. all parallel to the image plane) gets status
 * AB_E_INVALID; the other cameras are calibrated and the call returns AB_OK.  rvecs / tvecs ([total views][3] each, in camera
 * order, may be NULL) receive the pose of each view.  Runs on the context's stream and synchronises; AB_E_STATE while a batch
 * is in flight.                                                                                                         */
AB_API int ab_calibrate_cameras(ab_context* ctx, int n_cams, const ab_calib_camera* cams, ab_calib_result* out, double* rvecs,
                                double* tvecs);

/* ---- next row: marker / board rendering on the device ----------------------------------------------------- */
/* FiducidalMarkers::createMarkerImage (src/arucofidmarkers.cpp:213-263) without the text watermark (cv::putText
 * glyphs are OpenCV font data: not reproduced, addWaterMark must be false).  The image is square with side
 * size + 2*int(size*0.25f) when locked, else size; *out_side receives it; out == NULL only queries the side.   */
AB_API int ab_create_marker_image(ab_context* ctx, int id, int size, int locked, uint8_t* out, size_t out_stride, int* out_side);
/* createBoardImage (kind 0, :283-329), createBoardImage_ChessBoard (kind 1, :337-389), createBoardImage_Frame (kind 2,
 * :397-436) for a caller-supplied id list (the reference draws the ids with rand()).  Returns the image
 * (*out_w x *out_h; out == NULL only queries the size and the marker count) and the BoardConfiguration in pixels:
 * ids_out[i], corners_out[12*i..] (4 x (x,y,0)), *n_out markers.  kind 0 always centres the coordinates.          */
AB_API int ab_create_board_image(ab_context* ctx, int kind, int grid_w, int grid_h, int marker_size, int marker_distance,
                                 int center_data, const int32_t* ids, int n_ids, uint8_t* out, size_t out_stride, int* out_w,
                                 int* out_h, int32_t* ids_out, float* corners_out, int cap, int* n_out);
/* MarkerCode::getImg (src/highlyreliablemarkers.cpp:234-256): bits = n*n bytes (row-major, non-zero = white); pix_size
 * is rounded up to a multiple of n+2; *out_side receives the side; out == NULL only queries it.                   */
AB_API int ab_create_hrm_marker_image(ab_context* ctx, int n, const uint8_t* bits, int pix_size, uint8_t* out, size_t out_stride,
                                      int* out_side);

/* HighlyReliableMarkers::createBoardImage (src/highlyreliablemarkers.cpp:498-545) without the chromatic variant: a
 * grid_w x grid_h grid of the first grid_w*grid_h dictionary markers (bits: count*n*n bytes, row-major), marker side
 * (n+2)*20, gap side/5; ids_out = MarkerCode::getId() (the folded id of rotation 0), corners centred with y negated.
 * out == NULL only queries the size and the marker count.                                                        */
AB_API int ab_create_hrm_board_image(ab_context* ctx, int grid_w, int grid_h, int n, const uint8_t* bits, int count, uint8_t* out,
                                     size_t out_stride, int* out_w, int* out_h, int32_t* ids_out, float* corners_out, int cap,
                                     int* n_out);

/* pinned host memory for frame staging */
AB_API int ab_host_alloc(void** ptr, size_t bytes);
AB_API int ab_host_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* ARUCO_B200_H */
