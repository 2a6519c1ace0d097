// aruco::MarkerDetector -- header-only C++ facade over the C ABI (include/aruco_b200.h).
//
// Same class, method names, argument meaning and error behaviour as the reference's
// aruco::MarkerDetector (src/markerdetector.h:43-311), aruco::Marker (src/marker.h:46-141) and
// aruco::CameraParameters (src/cameraparameters.h:38-127), for the hot path only.  OpenCV C++ is not
// available in this image, so the facade carries a minimal cv-compatible view type (`aruco::GreyView`,
// `cv::Point2f`-like `Point2f`).  With OpenCV present, compile with -DARUCO_B200_WITH_OPENCV and pass cv::Mat
// directly (see INTEGRATION.md).  Errors: the reference throws cv::Exception from CV_Assert; this facade throws
// aruco::Exception (derives from std::runtime_error) with the C ABI's message.
#pragma once
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../aruco_b200.h"

#ifdef ARUCO_B200_WITH_OPENCV
#include <opencv2/core.hpp>
#endif

namespace aruco {

struct Exception : std::runtime_error {
    int code;
    Exception(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

struct Point2f {
    float x = 0, y = 0;
    Point2f() {}
    Point2f(float x_, float y_) : x(x_), y(y_) {}
};
struct Point {  // cv::Point (int)
    int x = 0, y = 0;
    Point() {}
    Point(int x_, int y_) : x(x_), y(y_) {}
};
struct Size {
    int width = 0, height = 0;
    Size() {}
    Size(int w, int h) : width(w), height(h) {}
};

// non-owning view of an 8-bit image (1 channel grey or 3 channel BGR), row stride in bytes
struct ImageView {
    const uint8_t* data = nullptr;
    int rows = 0, cols = 0, channels = 1;
    size_t step = 0;
    ImageView() {}
    ImageView(const uint8_t* d, int r, int c, int ch = 1, size_t s = 0) : data(d), rows(r), cols(c), channels(ch), step(s ? s : (size_t)c * ch) {}
#ifdef ARUCO_B200_WITH_OPENCV
    ImageView(const cv::Mat& m) : data(m.data), rows(m.rows), cols(m.cols), channels(m.channels()), step(m.step) {
        if (m.depth() != CV_8U) throw Exception(AB_E_INVALID, "8-bit image required");
    }
#endif
    bool empty() const { return data == nullptr || rows == 0 || cols == 0; }
};

// aruco::CameraParameters: f32 3x3 camera matrix, f32 1x5 distortion, calibration image size
class CameraParameters {
public:
    float CameraMatrix[9];
    float Distorsion[5];
    Size CamSize;
    CameraParameters() : valid_(false) { std::memset(CameraMatrix, 0, sizeof(CameraMatrix)); std::memset(Distorsion, 0, sizeof(Distorsion)); }
    CameraParameters(const float K[9], const float D[5], Size size) { setParams(K, D, size); }
    // setParams (cameraparameters.cpp:65-72): values are held as f32
    void setParams(const float K[9], const float D[5], Size size) {
        std::memcpy(CameraMatrix, K, sizeof(CameraMatrix));
        if (D) std::memcpy(Distorsion, D, sizeof(Distorsion));
        else std::memset(Distorsion, 0, sizeof(Distorsion));
        CamSize = size;
        valid_ = true;
    }
    bool isValid() const { return valid_ && CamSize.width > 0 && CamSize.height > 0; }
    // resize (cameraparameters.cpp:166-180)
    void resize(Size size) {
        if (!isValid()) throw Exception(AB_E_INVALID, "invalid camera parameters");
        if (size.width == CamSize.width && size.height == CamSize.height) return;
        float ax = float(size.width) / float(CamSize.width), ay = float(size.height) / float(CamSize.height);
        CameraMatrix[0] *= ax;
        CameraMatrix[2] *= ax;
        CameraMatrix[4] *= ay;
        CameraMatrix[5] *= ay;
    }

private:
    bool valid_;
};

// aruco::Marker: vector of 4 corners + id + ssize + Rvec/Tvec (f64; empty <=> hasPose == false)
class Marker : public std::vector<Point2f> {
public:
    int id = -1;
    float ssize = -1;
    double Rvec[3] = {0, 0, 0}, Tvec[3] = {0, 0, 0};
    bool hasPose = false;
    Marker() {}
    bool isValid() const { return id != -1 && size() == 4; }
    bool operator<(const Marker& o) const { return id < o.id; }  // src/marker.h:123
    Point2f getCenter() const {                                   // src/marker.cpp:128-138
        Point2f c;
        for (const auto& p : *this) { c.x += p.x; c.y += p.y; }
        c.x /= float(size());
        c.y /= float(size());
        return c;
    }
};

// MarkerDetector::MarkerCandidate (markerdetector.h:45-62): a marker plus the contour it came from
class MarkerCandidate : public Marker {
public:
    std::vector<Point> contour;  // all the points of its contour
    int idx = -1;                // index position in the global contour list
    MarkerCandidate() {}
    MarkerCandidate(const Marker& m) : Marker(m) {}
};

class MarkerDetector {
public:
    typedef aruco::MarkerCandidate MarkerCandidate;
    enum ThresholdMethods { FIXED_THRES, ADPT_THRES, CANNY };              // markerdetector.h:125
    enum CornerRefinementMethod { NONE, HARRIS, SUBPIX, LINES };           // markerdetector.h:186
    // MarkerdetectorFunc (markerdetector.h:78) on a raw S x S 8UC1 buffer
    typedef int (*MarkerdetectorFunc)(uint8_t* canonical, int size, int* nRotations, void* user);

    explicit MarkerDetector(int device = 0) : h_(nullptr), speed_(0), device_(device) {
        int rc = ab_create(device, &h_);
        if (rc != AB_OK) throw Exception(rc, "aruco_b200: no CUDA device (this library has no CPU path)");
        ab_default_params(&p_);
    }
    ~MarkerDetector() { if (h_) ab_destroy(h_); }
    // The reference holds detectors by value (e.g. BoardDetector, boarddetector.h:146): a copy is a new device context
    // with the same configuration (parameters, dictionary, decoder function); per-frame state is not copied.
    MarkerDetector(const MarkerDetector& o) : h_(nullptr), speed_(0), device_(o.device_) {
        int rc = ab_create(device_, &h_);
        if (rc != AB_OK) throw Exception(rc, "aruco_b200: no CUDA device (this library has no CPU path)");
        ab_default_params(&p_);
        copy_config(o);
    }
    MarkerDetector& operator=(const MarkerDetector& o) {
        if (this != &o) copy_config(o);
        return *this;
    }

    // detect (markerdetector.h:102-120)
    void detect(const ImageView& input, std::vector<Marker>& detectedMarkers, const float* camMatrix = nullptr,
                const float* distCoeff = nullptr, float markerSizeMeters = -1, bool setYPerpendicular = false) {
        if (input.empty() || (input.channels != 1 && input.channels != 3)) throw Exception(AB_E_INVALID, "detect: 8UC1 or 8UC3 image required");
        set([&](ab_params& q) { q.set_y_perpendicular = setYPerpendicular; });
        std::vector<ab_marker> buf(kCap);
        int32_t n = 0;
        int rc = input.channels == 1
                     ? ab_detect_batch(h_, input.data, input.cols, input.rows, input.step, input.step * input.rows, 1, camMatrix,
                                       distCoeff, markerSizeMeters, buf.data(), kCap, &n)
                     : ab_detect_batch_bgr(h_, input.data, input.cols, input.rows, input.step, input.step * input.rows, 1,
                                           camMatrix, distCoeff, markerSizeMeters, buf.data(), kCap, &n);
        check(rc);
        detectedMarkers.clear();
        for (int i = 0; i < n; i++) detectedMarkers.push_back(convert(buf[i]));
        last_rows_ = input.rows;
        last_cols_ = input.cols;
    }
    void detect(const ImageView& input, std::vector<Marker>& detectedMarkers, const CameraParameters& camParams,
                float markerSizeMeters = -1, bool setYPerpendicular = false) {
        if (camParams.isValid()) detect(input, detectedMarkers, camParams.CameraMatrix, camParams.Distorsion, markerSizeMeters, setYPerpendicular);
        else detect(input, detectedMarkers, nullptr, nullptr, markerSizeMeters, setYPerpendicular);
    }
    // n_frames images of first's geometry, frame_stride bytes apart (0: packed), in one batch, without camera; markers[f] of
    // frame f.  A board armed on this detector's context (BoardDetector::setParams) runs on every frame as well.
    void detectBatch(const ImageView& first, int n_frames, size_t frame_stride, std::vector<std::vector<Marker>>& markers) {
        if (first.empty() || (first.channels != 1 && first.channels != 3) || n_frames < 1)
            throw Exception(AB_E_INVALID, "detectBatch: 8UC1 or 8UC3 images required");
        const size_t fs = frame_stride ? frame_stride : first.step * first.rows;
        std::vector<ab_marker> buf((size_t)n_frames * kCap);
        std::vector<int32_t> n(n_frames);
        int rc = first.channels == 1
                     ? ab_detect_batch(h_, first.data, first.cols, first.rows, first.step, fs, n_frames, nullptr, nullptr, -1.f, buf.data(), kCap, n.data())
                     : ab_detect_batch_bgr(h_, first.data, first.cols, first.rows, first.step, fs, n_frames, nullptr, nullptr, -1.f, buf.data(), kCap, n.data());
        check(rc);
        markers.assign(n_frames, std::vector<Marker>());
        for (int f = 0; f < n_frames; f++)
            for (int i = 0; i < n[f]; i++) markers[f].push_back(convert(buf[(size_t)f * kCap + i]));
        last_rows_ = first.rows;
        last_cols_ = first.cols;
    }

    // every setter validates a COPY of the parameters and commits it only when the library accepts it (a rejected value
    // must not poison later calls)
    void setThresholdMethod(ThresholdMethods m) { set([&](ab_params& q) { q.thres_method = m; }); }
    ThresholdMethods getThresholdMethod() const { return (ThresholdMethods)p_.thres_method; }
    void setThresholdParams(double param1, double param2) { set([&](ab_params& q) { q.thres_param1 = param1; q.thres_param2 = param2; }); }
    void getThresholdParams(double& param1, double& param2) const { param1 = p_.thres_param1; param2 = p_.thres_param2; }
    void setThresholdParamRange(size_t r1 = 0, size_t /*r2*/ = 0) { set([&](ab_params& q) { q.thres_param1_range = (int)r1; }); }  // h:152
    void enableLockedCornersMethod(bool enable) {  // markerdetector.cpp:291-295
        set([&](ab_params& q) {
            q.locked_corners = enable;
            if (enable) q.corner_method = SUBPIX;
        });
    }
    void enableErosion(bool enable) { set([&](ab_params& q) { q.erosion = enable; }); }  // API-compat extension (removed upstream)
    void setCornerRefinementMethod(CornerRefinementMethod m) { set([&](ab_params& q) { q.corner_method = m; }); }
    CornerRefinementMethod getCornerRefinementMethod() const { return (CornerRefinementMethod)p_.corner_method; }
    // CV_Assert(min>0 && min<=1 && max>0 && max<=1 && min<max), cpp:1031-1038
    void setMinMaxSize(float min = 0.03f, float max = 0.5f) { set([&](ab_params& q) { q.min_size = min; q.max_size = max; }); }
    void getMinMaxSize(float& min, float& max) const { min = p_.min_size; max = p_.max_size; }
    void setDesiredSpeed(int val) {  // markerdetector.cpp:265-285
        if (val < 0) val = 0;
        else if (val > 3) val = 2;
        set([&](ab_params& q) {
            if (val == 0) { q.warp_size = 56; q.corner_method = SUBPIX; }
            else if (val == 1 || val == 2) { q.warp_size = 28; q.corner_method = NONE; }
        });
        speed_ = val;
    }
    int getDesiredSpeed() const { return speed_; }
    void setWarpSize(int val) { set([&](ab_params& q) { q.warp_size = val; }); }  // CV_Assert(val >= 10), cpp:1047-1051
    int getWarpSize() const { return p_.warp_size; }
    // setMakerDetectorFunction (markerdetector.h:243): built-ins run on the device, others are called back
    void useFiducidalMarkers() { set([&](ab_params& q) { q.decoder = AB_DECODER_FIDUCIDAL; }); }
    void useHighlyReliableMarkers(int n, int count, const uint8_t* bits, int tau0, float correctionDistanceRate = 1.f) {
        check(ab_load_hrm_dictionary(h_, n, count, bits, tau0, correctionDistanceRate));  // loadDictionary, hrm.cpp:312-328
        dict_bits_.assign(bits, bits + (size_t)count * n * n);
        dict_n_ = n; dict_count_ = count; dict_tau0_ = tau0; dict_rate_ = correctionDistanceRate;
        set([&](ab_params& q) { q.decoder = AB_DECODER_HRM; });
    }
    void setMakerDetectorFunction(MarkerdetectorFunc fn, void* user = nullptr) {
        check(ab_set_decoder_callback(h_, fn, user));
        cb_ = fn; cb_user_ = user;
        set([&](ab_params& q) { q.decoder = AB_DECODER_HOST_CALLBACK; });
    }

    // getThresholdedImage (h:183): copies the binarised image of the last detect into dst (rows x cols, step)
    void getThresholdedImage(uint8_t* dst, size_t step) { check(ab_get_thresholded(h_, 0, dst, step)); }
    // getCandidates (h:266): quads rejected by the decoder in the last detect
    std::vector<std::vector<Point2f>> getCandidates() {
        std::vector<float> q(8 * 1024);
        std::vector<int32_t> ids(1024);
        int32_t n = 0;
        check(ab_get_candidates(h_, 0, q.data(), ids.data(), nullptr, 1024, &n));
        std::vector<std::vector<Point2f>> out;
        for (int i = 0; i < n; i++)
            if (ids[i] < 0) {
                std::vector<Point2f> c;
                for (int k = 0; k < 4; k++) c.push_back(Point2f(q[8 * i + 2 * k], q[8 * i + 2 * k + 1]));
                out.push_back(c);
            }
        return out;
    }
    // public workers thresHold / detectRectangles / warp (h:255-275)
    void thresHold(int method, const ImageView& grey, uint8_t* out, size_t out_step, double param1 = -1, double param2 = -1) {
        if (grey.channels != 1) throw Exception(AB_E_INVALID, "thresHold: 8UC1 required");  // CV_Assert, cpp:644
        check(ab_threshold(h_, grey.data, grey.cols, grey.rows, grey.step, method, param1, param2, out, out_step));
    }
    void detectRectangles(const ImageView& thres, std::vector<std::vector<Point2f>>& candidates) {
        std::vector<float> q(8 * 1024);
        int32_t n = 0;
        check(ab_detect_rectangles(h_, thres.data, thres.cols, thres.rows, thres.step, q.data(), 1024, &n));
        candidates.clear();
        for (int i = 0; i < n; i++) {
            std::vector<Point2f> c;
            for (int k = 0; k < 4; k++) c.push_back(Point2f(q[8 * i + 2 * k], q[8 * i + 2 * k + 1]));
            candidates.push_back(c);
        }
    }
    void warp(const ImageView& in, uint8_t* out, Size size, const std::vector<Point2f>& points) {
        if (points.size() != 4 || size.width != size.height) throw Exception(AB_E_INVALID, "warp: 4 points and a square size");  // cpp:685
        float q[8];
        for (int k = 0; k < 4; k++) { q[2 * k] = points[k].x; q[2 * k + 1] = points[k].y; }
        check(ab_warp(h_, in.data, in.cols, in.rows, in.step, q, size.width, out));
    }
    // refineCandidateLines (h:280, cpp:931-997): LINES refinement of one candidate from its contour
    void refineCandidateLines(MarkerCandidate& candidate, const float* camMatrix = nullptr, const float* distCoeff = nullptr) {
        if (candidate.size() != 4 || candidate.contour.size() < 4) throw Exception(AB_E_INVALID, "refineCandidateLines: 4 corners and a contour");
        std::vector<int32_t> xy(2 * candidate.contour.size());
        for (size_t i = 0; i < candidate.contour.size(); i++) { xy[2 * i] = candidate.contour[i].x; xy[2 * i + 1] = candidate.contour[i].y; }
        float c[8];
        for (int k = 0; k < 4; k++) { c[2 * k] = candidate[k].x; c[2 * k + 1] = candidate[k].y; }
        check(ab_refine_candidate_lines(h_, xy.data(), (int)candidate.contour.size(), c, camMatrix, distCoeff));
        for (int k = 0; k < 4; k++) candidate[k] = Point2f(c[2 * k], c[2 * k + 1]);
    }
    ab_context* handle() { return h_; }
    static Marker convert(const ab_marker& m) {
        Marker r;
        r.id = m.id;
        for (int k = 0; k < 4; k++) r.push_back(Point2f(m.corners[2 * k], m.corners[2 * k + 1]));
        r.ssize = m.ssize;
        r.hasPose = m.has_pose != 0;
        for (int k = 0; k < 3; k++) { r.Rvec[k] = m.rvec[k]; r.Tvec[k] = m.tvec[k]; }
        return r;
    }

private:
    static const int kCap = 512;
    ab_context* h_;
    ab_params p_;
    int speed_;
    int device_;
    int last_rows_ = 0, last_cols_ = 0;
    MarkerdetectorFunc cb_ = nullptr;
    void* cb_user_ = nullptr;
    std::vector<uint8_t> dict_bits_;
    int dict_n_ = 0, dict_count_ = 0, dict_tau0_ = 0;
    float dict_rate_ = 1.f;
    void check(int rc) { if (rc != AB_OK) throw Exception(rc, ab_last_error(h_)); }
    template <class F>
    void set(F f) {
        ab_params q = p_;
        f(q);
        check(ab_set_params(h_, &q));
        p_ = q;
    }
    void copy_config(const MarkerDetector& o) {
        if (!o.dict_bits_.empty()) {
            check(ab_load_hrm_dictionary(h_, o.dict_n_, o.dict_count_, o.dict_bits_.data(), o.dict_tau0_, o.dict_rate_));
            dict_bits_ = o.dict_bits_;
            dict_n_ = o.dict_n_; dict_count_ = o.dict_count_; dict_tau0_ = o.dict_tau0_; dict_rate_ = o.dict_rate_;
        }
        if (o.cb_) {
            check(ab_set_decoder_callback(h_, o.cb_, o.cb_user_));
            cb_ = o.cb_; cb_user_ = o.cb_user_;
        }
        check(ab_set_params(h_, &o.p_));
        p_ = o.p_;
        speed_ = o.speed_;
    }
};

}  // namespace aruco
