// YAML wire formats of the reference (SURVEY 8(f) row 2), header-only, no OpenCV:
//   camera intrinsics      CameraParameters::readFromXMLFile / saveToFile   (src/cameraparameters.cpp:140-222)
//   marker lists / boards  cv::FileStorage << Marker / Board                 (src/serialization.cpp:24-68, test/filestorage_adapter.h)
//   BoardConfiguration     readFromFile / saveToFile                         (src/serialization.cpp:70-118, src/board.cpp:45-56)
//   HRM Dictionary         Dictionary::fromFile / toFile                     (src/serialization.cpp:120-152)
// The reference stores all of them through cv::FileStorage in its YAML 1.0 dialect.  `yaml::parse` reads the subset
// of that dialect cv::FileStorage writes (block maps and sequences, flow maps/sequences that may span lines, `key:value`
// without a space inside flow maps, `!!opencv-matrix`, quoted strings, comments); the writers emit text that
// cv::FileStorage reads back (tests/test_yaml.py checks both directions against cv2.FileStorage).
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <sstream>
#include <string>
#include <utility>
#include <vector>

#include "markerdetector.hpp"

namespace aruco {
namespace yaml {

struct Node {
    enum Type { NONE, SCALAR, SEQ, MAP } type = NONE;
    std::string scalar, tag;
    std::vector<Node> seq;
    std::vector<std::pair<std::string, Node>> map;
    bool empty() const { return type == NONE; }
    size_t size() const { return type == SEQ ? seq.size() : (type == MAP ? map.size() : 0); }
    const Node& operator[](const std::string& key) const {
        static const Node none;
        for (const auto& kv : map)
            if (kv.first == key) return kv.second;
        return none;
    }
    const Node& operator[](size_t i) const { return seq.at(i); }
    double as_double() const {
        if (type != SCALAR) throw Exception(AB_E_INVALID, "yaml: scalar expected");
        // cv::FileStorage writes ".Inf" / ".Nan"; plain strtod covers "1.", "0.", "-2.17e+00"
        if (scalar == ".Inf" || scalar == ".inf") return 1e308 * 10;
        if (scalar == "-.Inf" || scalar == "-.inf") return -1e308 * 10;
        char* end = nullptr;
        double v = std::strtod(scalar.c_str(), &end);
        if (end == scalar.c_str()) throw Exception(AB_E_INVALID, "yaml: number expected, got '" + scalar + "'");
        return v;
    }
    int as_int() const { return (int)as_double(); }
    const std::string& as_string() const { return scalar; }
};

class Parser {
public:
    explicit Parser(const std::string& text) {
        std::istringstream in(text);
        std::string l;
        while (std::getline(in, l)) {
            if (!l.empty() && l.back() == '\r') l.pop_back();
            std::string s = strip_comment(l);
            size_t ind = s.find_first_not_of(' ');
            if (ind == std::string::npos) continue;
            if (s.compare(ind, 1, "%") == 0 || s.compare(ind, 3, "---") == 0 || s.compare(ind, 3, "...") == 0) continue;
            lines_.push_back(Line{(int)ind, s.substr(ind)});
        }
    }
    Node parse() {
        if (lines_.empty()) return Node();
        return block(lines_[0].indent);
    }

private:
    struct Line {
        int indent;
        std::string text;
    };
    std::vector<Line> lines_;
    size_t li_ = 0;

    static std::string strip_comment(const std::string& l) {
        bool q = false;
        for (size_t i = 0; i < l.size(); i++) {
            if (l[i] == '"') q = !q;
            if (!q && l[i] == '#' && (i == 0 || l[i - 1] == ' ')) return rtrim(l.substr(0, i));
        }
        return rtrim(l);
    }
    static std::string rtrim(std::string s) {
        while (!s.empty() && (s.back() == ' ' || s.back() == '\t')) s.pop_back();
        return s;
    }
    static std::string trim(const std::string& s) {
        size_t a = s.find_first_not_of(" \t");
        if (a == std::string::npos) return "";
        return rtrim(s.substr(a));
    }
    static std::string unquote(const std::string& s) {
        if (s.size() >= 2 && s.front() == '"' && s.back() == '"') {
            std::string o;
            for (size_t i = 1; i + 1 < s.size(); i++) {
                if (s[i] == '\\' && i + 2 < s.size()) {
                    char c = s[++i];
                    o += c == 'n' ? '\n' : (c == 't' ? '\t' : c);
                } else {
                    o += s[i];
                }
            }
            return o;
        }
        return s;
    }
    static Node scalar_node(const std::string& s) {
        Node n;
        n.type = Node::SCALAR;
        n.scalar = unquote(trim(s));
        return n;
    }

    // value text that starts on the current line after "key:" or "-"; may continue on following lines (flow) or be a
    // nested block on deeper-indented lines (empty rest)
    Node value(std::string rest, int parent_indent) {
        rest = trim(rest);
        std::string tag;
        if (rest.compare(0, 2, "!!") == 0) {
            size_t sp = rest.find(' ');
            tag = rest.substr(2, sp == std::string::npos ? std::string::npos : sp - 2);
            rest = sp == std::string::npos ? "" : trim(rest.substr(sp));
        }
        Node n;
        if (rest.empty()) {
            li_++;
            if (li_ < lines_.size() && lines_[li_].indent > parent_indent) n = block(lines_[li_].indent);
            else if (li_ < lines_.size() && lines_[li_].indent == parent_indent && lines_[li_].text[0] == '-') n = block(parent_indent);  // "key:\n- a" at the same indent
        } else if (rest[0] == '[' || rest[0] == '{') {
            std::string flow = rest;
            while (!balanced(flow)) {
                li_++;
                if (li_ >= lines_.size()) throw Exception(AB_E_INVALID, "yaml: unterminated flow collection");
                flow += " " + lines_[li_].text;
            }
            li_++;
            size_t pos = 0;
            n = flow_value(flow, pos);
        } else {
            n = scalar_node(rest);
            li_++;
        }
        n.tag = tag;
        return n;
    }
    static bool balanced(const std::string& s) {
        int d = 0;
        bool q = false;
        for (char c : s) {
            if (c == '"') q = !q;
            if (q) continue;
            if (c == '[' || c == '{') d++;
            if (c == ']' || c == '}') d--;
        }
        return d == 0 && !q;
    }
    static void skip_ws(const std::string& s, size_t& p) {
        while (p < s.size() && (s[p] == ' ' || s[p] == '\t')) p++;
    }
    Node flow_value(const std::string& s, size_t& p) {
        skip_ws(s, p);
        Node n;
        if (p < s.size() && s[p] == '[') {
            n.type = Node::SEQ;
            p++;
            skip_ws(s, p);
            if (p < s.size() && s[p] == ':') p++;  // "[:" is cv::FileStorage's flow marker when writing, never written out
            for (;;) {
                skip_ws(s, p);
                if (p >= s.size()) throw Exception(AB_E_INVALID, "yaml: ']' expected");
                if (s[p] == ']') { p++; break; }
                n.seq.push_back(flow_value(s, p));
                skip_ws(s, p);
                if (p < s.size() && s[p] == ',') p++;
            }
        } else if (p < s.size() && s[p] == '{') {
            n.type = Node::MAP;
            p++;
            for (;;) {
                skip_ws(s, p);
                if (p >= s.size()) throw Exception(AB_E_INVALID, "yaml: '}' expected");
                if (s[p] == '}') { p++; break; }
                size_t c = s.find(':', p);
                if (c == std::string::npos) throw Exception(AB_E_INVALID, "yaml: ':' expected in flow map");
                std::string key = unquote(trim(s.substr(p, c - p)));
                p = c + 1;
                n.map.push_back(std::make_pair(key, flow_value(s, p)));
                skip_ws(s, p);
                if (p < s.size() && s[p] == ',') p++;
            }
        } else {
            size_t b = p;
            bool q = false;
            while (p < s.size() && (q || (s[p] != ',' && s[p] != ']' && s[p] != '}'))) {
                if (s[p] == '"') q = !q;
                p++;
            }
            n = scalar_node(s.substr(b, p - b));
        }
        return n;
    }
    static size_t key_colon(const std::string& t) {  // position of the ':' that ends a block-map key, npos if none
        bool q = false;
        for (size_t i = 0; i < t.size(); i++) {
            if (t[i] == '"') q = !q;
            if (!q && t[i] == ':' && (i + 1 == t.size() || t[i + 1] == ' ')) return i;
            if (!q && (t[i] == '[' || t[i] == '{')) return std::string::npos;
        }
        return std::string::npos;
    }
    Node block(int indent) {
        Node n;
        if (lines_[li_].text[0] == '-' && (lines_[li_].text.size() == 1 || lines_[li_].text[1] == ' ')) {
            n.type = Node::SEQ;
            while (li_ < lines_.size() && lines_[li_].indent == indent && lines_[li_].text[0] == '-') {
                std::string rest = trim(lines_[li_].text.substr(1));
                if (!rest.empty() && rest[0] != '[' && rest[0] != '{' && key_colon(rest) != std::string::npos) {
                    // "- key: value" starts an inline block map whose further keys sit at the key's column
                    int col = indent + (int)(lines_[li_].text.size() - rest.size());
                    lines_[li_].indent = col;
                    lines_[li_].text = rest;
                    n.seq.push_back(block(col));
                } else {
                    n.seq.push_back(value(rest, indent));
                }
            }
        } else {
            n.type = Node::MAP;
            while (li_ < lines_.size() && lines_[li_].indent == indent && lines_[li_].text[0] != '-') {
                const std::string& t = lines_[li_].text;
                size_t c = key_colon(t);
                if (c == std::string::npos) throw Exception(AB_E_INVALID, "yaml: 'key:' expected in '" + t + "'");
                std::string key = unquote(trim(t.substr(0, c)));
                n.map.push_back(std::make_pair(key, value(t.substr(c + 1), indent)));
            }
        }
        return n;
    }
};

inline Node parse(const std::string& text) { return Parser(text).parse(); }
inline std::string read_text(const std::string& path) {
    std::ifstream f(path.c_str(), std::ios::binary);
    if (!f) throw Exception(AB_E_INVALID, "cannot open " + path);
    std::ostringstream ss;
    ss << f.rdbuf();
    return ss.str();
}
inline Node load(const std::string& path) { return parse(read_text(path)); }
inline void write_text(const std::string& path, const std::string& text) {
    std::ofstream f(path.c_str(), std::ios::binary);
    if (!f) throw Exception(AB_E_INVALID, "cannot write " + path);
    f << text;
}
// numbers as cv::FileStorage prints them: %.16e for f64, %.8e for f32, integers plain
inline std::string num(double v) {
    char b[64];
    if (v == (double)(long long)v && v > -1e15 && v < 1e15) std::snprintf(b, sizeof b, "%lld.", (long long)v);
    else std::snprintf(b, sizeof b, "%.16e", v);
    return b;
}
inline std::string numf(float v) {
    char b[64];
    if (v == (float)(long long)v && v > -1e7f && v < 1e7f) std::snprintf(b, sizeof b, "%lld.", (long long)v);
    else std::snprintf(b, sizeof b, "%.8e", (double)v);
    return b;
}
// !!opencv-matrix (dt "d" or "f") -> row-major doubles
inline std::vector<double> matrix(const Node& n, int* rows = nullptr, int* cols = nullptr) {
    std::vector<double> out;
    if (n.empty()) return out;
    const Node& data = n["data"];
    if (n.type != Node::MAP || data.type != Node::SEQ) throw Exception(AB_E_INVALID, "yaml: opencv-matrix expected");
    if (rows) *rows = n["rows"].as_int();
    if (cols) *cols = n["cols"].as_int();
    for (const auto& v : data.seq) out.push_back(v.as_double());
    if ((int)out.size() != n["rows"].as_int() * n["cols"].as_int()) throw Exception(AB_E_INVALID, "yaml: matrix size mismatch");
    return out;
}

}  // namespace yaml

// ---- camera intrinsics ------------------------------------------------------------------------------------
// CameraParameters::readFromXMLFile (src/cameraparameters.cpp:187-222): values converted to f32, the first 5
// distortion coefficients kept; throws like the reference on a missing matrix / size / < 4 coefficients
inline CameraParameters readCameraParameters(const std::string& path) {
    const yaml::Node fs = yaml::load(path);
    int w = -1, h = -1;
    if (!fs["image_width"].empty()) w = fs["image_width"].as_int();
    if (!fs["image_height"].empty()) h = fs["image_height"].as_int();
    const std::vector<double> K = yaml::matrix(fs["camera_matrix"]), D = yaml::matrix(fs["distortion_coefficients"]);
    if (K.size() != 9) throw Exception(9007, "File :" + path + " does not contains valid camera matrix");
    if (w == -1 || h == 0) throw Exception(9007, "File :" + path + " does not contains valid camera dimensions");
    if (D.size() < 4) throw Exception(9007, "File :" + path + " does not contains valid distortion_coefficients");
    float Kf[9], Df[5] = {0, 0, 0, 0, 0};
    for (int i = 0; i < 9; i++) Kf[i] = (float)K[i];
    for (size_t i = 0; i < 5 && i < D.size(); i++) Df[i] = (float)D[i];
    return CameraParameters(Kf, Df, Size(w, h));
}
// CameraParameters::saveToFile (src/cameraparameters.cpp:140-162), YAML variant
inline void saveCameraParameters(const CameraParameters& cp, const std::string& path) {
    if (!cp.isValid()) throw Exception(9006, "invalid object");
    std::ostringstream o;
    o << "%YAML:1.0\n---\nimage_width: " << cp.CamSize.width << "\nimage_height: " << cp.CamSize.height << "\n";
    o << "camera_matrix: !!opencv-matrix\n   rows: 3\n   cols: 3\n   dt: f\n   data: [ ";
    for (int i = 0; i < 9; i++) o << yaml::numf(cp.CameraMatrix[i]) << (i < 8 ? ", " : " ]\n");
    o << "distortion_coefficients: !!opencv-matrix\n   rows: 1\n   cols: 5\n   dt: f\n   data: [ ";
    for (int i = 0; i < 5; i++) o << yaml::numf(cp.Distorsion[i]) << (i < 4 ? ", " : " ]\n");
    yaml::write_text(path, o.str());
}

// ---- markers ----------------------------------------------------------------------------------------------
inline std::string markerToYaml(const Marker& m, const std::string& indent) {  // serialization.cpp:24-45
    std::ostringstream o;
    o << indent << "-\n" << indent << "   id: " << m.id << "\n";
    if (m.hasPose) {
        o << indent << "   Tvec: [ " << yaml::num(m.Tvec[0]) << ", " << yaml::num(m.Tvec[1]) << ", " << yaml::num(m.Tvec[2]) << " ]\n";
        o << indent << "   Rvec: [ " << yaml::num(m.Rvec[0]) << ", " << yaml::num(m.Rvec[1]) << ", " << yaml::num(m.Rvec[2]) << " ]\n";
    }
    o << indent << "   corners: [ ";
    for (size_t i = 0; i < m.size(); i++) o << "[ " << yaml::numf(m[i].x) << ", " << yaml::numf(m[i].y) << " ]" << (i + 1 < m.size() ? ", " : "");
    o << " ]\n";
    return o.str();
}
inline Marker markerFromYaml(const yaml::Node& ms) {  // serialization.cpp:47-68
    Marker m;
    if (ms.empty()) return m;
    m.id = ms["id"].as_int();
    const yaml::Node &T = ms["Tvec"], &R = ms["Rvec"];
    if (T.size() == 3 && R.size() == 3) {
        for (int k = 0; k < 3; k++) {
            m.Tvec[k] = T[(size_t)k].as_double();
            m.Rvec[k] = R[(size_t)k].as_double();
        }
        m.hasPose = true;
    }
    const yaml::Node& c = ms["corners"];
    for (size_t i = 0; i < c.size(); i++) m.push_back(Point2f((float)c[i][(size_t)0].as_double(), (float)c[i][(size_t)1].as_double()));
    return m;
}
// the golden files of the reference's tests: "Markers: [ marker, ... ]" (test/core_tests.cpp:100-110)
inline void saveMarkers(const std::vector<Marker>& markers, const std::string& path, const std::string& key = "Markers") {
    std::ostringstream o;
    o << "%YAML:1.0\n---\n" << key << ":\n";
    for (const auto& m : markers) o << markerToYaml(m, "   ");
    yaml::write_text(path, o.str());
}
inline std::vector<Marker> readMarkers(const std::string& path, const std::string& key = "Markers") {
    const yaml::Node fs = yaml::load(path);
    std::vector<Marker> out;
    const yaml::Node& l = fs[key];
    for (size_t i = 0; i < l.size(); i++) out.push_back(markerFromYaml(l[i]));
    return out;
}

// ---- BoardConfiguration (src/board.h:56-97) ------------------------------------------------------------------
struct BoardConfiguration {
    enum MarkerInfoType { NONE = -1, PIX = 0, METERS = 1 };
    int mInfoType = NONE;
    std::vector<int> ids;
    std::vector<std::array<float, 12>> objPoints;  // 4 x (x, y, z) per marker
    size_t size() const { return ids.size(); }
    bool isExpressedInMeters() const { return mInfoType == METERS; }
    bool isExpressedInPixels() const { return mInfoType == PIX; }
    int getIndexOfMarkerId(int id) const {  // board.cpp:60-65
        for (size_t i = 0; i < ids.size(); i++)
            if (ids[i] == id) return (int)i;
        return -1;
    }
    // read (serialization.cpp:92-118)
    void readFromFile(const std::string& path) {
        const yaml::Node fn = yaml::load(path);
        if (fn["aruco_bc_nmarkers"].empty()) throw Exception(AB_E_INVALID, "invalid file type");
        const int n = fn["aruco_bc_nmarkers"].as_int();
        mInfoType = fn["aruco_bc_mInfoType"].as_int();
        const yaml::Node& markers = fn["aruco_bc_markers"];
        if (n != (int)markers.size()) throw Exception(AB_E_INVALID, "aruco_bc_nmarkers does not match the marker list");
        ids.assign(markers.size(), 0);
        objPoints.assign(markers.size(), std::array<float, 12>());
        for (size_t i = 0; i < markers.size(); i++) {
            ids[i] = markers[i]["id"].as_int();
            const yaml::Node& c = markers[i]["corners"];
            if (c.size() != 4) throw Exception(AB_E_INVALID, "4 corners per board marker expected");
            for (size_t k = 0; k < 4; k++)
                for (size_t d = 0; d < 3; d++) objPoints[i][3 * k + d] = (float)c[k][d].as_double();
        }
    }
    // operator<< (serialization.cpp:71-90)
    void saveToFile(const std::string& path) const {
        std::ostringstream o;
        o << "%YAML:1.0\n---\naruco_bc_nmarkers: " << ids.size() << "\naruco_bc_mInfoType: " << mInfoType << "\naruco_bc_markers:\n";
        for (size_t i = 0; i < ids.size(); i++) {
            o << "   - { id:" << ids[i] << ", corners:[ ";
            for (int k = 0; k < 4; k++)
                o << "[ " << yaml::numf(objPoints[i][3 * k]) << ", " << yaml::numf(objPoints[i][3 * k + 1]) << ", " << yaml::numf(objPoints[i][3 * k + 2]) << " ]"
                  << (k < 3 ? ", " : "");
            o << " ] }\n";
        }
        yaml::write_text(path, o.str());
    }
    ab_board_config abi() const {
        ab_board_config c;
        c.n_markers = (int32_t)ids.size();
        c.info_type = mInfoType;
        c.ids = ids.data();
        c.corners = objPoints.empty() ? nullptr : objPoints[0].data();
        return c;
    }
};

// ---- Board (src/board.h:103-140) and BoardDetector::detect (src/boarddetector.cpp:90-204) -------------------------
struct Board : std::vector<Marker> {
    BoardConfiguration conf;
    double Rvec[3] = {0, 0, 0}, Tvec[3] = {0, 0, 0};
    bool hasPose = false;
    float markerSizeMeters = -1;
};
inline void saveBoard(const Board& b, const std::string& path, const std::string& key = "Board") {  // filestorage_adapter.h:23-37
    std::ostringstream o;
    o << "%YAML:1.0\n---\n" << key << ":\n";
    o << "   Tvec: [ " << yaml::num(b.Tvec[0]) << ", " << yaml::num(b.Tvec[1]) << ", " << yaml::num(b.Tvec[2]) << " ]\n";
    o << "   Rvec: [ " << yaml::num(b.Rvec[0]) << ", " << yaml::num(b.Rvec[1]) << ", " << yaml::num(b.Rvec[2]) << " ]\n";
    o << "   Markers:\n";
    for (const auto& m : b) o << markerToYaml(m, "      ");
    yaml::write_text(path, o.str());
}
inline Board readBoard(const std::string& path, const std::string& key = "Board") {  // filestorage_adapter.h:39-60
    const yaml::Node fs = yaml::load(path);
    const yaml::Node& bs = fs[key];
    Board b;
    if (bs.empty()) return b;
    for (int k = 0; k < 3; k++) {
        b.Tvec[k] = bs["Tvec"][(size_t)k].as_double();
        b.Rvec[k] = bs["Rvec"][(size_t)k].as_double();
    }
    b.hasPose = true;
    const yaml::Node& ms = bs["Markers"];
    for (size_t i = 0; i < ms.size(); i++) b.push_back(markerFromYaml(ms[i]));
    return b;
}

class BoardDetector {
public:
    explicit BoardDetector(MarkerDetector& md, bool setYPerpendicular = false) : md_(md), y_perp_(setYPerpendicular) {}  // boarddetector.h:68
    void setYPerpendicular(bool enable) { y_perp_ = enable; arm(); }   // boarddetector.h:126
    bool isYPerpendicular() const { return y_perp_; }
    void set_repj_err_thres(float v) { repj_err_thres_ = v; arm(); }    // boarddetector.h:134
    // setParams (boarddetector.h): the configuration and camera detectBatch uses.  Arms the board on the marker detector's
    // context, so its batches run BoardDetector::detect on every frame.
    void setParams(const BoardConfiguration& conf, const CameraParameters& cp, float markerSizeMeters = -1) {
        conf_ = conf;
        cp_ = cp;
        size_ = markerSizeMeters;
        armed_ = true;
        arm();
    }
    // BoardDetector::detect(const cv::Mat&) (boarddetector.cpp:66-78) over n_frames images of first's geometry, frame_stride
    // bytes apart (0: packed): markers without camera, then the board of setParams on each frame, in one batch.
    // Returns the board of every frame; markers[f] receives frame f's markers, prob[f] (when given) the detect return value.
    std::vector<Board> detectBatch(const ImageView& first, int n_frames, size_t frame_stride, std::vector<std::vector<Marker>>& markers,
                                   std::vector<float>* prob = nullptr) {
        if (!armed_) throw Exception(AB_E_STATE, "BoardDetector::detectBatch: setParams first");
        md_.detectBatch(first, n_frames, frame_stride, markers);
        size_t cap = 1;
        for (const auto& m : markers) cap = std::max(cap, m.size());
        std::vector<ab_board> res(n_frames);
        std::vector<ab_marker> bm((size_t)n_frames * cap);
        int rc = ab_get_boards(md_.handle(), n_frames, res.data(), bm.data(), (int)cap);
        if (rc != AB_OK) throw Exception(rc, ab_last_error(md_.handle()));
        std::vector<Board> out(n_frames);
        if (prob) prob->assign(n_frames, 0.f);
        for (int f = 0; f < n_frames; f++) {
            fill(out[f], res[f], bm.data() + (size_t)f * cap, conf_);
            if (prob) (*prob)[f] = res[f].prob;
        }
        return out;
    }
    float get_repj_err_thres() const { return repj_err_thres_; }
    // The calibration views of detectBatch's boards (the reference's utils/aruco_calibration): boards with at least min_markers
    // markers, stacked as the board stage stacks them -- per marker its 4 configuration corners (times metres per pixel for a
    // PIX configuration with a marker size) and its 4 image corners.
    void stackViews(const std::vector<Board>& boards, std::vector<std::vector<std::array<float, 3>>>& objPoints,
                    std::vector<std::vector<Point2f>>& imgPoints, size_t min_markers = 4) const {
        if (!armed_) throw Exception(AB_E_STATE, "BoardDetector::stackViews: setParams first");
        double mpp = 1.0;
        if (conf_.mInfoType == BoardConfiguration::PIX && size_ > 0) {
            const float* c = conf_.objPoints[0].data();
            mpp = (double)size_ / std::sqrt((double)(c[0] - c[3]) * (c[0] - c[3]) + (double)(c[1] - c[4]) * (c[1] - c[4]) +
                                            (double)(c[2] - c[5]) * (c[2] - c[5]));
        }
        objPoints.clear();
        imgPoints.clear();
        for (const Board& b : boards) {
            std::vector<std::array<float, 3>> o;
            std::vector<Point2f> im;
            for (const Marker& m : b) {
                const int k = conf_.getIndexOfMarkerId(m.id);
                if (k < 0 || m.size() != 4) continue;
                for (int p = 0; p < 4; p++) {
                    o.push_back({(float)((double)conf_.objPoints[k][3 * p] * mpp), (float)((double)conf_.objPoints[k][3 * p + 1] * mpp),
                                 (float)((double)conf_.objPoints[k][3 * p + 2] * mpp)});
                    im.push_back(m[p]);
                }
            }
            if (o.size() < 4 * min_markers) continue;
            objPoints.push_back(o);
            imgPoints.push_back(im);
        }
    }
    // The stereo calibration views of two cameras' detectBatch boards of the same frames (boards1[f] and boards2[f]): per frame
    // the configuration markers matched by both cameras, in camera 1's detection order (each id once), stacked as stackViews
    // stacks them; frames with fewer than min_markers common markers are skipped.
    void stackStereoViews(const std::vector<Board>& boards1, const std::vector<Board>& boards2,
                          std::vector<std::vector<std::array<float, 3>>>& objPoints, std::vector<std::vector<Point2f>>& imgPoints1,
                          std::vector<std::vector<Point2f>>& imgPoints2, size_t min_markers = 4) const {
        if (boards1.size() != boards2.size()) throw Exception(AB_E_INVALID, "BoardDetector::stackStereoViews: the cameras' frame counts differ");
        objPoints.clear();
        imgPoints1.clear();
        imgPoints2.clear();
        for (size_t f = 0; f < boards1.size(); f++) {
            Board b1, b2;
            for (const Marker& m : boards1[f]) {
                if (conf_.getIndexOfMarkerId(m.id) < 0 || m.size() != 4) continue;
                bool seen = false;
                for (const Marker& x : b1) seen = seen || x.id == m.id;
                const Marker* other = nullptr;
                for (const Marker& x : boards2[f])
                    if (!other && x.id == m.id && x.size() == 4) other = &x;
                if (seen || !other) continue;
                b1.push_back(m);
                b2.push_back(*other);
            }
            std::vector<std::vector<std::array<float, 3>>> o;
            std::vector<std::vector<Point2f>> i1, i2;
            stackViews({b1}, o, i1, min_markers);
            if (o.empty()) continue;
            stackViews({b2}, o, i2, min_markers);
            objPoints.push_back(o[0]);
            imgPoints1.push_back(i1[0]);
            imgPoints2.push_back(i2[0]);
        }
    }
    // detect (boarddetector.cpp:90-204): returns the fraction of the board's markers that were found
    float detect(const std::vector<Marker>& detectedMarkers, const BoardConfiguration& conf, Board& out, const CameraParameters& cp,
                 float markerSizeMeters = -1) {
        std::vector<ab_marker> in(detectedMarkers.size()), matched(detectedMarkers.size());
        for (size_t i = 0; i < detectedMarkers.size(); i++) {
            const Marker& m = detectedMarkers[i];
            ab_marker a;
            std::memset(&a, 0, sizeof(a));
            a.id = m.id;
            for (size_t k = 0; k < 4 && k < m.size(); k++) {
                a.corners[2 * k] = m[k].x;
                a.corners[2 * k + 1] = m[k].y;
            }
            a.ssize = m.ssize;
            a.has_pose = m.hasPose;
            for (int k = 0; k < 3; k++) {
                a.rvec[k] = m.Rvec[k];
                a.tvec[k] = m.Tvec[k];
            }
            in[i] = a;
        }
        const ab_board_config cfg = conf.abi();
        ab_board res;
        const bool cam = cp.isValid();
        int rc = ab_detect_board(md_.handle(), in.data(), (int)in.size(), &cfg, cam ? cp.CameraMatrix : nullptr, cam ? cp.Distorsion : nullptr,
                                 markerSizeMeters, repj_err_thres_, y_perp_ ? 1 : 0, matched.data(), &res);
        if (rc != AB_OK) throw Exception(rc, ab_last_error(md_.handle()));
        fill(out, res, matched.data(), conf);
        return res.prob;
    }

private:
    MarkerDetector& md_;
    bool y_perp_;
    float repj_err_thres_ = -1;  // boarddetector.cpp:38-41
    BoardConfiguration conf_;
    CameraParameters cp_;
    float size_ = -1;
    bool armed_ = false;
    void arm() {
        if (!armed_) return;
        const ab_board_config cfg = conf_.abi();
        const bool cam = cp_.isValid();
        int rc = ab_set_board(md_.handle(), &cfg, cam ? cp_.CameraMatrix : nullptr, cam ? cp_.Distorsion : nullptr, size_, repj_err_thres_,
                              y_perp_ ? 1 : 0);
        if (rc != AB_OK) throw Exception(rc, ab_last_error(md_.handle()));
    }
    static void fill(Board& out, const ab_board& res, const ab_marker* matched, const BoardConfiguration& conf) {
        out.clear();
        out.conf = conf;
        out.markerSizeMeters = res.ssize;
        out.hasPose = res.has_pose != 0;
        for (int k = 0; k < 3; k++) {
            out.Rvec[k] = res.rvec[k];
            out.Tvec[k] = res.tvec[k];
        }
        for (int i = 0; i < res.n_markers; i++) out.push_back(MarkerDetector::convert(matched[i]));
    }
};

// cv::calibrateCamera(objectPoints, imagePoints, imageSize, K, D, rvecs, tvecs) with flags 0 on the device (ab_calibrate_cameras):
// object points on the z = 0 plane.  Returns the rms reprojection error; `out` receives K and D (f32, as CameraParameters holds
// them) and the image size; rvecs / tvecs (optional) the f64 pose of each view.  Throws on degenerate input.
inline double calibrateCamera(MarkerDetector& md, const std::vector<std::vector<std::array<float, 3>>>& objPoints,
                              const std::vector<std::vector<Point2f>>& imgPoints, Size imageSize, CameraParameters& out,
                              std::vector<std::array<double, 3>>* rvecs = nullptr, std::vector<std::array<double, 3>>* tvecs = nullptr) {
    if (objPoints.size() != imgPoints.size()) throw Exception(AB_E_INVALID, "calibrateCamera: objPoints and imgPoints differ in size");
    std::vector<int32_t> n;
    std::vector<float> obj, img;
    for (size_t v = 0; v < objPoints.size(); v++) {
        if (objPoints[v].size() != imgPoints[v].size()) throw Exception(AB_E_INVALID, "calibrateCamera: a view's point counts differ");
        n.push_back((int32_t)objPoints[v].size());
        for (size_t i = 0; i < objPoints[v].size(); i++) {
            obj.insert(obj.end(), objPoints[v][i].begin(), objPoints[v][i].end());
            img.push_back(imgPoints[v][i].x);
            img.push_back(imgPoints[v][i].y);
        }
    }
    const ab_calib_camera cam = {imageSize.width, imageSize.height, (int32_t)n.size(), n.data(), obj.data(), img.data()};
    ab_calib_result res;
    std::vector<double> r(3 * std::max<size_t>(n.size(), 1)), t(r.size());
    int rc = ab_calibrate_cameras(md.handle(), 1, &cam, &res, r.data(), t.data());
    if (rc != AB_OK) throw Exception(rc, ab_last_error(md.handle()));
    if (res.status != AB_OK) throw Exception(res.status, "calibrateCamera: degenerate input (non-planar object points, fewer than 2 views, "
                                                         "a view with fewer than 4 points, or views that do not determine the focal lengths)");
    float K[9], D[5];
    for (int i = 0; i < 9; i++) K[i] = (float)res.K[i];
    for (int i = 0; i < 5; i++) D[i] = (float)res.D[i];
    out.setParams(K, D, imageSize);
    for (size_t v = 0; v < n.size(); v++) {
        if (rvecs) rvecs->push_back({r[3 * v], r[3 * v + 1], r[3 * v + 2]});
        if (tvecs) tvecs->push_back({t[3 * v], t[3 * v + 1], t[3 * v + 2]});
    }
    return res.rms;
}

// The result of stereoCalibrate: camera 1 -> camera 2 (x2 = R x1 + T), E = [T]x R, F = K2^-T E K1^-1 (F[8] = 1), row-major.
struct StereoParameters {
    double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, T[3] = {0, 0, 0}, E[9] = {0}, F[9] = {0};
    double rms = -1;
};

// cv::stereoCalibrate(objectPoints, imagePoints1, imagePoints2, K1, D1, K2, D2, size, R, T, E, F, CALIB_FIX_INTRINSIC) on the
// device (ab_stereo_calibrate): the cameras' f32 K and D are widened to f64 and kept fixed; object points on the z = 0
// plane; TermCriteria(COUNT + EPS, max_iter, eps).  Returns the rms reprojection error over both cameras.  Throws on
// degenerate input.
inline double stereoCalibrate(MarkerDetector& md, const std::vector<std::vector<std::array<float, 3>>>& objPoints,
                              const std::vector<std::vector<Point2f>>& imgPoints1, const std::vector<std::vector<Point2f>>& imgPoints2,
                              const CameraParameters& cam1, const CameraParameters& cam2, StereoParameters& out, int max_iter = 30,
                              double eps = 1e-6) {
    if (objPoints.size() != imgPoints1.size() || objPoints.size() != imgPoints2.size())
        throw Exception(AB_E_INVALID, "stereoCalibrate: objPoints, imgPoints1 and imgPoints2 differ in size");
    if (!cam1.isValid() || !cam2.isValid()) throw Exception(AB_E_INVALID, "stereoCalibrate: both cameras need valid parameters");
    std::vector<int32_t> n;
    std::vector<float> obj, i1, i2;
    for (size_t v = 0; v < objPoints.size(); v++) {
        if (objPoints[v].size() != imgPoints1[v].size() || objPoints[v].size() != imgPoints2[v].size())
            throw Exception(AB_E_INVALID, "stereoCalibrate: a view's point counts differ");
        n.push_back((int32_t)objPoints[v].size());
        for (size_t i = 0; i < objPoints[v].size(); i++) {
            obj.insert(obj.end(), objPoints[v][i].begin(), objPoints[v][i].end());
            i1.push_back(imgPoints1[v][i].x);
            i1.push_back(imgPoints1[v][i].y);
            i2.push_back(imgPoints2[v][i].x);
            i2.push_back(imgPoints2[v][i].y);
        }
    }
    ab_stereo_pair pr;
    std::memset(&pr, 0, sizeof(pr));
    pr.width = cam1.CamSize.width;
    pr.height = cam1.CamSize.height;
    pr.n_views = (int32_t)n.size();
    pr.n_points = n.data();
    pr.obj = obj.data();
    pr.img1 = i1.data();
    pr.img2 = i2.data();
    for (int i = 0; i < 9; i++) {
        pr.K1[i] = cam1.CameraMatrix[i];
        pr.K2[i] = cam2.CameraMatrix[i];
    }
    for (int i = 0; i < 5; i++) {
        pr.D1[i] = cam1.Distorsion[i];
        pr.D2[i] = cam2.Distorsion[i];
    }
    ab_stereo_result res;
    int rc = ab_stereo_calibrate(md.handle(), 1, &pr, max_iter, eps, &res, nullptr, nullptr, nullptr);
    if (rc != AB_OK) throw Exception(rc, ab_last_error(md.handle()));
    if (res.status != AB_OK) throw Exception(res.status, "stereoCalibrate: degenerate input (no view, a view with fewer than 4 or collinear "
                                                         "points, object points off the z = 0 plane, or a pose that is not determined)");
    for (int i = 0; i < 9; i++) {
        out.R[i] = res.R[i];
        out.E[i] = res.E[i];
        out.F[i] = res.F[i];
    }
    for (int i = 0; i < 3; i++) out.T[i] = res.T[i];
    out.rms = res.rms;
    return res.rms;
}

// R, T, E, F as cv::FileStorage writes CV_64F matrices (!!opencv-matrix, dt: d), every value with %.17g so that it reads back
// exactly; rms as a plain value.
inline void saveStereoParameters(const StereoParameters& sp, const std::string& path) {
    std::ostringstream o;
    auto mat = [&](const char* name, const double* v, int rows, int cols) {
        o << name << ": !!opencv-matrix\n   rows: " << rows << "\n   cols: " << cols << "\n   dt: d\n   data: [ ";
        for (int i = 0; i < rows * cols; i++) {
            char b[40];
            std::snprintf(b, sizeof b, "%.17g", v[i]);
            o << b << (i + 1 < rows * cols ? ", " : " ]\n");
        }
    };
    o << "%YAML:1.0\n---\n";
    mat("R", sp.R, 3, 3);
    mat("T", sp.T, 3, 1);
    mat("E", sp.E, 3, 3);
    mat("F", sp.F, 3, 3);
    char b[40];
    std::snprintf(b, sizeof b, "%.17g", sp.rms);
    o << "rms: " << b << "\n";
    yaml::write_text(path, o.str());
}

// ---- HRM dictionary (src/highlyreliablemarkers.h:95-112) -------------------------------------------------------------
struct Dictionary {
    int markersize = 0;  // n
    int tau0 = 0;
    std::vector<std::string> codes;  // n*n characters '0'/'1', row-major (MarkerCode::toString / fromString)
    size_t size() const { return codes.size(); }
    void fromFile(const std::string& path) {  // Dictionary::fromFile, serialization.cpp:133-151
        const yaml::Node fs = yaml::load(path);
        const int nmarkers = fs["nmarkers"].as_int();
        markersize = fs["markersize"].as_int();
        tau0 = fs["tau0"].as_int();
        codes.clear();
        for (int i = 0; i < nmarkers; i++) {
            std::string s = fs["marker_" + std::to_string(i)].as_string();
            if ((int)s.size() != markersize * markersize) throw Exception(AB_E_INVALID, "dictionary marker " + std::to_string(i) + " has the wrong length");
            codes.push_back(s);
        }
    }
    void toFile(const std::string& path) const {  // serialization.cpp:121-131
        std::ostringstream o;
        o << "%YAML:1.0\n---\nnmarkers: " << codes.size() << "\nmarkersize: " << markersize << "\ntau0: " << tau0 << "\n";
        for (size_t i = 0; i < codes.size(); i++) o << "marker_" << i << ": \"" << codes[i] << "\"\n";
        yaml::write_text(path, o.str());
    }
    // HighlyReliableMarkers::loadDictionary (src/highlyreliablemarkers.cpp:312-328) on a detector
    void loadInto(MarkerDetector& md, float correctionDistanceRate = 1.f) const {
        std::vector<uint8_t> bits;
        for (const auto& c : codes)
            for (char ch : c) bits.push_back(ch == '1');
        md.useHighlyReliableMarkers(markersize, (int)codes.size(), bits.data(), tau0, correctionDistanceRate);
    }
};

}  // namespace aruco
