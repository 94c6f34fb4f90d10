// C++ façade of the event front end and the spline calibration over the C ABI, mirroring the reference's classes
// (names, argument meaning, error behaviour) without its Eigen / OpenCV / Ceres dependencies:
//
//   opengv2::EventContainer        EV/include/opengv2/event/EventContainer.hpp:15-30   (time-ordered event store)
//   opengv2::CirclePatternParameters  ECC/include/.../parameters.hpp:12-27
//   opengv2::CirclesEventFrame     ECC/include/.../CirclesEventFrame.hpp:21-95: Params, ctor(container, duration, pattern,
//                                  params), bool extractFeatures(), eventsNum(), findCenter(p), fitCircle(...)
//   opengv2::EventCalibSpline      ECC/include/.../EventCalibSpline.hpp:17-357: optimize(), intrinsics OFFSET_* enum
//
// The batched entry point the reference lacks — many windows per launch — is ecb::FrontEnd below; the per-frame class
// is kept so that the reference's MultiProcess loop (ECC/test/eventCameraCalib.cpp:34-97) compiles unchanged against it.
//   opengv2::EventStream::txt2bin  EV/src/EventStream.cpp:25-67 (text -> 25-byte records)
//   EventCalibSpline::evaluate / time2splineIdx / saveKeyFrameTrajectoryTUM   ECC/.../EventCalibSpline.hpp:295-330,
//                                  CORE/system/src/SystemBase.cpp:122-150 (TUM lines `t tx ty tz qx qy qz qw`, fixed, precision 10)
// extractFeatures() orders the candidates with include/ecb/circles_grid.hpp (the canonical result of the reference's
// findCirclesGrid call, CirclesEventFrame.cpp:332-356) and reports success when the grid is found.
#ifndef ECB_EVENT_CALIB_HPP
#define ECB_EVENT_CALIB_HPP

#include <algorithm>
#include <array>
#include <cmath>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <limits>
#include <map>
#include <cstdint>
#include <cstring>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_set>
#include <utility>
#include <vector>

#include "../eventcalib_b200.h"
#include "../../eventcalib_b200/csrc/ecb_so3.h"  // plain host/device header: the SO(3) spline of the useSO3 variant
#include "calib_init.hpp"
#include "circles_grid.hpp"
#include "compat/opengv2_lite.hpp"
#include "dbscan.h"
#include "image_lite.hpp"

namespace ecb {
// Constant intrinsics of the spline stage (ecb_cost_set_constant_intrinsics) from comma- or space-separated names of
// fx fy cx cy k1 k2 k3 k4 k5 (k1 .. k5: the inverse radial polynomial, not OpenCV's coefficients).  Returns the mask (0 for no
// names), or -1 with the first unknown token in *unknown.
inline int constantIntrinsicsMask(const std::string &names, std::string *unknown = nullptr) {
    static const char *const kNames[9] = {"fx", "fy", "cx", "cy", "k1", "k2", "k3", "k4", "k5"};
    std::string list = names;
    std::replace(list.begin(), list.end(), ',', ' ');
    std::istringstream is(list);
    std::string tok;
    int mask = 0;
    while (is >> tok) {
        int i = 0;
        while (i < 9 && tok != kNames[i]) ++i;
        if (i == 9) {
            if (unknown) *unknown = tok;
            return -1;
        }
        mask |= 1 << i;
    }
    return mask;
}
// Outlier policy over the residual statistics per key frame (ECB_RESIDUALS_BY_KEYFRAME, all shards combined): s = the lower median
// (element floor((n - 1) / 2) after sorting) of the RMS sqrt(sum_sq / count) of the n key frames with count > 0; a key frame whose
// RMS > k s is dropped, and a record is removed when |r| > k s.  The median over key frames keeps a minority of mislabelled
// frames from inflating the scale, which a global RMS would not.  Empty key frames take no part and are never dropped.  Returns s
// (0 without records); *threshold = k s, *drop = one flag per key frame (the arguments of ecb_cost_reject).
inline double outlierRejection(const std::vector<ecb_residual_group> &byKeyframe, double k, double *threshold,
                               std::vector<uint8_t> *drop) {
    std::vector<double> rms(byKeyframe.size(), 0.0), sorted;
    for (size_t j = 0; j < byKeyframe.size(); ++j)
        if (byKeyframe[j].count > 0) {
            rms[j] = std::sqrt(byKeyframe[j].sum_sq / (double) byKeyframe[j].count);
            sorted.push_back(rms[j]);
        }
    std::sort(sorted.begin(), sorted.end());
    const double s = sorted.empty() ? 0.0 : sorted[(sorted.size() - 1) / 2];
    const double t = k * s;
    if (threshold) *threshold = t;
    if (drop) {
        drop->assign(byKeyframe.size(), 0);
        for (size_t j = 0; j < byKeyframe.size(); ++j) (*drop)[j] = byKeyframe[j].count > 0 && rms[j] > t ? 1 : 0;
    }
    return s;
}
}  // namespace ecb

namespace opengv2 {

struct Vec2 {
    double v[2];
    double &operator[](int i) { return v[i]; }
    const double &operator[](int i) const { return v[i]; }
};

// the reference's 25-byte record (Event.hpp:36-47), packed
#pragma pack(push, 1)
struct EventRecord {
    double t, x, y;
    uint8_t polarity;
};
#pragma pack(pop)
static_assert(sizeof(EventRecord) == 25, "reference record is 25 bytes");

struct CirclePatternParameters {
    typedef std::shared_ptr<CirclePatternParameters> Ptr;
    bool isAsymmetric = true;
    int rows = 9, cols = 4;
    double circleRadius = 1.75, squareSize = 5.5;
};

// EventStream::txt2bin (EV/src/EventStream.cpp:25-67): "timeStamp x y polarity" lines -> packed records next to the text
// file (same name, .bin).  timeBase / endTime: LLONG_MIN = "first stamp" / "no limit" like the reference's defaults.
struct EventStream {
    static long long txt2bin(const std::string &txtFilePath, double timeMagnitude,
                             long long timeBase_in = std::numeric_limits<long long>::min(),
                             long long endTime_in = std::numeric_limits<long long>::min()) {
        std::ifstream is(txtFilePath, std::ifstream::in);
        if (!is.is_open()) throw std::invalid_argument("No such file: " + txtFilePath);
        const auto lastIndex = txtFilePath.find_last_of('.');
        std::ofstream os(txtFilePath.substr(0, lastIndex) + ".bin", std::ofstream::binary | std::ofstream::out | std::ofstream::trunc);
        long long counter = 0, timeStamp = 0, timeBase = timeBase_in;
        double x = 0, y = 0;
        bool polarity = false;
        while (is.good()) {
            is >> timeStamp >> x >> y >> polarity;
            if (counter == 0 && timeBase_in == std::numeric_limits<long long>::min()) timeBase = timeStamp;
            if (endTime_in != std::numeric_limits<long long>::min() && timeStamp > endTime_in) break;
            const double t = ((timeStamp - timeBase) * timeMagnitude);  // convert to second
            if (t < 0) continue;
            os.write((const char *) &t, sizeof t);
            os.write((const char *) &x, sizeof x);
            os.write((const char *) &y, sizeof y);
            os.write((const char *) &polarity, sizeof polarity);
            counter++;
        }
        std::cout << counter << " data processed." << std::endl;
        std::cout.precision(30);
        std::cout << "TimeBase :" << timeBase << std::endl;
        std::cout.precision(15);
        std::cout << "Last data is :" << timeStamp << " " << x << " " << y << " " << polarity << std::endl;
        std::cout << "Duration :" << ((timeStamp - timeBase) * timeMagnitude) << std::endl;
        return counter;
    }
};

// cubic B-spline span / basis on the host (BsplineReal::findSpan :208-231, dersBasisFuns :107-145, derivative 0)
inline int bspline_find_span(const std::vector<double> &kn, double u) {
    const int degree = 3, n = (int) kn.size() - 2 - degree;
    if (u == kn[(size_t) n + 1]) return n;
    int low = degree, high = n + 1, mid = (low + high) / 2;
    while (u < kn[(size_t) mid] || u >= kn[(size_t) mid + 1]) {
        if (u < kn[(size_t) mid]) high = mid; else low = mid;
        mid = (low + high) / 2;
    }
    return mid;
}
inline void bspline_basis(const std::vector<double> &kn, int span, double u, double N[4]) {
    double ndu[4][4] = {{0}}, left[4] = {0}, right[4] = {0};
    ndu[0][0] = 1.0;
    for (int j = 1; j <= 3; ++j) {
        left[j] = u - kn[(size_t) (span + 1 - j)];
        right[j] = kn[(size_t) (span + j)] - u;
        double saved = 0.0;
        for (int r = 0; r < j; ++r) {
            ndu[j][r] = right[r + 1] + left[j - r];
            const double temp = ndu[r][j - 1] / ndu[j][r];
            ndu[r][j] = saved + right[r + 1] * temp;
            saved = left[j - r] * temp;
        }
        ndu[j][j] = saved;
    }
    for (int j = 0; j <= 3; ++j) N[j] = ndu[j][3];
}

// Time-ordered events resident on the device (replaces std::multimap<double, Event_loc_pol>, EventContainer.hpp:26)
struct EventContainer {
    typedef std::shared_ptr<EventContainer> Ptr;
    ecb_ctx *ctx = nullptr;
    int width = 0, height = 0;
    int64_t size = 0;
    double firstTime = 0, lastTime = 0;

    EventContainer(int device, int w, int h) : width(w), height(h) {
        if (ecb_ctx_create(device, nullptr, &ctx) != ECB_OK) throw std::runtime_error("ecb: no usable CUDA device");
        if (ecb_set_sensor(ctx, w, h) != ECB_OK) throw std::invalid_argument(ecb_last_error(ctx));
    }
    ~EventContainer() { ecb_ctx_destroy(ctx); }
    EventContainer(const EventContainer &) = delete;
    EventContainer &operator=(const EventContainer &) = delete;

    // records: time-sorted reference records (the caller applies StartTime / EndTime like eventCameraCalib.cpp:154-163)
    void load(const EventRecord *records, int64_t n) {
        if (ecb_load_events_host(ctx, records, n) != ECB_OK) throw std::invalid_argument(ecb_last_error(ctx));
        size = n;
        if (n > 0) {
            firstTime = records[0].t;
            lastTime = records[n - 1].t;
        }
    }
};

struct CalibCircleLite {
    Vec2 center;
    double radius;
    int pCluster, nCluster;
};

// ---- batched front end: all windows of a piece in one launch ----
class FrontEnd {
public:
    struct Params {  // CirclesEventFrame::Params (CirclesEventFrame.cpp:35-48)
        double dbscan_eps = 4;
        int dbscan_startMinSample = 2;
        int clusterMinSample = 5;
        int knn_num = 3;
        bool fitCircle = false;
    };
    FrontEnd(EventContainer::Ptr c, CirclePatternParameters::Ptr pattern, Params p) : c_(c), pattern_(pattern), p_(p) {
        // circleRadiusThreshold_ (CirclesEventFrame.cpp:16-33)
        const double W = c->width, H = c->height;
        const double c2 = pattern->isAsymmetric ? 2.0 * pattern->cols : (double) pattern->cols;
        rthr_ = std::min(std::max(W, H) / std::max((double) pattern->rows, c2), std::min(W, H) / std::min((double) pattern->rows, c2)) /
                pattern->squareSize * pattern->circleRadius * 1.5;
    }
    // windows: closed intervals [first, second] (EventFrame.cpp:14-15)
    void run(const std::vector<std::pair<double, double>> &windows) {
        ecb_frontend_params fp;
        std::memset(&fp, 0, sizeof fp);
        fp.dbscan_eps = p_.dbscan_eps;
        fp.dbscan_min_pts = (uint32_t) p_.dbscan_startMinSample;
        fp.cluster_min = (uint32_t) p_.clusterMinSample;
        fp.knn_num = p_.knn_num;
        fp.fit_circle = p_.fitCircle ? 1 : 0;
        fp.radius_threshold = rthr_;
        fp.rows_cols = (uint32_t) (pattern_->rows * pattern_->cols);
        fp.order_mode = 1;   // pid order = iteration order of EventFrame's unordered_sets (EventFrame.cpp:12-35)
        fp.median_mode = 1;  // cluster centre = std::nth_element's pick over the BFS-ordered members (CirclesEventFrame.cpp:137-147)
        std::vector<double> w(2 * windows.size());
        for (size_t i = 0; i < windows.size(); ++i) {
            w[2 * i] = windows[i].first;
            w[2 * i + 1] = windows[i].second;
        }
        if (ecb_frontend_run(c_->ctx, w.data(), (int) windows.size(), &fp) != ECB_OK)
            throw std::runtime_error(ecb_last_error(c_->ctx));
        pts_valid_[0] = pts_valid_[1] = false;
        summary_.resize(windows.size());
        stride_ = 1;
        if (!windows.empty()) {
            if (ecb_frontend_summary(c_->ctx, summary_.data(), (int) windows.size()) != ECB_OK)
                throw std::runtime_error(ecb_last_error(c_->ctx));
            // max_clusters = 0: the kept-cluster tables grow with the data, so a window is never truncated
            // (CirclesEventFrame.cpp:89-312 has no cap); anything else the kernels flag is an error, not a shorter list
            for (const auto &s : summary_) {
                if (s.status & (ECB_PB_CLUSTER_CAP | ECB_PB_RANGE))
                    throw std::runtime_error("front end: window result incomplete (status bits " + std::to_string(s.status) + ")");
                stride_ = std::max(stride_, (int) s.n_candidates);
            }
        }
        cand_.assign(windows.size() * (size_t) stride_ * 5, 0.0);
        if (!windows.empty() && ecb_frontend_candidates(c_->ctx, cand_.data(), stride_) != ECB_OK)
            throw std::runtime_error(ecb_last_error(c_->ctx));
    }
    const ecb_window_summary &summary(size_t w) const { return summary_[w]; }
    int eventsNum(size_t w) const { return summary_[w].n_points[0] + summary_[w].n_points[1]; }
    std::vector<CalibCircleLite> candidates(size_t w) const {
        std::vector<CalibCircleLite> out;
        for (int k = 0; k < summary_[w].n_candidates && k < stride_; ++k) {
            const double *c = &cand_[(w * (size_t) stride_ + k) * 5];
            out.push_back(CalibCircleLite{{{c[2], c[3]}}, c[4], (int) c[0], (int) c[1]});
        }
        return out;
    }
    double circleRadiusThreshold() const { return rthr_; }
    ecb_ctx *context() const { return c_->ctx; }
    int width() const { return c_->width; }
    int height() const { return c_->height; }
    // positiveEvents_ / negativeEvents_ of window w (pol 1 / 0) in pid order with their raw DBSCAN labels (-1 = Noise)
    void windowPoints(size_t w, int pol, std::vector<Vec2> &xy, std::vector<int32_t> &labels) {
        if (!pts_valid_[pol]) {
            const int64_t n = ecb_frontend_total_points(c_->ctx, pol);
            pts_xy_[pol].assign((size_t) std::max<int64_t>(n, 1) * 2, 0.0);
            pts_lab_[pol].assign((size_t) std::max<int64_t>(n, 1), -1);
            if (ecb_frontend_points(c_->ctx, pol, pts_xy_[pol].data(), pts_lab_[pol].data()) != ECB_OK)
                throw std::runtime_error(ecb_last_error(c_->ctx));
            pts_valid_[pol] = true;
        }
        const size_t off = (size_t) summary_[w].point_offset[pol], n = (size_t) summary_[w].n_points[pol];
        xy.resize(n);
        labels.assign(pts_lab_[pol].begin() + off, pts_lab_[pol].begin() + off + n);
        for (size_t i = 0; i < n; ++i) xy[i] = Vec2{{pts_xy_[pol][2 * (off + i)], pts_xy_[pol][2 * (off + i) + 1]}};
    }
    // clusters that pass clusterMinSample (CirclesEventFrame.cpp:89-117), in kept order: raw cluster id, size, median pid
    void keptClusters(size_t w, int pol, std::vector<int32_t> &raw_id, std::vector<int32_t> &size, std::vector<int32_t> &median_pid) {
        const int cap = std::max(1, (int) summary_[w].n_kept[pol]);
        raw_id.assign((size_t) cap, 0), size.assign((size_t) cap, 0), median_pid.assign((size_t) cap, 0);
        const int n = ecb_frontend_clusters(c_->ctx, (int) w, pol, raw_id.data(), size.data(), median_pid.data(), cap);
        if (n < 0) throw std::runtime_error(ecb_last_error(c_->ctx));
        raw_id.resize((size_t) n), size.resize((size_t) n), median_pid.resize((size_t) n);
    }
    // rectifyFeatures (CirclesEventFrame.cpp:417-609) for windows of the last run, batched: image_points = 5 projected points
    // (landmark + four quadrant points, :431-456) per frame and circle; out[frame][circle] = cx, cy, r (r < 0: deleted)
    void rectify(const std::vector<int32_t> &window_index, int n_circles, const std::vector<double> &image_points, double inlier,
                 int rows, int cols, bool asymmetric, std::vector<double> &out, std::vector<int32_t> &verdict) {
        out.assign(window_index.size() * (size_t) n_circles * 3, 0.0);
        verdict.assign(window_index.size(), 0);
        if (window_index.empty()) return;
        if (ecb_frontend_rectify(c_->ctx, window_index.data(), (int) window_index.size(), n_circles, image_points.data(), inlier, rows,
                                 cols, asymmetric ? 1 : 0, out.data(), verdict.data()) != ECB_OK)
            throw std::runtime_error(ecb_last_error(c_->ctx));
    }

private:
    int stride_ = 1;  // candidate slots per window of the last run = its largest candidate count
    EventContainer::Ptr c_;
    CirclePatternParameters::Ptr pattern_;
    Params p_;
    double rthr_;
    std::vector<ecb_window_summary> summary_;
    std::vector<double> cand_;
    std::vector<double> pts_xy_[2];
    std::vector<int32_t> pts_lab_[2];
    bool pts_valid_[2] = {false, false};
};

// The reference's debug rendering of a frame (CirclesEventFrame.cpp:74-126,150-157,314-318,623-627): kept clusters coloured
// by their index (20 * k -> B = c / 256, G = c % 256, R = 200 for positive / 100 for negative clusters), white radius-2 circles
// at the cluster medians, green candidate circles, and — after rectifyFeatures — white circles at the rectified features.
// eventImage (positive events red, negative green) and clusterImage (the clusters alone) are the public debug members of
// CirclesEventFrame.hpp:69.  FE: FrontEnd or ShardedFrontEnd.
template <class FE>
inline ecb::Image8UC3 renderFrameImage(FE &fe, size_t w, const std::vector<std::array<double, 3>> *rectified = nullptr,
                                       ecb::Image8UC3 *eventImage = nullptr, ecb::Image8UC3 *clusterImage = nullptr) {
    ecb::Image8UC3 img(fe.height(), fe.width());
    std::vector<Vec2> xy[2];
    std::vector<int32_t> lab[2], raw[2], size[2], med[2];
    for (int pol = 0; pol < 2; ++pol) {
        fe.windowPoints(w, pol, xy[pol], lab[pol]);
        fe.keptClusters(w, pol, raw[pol], size[pol], med[pol]);
    }
    if (eventImage) {
        *eventImage = ecb::Image8UC3(fe.height(), fe.width());
        for (const Vec2 &p : xy[1]) eventImage->set((int) p[0], (int) p[1], 0, 0, 255);
        for (const Vec2 &p : xy[0]) eventImage->set((int) p[0], (int) p[1], 0, 255, 0);
    }
    for (int pol = 1; pol >= 0; --pol) {  // positive clusters first (:89-102), then negative (:104-117)
        std::map<int32_t, unsigned> kept_of;
        for (size_t k = 0; k < raw[pol].size(); ++k) kept_of[raw[pol][k]] = (unsigned) k;
        for (size_t i = 0; i < xy[pol].size(); ++i) {
            const auto it = kept_of.find(lab[pol][i]);
            if (lab[pol][i] < 0 || it == kept_of.end()) continue;
            const unsigned color = 20 * it->second;
            img.set((int) xy[pol][i][0], (int) xy[pol][i][1], (uint8_t) (color / 256), (uint8_t) (color % 256), pol ? 200 : 100);
        }
    }
    if (clusterImage) *clusterImage = img;
    for (int pol = 1; pol >= 0; --pol)
        for (int32_t m : med[pol])
            if (m >= 0 && (size_t) m < xy[pol].size()) img.circle((int) xy[pol][(size_t) m][0], (int) xy[pol][(size_t) m][1], 2, 255, 255, 255);
    for (const CalibCircleLite &c : fe.candidates(w)) img.circle((int) c.center[0], (int) c.center[1], (int) c.radius, 0, 255, 0);
    if (rectified)
        for (const auto &c : *rectified)
            if (c[2] >= 0) img.circle((int) c[0], (int) c[1], (int) c[2], 255, 255, 255);
    return img;
}

// ---- per-frame class with the reference's interface ----
class CirclesEventFrame {
public:
    typedef FrontEnd::Params Params;
    CirclesEventFrame(EventContainer::Ptr container, const std::pair<double, double> &duration,
                      CirclePatternParameters::Ptr pattern, Params params = Params())
        : fe_(container, pattern, params), duration_(duration), pattern_(pattern) {
        fe_.run({duration_});  // the EventFrame ctor does the window / dedupe / cancel work (EventFrame.cpp:10-36)
    }
    bool extractFeatures() {  // CirclesEventFrame.cpp:61-359
        const ecb_window_summary &s = fe_.summary(0);
        if (s.n_points[0] == 0 || s.n_points[1] == 0) return false;  // :62-64
        if (debugImages) image_ = renderFrameImage(fe_, 0, nullptr, &eventImage, &clusterImage);
        const bool found = orderFeatures(fe_.candidates(0), *pattern_, features_);
        lm_of_feature_.clear();
        for (size_t k = 0; k < features_.size(); ++k) lm_of_feature_.push_back((int) k);  // feature k observes board point k (:340-352)
        return found;
    }
    // DEBUG images like the reference's public members (CirclesEventFrame.hpp:69) and Bodyframe's image(); filled by
    // extractFeatures / rectifyFeatures when debugImages is set (they cost a device -> host copy of the frame's points)
    bool debugImages = false;
    ecb::Image8UC3 eventImage, clusterImage;
    const ecb::Image8UC3 &image() const { return image_; }
    // :320-356: the candidates in pattern order (findCirclesGrid, CALIB_CB_ASYMMETRIC_GRID) -> features_; false when the grid
    // is not found.  Grid ordering: include/ecb/circles_grid.hpp (the canonical RESULT of OpenCV's finder).
    static bool orderFeatures(const std::vector<CalibCircleLite> &cand, const CirclePatternParameters &pattern,
                              std::vector<CalibCircleLite> &features) {
        features.clear();
        // the reference calls findCirclesGrid with CALIB_CB_ASYMMETRIC_GRID whatever Is_Pattern_Asymmetric says (:332-336)
        if ((int) cand.size() < pattern.rows * pattern.cols) return false;
        std::vector<ecb::Pt2> pts;
        for (const auto &c : cand) pts.push_back(ecb::Pt2{(double) (float) c.center[0], (double) (float) c.center[1]});  // cv::Point2f (:322-324)
        std::vector<int> order;
        if (!ecb::find_asymmetric_circles_grid(pts, pattern.rows, pattern.cols, order) &&
            !ecb::find_asymmetric_circles_grid_clustering(pts, pattern.rows, pattern.cols, order))  // the CALIB_CB_CLUSTERING retry (:334-336)
            return false;
        for (int idx : order) features.push_back(cand[(size_t) idx]);
        return true;
    }
    // rectifyFeatures (CirclesEventFrame.cpp:417-609).  The reference projects every feature's landmark and four quadrant
    // points with cv::projectPoints (:431-456) from (outlierIdxs, Rcw, tcw); that projection needs the OpenCV initialisation
    // and stays with the caller, who passes the 5 image points per feature (board order).  Radius search, quadrant band,
    // cluster expansion, refit and the gates run batched on the GPU; deleted features are erased like :585-594.
    bool rectifyFeatures(const std::vector<std::array<Vec2, 5>> &imagePoints) {
        const int n = (int) imagePoints.size();
        std::vector<double> img((size_t) n * 10), out((size_t) n * 3);
        for (int k = 0; k < n; ++k)
            for (int i = 0; i < 5; ++i) {
                img[(size_t) k * 10 + 2 * i] = imagePoints[(size_t) k][(size_t) i][0];
                img[(size_t) k * 10 + 2 * i + 1] = imagePoints[(size_t) k][(size_t) i][1];
            }
        const int32_t w = 0;
        int32_t ok = 0;
        if (ecb_frontend_rectify(fe_.context(), &w, 1, n, img.data(), 3.0, pattern_->rows, pattern_->cols,
                                 pattern_->isAsymmetric ? 1 : 0, out.data(), &ok) != ECB_OK)
            return false;
        std::vector<CalibCircleLite> kept;
        std::vector<int> lm_kept;
        std::vector<std::array<double, 3>> circles;
        for (int k = 0; k < n; ++k) {
            circles.push_back({out[(size_t) k * 3], out[(size_t) k * 3 + 1], out[(size_t) k * 3 + 2]});
            if (out[(size_t) k * 3 + 2] >= 0) {
                kept.push_back(CalibCircleLite{{{out[(size_t) k * 3], out[(size_t) k * 3 + 1]}}, out[(size_t) k * 3 + 2], -1, -1});
                lm_kept.push_back((size_t) k < lm_of_feature_.size() ? lm_of_feature_[(size_t) k] : k);
            }
        }
        features_ = kept;
        lm_of_feature_ = lm_kept;
        if (debugImages && ok) image_ = renderFrameImage(fe_, 0, &circles);  // :623-627
        return ok != 0;
    }
    // ---- the reference's own argument lists (CirclesEventFrame.hpp:43-65) ----
    // The reference reaches the camera through the frame's sensor_ and the board points through each feature's landmark();
    // here both are handed over once.  Landmark k belongs to feature k of the ordered grid (EventCalibIni.cpp:99-113).
    void setSensor(const ecb::CameraModel &camera) { camera_ = camera; }
    void setLandmarks(const std::vector<LandmarkBase::Ptr> &landmarks) { landmarks_ = landmarks; }
    // CirclesEventFrame.cpp:417-456: Rcw / tcw -> rvec / tvec, the landmark and its four quadrant points (cv::Point3f) projected
    // with the camera (cv::projectPoints, cv::Point2f), then the batched GPU part.  outlierIdxs is not read by the reference's
    // implementation either.
    bool rectifyFeatures(const std::unordered_set<int> &outlierIdxs, const Eigen::Ref<const Eigen::Matrix3d> &Rcw,
                         const Eigen::Ref<const Eigen::Vector3d> &tcw) {
        (void) outlierIdxs;
        double R[9], rvec[3], tvec[3] = {tcw[0], tcw[1], tcw[2]};
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) R[3 * r + c] = Rcw(r, c);
        ecb::rodriguesInverse(R, rvec);
        const double skewR = pattern_->circleRadius / std::sqrt(2.0);
        std::vector<std::array<Vec2, 5>> imagePoints;
        for (size_t k = 0; k < features_.size(); ++k) {
            const int li = k < lm_of_feature_.size() ? lm_of_feature_[k] : (int) k;
            if (li < 0 || (size_t) li >= landmarks_.size() || !landmarks_[(size_t) li])
                throw std::logic_error("CirclesEventFrame::rectifyFeatures: setLandmarks() first (one landmark per board point)");
            const Eigen::Vector3d c = landmarks_[(size_t) li]->position();
            const double o5[15] = {(double) (float) c[0], (double) (float) c[1], (double) (float) c[2],
                                   (double) (float) (c[0] + skewR), (double) (float) (c[1] + skewR), (double) (float) c[2],
                                   (double) (float) (c[0] + skewR), (double) (float) (c[1] - skewR), (double) (float) c[2],
                                   (double) (float) (c[0] - skewR), (double) (float) (c[1] - skewR), (double) (float) c[2],
                                   (double) (float) (c[0] - skewR), (double) (float) (c[1] + skewR), (double) (float) c[2]};
            double p5[10];
            ecb::projectPoints(o5, 5, rvec, tvec, camera_, p5);
            std::array<Vec2, 5> ip;
            for (int i = 0; i < 5; ++i) ip[(size_t) i] = Vec2{{(double) (float) p5[2 * i], (double) (float) p5[2 * i + 1]}};
            imagePoints.push_back(ip);
        }
        return rectifyFeatures(imagePoints);
    }
    // CirclesEventFrame.hpp:50-65: the landmark of the nearest feature if the event lies within 5 px of its rim, else nullptr
    LandmarkBase::Ptr findCenter(const Eigen::Vector2d &p) const {
        const int k = findCenter(Vec2{{p[0], p[1]}});
        if (k < 0) return nullptr;
        const int li = (size_t) k < lm_of_feature_.size() ? lm_of_feature_[(size_t) k] : k;
        return li >= 0 && (size_t) li < landmarks_.size() ? landmarks_[(size_t) li] : nullptr;
    }
    int eventsNum() const { return fe_.eventsNum(0); }
    const std::vector<CalibCircleLite> &features() const { return features_; }
    // CirclesEventFrame.hpp:50-65: nearest circle, accepted iff | ||p-c|| - r | < 5 px; returns the feature index or -1
    int findCenter(const Vec2 &p) const {
        int best = -1;
        double bd = 0;
        for (size_t i = 0; i < features_.size(); ++i) {
            const double dx = p[0] - features_[i].center[0], dy = p[1] - features_[i].center[1], d2 = dx * dx + dy * dy;
            if (best < 0 || d2 < bd) {
                best = (int) i;
                bd = d2;
            }
        }
        if (best < 0) return -1;
        return std::abs(std::sqrt(bd) - features_[(size_t) best].radius) < 5 ? best : -1;
    }

private:
    FrontEnd fe_;
    std::pair<double, double> duration_;
    CirclePatternParameters::Ptr pattern_;
    std::vector<CalibCircleLite> features_;
    std::vector<int> lm_of_feature_;  // board point / landmark index of every feature still alive
    std::vector<LandmarkBase::Ptr> landmarks_;
    ecb::CameraModel camera_;
    ecb::Image8UC3 image_;
};

// ---- the tracking gate: TrackingBase::process (core/tracking/src/TrackingBase.cpp:16-46) + EventCalibIni::track
// (event_camera_calib/src/EventCalibIni.cpp:23-97).  The first frame initialises the map; a later frame is accepted when the
// median angle between the directions of its grid rows and those of the neighbouring key frame (lower_bound of its time
// stamp, else the last one), divided by the time between them, stays below 5e-4*pi / MotionTimeStep rad/s.
// Row direction: total-least-squares line through the row's centres (the reference takes the last right singular vector of
// [x y 1]; here the eigenvector of the 3x3 normal matrix, same line).  Host only.
class TrackingGate {
public:
    TrackingGate(int rows, int cols, double motionTimeStep) : rows_(rows), cols_(cols), step_(motionTimeStep) {}
    bool process(double timeStamp, const std::vector<CalibCircleLite> &features) {
        if (keyframes_.empty()) {  // initialization(): addFrame, state = OK
            keyframes_[timeStamp] = features;
            return true;
        }
        auto itr = keyframes_.lower_bound(timeStamp);
        const auto &ref = itr != keyframes_.end() ? *itr : *keyframes_.rbegin();
        const double duration = std::abs(timeStamp - ref.first);
        std::vector<double> theta;
        for (int i = 0; i < rows_; ++i) {
            double r[2], c[2];
            rowDirection(ref.second, i, r);
            rowDirection(features, i, c);
            theta.push_back(std::acos((r[0] * c[0] + r[1] * c[1]) / (std::sqrt(r[0] * r[0] + r[1] * r[1]) * std::sqrt(c[0] * c[0] + c[1] * c[1]))));
        }
        std::nth_element(theta.begin(), theta.begin() + theta.size() / 2, theta.end());
        if (theta[theta.size() / 2] / duration < (5e-4 * M_PI) / step_) {
            keyframes_.emplace(timeStamp, features);  // MapBase::addFrame
            return true;
        }
        return false;
    }
    const std::map<double, std::vector<CalibCircleLite>> &keyframes() const { return keyframes_; }

private:
    // direction (B, -A) of the line A x + B y + C = 0 through row i, pointing from its first to its last centre
    void rowDirection(const std::vector<CalibCircleLite> &f, int i, double d[2]) const {
        double M[3][3] = {{0}};
        for (int j = 0; j < cols_; ++j) {
            const double v[3] = {f[(size_t) (i * cols_ + j)].center[0], f[(size_t) (i * cols_ + j)].center[1], 1.0};
            for (int a = 0; a < 3; ++a)
                for (int b = 0; b < 3; ++b) M[a][b] += v[a] * v[b];
        }
        double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
        for (int sweep = 0; sweep < 60; ++sweep) {  // cyclic Jacobi on the symmetric 3x3
            double off = 0;
            for (int p = 0; p < 3; ++p)
                for (int q = p + 1; q < 3; ++q) off += M[p][q] * M[p][q];
            if (off < 1e-300) break;
            for (int p = 0; p < 3; ++p)
                for (int q = p + 1; q < 3; ++q) {
                    if (M[p][q] == 0) continue;
                    const double th = (M[q][q] - M[p][p]) / (2 * M[p][q]);
                    const double t = (th >= 0 ? 1.0 : -1.0) / (std::abs(th) + std::sqrt(th * th + 1));
                    const double c = 1 / std::sqrt(t * t + 1), s = t * c;
                    for (int k = 0; k < 3; ++k) {
                        const double mkp = M[k][p], mkq = M[k][q];
                        M[k][p] = c * mkp - s * mkq;
                        M[k][q] = s * mkp + c * mkq;
                    }
                    for (int k = 0; k < 3; ++k) {
                        const double mpk = M[p][k], mqk = M[q][k];
                        M[p][k] = c * mpk - s * mqk;
                        M[q][k] = s * mpk + c * mqk;
                    }
                    for (int k = 0; k < 3; ++k) {
                        const double vkp = V[k][p], vkq = V[k][q];
                        V[k][p] = c * vkp - s * vkq;
                        V[k][q] = s * vkp + c * vkq;
                    }
                }
        }
        int m = 0;
        for (int k = 1; k < 3; ++k)
            if (M[k][k] < M[m][m]) m = k;
        d[0] = V[1][m];
        d[1] = -V[0][m];
        const double ex = f[(size_t) (i * cols_ + cols_ - 1)].center[0] - f[(size_t) (i * cols_)].center[0];
        const double ey = f[(size_t) (i * cols_ + cols_ - 1)].center[1] - f[(size_t) (i * cols_)].center[1];
        if (d[0] * ex + d[1] * ey < 0) d[0] = -d[0], d[1] = -d[1];
    }
    int rows_, cols_;
    double step_;
    std::map<double, std::vector<CalibCircleLite>> keyframes_;
};

// PinholeCamera::inverseRadialDistortion (core/sensor/src/PinholeCamera.cpp:70-95): the 5-term inverse of the radial
// polynomial 1 + k0 r^2 + k1 r^4 + k2 r^6 + k3 r^8 — the initial intrinsics_[4..8] of the spline problem
// (EventCalibSpline.cpp:101-105: k = (distCoeffs(0), distCoeffs(1), distCoeffs(4), 0)).
inline std::array<double, 5> inverseRadialDistortion(const std::array<double, 4> &k) {
    const double k00 = k[0] * k[0], k000 = k[0] * k00, k0000 = k[0] * k000, k00000 = k[0] * k0000;
    const double k01 = k[0] * k[1], k001 = k[0] * k01, k0001 = k[0] * k001;
    const double k11 = k[1] * k[1], k011 = k[0] * k11;
    const double k02 = k[0] * k[2], k002 = k[0] * k02;
    const double k12 = k[1] * k[2], k03 = k[0] * k[3];
    std::array<double, 5> b;
    b[0] = -k[0];
    b[1] = 3 * k00 - k[1];
    b[2] = -12 * k000 + 8 * k01 - k[2];
    b[3] = 55 * k0000 - 55 * k001 + 5 * k11 + 10 * k02 - k[3];
    b[4] = -273 * k00000 + 364 * k0001 - 78 * k011 - 78 * k002 + 12 * k12 + 12 * k03;
    return b;
}

// ---- initialisation stage: EventCalibIni::cvCalibration (event_camera_calib/src/EventCalibIni.cpp:143-327) ----
struct CalibrationSetting {  // include/opengv2/event_camera_calib/parameters.hpp:29-86 (same member names)
    CirclePatternParameters::Ptr circlePatternParameters;
    int NumOfFrameToUse = 200;
    float aspectRatio = 1;
    bool calibZeroTangentDist = true, calibFixPrincipalPoint = true, useFisheye = false;
    bool fixK1 = false, fixK2 = false, fixK3 = false, fixK4 = true, fixK5 = true;
    ecb::CalibFlags flags() const {  // validate(): the cv::CALIB_* bits; K4..K6 do not exist in the 5-coefficient model
        ecb::CalibFlags f;
        f.fixPrincipalPoint = calibFixPrincipalPoint;
        f.zeroTangentDist = calibZeroTangentDist;
        f.fixAspectRatio = aspectRatio != 0;
        f.aspectRatio = aspectRatio != 0 ? aspectRatio : 1.0;  // cameraMatrix(0,0) = aspectRatio over (1,1) = 1 (:147-149)
        f.fixK1 = fixK1, f.fixK2 = fixK2, f.fixK3 = fixK3;
        return f;
    }
};

// Eigen's default stream format for a dense matrix: every coefficient right-aligned to the widest one, rows on lines
inline void printEigenLike(std::ostream &os, const double *m, int rows, int cols) {
    std::vector<std::string> cell((size_t) rows * cols);
    size_t width = 0;
    for (int i = 0; i < rows * cols; ++i) {
        std::ostringstream ss;
        ss.precision(os.precision());
        ss << m[i];
        cell[(size_t) i] = ss.str();
        width = std::max(width, cell[(size_t) i].size());
    }
    for (int r = 0; r < rows; ++r) {
        for (int c = 0; c < cols; ++c) os << (c ? " " : "") << std::setw((int) width) << cell[(size_t) r * cols + c];
        if (r + 1 < rows) os << "\n";
    }
}

class EventCalibIni {
public:
    struct KeyFrame {
        double timeStamp = 0;
        std::pair<double, double> duration;        // the window of the frame (EventFrame ctor)
        int eventsNum = 0;
        std::vector<CalibCircleLite> features;     // board order, rows * cols
        double unitQwb[4] = {0, 0, 0, 1}, twb[3] = {0, 0, 0};
        std::vector<std::array<double, 3>> circles;  // after rectifyFeatures: (cx, cy, r) per board point, r < 0 = deleted
    };
    EventCalibIni(const CalibrationSetting &setting, double motionTimeStep, int width, int height)
        : setting_(setting), step_(motionTimeStep), width_(width), height_(height) {}
    // calcBoardCornerPositions (:99-113), as cv::Point3f
    std::vector<double> boardPoints() const {
        const CirclePatternParameters &p = *setting_.circlePatternParameters;
        std::vector<double> c;
        for (int i = 0; i < p.rows; ++i)
            for (int j = 0; j < p.cols; ++j) {
                c.push_back((double) (float) ((p.isAsymmetric ? (2 * j + i % 2) : j) * p.squareSize));
                c.push_back((double) (float) (i * p.squareSize));
                c.push_back(0.0);
            }
        return c;
    }
    // cvCalibration(): intrinsics from NumOfFrameToUse evenly spaced key frames, then for every key frame in time order the
    // planar PnP pose, checkPose against the last frame kept, rectifyFeatures (one batched GPU call over all frames — its
    // verdict does not depend on the other frames) -> `frames` is replaced by the frames that stay in the map.
    // FE: FrontEnd (one GPU) or ShardedFrontEnd (multi_gpu.hpp)
    template <class FE>
    bool cvCalibration(FE &fe, std::map<double, KeyFrame> &frames, std::ostream &os) {
        if (setting_.useFisheye) {
            os << "Calibration failed: the fisheye model (cv::fisheye::calibrate) is not part of this build" << std::endl;
            return false;
        }
        if (frames.empty()) return false;
        const CirclePatternParameters &pat = *setting_.circlePatternParameters;
        const int nc = pat.rows * pat.cols, frameNum = (int) frames.size();
        int use = setting_.NumOfFrameToUse, step = use > 0 ? frameNum / use : 0;
        if (step == 0) {
            use = frameNum;
            step = 1;
        }
        std::vector<std::vector<double>> imagePoints;
        auto itr = frames.cbegin();
        for (int counter = 0; counter < use; ++counter) {
            std::vector<double> ip;
            for (const auto &f : itr->second.features) {  // cv::Point2f
                ip.push_back((double) (float) f.center[0]);
                ip.push_back((double) (float) f.center[1]);
            }
            imagePoints.push_back(std::move(ip));
            for (int k = 0; k < step && itr != frames.cend(); ++k) ++itr;
        }
        const std::vector<double> obj = boardPoints();
        std::vector<std::array<double, 3>> rvecs, tvecs;
        const double rms = ecb::calibrateCamera(obj, imagePoints, width_, height_, setting_.flags(), camera, rvecs, tvecs);
        os << "Re-projection error reported by calibrateCamera: " << rms << std::endl;
        bool ok = rms >= 0 && std::isfinite(camera.fx) && std::isfinite(camera.fy);
        for (double d : camera.dist) ok = ok && std::isfinite(d);
        std::vector<float> perView;
        const double totalAvgErr = ok ? ecb::computeReprojectionErrors(obj, imagePoints, rvecs, tvecs, camera, perView) : 0.0;
        os << (ok ? "Calibration succeeded" : "Calibration failed") << ". avg re projection error = " << totalAvgErr << std::endl;
        int counter1 = 0, counter2 = 0;
        if (ok) {
            const double K[9] = {camera.fx, 0, camera.cx, 0, camera.fy, camera.cy, 0, 0, 1};
            printEigenLike(os, K, 3, 3);
            os << std::endl;
            printEigenLike(os, camera.dist, 1, 5);
            os << std::endl;
            // poses of all frames (:246-275)
            std::vector<KeyFrame *> all;
            std::vector<std::pair<double, double>> windows;
            std::vector<double> img;  // frames x circles x 5 x 2 projected points (CirclesEventFrame.cpp:431-456)
            const double skewR = pat.circleRadius / std::sqrt(2.0);
            for (auto &kv : frames) {
                KeyFrame &kf = kv.second;
                std::vector<double> ip;
                for (const auto &f : kf.features) {
                    ip.push_back((double) (float) f.center[0]);
                    ip.push_back((double) (float) f.center[1]);
                }
                double rvec[3], tvec[3];
                std::vector<int> inliers;
                const bool solved = (int) kf.features.size() == nc && ecb::solvePnPPlanar(obj, ip, camera, 4.0, rvec, tvec, inliers);
                if (!solved) {  // OpenCV leaves rvec / tvec empty and the reference would fail in cv::Rodrigues; drop the frame
                    ++counter1;
                    continue;
                }
                ecb::bodyPoseFromPnP(rvec, tvec, kf.unitQwb, kf.twb);
                for (int k = 0; k < nc; ++k) {
                    const double *c = &obj[(size_t) 3 * k];
                    const double o5[15] = {c[0], c[1], c[2],
                                           (double) (float) (c[0] + skewR), (double) (float) (c[1] + skewR), c[2],
                                           (double) (float) (c[0] + skewR), (double) (float) (c[1] - skewR), c[2],
                                           (double) (float) (c[0] - skewR), (double) (float) (c[1] - skewR), c[2],
                                           (double) (float) (c[0] - skewR), (double) (float) (c[1] + skewR), c[2]};
                    double p5[10];
                    ecb::projectPoints(o5, 5, rvec, tvec, camera, p5);
                    for (double v : p5) img.push_back((double) (float) v);  // vector<cv::Point2f>
                }
                all.push_back(&kf);
                windows.push_back(kf.duration);
            }
            std::vector<double> out(all.size() * (size_t) nc * 3);
            std::vector<int32_t> verdict(all.size(), 0), widx(all.size());
            if (!all.empty()) {
                fe.run(windows);
                for (size_t i = 0; i < all.size(); ++i) widx[i] = (int32_t) i;
                fe.rectify(widx, nc, img, 3.0, pat.rows, pat.cols, pat.isAsymmetric, out, verdict);
            }
            // replay of the sequential loop (:246-300): checkPose against the last frame kept, then the rectify verdict
            std::vector<const KeyFrame *> seq(all.begin(), all.end());
            const std::vector<char> keep = replayKeep(seq, verdict, step_, counter1, counter2);
            std::map<double, KeyFrame> kept;
            for (size_t i = 0; i < all.size(); ++i) {
                if (!keep[i]) continue;
                KeyFrame &kf = *all[i];
                kf.circles.resize((size_t) nc);
                for (int k = 0; k < nc; ++k)
                    for (int a = 0; a < 3; ++a) kf.circles[(size_t) k][(size_t) a] = out[(i * nc + (size_t) k) * 3 + (size_t) a];
                kept.emplace(kf.timeStamp, kf);
            }
            frames.swap(kept);
        }
        os << counter1 << " frames discard by checkPose." << std::endl;
        os << counter2 << " frames discard by rectifyFeature." << std::endl;
        return ok;
    }
    // The reference adds the frames back one by one in time order (:246-300): a frame is dropped when checkPose against the
    // LAST FRAME KEPT fails (counter1), else when its rectifyFeatures verdict is false (counter2).  The verdicts do not depend
    // on the other frames, so they can be computed for all frames at once and the loop replayed afterwards.
    static std::vector<char> replayKeep(const std::vector<const KeyFrame *> &framesInTimeOrder, const std::vector<int32_t> &verdict,
                                        double motionTimeStep, int &counter1, int &counter2) {
        std::vector<char> keep(framesInTimeOrder.size(), 0);
        const KeyFrame *last = nullptr;
        for (size_t i = 0; i < framesInTimeOrder.size(); ++i) {
            const KeyFrame &kf = *framesInTimeOrder[i];
            if (last && !ecb::checkPose(last->timeStamp, last->unitQwb, last->twb, kf.timeStamp, kf.unitQwb, kf.twb, motionTimeStep)) {
                ++counter1;
                continue;
            }
            if (!verdict[i]) {
                ++counter2;
                continue;
            }
            keep[i] = 1;
            last = &kf;
        }
        return keep;
    }
    ecb::CameraModel camera;  // K and distCoeffs (k1 k2 p1 p2 k3) after cvCalibration

private:
    CalibrationSetting setting_;
    double step_;
    int width_, height_;
};

// ---- spline calibration: EventCalibSpline::optimize on the GPU ----
class EventCalibSpline {
public:
    enum {  // EventCalibSpline.hpp:24-34
        OFFSET_FOCAL_LENGTH_X, OFFSET_FOCAL_LENGTH_Y, OFFSET_PRINCIPAL_POINT_X, OFFSET_PRINCIPAL_POINT_Y,
        OFFSET_K1, OFFSET_K2, OFFSET_K3, OFFSET_K4, OFFSET_K5,
    };
    struct Segment {            // one spline (EventCalibSpline.cpp:63-91)
        std::vector<double> knots;      // n_cp + 4, clamped cubic
        std::vector<double> rot_cp;     // n_cp x (x,y,z,w)
        std::vector<double> trans_cp;   // n_cp x 3
    };
    struct KeyFrame {
        double timeStamp;
        std::vector<std::array<double, 3>> circles;  // (cx, cy, r) per board point; r < 0: absent
    };
    // useSO3 (eventCameraCalib.cpp:204-209): false = CalibReprojectionError (normalised quaternion spline), true =
    // CalibReprojectionError_SO3 (cumulative SO(3) spline, LocalParameterizationSO3); rot_cp are x,y,z,w coefficients either way
    EventCalibSpline(EventContainer::Ptr events, std::vector<Segment> segments, std::array<double, 9> intrinsics,
                     double motionTimeStep, double circleRadius, bool useSO3 = false)
        : ev_(events), seg_(std::move(segments)), intr_(intrinsics), step_(motionTimeStep), radius_(circleRadius), useSO3_(useSO3) {
        if (seg_.empty()) throw std::logic_error("sampleSets not filtered");  // EventCalibSpline.cpp:78-80
        std::vector<double> kn;
        for (auto &s : seg_) {
            n_cp_.push_back((int32_t) (s.rot_cp.size() / 4));
            kn.insert(kn.end(), s.knots.begin(), s.knots.end());
        }
        if (ecb_cost_setup(ev_->ctx, (int) seg_.size(), n_cp_.data(), kn.data(), radius_, 0.2 * radius_) != ECB_OK)
            throw std::logic_error(ecb_last_error(ev_->ctx));  // HuberLoss(0.2 r), EventCalibSpline.cpp:197
        ecb_cost_set_rotation_model(ev_->ctx, useSO3_ ? 1 : 0);
    }
    // Intrinsics held at their current values by optimize() (bit i = intrinsic i in the OFFSET_* order, see
    // ecb::constantIntrinsicsMask); covariance() is then conditional on them.  0 (default): all 9 free, as in the reference.
    int setConstantIntrinsics(uint32_t mask) { return ecb_cost_set_constant_intrinsics(ev_->ctx, mask); }
    // ---- the reference constructor's own set-up (EventCalibSpline.cpp:14-113) from the key frames of the map ----
    struct KeyPose {
        double timeStamp;
        double unitQwb[4];  // x y z w
        double twb[3];
    };
    // The reference's constructor, argument for argument (EventCalibSpline.hpp:19, EventCalibSpline.cpp:14-113): frame-count
    // check, reduceMap() (segments at gaps > 50 steps; segments with fewer than degree + 1 frames are REMOVED from the map),
    // spline fits, intrinsics_ from the camera (K + 5-term inverse of the radial part of distCoeffs), the two report lines,
    // optimize() (association + LM on the GPU) and updateMap() (K, inverseRadialPoly, every key frame's pose <- spline pose).
    // The camera and the board landmarks come from the map (compat/opengv2_lite.hpp); `reduceMap` only enables the part of
    // reduceMap() the reference itself has disabled (:346-348), so it is accepted and has no further effect.
    EventCalibSpline(MapBase::Ptr map, EventContainer::Ptr eventContainer, bool useSO3, bool reduceMap, double motionTimeStep,
                     double circleRadius)
        : EventCalibSpline(eventContainer, segmentsOfMap(map, motionTimeStep, useSO3), intrinsicsOfMap(map), motionTimeStep, circleRadius,
                           useSO3) {
        (void) reduceMap;
        map_ = map;
        std::vector<KeyFrame> kfs;
        for (const auto &kv : map->keyframes()) kfs.push_back(KeyFrame{kv.second->timeStamp(), kv.second->circles});
        std::vector<std::array<double, 3>> landmarks;
        for (const auto &kv : map->landmarks()) {
            const Eigen::Vector3d p = kv.second->position();
            landmarks.push_back({p[0], p[1], p[2]});
        }
        associate(kfs, landmarks);
        if (!optimize()) throw std::runtime_error(ecb_last_error(ev_->ctx));
        updateMap();
    }
    void updateMap() {  // EventCalibSpline.cpp:253-317
        if (!map_) return;
        map_->camera.fx = intr_[0], map_->camera.fy = intr_[1], map_->camera.cx = intr_[2], map_->camera.cy = intr_[3];
        for (int k = 0; k < 5; ++k) map_->inverseRadialPoly[(size_t) k] = intr_[(size_t) (4 + k)];
        std::cout.precision(12);
        std::cout << "Intrinsics after optimization:";
        printEigenLikeRow(std::cout, intr_.data(), 9);
        std::cout << std::endl;
        for (const auto &kv : map_->keyframes()) {
            Bodyframe &bf = *kv.second;
            double q[4], t[3];
            if (!evaluate(bf.timeStamp(), q, t)) continue;  // time2splineIdx < 0
            const Eigen::Quaterniond Qwb_old = bf.unitQwb();
            const Eigen::Vector3d twb_old = bf.twb();
            bf.setPose(Eigen::Vector3d(t[0], t[1], t[2]), Eigen::Quaterniond(q[3], q[0], q[1], q[2]));
            const Eigen::Quaterniond Qbw_old = Qwb_old.conjugate();  // real -> opt (:310-315)
            bf.optT = {Qbw_old.x(), Qbw_old.y(), Qbw_old.z(), Qbw_old.w(), twb_old[0], twb_old[1], twb_old[2]};
        }
    }
    // reduceMap() :319-348: segments at gaps > 50 * MotionTimeStep, segments with fewer than degree + 1 frames dropped
    static std::vector<std::vector<KeyPose>> segmentKeyframes(const std::vector<KeyPose> &kf, double motionTimeStep) {
        std::vector<std::vector<KeyPose>> sets(1);
        if (kf.empty()) return {};
        double last = kf.front().timeStamp;
        for (const auto &k : kf) {
            if (k.timeStamp - last > 50 * motionTimeStep) sets.emplace_back();
            sets.back().push_back(k);
            last = k.timeStamp;
        }
        std::vector<std::vector<KeyPose>> out;
        for (auto &s : sets)
            if (s.size() >= 4) out.push_back(s);
        return out;
    }
    // BsplineReal(dim, samples, cpNum, timestamps) (BsplineReal.hpp:31-100,329-449 without derivative samples): clamped
    // knots by NURBS-book eq. 9.68, first / last control point = first / last sample, interior ones by least squares
    static void fitSpline(const std::vector<double> &us, const std::vector<double> &data, int dim, int cpNum,
                          std::vector<double> &knots, std::vector<double> &cp) {
        const int degree = 3, n = (int) us.size();
        knots.assign((size_t) cpNum + degree + 1, 0.0);
        for (int i = 0; i <= degree; ++i) knots[(size_t) i] = us.front(), knots[knots.size() - 1 - (size_t) i] = us.back();
        const double d = n / double(cpNum - degree);
        for (int j = 1; j <= cpNum - 1 - degree; ++j) {
            const int i = (int) std::floor(j * d);
            const double alpha = j * d - i;
            knots[(size_t) (degree + j)] = (1 - alpha) * us[(size_t) i - 1] + alpha * us[(size_t) i];
        }
        cp.assign((size_t) cpNum * dim, 0.0);
        for (int c = 0; c < dim; ++c) cp[(size_t) c] = data[(size_t) c], cp[(size_t) (cpNum - 1) * dim + c] = data[(size_t) (n - 1) * dim + c];
        const int m = cpNum - 2;
        if (m <= 0) return;
        std::vector<double> A((size_t) m * m, 0.0), B((size_t) m * dim, 0.0);
        for (int k = 1; k < n - 1; ++k) {  // interior samples (rows 1 .. n-2 of N)
            const int span = bspline_find_span(knots, us[(size_t) k]);
            double N[4];
            bspline_basis(knots, span, us[(size_t) k], N);
            double n0 = 0, nl = 0;  // N_{0,p}(u_k), N_{cpNum-1,p}(u_k)
            for (int j = 0; j <= degree; ++j) {
                if (span - degree + j == 0) n0 = N[j];
                if (span - degree + j == cpNum - 1) nl = N[j];
            }
            for (int a = 0; a <= degree; ++a) {
                const int ia = span - degree + a - 1;  // interior control point index 0 .. m-1
                if (ia < 0 || ia >= m || N[a] == 0) continue;
                for (int b = 0; b <= degree; ++b) {
                    const int ib = span - degree + b - 1;
                    if (ib < 0 || ib >= m) continue;
                    A[(size_t) ia * m + ib] += N[a] * N[b];
                }
                for (int c = 0; c < dim; ++c)
                    B[(size_t) ia * dim + c] += N[a] * (data[(size_t) k * dim + c] - n0 * data[(size_t) c] - nl * data[(size_t) (n - 1) * dim + c]);
            }
        }
        // A = L L^T (dense Cholesky; cpNum is a few hundred at most), then the dim right-hand sides
        for (int j = 0; j < m; ++j) {
            for (int k = 0; k < j; ++k)
                for (int i = j; i < m; ++i) A[(size_t) i * m + j] -= A[(size_t) i * m + k] * A[(size_t) j * m + k];
            const double dgl = std::sqrt(A[(size_t) j * m + j]);
            if (!(dgl > 0)) throw std::logic_error("Function optimization: decomposition failed!");
            for (int i = j; i < m; ++i) A[(size_t) i * m + j] /= dgl;
        }
        for (int c = 0; c < dim; ++c) {
            std::vector<double> y((size_t) m);
            for (int i = 0; i < m; ++i) {
                double v = B[(size_t) i * dim + c];
                for (int k = 0; k < i; ++k) v -= A[(size_t) i * m + k] * y[(size_t) k];
                y[(size_t) i] = v / A[(size_t) i * m + i];
            }
            for (int i = m - 1; i >= 0; --i) {
                double v = y[(size_t) i];
                for (int k = i + 1; k < m; ++k) v -= A[(size_t) k * m + i] * cp[(size_t) (k + 1) * dim + c];
                cp[(size_t) (i + 1) * dim + c] = v / A[(size_t) i * m + i];
            }
        }
    }
    // Spline segments from the map's key frames like the reference constructor (:25-91): frame count check, segmentation,
    // time bounds extended by 3 steps, cpNum = floor(T / (50 step)) clamped, spline fits.  useSO3: the reference fits the
    // SO(3) control points with Ceres (BsplineSO3::optimizeCP); here they start from the normalised quaternion-spline fit.
    static std::vector<Segment> segmentsFromKeyframes(const std::vector<KeyPose> &kf, double motionTimeStep, bool useSO3 = false,
                                                      bool checkFrameCount = true) {
        if (checkFrameCount && kf.size() <= 10) throw std::logic_error("too few frames in the map.");
        std::vector<Segment> out;
        for (auto &set : segmentKeyframes(kf, motionTimeStep)) {
            std::vector<double> us, tw, qw;
            for (auto &k : set) {
                us.push_back(k.timeStamp);
                tw.insert(tw.end(), k.twb, k.twb + 3);
                qw.insert(qw.end(), k.unitQwb, k.unitQwb + 4);
            }
            us.front() -= 3 * motionTimeStep;
            us.back() += 3 * motionTimeStep;
            int cpNum = (int) std::floor((us.back() - us.front()) / (50 * motionTimeStep));
            if (cpNum > (int) us.size()) cpNum = (int) us.size() - 1;
            if (cpNum < 4) cpNum = 4;  // become a bezier curve
            Segment sg;
            std::vector<double> kn2;
            fitSpline(us, tw, 3, cpNum, sg.knots, sg.trans_cp);
            fitSpline(us, qw, 4, cpNum, kn2, sg.rot_cp);
            if (useSO3)
                for (size_t c = 0; c + 3 < sg.rot_cp.size(); c += 4) {
                    const double nq = std::sqrt(sg.rot_cp[c] * sg.rot_cp[c] + sg.rot_cp[c + 1] * sg.rot_cp[c + 1] +
                                                sg.rot_cp[c + 2] * sg.rot_cp[c + 2] + sg.rot_cp[c + 3] * sg.rot_cp[c + 3]);
                    for (int a = 0; a < 4; ++a) sg.rot_cp[c + (size_t) a] /= nq;
                }
            out.push_back(std::move(sg));
        }
        if (out.empty()) throw std::logic_error("sampleSets not filtered");
        return out;
    }
    // association loop, EventCalibSpline.cpp:157-192; landmarks: board points (EventCalibIni.cpp:99-113)
    int64_t associate(const std::vector<KeyFrame> &kf, const std::vector<std::array<double, 3>> &landmarks) {
        const int nc = (int) landmarks.size();
        std::vector<double> t(kf.size()), c(kf.size() * nc * 3);
        for (size_t i = 0; i < kf.size(); ++i) {
            t[i] = kf[i].timeStamp;
            for (int q = 0; q < nc; ++q)
                for (int a = 0; a < 3; ++a) c[(i * nc + q) * 3 + a] = q < (int) kf[i].circles.size() ? kf[i].circles[q][a] : -1.0;
        }
        int64_t n = 0;
        if (ecb_cost_associate(ev_->ctx, t.data(), c.data(), (int) kf.size(), nc, &landmarks[0][0], step_, &n) != ECB_OK)
            throw std::runtime_error(ecb_last_error(ev_->ctx));
        kfTime_ = t;  // residualGroups(ECB_RESIDUALS_BY_KEYFRAME) groups by these stamps
        kfCircles_ = c;  // keyframeReprojection reprojects these centres
        landmarks_ = landmarks;
        return n;
    }
    bool optimize(ecb_lm_summary *summary = nullptr) {  // EventCalibSpline.cpp:115-251
        std::vector<double> rot, trans;
        flatten(seg_, rot, trans);
        ecb_lm_options opt;
        ecb_lm_default_options(&opt);
        opt.rotation_model = useSO3_ ? 1 : 0;
        ecb_lm_summary sum;
        if (ecb_calibrate(ev_->ctx, (int) seg_.size(), n_cp_.data(), intr_.data(), rot.data(), trans.data(), &opt, &sum, nullptr, 0) != ECB_OK)
            return false;
        size_t ro = 0, to = 0;
        for (auto &s : seg_) {
            std::copy(rot.begin() + ro, rot.begin() + ro + s.rot_cp.size(), s.rot_cp.begin());
            std::copy(trans.begin() + to, trans.begin() + to + s.trans_cp.size(), s.trans_cp.begin());
            ro += s.rot_cp.size();
            to += s.trans_cp.size();
        }
        if (summary) *summary = sum;
        return true;
    }
    // Uncertainty of the calibration (ecb_covariance): Z = H^-1 at the current point (where optimize() left it) on the band /
    // arrow pattern, sigma^2 = 2 cost / (residuals - parameters), standard deviation of parameter i = sqrt(sigma^2 Z_ii).  With
    // constant intrinsics (setConstantIntrinsics) Z is conditional on them: their rows / columns are 0, and so their deviation.
    struct Covariance {
        std::array<double, 81> intrinsics{};  // Z of fx fy cx cy k1 .. k5, row major
        std::vector<double> band;             // 6C x 24: Z(j + r, j) at [j * 24 + r], control point c owns rows 6c .. 6c+5
        std::vector<double> cross;            // 9 x 6C: Z(intrinsic i, j) at [i * 6C + j]
        ecb_covariance_summary summary{};
        std::array<double, 9> stdIntrinsics() const {
            std::array<double, 9> s{};
            for (int i = 0; i < 9; ++i) s[(size_t) i] = std::sqrt(summary.sigma2 * intrinsics[(size_t) (10 * i)]);
            return s;
        }
    };
    // ECB_OK, ECB_FAILED for rank-deficient normal equations (out.summary.deficient_index names the parameter), < 0 on errors
    int covariance(Covariance &out) const { return covarianceAt(ev_->ctx, n_cp_, intr_, seg_, nullptr, 0, out); }
    // the same at a given point; d_packed / n_residuals_total as ecb_covariance (an already-summed buffer of several GPUs)
    static int covarianceAt(ecb_ctx *ctx, const std::vector<int32_t> &n_cp, const std::array<double, 9> &intr,
                            const std::vector<Segment> &seg, const void *d_packed, int64_t n_residuals_total, Covariance &out) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        const size_t n = trans.size() * 2;  // 6 C
        out.band.assign(n * 24, 0.0);
        out.cross.assign(9 * n, 0.0);
        return ecb_covariance(ctx, (int) n_cp.size(), n_cp.data(), intr.data(), rot.data(), trans.data(), d_packed, n_residuals_total,
                              out.intrinsics.data(), out.band.data(), out.cross.data(), &out.summary);
    }
    // Uncertainty of the trajectory (ecb_pose_covariance), after covariance(): pose[7 n] = tx ty tz qx qy qz qw and cov[36 n] =
    // Sigma(t) row major over (dtheta body frame, dp world frame) at each time; NaN rows for times outside every segment.
    // The covariance is cov.summary.sigma2 Sigma.  ECB_OK, or < 0 (ECB_ERR_STATE without a successful covariance()).
    int poseCovariance(const std::vector<double> &times, std::vector<double> &pose, std::vector<double> &cov,
                       int64_t *n_valid = nullptr) const {
        return poseCovarianceAt(ev_->ctx, times, pose, cov, n_valid);
    }
    static int poseCovarianceAt(ecb_ctx *ctx, const std::vector<double> &times, std::vector<double> &pose, std::vector<double> &cov,
                                int64_t *n_valid) {
        pose.assign(7 * times.size(), 0.0);
        cov.assign(36 * times.size(), 0.0);
        return ecb_pose_covariance(ctx, times.data(), (int64_t) times.size(), pose.data(), cov.data(), n_valid);
    }
    // Motion of the trajectory (ecb_trajectory_motion) at the current control points: motion[16 n] = tx ty tz qx qy qz qw, body
    // angular velocity wx wy wz (rad per time unit), world velocity vx vy vz and acceleration ax ay az at each time; NaN rows for
    // times outside every segment.  ECB_OK, or < 0.
    int trajectoryMotion(const std::vector<double> &times, std::vector<double> &motion, int64_t *n_valid = nullptr) const {
        return trajectoryMotionAt(ev_->ctx, seg_, times, motion, n_valid);
    }
    static int trajectoryMotionAt(ecb_ctx *ctx, const std::vector<Segment> &seg, const std::vector<double> &times,
                                  std::vector<double> &motion, int64_t *n_valid) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        motion.assign(16 * times.size(), 0.0);
        return ecb_trajectory_motion(ctx, rot.data(), trans.data(), times.data(), (int64_t) times.size(), motion.data(), n_valid);
    }
    // Camera-gyroscope calibration (ecb_gyro_calibrate) at the current control points: gyro[4 n] = t wx wy wz (gyroscope stamps
    // and readings, rad per time unit), the offset scanned on nOffsets points over [-maxOffset, maxOffset] (nOffsets 1 with
    // maxOffset 0: held at 0).  offsetCost (nOffsets) and residuals (3 n) are filled when non-null.  ECB_OK, ECB_FAILED with
    // result.status (too few samples, the scan's minimum at the grid's edge, a rank-deficient system), or < 0.
    int calibrateGyroscope(const std::vector<double> &gyro, double maxOffset, int nOffsets, ecb_gyro_calibration &result,
                           std::vector<double> *offsetCost = nullptr, std::vector<double> *residuals = nullptr) const {
        return calibrateGyroscopeAt(ev_->ctx, seg_, gyro, maxOffset, nOffsets, result, offsetCost, residuals);
    }
    static int calibrateGyroscopeAt(ecb_ctx *ctx, const std::vector<Segment> &seg, const std::vector<double> &gyro, double maxOffset,
                                    int nOffsets, ecb_gyro_calibration &result, std::vector<double> *offsetCost,
                                    std::vector<double> *residuals) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        if (offsetCost) offsetCost->assign((size_t) std::max(nOffsets, 0), 0.0);
        if (residuals) residuals->assign(3 * (gyro.size() / 4), 0.0);
        return ecb_gyro_calibrate(ctx, rot.data(), gyro.data(), (int64_t) (gyro.size() / 4), maxOffset, nOffsets, &result,
                                  offsetCost ? offsetCost->data() : nullptr, residuals ? residuals->data() : nullptr);
    }
    // The same motion with its covariance (ecb_motion_covariance), after covariance(): cov[81 n] = Sigma_m(t) row major over
    // (w body frame, v, a world frame).  The covariance is cov.summary.sigma2 Sigma_m.  ECB_OK, or < 0 (ECB_ERR_STATE without a
    // successful covariance()).
    int motionCovariance(const std::vector<double> &times, std::vector<double> &motion, std::vector<double> &cov,
                         int64_t *n_valid = nullptr) const {
        return motionCovarianceAt(ev_->ctx, times, motion, cov, n_valid);
    }
    static int motionCovarianceAt(ecb_ctx *ctx, const std::vector<double> &times, std::vector<double> &motion,
                                  std::vector<double> &cov, int64_t *n_valid) {
        motion.assign(16 * times.size(), 0.0);
        cov.assign(81 * times.size(), 0.0);
        return ecb_motion_covariance(ctx, times.data(), (int64_t) times.size(), motion.data(), cov.data(), n_valid);
    }
    // How well the model fits (ecb_cost_residuals / ecb_cost_residual_groups) at the current point, where optimize() left it.
    // r is the raw residual ||X_w - L|| - radius: a distance on the board plane in the units of the board points, NOT pixels.
    // residuals: r of every record in the association's order.  residualGroups: statistics per key frame (the stamps of the last
    // associate()), per circle or per sensor cell of cellPx pixels (by = ECB_RESIDUALS_BY_*); total (may be null) over every record.
    int residuals(std::vector<double> &r) const { return residualsAt(ev_->ctx, intr_, seg_, r); }
    int residualGroups(int by, int cellPx, std::vector<ecb_residual_group> &groups, ecb_residual_group *total) const {
        return residualGroupsAt(ev_->ctx, intr_, seg_, kfTime_, by, cellPx, groups, total);
    }
    static int residualsAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg, std::vector<double> &r) {
        return recordReportAt(ctx, intr, seg, false, r, nullptr);
    }
    static int residualGroupsAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg,
                                const std::vector<double> &kfTime, int by, int cellPx, std::vector<ecb_residual_group> &groups,
                                ecb_residual_group *total) {
        return groupReportAt(ecb_cost_residual_groups, ctx, intr, seg, kfTime, by, cellPx, groups, total);
    }
    // Outlier rejection (ecb_cost_reject) at the current point: removes the records with !(|r| <= maxAbsR) and those of the key
    // frames flagged in dropKeyframe (one flag per key frame of the last associate(); empty: no key-frame criterion).  A following
    // optimize(), the reports and covariance() see only the kept records, until the next associate().  See ecb::outlierRejection.
    int rejectResiduals(double maxAbsR, const std::vector<uint8_t> &dropKeyframe, int64_t *kept, int64_t *removed) {
        return rejectResidualsAt(ev_->ctx, intr_, seg_, kfTime_, maxAbsR, dropKeyframe, kept, removed);
    }
    static int rejectResidualsAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg,
                                 const std::vector<double> &kfTime, double maxAbsR, const std::vector<uint8_t> &dropKeyframe,
                                 int64_t *kept, int64_t *removed) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        const bool mask = !dropKeyframe.empty();
        if (mask && dropKeyframe.size() != kfTime.size()) return ECB_ERR_ARG;
        return ecb_cost_reject(ctx, intr.data(), rot.data(), trans.data(), maxAbsR, mask ? kfTime.data() : nullptr,
                               mask ? dropKeyframe.data() : nullptr, (int) dropKeyframe.size(), kept, removed);
    }
    // Re-association (ecb_cost_reassociate) at the current point: every event near a key frame of the last associate() (maxDt = 0:
    // the association's window) is matched to the board circle nearest to its back-projection at its own pose and kept when its
    // event-to-rim error is below gatePx pixels (5: the association's tolerance).  The kept events replace the records; a following
    // optimize() solves again on them.  Counts (each may be null): the new records, and against the records before the call the
    // events with the same circle, another circle, newly recorded, and records lost.
    struct ReassociationCounts {
        int64_t residuals = 0, same = 0, changed = 0, added = 0, lost = 0;
    };
    int reassociate(double gatePx, double maxDt, ReassociationCounts *counts) {
        return reassociateAt(ev_->ctx, intr_, seg_, gatePx, maxDt, counts);
    }
    static int reassociateAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg, double gatePx,
                             double maxDt, ReassociationCounts *counts) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        ReassociationCounts c;
        const int rc = ecb_cost_reassociate(ctx, intr.data(), rot.data(), trans.data(), gatePx, maxDt, &c.residuals, &c.same,
                                            &c.changed, &c.added, &c.lost);
        if (rc == ECB_OK && counts) *counts = c;
        return rc;
    }
    // adds group b into a: counts and sums added, max_abs the max (shards combine in rank order)
    static void accumulateResidualGroup(ecb_residual_group &a, const ecb_residual_group &b) {
        a.count += b.count;
        a.n_downweighted += b.n_downweighted;
        a.sum += b.sum;
        a.sum_sq += b.sum_sq;
        a.max_abs = std::max(a.max_abs, b.max_abs);
        a.cost += b.cost;
    }
    // The same fit in pixels, through the forward camera model (ecb_cost_reprojection_errors / ecb_cost_reprojection_groups /
    // ecb_keyframe_reprojection), at the current point.  e_k = sign(|d| - radius) |q - o|: o the event pixel, q the projection of
    // the rim point the residual measures; NaN where it cannot be projected.  reprojectionErrors: e of every record in the
    // association's order; reprojectionGroups: the groups of residualGroups; keyframeReprojection: the board points at the stamps
    // of the last associate() against the detected centres, proj[K][n][2] and err[K][n] (pixels, NaN for an absent feature).
    int reprojectionErrors(std::vector<double> &e, int64_t *nInvalid = nullptr) const {
        return reprojectionErrorsAt(ev_->ctx, intr_, seg_, e, nInvalid);
    }
    int reprojectionGroups(int by, int cellPx, std::vector<ecb_reprojection_group> &groups, ecb_reprojection_group *total) const {
        return reprojectionGroupsAt(ev_->ctx, intr_, seg_, kfTime_, by, cellPx, groups, total);
    }
    int keyframeReprojection(std::vector<double> &proj, std::vector<double> &err, ecb_reprojection_group *total) const {
        return keyframeReprojectionAt(ev_->ctx, intr_, seg_, kfTime_, kfCircles_, landmarks_, proj, err, total);
    }
    static int reprojectionErrorsAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg,
                                    std::vector<double> &e, int64_t *nInvalid) {
        return recordReportAt(ctx, intr, seg, true, e, nInvalid);
    }
    static int reprojectionGroupsAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg,
                                    const std::vector<double> &kfTime, int by, int cellPx, std::vector<ecb_reprojection_group> &groups,
                                    ecb_reprojection_group *total) {
        return groupReportAt(ecb_cost_reprojection_groups, ctx, intr, seg, kfTime, by, cellPx, groups, total);
    }
    // kfCircles[K][n][3] (cx cy r, r < 0 absent) and landmarks[n] as given to ecb_cost_associate
    static int keyframeReprojectionAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg,
                                      const std::vector<double> &kfTime, const std::vector<double> &kfCircles,
                                      const std::vector<std::array<double, 3>> &landmarks, std::vector<double> &proj,
                                      std::vector<double> &err, ecb_reprojection_group *total) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        const size_t m = kfTime.size() * landmarks.size();
        if (m == 0 || kfCircles.size() != 3 * m) return ECB_ERR_STATE;  // no associate() yet
        proj.assign(2 * m, 0.0);
        err.assign(m, 0.0);
        return ecb_keyframe_reprojection(ctx, intr.data(), rot.data(), trans.data(), kfTime.data(), kfCircles.data(),
                                         (int) kfTime.size(), (int) landmarks.size(), &landmarks[0][0], proj.data(), err.data(),
                                         total);
    }
    // adds group b into a: counts and sums added, max_abs the max (shards combine in rank order)
    static void accumulateReprojectionGroup(ecb_reprojection_group &a, const ecb_reprojection_group &b) {
        a.count += b.count;
        a.n_invalid += b.n_invalid;
        a.sum += b.sum;
        a.sum_sq += b.sum_sq;
        a.max_abs = std::max(a.max_abs, b.max_abs);
    }
    const std::vector<double> &keyframeTimes() const { return kfTime_; }
    const std::vector<double> &keyframeCircles() const { return kfCircles_; }
    const std::vector<std::array<double, 3>> &landmarks() const { return landmarks_; }
    const std::array<double, 9> &intrinsics() const { return intr_; }
    const std::vector<Segment> &segments() const { return seg_; }
    // the control points of all segments in order: rotation (4 per point) and translation (3 per point), as the C ABI takes them
    static void flatten(const std::vector<Segment> &seg, std::vector<double> &rot, std::vector<double> &trans) {
        for (auto &s : seg) {
            rot.insert(rot.end(), s.rot_cp.begin(), s.rot_cp.end());
            trans.insert(trans.end(), s.trans_cp.begin(), s.trans_cp.end());
        }
    }
    // EventCalibSpline.hpp:286-303: index of the segment whose knot range holds t, else -1
    int time2splineIdx(double t) const { return time2splineIdx(seg_, t); }
    static int time2splineIdx(const std::vector<Segment> &seg, double t) {
        for (size_t i = 0; i < seg.size(); ++i)
            if (t >= seg[i].knots.front() && t <= seg[i].knots.back()) return (int) i;
        return -1;
    }
    // EventCalibSpline.hpp:305-330: pose of the spline at t — unitQwb as x,y,z,w and twb
    bool evaluate(double t, double unitQwb[4], double twb[3]) const { return evaluate(seg_, useSO3_, t, unitQwb, twb); }
    static bool evaluate(const std::vector<Segment> &seg, bool useSO3, double t, double unitQwb[4], double twb[3]) {
        const int idx = time2splineIdx(seg, t);
        if (idx < 0) return false;
        const Segment &s = seg[(size_t) idx];
        const int span = bspline_find_span(s.knots, t);
        double N[4];
        bspline_basis(s.knots, span, t, N);
        for (int c = 0; c < 3; ++c) {
            twb[c] = 0;
            for (int j = 0; j < 4; ++j) twb[c] += N[j] * s.trans_cp[(size_t) (3 * (span - 3 + j) + c)];
        }
        const double *Q = &s.rot_cp[(size_t) (4 * (span - 3))];
        if (useSO3) {  // BsplineSO3::evaluate: R0 * prod exp(beta_j log(R_{j-1}^-1 R_j))
            double beta[3];
            ecb_so3::cumulative_basis(N, beta);
            ecb_so3::rotation_value(Q, beta, unitQwb);
        } else {  // BsplineReal<4>::evaluate + normalize() (EventCalibSpline.cpp:283-286)
            double n2 = 0;
            for (int c = 0; c < 4; ++c) {
                unitQwb[c] = 0;
                for (int j = 0; j < 4; ++j) unitQwb[c] += N[j] * Q[4 * j + c];
                n2 += unitQwb[c] * unitQwb[c];
            }
            const double n = std::sqrt(n2);
            for (int c = 0; c < 4; ++c) unitQwb[c] /= n;
        }
        return true;
    }
    // SystemBase::saveKeyFrameTrajectoryTUM (SystemBase.cpp:122-150) for the key-frame stamps after updateMap() (:253-317);
    // sensor = body (identity extrinsics, eventCameraCalib.cpp:133-134).  Returns the number of lines written.
    int saveKeyFrameTrajectoryTUM(const std::string &filename, const std::vector<double> &keyframeStamps) const {
        return saveKeyFrameTrajectoryTUM(seg_, useSO3_, filename, keyframeStamps);
    }
    static int saveKeyFrameTrajectoryTUM(const std::vector<Segment> &seg, bool useSO3, const std::string &filename,
                                         const std::vector<double> &keyframeStamps) {
        std::ofstream f(filename.c_str());
        f << std::fixed;
        int num = 0;
        for (double ts : keyframeStamps) {
            double q[4], t[3];
            if (!evaluate(seg, useSO3, ts, q, t)) continue;
            f << std::setprecision(10) << ts << " " << t[0] << " " << t[1] << " " << t[2] << " " << q[0] << " " << q[1] << " "
              << q[2] << " " << q[3] << std::endl;
            ++num;
        }
        return num;
    }

private:
    static void printEigenLikeRow(std::ostream &os, const double *v, int n);
    // reduceMap() :319-344 + the set-up of :36-91 on the map's key frames
    static std::vector<Segment> segmentsOfMap(const MapBase::Ptr &map, double motionTimeStep, bool useSO3) {
        if (!map || map->frameNum() <= 10) throw std::logic_error("too few frames in the map.");
        std::vector<KeyPose> kf;
        for (const auto &kv : map->keyframes()) {
            const Eigen::Quaterniond q = kv.second->unitQwb();
            const Eigen::Vector3d t = kv.second->twb();
            kf.push_back(KeyPose{kv.second->timeStamp(), {q.x(), q.y(), q.z(), q.w()}, {t[0], t[1], t[2]}});
        }
        std::vector<double> drop;  // frames of segments shorter than degree + 1 leave the map
        {
            std::vector<std::vector<double>> sets(1);
            double last = kf.front().timeStamp;
            for (const auto &k : kf) {
                if (k.timeStamp - last > 50 * motionTimeStep) sets.emplace_back();
                sets.back().push_back(k.timeStamp);
                last = k.timeStamp;
            }
            for (const auto &st : sets)
                if (st.size() < 4) drop.insert(drop.end(), st.begin(), st.end());
        }
        for (double id : drop) map->removeFrame(id);
        for (size_t i = 1; i < kf.size(); ++i) {  // one sign per quaternion so that the real-valued spline fit sees a continuous curve
            double d = 0;
            for (int a = 0; a < 4; ++a) d += kf[i].unitQwb[a] * kf[i - 1].unitQwb[a];
            if (d < 0)
                for (int a = 0; a < 4; ++a) kf[i].unitQwb[a] = -kf[i].unitQwb[a];
        }
        return segmentsFromKeyframes(kf, motionTimeStep, useSO3, false);
    }
    static std::array<double, 9> intrinsicsOfMap(const MapBase::Ptr &map) {  // :93-108
        const ecb::CameraModel &cam = map->camera;
        const std::array<double, 4> radial = {cam.dist[0], cam.dist[1], cam.dist[4], 0.0};
        const std::array<double, 5> inv = inverseRadialDistortion(radial);
        const std::array<double, 9> intrinsics = {cam.fx, cam.fy, cam.cx, cam.cy, inv[0], inv[1], inv[2], inv[3], inv[4]};
        std::cout << "OpenCV Distortion before optimization:";
        printEigenLikeRow(std::cout, radial.data(), 4);
        std::cout << std::endl << "Intrinsics before optimization:";
        printEigenLikeRow(std::cout, intrinsics.data(), 9);
        std::cout << std::endl;
        return intrinsics;
    }
    MapBase::Ptr map_;
    EventContainer::Ptr ev_;
    std::vector<Segment> seg_;
    std::vector<int32_t> n_cp_;
    std::array<double, 9> intr_;
    std::vector<double> kfTime_;  // key-frame stamps of the last associate()
    std::vector<double> kfCircles_;  // ... its circles [K][n][3], r < 0 absent
    std::vector<std::array<double, 3>> landmarks_;  // ... and its board points
    double step_, radius_;
    bool useSO3_ = false;
    // one value per record (ecb_cost_reprojection_errors when pixels, else ecb_cost_residuals) -> out, sized from ecb_cost_layout
    static int recordReportAt(ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg, bool pixels,
                              std::vector<double> &out, int64_t *nInvalid) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        int64_t n = 0;
        int rc = ecb_cost_layout(ctx, nullptr, nullptr, &n, nullptr);
        if (rc != ECB_OK) return rc;
        out.assign((size_t) n, 0.0);
        double *h = n > 0 ? out.data() : nullptr;
        return pixels ? ecb_cost_reprojection_errors(ctx, intr.data(), rot.data(), trans.data(), nullptr, h, nInvalid)
                      : ecb_cost_residuals(ctx, intr.data(), rot.data(), trans.data(), nullptr, h);
    }
    // the groups of one report (fn: ecb_cost_residual_groups or ecb_cost_reprojection_groups): the size query, then the filled call
    template <class Group>
    static int groupReportAt(int (*fn)(ecb_ctx *, const double *, const double *, const double *, int, const double *, int, int, Group *,
                                       int, int *, Group *),
                             ecb_ctx *ctx, const std::array<double, 9> &intr, const std::vector<Segment> &seg,
                             const std::vector<double> &kfTime, int by, int cellPx, std::vector<Group> &groups, Group *total) {
        std::vector<double> rot, trans;
        flatten(seg, rot, trans);
        const double *kf = kfTime.empty() ? nullptr : kfTime.data();
        int ng = 0;
        int rc = fn(ctx, intr.data(), rot.data(), trans.data(), by, kf, (int) kfTime.size(), cellPx, nullptr, 0, &ng, nullptr);
        if (rc != ECB_OK) return rc;
        groups.assign((size_t) ng, Group{});
        Group dummy;
        return fn(ctx, intr.data(), rot.data(), trans.data(), by, kf, (int) kfTime.size(), cellPx, ng > 0 ? groups.data() : &dummy, ng, &ng,
                  total);
    }
};
inline void EventCalibSpline::printEigenLikeRow(std::ostream &os, const double *v, int n) { printEigenLike(os, v, 1, n); }

}  // namespace opengv2
#endif  // ECB_EVENT_CALIB_HPP
