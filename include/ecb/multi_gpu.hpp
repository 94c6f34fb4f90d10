// Several GPUs driven from ONE C++ process — the host side of the reference's own parallelism.
//
// The reference parallelises inside its CLI: the event stream is cut into time pieces and hardware_concurrency() - 2 worker
// threads run the window loop on them (ECC/test/eventCameraCalib.cpp:172-190).  Here the same time pieces are dealt out to
// the visible GPUs in contiguous blocks: every GPU holds the records of its own time range (a contiguous byte range of the
// time-sorted .bin), one host thread + one context per GPU, no data-path collective for the detection.  The spline
// optimisation shards the residuals the same way; the one exchange step of the path — the sum of the packed normal
// equations and of the candidate costs — runs inside the kernels over peer-mapped buffers (ecb_lm_device_set_exchange,
// include/eventcalib_b200.h), so every GPU takes bit-identical decisions.
//
//   opengv2::ShardedEventContainer   G x EventContainer, events partitioned by time at given cut points
//   opengv2::ShardedFrontEnd         FrontEnd::run / summary / candidates / rectify over the shards (window -> owning shard)
//   opengv2::ShardedCalibSpline      EventCalibSpline::associate + optimize over the shards
//
// Results do not depend on the number of shards: a window is evaluated by exactly one GPU from exactly the events the single
// GPU would use (tests/test_host_cli.py::test_cli_multi_gpu_equals_single_gpu).  Devices: ECB_DEVICES = "0,1,2" / "all"
// (default: all visible devices; ECB_DEVICE = one device like the single-GPU build).
#ifndef ECB_MULTI_GPU_HPP
#define ECB_MULTI_GPU_HPP

#include <thread>

#include "event_calib.hpp"

namespace opengv2 {

inline std::vector<int> ecbDevices() {
    std::vector<int> dev;
    const char *list = getenv("ECB_DEVICES");
    if (list && std::string(list) != "all") {
        std::stringstream ss(list);
        std::string tok;
        while (std::getline(ss, tok, ','))
            if (!tok.empty()) dev.push_back(atoi(tok.c_str()));
    } else if (!list && getenv("ECB_DEVICE")) {
        dev.push_back(atoi(getenv("ECB_DEVICE")));
    } else {
        const int n = ecb_device_count();
        for (int d = 0; d < n; ++d) dev.push_back(d);
    }
    if (dev.empty()) dev.push_back(0);
    return dev;
}

// runs f(g) for g = 0 .. n-1 on n host threads (one per GPU, like the reference's worker threads); rethrows the first error
template <class F>
inline void forEachShard(int n, F &&f) {
    if (n == 1) {
        f(0);
        return;
    }
    std::vector<std::thread> th;
    std::vector<std::exception_ptr> err((size_t) n);
    for (int g = 0; g < n; ++g)
        th.emplace_back([&, g]() {
            try {
                f(g);
            } catch (...) {
                err[(size_t) g] = std::current_exception();
            }
        });
    for (auto &t : th) t.join();
    for (auto &e : err)
        if (e) std::rethrow_exception(e);
}

struct ShardedEventContainer {
    typedef std::shared_ptr<ShardedEventContainer> Ptr;
    std::vector<EventContainer::Ptr> shard;
    std::vector<int> device;
    std::vector<double> cut;        // shard g holds the events with cut[g] <= t < cut[g+1]  (cut[0] = -inf, cut[G] = +inf)
    std::vector<int64_t> base;      // index of shard g's first event in the whole stream (G + 1 entries)
    int width = 0, height = 0;
    double firstTime = 0, lastTime = 0;

    ShardedEventContainer(const std::vector<int> &devices, int w, int h) : device(devices), width(w), height(h) {
        for (int d : devices) shard.push_back(std::make_shared<EventContainer>(d, w, h));
    }
    int shards() const { return (int) shard.size(); }
    // records: time-sorted; cuts: G - 1 ascending stamps (normally boundaries of the CLI's time pieces)
    void load(const EventRecord *rec, int64_t n, const std::vector<double> &cuts) {
        const int G = shards();
        if ((int) cuts.size() != G - 1) throw std::invalid_argument("ShardedEventContainer::load: need one cut per shard boundary");
        cut.assign(1, -std::numeric_limits<double>::infinity());
        base.assign(1, 0);
        for (int g = 0; g + 1 < G; ++g) {
            const EventRecord *it = std::lower_bound(rec, rec + n, cuts[(size_t) g], [](const EventRecord &r, double t) { return r.t < t; });
            cut.push_back(cuts[(size_t) g]);
            base.push_back(std::max<int64_t>(base.back(), it - rec));
        }
        cut.push_back(std::numeric_limits<double>::infinity());
        base.push_back(n);
        forEachShard(G, [&](int g) { shard[(size_t) g]->load(rec + base[(size_t) g], base[(size_t) g + 1] - base[(size_t) g]); });
        if (n > 0) {
            firstTime = rec[0].t;
            lastTime = rec[n - 1].t;
        }
    }
    // the shard that holds every event of the closed window [first, second], or -1 if it straddles a cut
    int owner(double first, double second) const {
        const int g = (int) (std::upper_bound(cut.begin(), cut.end(), first) - cut.begin()) - 1;
        return second < cut[(size_t) g + 1] ? g : -1;
    }
};

class ShardedFrontEnd {
public:
    typedef FrontEnd::Params Params;
    ShardedFrontEnd(ShardedEventContainer::Ptr c, CirclePatternParameters::Ptr pattern, Params p) : c_(c) {
        for (auto &s : c->shard) fe_.emplace_back(new FrontEnd(s, pattern, p));
    }
    void run(const std::vector<std::pair<double, double>> &windows) {
        const int G = c_->shards();
        std::vector<std::vector<std::pair<double, double>>> sub((size_t) G);
        where_.assign(windows.size(), {0, 0});
        for (size_t w = 0; w < windows.size(); ++w) {
            const int g = c_->owner(windows[w].first, windows[w].second);
            if (g < 0) throw std::invalid_argument("window straddles two GPU shards (windows must lie inside one time piece)");
            where_[w] = {g, (int) sub[(size_t) g].size()};
            sub[(size_t) g].push_back(windows[w]);
        }
        forEachShard(G, [&](int g) {
            if (!sub[(size_t) g].empty()) fe_[(size_t) g]->run(sub[(size_t) g]);
        });
    }
    // summary in whole-stream event indices (point_offset stays shard-local)
    ecb_window_summary summary(size_t w) const {
        ecb_window_summary s = fe_[(size_t) where_[w].first]->summary((size_t) where_[w].second);
        s.ev_lo += c_->base[(size_t) where_[w].first];
        s.ev_hi += c_->base[(size_t) where_[w].first];
        return s;
    }
    int eventsNum(size_t w) const { return fe_[(size_t) where_[w].first]->eventsNum((size_t) where_[w].second); }
    std::vector<CalibCircleLite> candidates(size_t w) const { return fe_[(size_t) where_[w].first]->candidates((size_t) where_[w].second); }
    // rectifyFeatures over windows of the last run (FrontEnd::rectify), routed to the owning shards
    void rectify(const std::vector<int32_t> &window_index, int n_circles, const std::vector<double> &image_points, double inlier,
                 int rows, int cols, bool asymmetric, std::vector<double> &out, std::vector<int32_t> &verdict) {
        const int G = c_->shards();
        const size_t per = (size_t) n_circles * 10, per_out = (size_t) n_circles * 3;
        std::vector<std::vector<int32_t>> idx((size_t) G), local((size_t) G), v((size_t) G);
        std::vector<std::vector<double>> img((size_t) G), o((size_t) G);
        for (size_t i = 0; i < window_index.size(); ++i) {
            const auto &wh = where_[(size_t) window_index[i]];
            idx[(size_t) wh.first].push_back((int32_t) i);
            local[(size_t) wh.first].push_back(wh.second);
            img[(size_t) wh.first].insert(img[(size_t) wh.first].end(), image_points.begin() + i * per, image_points.begin() + (i + 1) * per);
        }
        forEachShard(G, [&](int g) {
            if (local[(size_t) g].empty()) return;
            fe_[(size_t) g]->rectify(local[(size_t) g], n_circles, img[(size_t) g], inlier, rows, cols, asymmetric, o[(size_t) g], v[(size_t) g]);
        });
        out.assign(window_index.size() * per_out, 0.0);
        verdict.assign(window_index.size(), 0);
        for (int g = 0; g < G; ++g)
            for (size_t k = 0; k < idx[(size_t) g].size(); ++k) {
                const size_t i = (size_t) idx[(size_t) g][k];
                std::copy(o[(size_t) g].begin() + k * per_out, o[(size_t) g].begin() + (k + 1) * per_out, out.begin() + i * per_out);
                verdict[i] = v[(size_t) g][k];
            }
    }
    int shards() const { return c_->shards(); }
    int width() const { return c_->width; }
    int height() const { return c_->height; }
    void windowPoints(size_t w, int pol, std::vector<Vec2> &xy, std::vector<int32_t> &labels) {
        fe_[(size_t) where_[w].first]->windowPoints((size_t) where_[w].second, pol, xy, labels);
    }
    void keptClusters(size_t w, int pol, std::vector<int32_t> &raw_id, std::vector<int32_t> &size, std::vector<int32_t> &median_pid) {
        fe_[(size_t) where_[w].first]->keptClusters((size_t) where_[w].second, pol, raw_id, size, median_pid);
    }

private:
    ShardedEventContainer::Ptr c_;
    std::vector<std::unique_ptr<FrontEnd>> fe_;
    std::vector<std::pair<int, int>> where_;  // window -> (shard, index in the shard's batch)
};

// EventCalibSpline over the shards: every GPU associates ITS events with all key frames and evaluates its residuals; the LM
// loop runs replicated on the devices (ecb_lm_device_*), the normal equations and candidate costs summed over NVLink inside
// the kernels.  One shard: the single-GPU EventCalibSpline (host state machine), unchanged.
class ShardedCalibSpline {
public:
    typedef EventCalibSpline::Segment Segment;
    typedef EventCalibSpline::KeyFrame KeyFrame;
    ShardedCalibSpline(ShardedEventContainer::Ptr events, std::vector<Segment> segments, std::array<double, 9> intrinsics,
                       double motionTimeStep, double circleRadius, bool useSO3 = false)
        : ev_(events), useSO3_(useSO3) {
        for (auto &s : events->shard) sp_.emplace_back(new EventCalibSpline(s, segments, intrinsics, motionTimeStep, circleRadius, useSO3));
        for (auto &s : segments) n_cp_.push_back((int32_t) (s.rot_cp.size() / 4));
    }
    // constant intrinsics (EventCalibSpline::setConstantIntrinsics) on every shard's context: every rank zeroes the same rows of
    // the same summed normal equations, so the replicated state machine and the covariance stay bit-identical across ranks
    int setConstantIntrinsics(uint32_t mask) {
        for (auto &s : sp_) {
            const int rc = s->setConstantIntrinsics(mask);
            if (rc != ECB_OK) return rc;
        }
        return ECB_OK;
    }
    int64_t associate(const std::vector<KeyFrame> &kf, const std::vector<std::array<double, 3>> &landmarks) {
        std::vector<int64_t> n(sp_.size(), 0);
        forEachShard((int) sp_.size(), [&](int g) { n[(size_t) g] = sp_[(size_t) g]->associate(kf, landmarks); });
        int64_t tot = 0;
        for (int64_t v : n) tot += v;
        return tot;
    }
    bool optimize(ecb_lm_summary *summary = nullptr) {
        const int G = (int) sp_.size();
        if (G == 1) return sp_[0]->optimize(summary);
        for (int g = 0; g < G; ++g)
            for (int h = 0; h < g; ++h)
                if (ev_->device[(size_t) g] == ev_->device[(size_t) h])
                    throw std::invalid_argument("ShardedCalibSpline::optimize: the shards must live on distinct devices");
        std::vector<double> rot, trans;  // from the current point: a second optimize() continues from the first solution
        EventCalibSpline::flatten(segments(), rot, trans);
        std::array<double, 9> intr = intrinsics();
        ecb_lm_options opt;
        ecb_lm_default_options(&opt);
        opt.rotation_model = useSO3_ ? 1 : 0;
        std::vector<ecb_lm_device *> lm((size_t) G, nullptr);
        std::vector<void *> buf((size_t) G, nullptr);
        auto ctx = [&](int g) { return ev_->shard[(size_t) g]->ctx; };
        bool ok = true;
        ecb_lm_summary sum;
        std::memset(&sum, 0, sizeof sum);
        try {
            for (int g = 0; g < G; ++g) {
                for (int h = 0; h < G; ++h)
                    if (h != g && ecb_enable_peer_access(ctx(g), ev_->device[(size_t) h]) != ECB_OK) throw std::runtime_error(ecb_last_error(ctx(g)));
                if (ecb_device_alloc(ctx(g), ecb_exchange_buffer_bytes(ctx(g), G), &buf[(size_t) g]) != ECB_OK)
                    throw std::runtime_error(ecb_last_error(ctx(g)));
            }
            for (int g = 0; g < G; ++g) {
                if (ecb_lm_device_create(ctx(g), (int) n_cp_.size(), n_cp_.data(), &opt, &lm[(size_t) g]) != ECB_OK ||
                    ecb_lm_device_set_exchange(lm[(size_t) g], g, G, buf.data()) != ECB_OK)
                    throw std::runtime_error(ecb_last_error(ctx(g)));
            }
            // every GPU's whole loop is enqueued by its own host thread; the kernels wait for each other over the peer buffers
            std::vector<std::vector<double>> r((size_t) G, rot), t((size_t) G, trans);
            std::vector<std::array<double, 9>> in((size_t) G, intr);
            std::vector<ecb_lm_summary> sm((size_t) G);
            forEachShard(G, [&](int g) {
                if (ecb_calibrate_device(lm[(size_t) g], in[(size_t) g].data(), r[(size_t) g].data(), t[(size_t) g].data(), &sm[(size_t) g], nullptr, 0) != ECB_OK)
                    throw std::runtime_error(ecb_last_error(ctx(g)));
            });
            for (int g = 1; g < G; ++g)  // replicated state machine: bit-identical on every rank
                if (in[(size_t) g] != in[0] || r[(size_t) g] != r[0] || t[(size_t) g] != t[0])
                    throw std::runtime_error("multi-GPU LM: the ranks' results differ");
            sum = sm[0];
            result_intr_ = in[0];
            result_rot_ = r[0];
            result_trans_ = t[0];
        } catch (...) {
            ok = false;
            cleanup(lm, buf);
            throw;
        }
        cleanup(lm, buf);
        if (summary) *summary = sum;
        // write the solution back into the segments
        seg_ = segments();
        size_t ro = 0, to = 0;
        for (auto &s : seg_) {
            std::copy(result_rot_.begin() + ro, result_rot_.begin() + ro + s.rot_cp.size(), s.rot_cp.begin());
            std::copy(result_trans_.begin() + to, result_trans_.begin() + to + s.trans_cp.size(), s.trans_cp.begin());
            ro += s.rot_cp.size();
            to += s.trans_cp.size();
        }
        solved_ = true;
        return ok;
    }
    // Covariance at the current point (EventCalibSpline::covariance).  Several GPUs: the normal equations are summed over the
    // shards by the exchange into a device buffer on every shard, and every shard factorises and inverts the same sum; the ranks'
    // results are bit-identical (checked), rank 0's is returned.
    int covariance(EventCalibSpline::Covariance &out) {
        const int G = (int) sp_.size();
        if (G == 1) return EventCalibSpline::covarianceAt(ev_->shard[0]->ctx, n_cp_, intrinsics(), segments(), nullptr, 0, out);
        auto ctx = [&](int g) { return ev_->shard[(size_t) g]->ctx; };
        std::vector<double> rot, trans;
        EventCalibSpline::flatten(segments(), rot, trans);
        const std::array<double, 9> intr = intrinsics();
        std::vector<void *> buf((size_t) G, nullptr), packed((size_t) G, nullptr);
        std::vector<EventCalibSpline::Covariance> cov((size_t) G);
        std::vector<int> rc((size_t) G, ECB_OK);
        int64_t n_total = 0;
        auto release = [&]() {
            for (int g = 0; g < G; ++g) {
                ecb_synchronize(ctx(g));
                if (buf[(size_t) g]) ecb_device_free(ctx(g), buf[(size_t) g]);
                if (packed[(size_t) g]) ecb_device_free(ctx(g), packed[(size_t) g]);
            }
        };
        try {
            for (int g = 0; g < G; ++g) {
                int64_t nr = 0, nd = 0;
                if (ecb_cost_layout(ctx(g), nullptr, nullptr, &nr, &nd) != ECB_OK) throw std::runtime_error(ecb_last_error(ctx(g)));
                n_total += nr;
                for (int h = 0; h < G; ++h)
                    if (h != g && ecb_enable_peer_access(ctx(g), ev_->device[(size_t) h]) != ECB_OK) throw std::runtime_error(ecb_last_error(ctx(g)));
                if (ecb_device_alloc(ctx(g), ecb_exchange_buffer_bytes(ctx(g), G), &buf[(size_t) g]) != ECB_OK ||
                    ecb_device_alloc(ctx(g), (size_t) nd * 8, &packed[(size_t) g]) != ECB_OK)
                    throw std::runtime_error(ecb_last_error(ctx(g)));
            }
            forEachShard(G, [&](int g) {  // the receive side waits for the peers: one host thread per shard
                if (ecb_cost_normal_eq_exchange(ctx(g), intr.data(), rot.data(), trans.data(), g, G, buf.data(), 1, ECB_EXCHANGE_BOTH,
                                                packed[(size_t) g], nullptr) != ECB_OK ||
                    ecb_synchronize(ctx(g)) != ECB_OK)
                    throw std::runtime_error(ecb_last_error(ctx(g)));
                rc[(size_t) g] = EventCalibSpline::covarianceAt(ctx(g), n_cp_, intr, segments(), packed[(size_t) g], n_total, cov[(size_t) g]);
                if (rc[(size_t) g] < 0) throw std::runtime_error(ecb_last_error(ctx(g)));
            });
        } catch (...) {
            release();
            throw;
        }
        release();
        for (int g = 1; g < G; ++g)
            if (rc[(size_t) g] != rc[0] || cov[(size_t) g].intrinsics != cov[0].intrinsics || cov[(size_t) g].band != cov[0].band ||
                cov[(size_t) g].cross != cov[0].cross)
                throw std::runtime_error("multi-GPU covariance: the ranks' results differ");
        out = cov[0];
        return rc[0];
    }
    // Pose covariance (EventCalibSpline::poseCovariance) after covariance(): every rank holds the same Z bit for bit, rank 0's
    // context answers.
    int poseCovariance(const std::vector<double> &times, std::vector<double> &pose, std::vector<double> &cov,
                       int64_t *n_valid = nullptr) const {
        return EventCalibSpline::poseCovarianceAt(ev_->shard[0]->ctx, times, pose, cov, n_valid);
    }
    // Motion of the trajectory at the current control points (EventCalibSpline::trajectoryMotion) and, after covariance(), with
    // its covariance (EventCalibSpline::motionCovariance): rank 0's context answers.
    int trajectoryMotion(const std::vector<double> &times, std::vector<double> &motion, int64_t *n_valid = nullptr) const {
        return EventCalibSpline::trajectoryMotionAt(ev_->shard[0]->ctx, segments(), times, motion, n_valid);
    }
    int motionCovariance(const std::vector<double> &times, std::vector<double> &motion, std::vector<double> &cov,
                         int64_t *n_valid = nullptr) const {
        return EventCalibSpline::motionCovarianceAt(ev_->shard[0]->ctx, times, motion, cov, n_valid);
    }
    // Camera-gyroscope calibration at the current control points (EventCalibSpline::calibrateGyroscope): rank 0's context answers.
    int calibrateGyroscope(const std::vector<double> &gyro, double maxOffset, int nOffsets, ecb_gyro_calibration &result,
                           std::vector<double> *offsetCost = nullptr, std::vector<double> *residuals = nullptr) const {
        return EventCalibSpline::calibrateGyroscopeAt(ev_->shard[0]->ctx, segments(), gyro, maxOffset, nOffsets, result, offsetCost,
                                                      residuals);
    }
    // Residual statistics at the current point (EventCalibSpline::residualGroups): every shard reports its own records (one host
    // thread each), the groups are combined in rank order (counts and sums added, max_abs the max).
    int residualGroups(int by, int cellPx, std::vector<ecb_residual_group> &groups, ecb_residual_group *total) const {
        return combineGroups(EventCalibSpline::residualGroupsAt, EventCalibSpline::accumulateResidualGroup, by, cellPx, groups, total);
    }
    // Outlier rejection at the current point: the shards' statistics per key frame combined in rank order (residualGroups), the
    // policy applied once on the host (ecb::outlierRejection with factor k), then every shard removes its records with the same
    // threshold and key-frame mask (EventCalibSpline::rejectResiduals, one host thread each), so the kept records do not depend
    // on the sharding.  Outputs (each may be null): scale s, threshold k s, the mask, and the kept / removed records of all shards.
    int rejectOutliers(double k, double *scale, double *threshold, std::vector<uint8_t> *drop, int64_t *kept, int64_t *removed) {
        std::vector<ecb_residual_group> byKf;
        int rc0 = residualGroups(ECB_RESIDUALS_BY_KEYFRAME, 16, byKf, nullptr);
        if (rc0 != ECB_OK) return rc0;
        double t = 0.0;
        std::vector<uint8_t> mask;
        const double s = ecb::outlierRejection(byKf, k, &t, &mask);
        const int G = (int) sp_.size();
        std::vector<int64_t> kp((size_t) G, 0), rm((size_t) G, 0);
        std::vector<int> rc((size_t) G, ECB_OK);
        forEachShard(G, [&](int g) {
            rc[(size_t) g] = EventCalibSpline::rejectResidualsAt(ev_->shard[(size_t) g]->ctx, intrinsics(), segments(),
                                                                 sp_[(size_t) g]->keyframeTimes(), t, mask, &kp[(size_t) g],
                                                                 &rm[(size_t) g]);
        });
        for (int g = 0; g < G; ++g)
            if (rc[(size_t) g] != ECB_OK) return rc[(size_t) g];
        int64_t nk = 0, nr = 0;
        for (int g = 0; g < G; ++g) nk += kp[(size_t) g], nr += rm[(size_t) g];
        if (scale) *scale = s;
        if (threshold) *threshold = t;
        if (drop) *drop = mask;
        if (kept) *kept = nk;
        if (removed) *removed = nr;
        return ECB_OK;
    }
    // Re-association at the current point (EventCalibSpline::reassociate): every shard re-associates its own events (one host
    // thread each); the counts are summed in rank order.
    int reassociate(double gatePx, double maxDt, EventCalibSpline::ReassociationCounts *counts) {
        const int G = (int) sp_.size();
        std::vector<EventCalibSpline::ReassociationCounts> part((size_t) G);
        std::vector<int> rc((size_t) G, ECB_OK);
        forEachShard(G, [&](int g) {
            rc[(size_t) g] = EventCalibSpline::reassociateAt(ev_->shard[(size_t) g]->ctx, intrinsics(), segments(), gatePx, maxDt,
                                                             &part[(size_t) g]);
        });
        for (int g = 0; g < G; ++g)
            if (rc[(size_t) g] != ECB_OK) return rc[(size_t) g];
        EventCalibSpline::ReassociationCounts t;
        for (const auto &p : part) {
            t.residuals += p.residuals;
            t.same += p.same;
            t.changed += p.changed;
            t.added += p.added;
            t.lost += p.lost;
        }
        if (counts) *counts = t;
        return ECB_OK;
    }
    // Reprojection statistics in pixels (EventCalibSpline::reprojectionGroups), combined as residualGroups
    int reprojectionGroups(int by, int cellPx, std::vector<ecb_reprojection_group> &groups, ecb_reprojection_group *total) const {
        return combineGroups(EventCalibSpline::reprojectionGroupsAt, EventCalibSpline::accumulateReprojectionGroup, by, cellPx, groups,
                             total);
    }
    // Key-frame centres reprojected (EventCalibSpline::keyframeReprojection): they read no records, rank 0's context answers
    int keyframeReprojection(std::vector<double> &proj, std::vector<double> &err, ecb_reprojection_group *total) const {
        return EventCalibSpline::keyframeReprojectionAt(ev_->shard[0]->ctx, intrinsics(), segments(), sp_[0]->keyframeTimes(),
                                                        sp_[0]->keyframeCircles(), sp_[0]->landmarks(), proj, err, total);
    }
    const std::array<double, 9> &intrinsics() const { return solved_ ? result_intr_ : sp_[0]->intrinsics(); }
    const std::vector<Segment> &segments() const { return solved_ ? seg_ : sp_[0]->segments(); }
    int saveKeyFrameTrajectoryTUM(const std::string &filename, const std::vector<double> &keyframeStamps) const {
        return EventCalibSpline::saveKeyFrameTrajectoryTUM(segments(), useSO3_, filename, keyframeStamps);
    }
    const char *lastError() const { return ecb_last_error(ev_->shard[0]->ctx); }

private:
    // the groups of one report, every shard its own records (at: EventCalibSpline::residualGroupsAt or reprojectionGroupsAt, one
    // host thread each), combined in rank order by add
    template <class Group, class At, class Add>
    int combineGroups(At at, Add add, int by, int cellPx, std::vector<Group> &groups, Group *total) const {
        const int G = (int) sp_.size();
        std::vector<std::vector<Group>> part((size_t) G);
        std::vector<Group> tot((size_t) G);
        std::vector<int> rc((size_t) G, ECB_OK);
        forEachShard(G, [&](int g) {
            rc[(size_t) g] = at(ev_->shard[(size_t) g]->ctx, intrinsics(), segments(), sp_[(size_t) g]->keyframeTimes(), by, cellPx,
                                part[(size_t) g], &tot[(size_t) g]);
        });
        for (int g = 0; g < G; ++g)
            if (rc[(size_t) g] != ECB_OK) return rc[(size_t) g];
        groups = part[0];
        Group t = tot[0];
        for (int g = 1; g < G; ++g) {
            for (size_t i = 0; i < groups.size(); ++i) add(groups[i], part[(size_t) g][i]);
            add(t, tot[(size_t) g]);
        }
        if (total) *total = t;
        return ECB_OK;
    }
    void cleanup(std::vector<ecb_lm_device *> &lm, std::vector<void *> &buf) {
        for (size_t g = 0; g < lm.size(); ++g) {
            if (lm[g]) ecb_lm_device_destroy(lm[g]);
            if (buf[g]) {
                ecb_synchronize(ev_->shard[g]->ctx);
                ecb_device_free(ev_->shard[g]->ctx, buf[g]);
            }
        }
    }
    ShardedEventContainer::Ptr ev_;
    std::vector<std::unique_ptr<EventCalibSpline>> sp_;
    std::vector<int32_t> n_cp_;
    bool useSO3_ = false, solved_ = false;
    std::array<double, 9> result_intr_{};
    std::vector<double> result_rot_, result_trans_;
    std::vector<Segment> seg_;
};

}  // namespace opengv2
#endif  // ECB_MULTI_GPU_HPP
