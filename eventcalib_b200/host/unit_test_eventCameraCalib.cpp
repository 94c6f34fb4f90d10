// unit_test_eventCameraCalib settingFilePath binFilePath SavePath
//
// Drop-in for the reference CLI (ECC/test/eventCameraCalib.cpp:104-233): same 3 positional arguments, same usage / exit
// codes, same `parameter/event_calibration/example.yaml` keys, same stdout lines ("Events from ... loaded.", "N frames in
// Map.", "Frame t contain n events.", the calibrateCamera report, "N frames in Map after Initialization.", the intrinsics
// before / after the optimisation) and the same SavePath/TrajectoryByEvent.txt — with the window loop running as ONE batched
// GPU launch per lattice instead of hardware_concurrency()-2 CPU threads, rectifyFeatures batched over all key frames, and the
// spline optimisation's residuals / Jacobians / normal equations on the GPU.  Headless (the reference opens a Pangolin
// viewer, :129).  SavePath/image/<timestamp>.png holds every key frame's debug image like :214-227 (cluster colours, medians,
// candidate and rectified circles; include/ecb/image_lite.hpp — ECB_NO_IMAGES=1 skips them).
//
// The window loop is the reference's adaptive one (accept -> jump by length + 5 steps, else grow by one step until the
// window holds FrameEventNumThreshold events or exceeds 3 lengths, then slide; :49-81) over the reference's time pieces.
// A window becomes a key frame when the candidate circles are found, ordered as the rows x cols grid, and pass the tracking
// gate (EventCalibIni::track: row directions vs the neighbouring key frame; the reference's worker threads race on the
// shared map, here the pieces of one round are gated in piece order).  The initialisation (EventCalibIni::cvCalibration)
// runs without OpenCV (include/ecb/calib_init.hpp); the ordered circles of the key frames are also written to
// SavePath/candidates.txt.
//
// Several GPUs (ECB_DEVICES, default: all visible): the reference's time pieces are dealt out to the GPUs in contiguous blocks,
// every GPU holds the records of its block, one host thread + context per GPU (include/ecb/multi_gpu.hpp); the spline
// optimisation shards the residuals the same way and sums the normal equations over NVLink inside the kernels.  The frames,
// candidates and key-frame map do not depend on the number of GPUs.
//
// ECB_CONSTANT_INTRINSICS=k3,k4,k5 (comma- or space-separated names of fx fy cx cy k1 .. k5; k1 .. k5 are the spline stage's
// inverse radial polynomial, not the YAML's Fix_K* OpenCV coefficients) holds those intrinsics at their initial values in the
// spline optimisation, which the reference does not offer: it prints a "Constant intrinsics:" line before the optimisation, and
// the covariance files (ECB_COVARIANCE, ECB_TRAJECTORY_COVARIANCE) are conditional on them.  An unknown name, or the variable
// together with ECB_REFERENCE_SIGNATURES (the reference's constructor frees all nine), ends the program with exit code 1.
//
// ECB_RESIDUALS=1 reports how well the model fits after the optimisation, which the reference does not: a "Residuals:" line (count,
// RMS, mean, max |r|, down-weighted share) and SavePath/ResidualsByKeyframe.txt, ResidualsByCircle.txt and ResidualMap.txt
// (statistics per key frame, per board circle and per sensor cell of ECB_RESIDUAL_CELL pixels, default 16).  r is the raw
// residual ||X_w - L|| - circleRadius, a distance on the board plane in the units of the board points, not pixels.  A cell size
// that is not a positive integer ends the program with exit code 1 before any GPU work.
//
// ECB_REJECT=k (a positive finite number) rejects outliers after the first optimisation, which the reference does not: the
// statistics per key frame give s, the lower median of the key frames' RMS residuals; the key frames whose RMS exceeds k s and the
// records with |r| > k s are removed (ecb::outlierRejection), an "Outlier rejection:" line is printed, and the optimisation runs
// again from the first solution on the kept records ("Solver Summary (after rejection):").  The intrinsics, the trajectory and
// every report and covariance file then describe the second solve.  An invalid value, or the variable together with
// ECB_REFERENCE_SIGNATURES, ends the program with exit code 1 before any GPU work.
//
// ECB_REASSOCIATE=n (a positive integer, at most 1000) refines the association after the first optimisation, which the
// reference does not: n rounds, each re-associating every event near a key frame with the board circle nearest to its
// back-projection at its own pose on the current spline (kept when its event-to-rim error is below 5 px, the association's
// tolerance), printing a "Re-association r:" line with the record counts against the previous records, and optimising again from the current solution
// ("Solver Summary (after re-association r):").  ECB_REJECT then applies after the last round; the intrinsics, the trajectory and
// every report and covariance file describe the final solve.  An invalid value, or the variable together with
// ECB_REFERENCE_SIGNATURES, ends the program with exit code 1 before any GPU work.
//
// ECB_REPROJECTION=1 reports the same fit in pixels after the optimisation, through the forward camera model: a "Reprojection:"
// line (event-to-rim count, RMS, mean, max |e|, invalid count; key-frame-centre count and RMS; rho_fold * fx next to the farthest
// sensor corner's distorted radius, in pixels) and SavePath/ReprojectionByKeyframe.txt, ReprojectionByCircle.txt and
// ReprojectionMap.txt (cells of ECB_RESIDUAL_CELL pixels).
//
// ECB_TRAJECTORY_MOTION=rate (Hz, a positive finite number) samples the motion of the final trajectory, which the reference does
// not: SavePath/TrajectoryMotion.txt has one line per stamp t0 + k / rate from the first knot of the first segment to the last
// knot of the last (stamps in the gaps between segments are skipped): the stamp, the body-frame angular velocity, the world-frame
// velocity and acceleration, then their 9 standard deviations sqrt(sigma2 Sigma_m,ii) (NaN when the covariance is rank
// deficient).  A "Trajectory motion:" line gives the sample count, the rate, max |omega| and max |v|.  An invalid value ends the
// program with exit code 1 before any file or GPU work.
//
// ECB_GYRO=path calibrates a gyroscope against the final trajectory, which the reference does not.  The file has one sample per
// line, "t wx wy wz" (s, rad/s; further columns, e.g. an accelerometer, are ignored; lines starting with '#' and blank lines are
// skipped).  ECB_GYRO_MAX_OFFSET=seconds (finite, >= 0, default 0.05) bounds the time offset, scanned on 1001 points (held at 0
// when it is 0).  The model is w_g = R_gc w_c(t + offset) + bias (ecb_gyro_calibrate).  SavePath/CameraGyroscope.txt gets the
// estimate, its standard deviations and the scan curve, and a "Camera-gyroscope:" line is printed.  A failed calibration (too
// few samples, the offset at the edge of the search window, rotation about one axis only) is reported on stderr and writes no
// file.  A missing or malformed file, or an invalid offset, ends the program with exit code 1 before any file or GPU work.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <map>
#include <sstream>
#include <string>
#include <sys/stat.h>
#include <thread>
#include <vector>

#include "../../include/ecb/multi_gpu.hpp"

using namespace opengv2;

// the subset of OpenCV FileStorage YAML 1.0 the reference's config uses: `key: scalar` and `key: [ a, b, ... ]`
struct Settings {
    std::map<std::string, std::string> kv;
    bool open(const std::string &path) {
        std::ifstream is(path);
        if (!is.is_open()) return false;
        std::string line;
        while (std::getline(is, line)) {
            const size_t h = line.find('#');
            if (h != std::string::npos) line = line.substr(0, h);
            if (line.rfind("%YAML", 0) == 0 || line.rfind("---", 0) == 0) continue;
            const size_t c = line.find(':');
            if (c == std::string::npos) continue;
            auto trim = [](std::string s) {
                const char *ws = " \t\r\n\"";
                const size_t b = s.find_first_not_of(ws);
                if (b == std::string::npos) return std::string();
                return s.substr(b, s.find_last_not_of(ws) - b + 1);
            };
            const std::string k = trim(line.substr(0, c)), v = trim(line.substr(c + 1));
            if (!k.empty()) kv[k] = v;
        }
        return true;
    }
    bool has(const std::string &k) const { return kv.count(k) && !kv.at(k).empty(); }
    double num(const std::string &k, double dflt = 0) const { return has(k) ? atof(kv.at(k).c_str()) : dflt; }
};

int main(int argc, char **argv) {
    if (argc != 4) {
        std::cerr << std::endl << "Usage: ./unit_test_eventCameraCalib settingFilePath binFilePath SavePath" << std::endl;
        return 1;
    }
    std::cout.precision(8);
    uint32_t constIntrinsics = 0;  // checked before any file or GPU work
    if (const char *ci = getenv("ECB_CONSTANT_INTRINSICS")) {
        if (getenv("ECB_REFERENCE_SIGNATURES")) {
            std::cerr << "ecb: ECB_CONSTANT_INTRINSICS cannot be combined with ECB_REFERENCE_SIGNATURES (the reference's "
                         "EventCalibSpline frees all 9 intrinsics)" << std::endl;
            return 1;
        }
        std::string unknown;
        const int m = ecb::constantIntrinsicsMask(ci, &unknown);
        if (m < 0) {
            std::cerr << "ecb: ECB_CONSTANT_INTRINSICS: unknown intrinsic '" << unknown << "' (names: fx fy cx cy k1 k2 k3 k4 k5)"
                      << std::endl;
            return 1;
        }
        constIntrinsics = (uint32_t) m;
    }
    double rejectK = 0.0;  // checked before any file or GPU work; 0: no outlier rejection
    if (const char *rk = getenv("ECB_REJECT")) {
        if (getenv("ECB_REFERENCE_SIGNATURES")) {
            std::cerr << "ecb: ECB_REJECT cannot be combined with ECB_REFERENCE_SIGNATURES (the reference's EventCalibSpline "
                         "optimises once on every residual)" << std::endl;
            return 1;
        }
        char *end = nullptr;
        const double v = strtod(rk, &end);
        if (end == rk || *end != '\0' || !(v > 0.0) || !std::isfinite(v)) {
            std::cerr << "ecb: ECB_REJECT must be a positive finite number (the factor k of the threshold k s), got '" << rk << "'"
                      << std::endl;
            return 1;
        }
        rejectK = v;
    }
    int reassociateRounds = 0;  // checked before any file or GPU work; 0: no re-association
    if (const char *ra = getenv("ECB_REASSOCIATE")) {
        if (getenv("ECB_REFERENCE_SIGNATURES")) {
            std::cerr << "ecb: ECB_REASSOCIATE cannot be combined with ECB_REFERENCE_SIGNATURES (the reference's EventCalibSpline "
                         "associates once, from the detected circles)" << std::endl;
            return 1;
        }
        char *end = nullptr;
        const long v = strtol(ra, &end, 10);
        if (end == ra || *end != '\0' || v < 1 || v > 1000) {
            std::cerr << "ecb: ECB_REASSOCIATE must be a positive integer (rounds, at most 1000), got '" << ra << "'" << std::endl;
            return 1;
        }
        reassociateRounds = (int) v;
    }
    int residualCell = 16;  // checked before any file or GPU work
    if (const char *rc = getenv("ECB_RESIDUAL_CELL")) {
        char *end = nullptr;
        const long v = strtol(rc, &end, 10);
        if (end == rc || *end != '\0' || v < 1 || v > 32767) {
            std::cerr << "ecb: ECB_RESIDUAL_CELL must be a positive integer (pixels), got '" << rc << "'" << std::endl;
            return 1;
        }
        residualCell = (int) v;
    }
    double motionRate = 0.0;  // checked before any file or GPU work; 0: no motion file
    if (const char *mr = getenv("ECB_TRAJECTORY_MOTION")) {
        char *end = nullptr;
        const double v = strtod(mr, &end);
        if (end == mr || *end != '\0' || !(v > 0.0) || !std::isfinite(v)) {
            std::cerr << "ecb: ECB_TRAJECTORY_MOTION must be a positive finite number (samples per second), got '" << mr << "'"
                      << std::endl;
            return 1;
        }
        motionRate = v;
    }
    std::vector<double> gyro;  // t wx wy wz per sample; read and checked before any file or GPU work
    double gyroMaxOffset = 0.05;
    if (const char *gp = getenv("ECB_GYRO")) {
        if (const char *mo = getenv("ECB_GYRO_MAX_OFFSET")) {
            char *end = nullptr;
            const double v = strtod(mo, &end);
            if (end == mo || *end != '\0' || !(v >= 0.0) || !std::isfinite(v)) {
                std::cerr << "ecb: ECB_GYRO_MAX_OFFSET must be a finite number >= 0 (seconds), got '" << mo << "'" << std::endl;
                return 1;
            }
            gyroMaxOffset = v;
        }
        std::ifstream gf(gp);
        if (!gf.is_open()) {
            std::cerr << "ecb: ECB_GYRO: cannot open '" << gp << "'" << std::endl;
            return 1;
        }
        std::string line;
        for (long no = 1; std::getline(gf, line); ++no) {
            const size_t b = line.find_first_not_of(" \t\r");
            if (b == std::string::npos || line[b] == '#') continue;
            std::istringstream ls(line);
            double v[4];
            if (!(ls >> v[0] >> v[1] >> v[2] >> v[3])) {
                std::cerr << "ecb: ECB_GYRO: line " << no << " of '" << gp << "' is not \"t wx wy wz\" (4 numbers)" << std::endl;
                return 1;
            }
            gyro.insert(gyro.end(), v, v + 4);
        }
    }
    Settings fs;
    if (!fs.open(argv[1])) {
        std::cerr << "Failed to open settings file at: " << argv[1] << std::endl;
        exit(-1);
    }
    auto pattern = std::make_shared<CirclePatternParameters>();
    pattern->cols = (int) fs.num("BoardSize_Cols", 4);
    pattern->rows = (int) fs.num("BoardSize_Rows", 9);
    pattern->squareSize = fs.num("Square_Size", 5.5);
    pattern->isAsymmetric = fs.num("Is_Pattern_Asymmetric", 1) != 0;
    pattern->circleRadius = fs.num("Circles_Radius", 1.75);
    CalibrationSetting setting;  // parameters.hpp:32-46
    setting.circlePatternParameters = pattern;
    setting.aspectRatio = (float) fs.num("Calibrate_FixAspectRatio", 1);
    setting.calibZeroTangentDist = fs.num("Calibrate_AssumeZeroTangentialDistortion", 1) != 0;
    setting.calibFixPrincipalPoint = fs.num("Calibrate_FixPrincipalPointAtTheCenter", 1) != 0;
    setting.useFisheye = fs.num("Calibrate_UseFisheyeModel", 0) != 0;
    setting.fixK1 = fs.num("Fix_K1", 0) != 0;
    setting.fixK2 = fs.num("Fix_K2", 0) != 0;
    setting.fixK3 = fs.num("Fix_K3", 0) != 0;
    setting.fixK4 = fs.num("Fix_K4", 1) != 0;
    setting.fixK5 = fs.num("Fix_K5", 1) != 0;
    setting.NumOfFrameToUse = (int) fs.num("Calibrate_NrOfFrameToUse", 200);
    const double motionTimeStep = fs.num("MotionTimeStep");
    const int width = (int) fs.num("Camera.width"), height = (int) fs.num("Camera.height");
    if (!(motionTimeStep > 0) || width <= 0 || height <= 0) {
        std::cerr << "settings: MotionTimeStep / Camera.width / Camera.height missing" << std::endl;
        exit(-1);
    }

    // load: keep t >= StartTime, stop at the first t >= EndTime (eventCameraCalib.cpp:154-163)
    std::ifstream is(argv[2], std::ifstream::binary | std::ifstream::in);
    if (!is.is_open()) {
        std::cerr << "No such file: " << argv[2] << std::endl;  // EventStream ctor throws invalid_argument (EventStream.cpp:15)
        return 1;
    }
    is.seekg(0, std::ios::end);
    const int64_t n_all = (int64_t) is.tellg() / 25;
    is.seekg(0);
    std::vector<EventRecord> rec((size_t) n_all);
    is.read((char *) rec.data(), n_all * 25);
    const bool customEnd = fs.has("EndTime");
    const double startTime = fs.num("StartTime");
    double endTime = fs.num("EndTime");
    int64_t b = 0, e = n_all;
    while (b < n_all && rec[(size_t) b].t < startTime) ++b;
    if (customEnd)
        for (e = b; e < n_all && rec[(size_t) e].t < endTime; ++e) {}
    if (e <= b) {
        std::cerr << "no events in [StartTime, EndTime)" << std::endl;
        return 1;
    }
    // the reference sets endTime to the last loaded stamp (:165) and cuts [startTime, endTime] into its time pieces (:172-180)
    endTime = rec[(size_t) e - 1].t;

    FrontEnd::Params params;
    params.dbscan_eps = fs.num("dbscan_eps", 4);
    params.dbscan_startMinSample = (int) fs.num("dbscan_startMinSample", 2);
    params.clusterMinSample = (int) fs.num("clusterMinSample", 5);
    params.knn_num = (int) fs.num("knn_num", 3);
    params.fitCircle = fs.num("fitCircle", 0) != 0;
    // The reference's adaptive window loop (MultiProcess::process, eventCameraCalib.cpp:34-97) over its time pieces (:172-180),
    // run as a wavefront: every round evaluates the CURRENT window of every unfinished piece in one batched GPU call, then
    // each piece applies the reference's accept / grow / slide rule to its own result.  The pieces are independent, so the
    // frames found are those of the reference run with one worker per piece.  pieceNum = 5 * (hardware_concurrency() - 2)
    // like the reference (:172-174), or ECB_PIECES.
    const double len = 3 * motionTimeStep, frameGap = 5 * motionTimeStep;
    const int frameEventNumThreshold = (int) fs.num("FrameEventNumThreshold", 4000);
    int pieceNum = 5 * std::max(1, (int) std::thread::hardware_concurrency() - 2);
    if (getenv("ECB_PIECES")) pieceNum = std::max(1, atoi(getenv("ECB_PIECES")));
    const double pstep = (endTime - startTime) / pieceNum;
    struct Piece {
        double lo, hi, first, second;
        bool done;
    };
    std::vector<Piece> pieces;
    for (int k = 0; k < pieceNum; ++k) {
        Piece pc{endTime - pstep * (k + 1), endTime - pstep * k, 0, 0, false};
        pc.first = pc.lo;
        pc.second = pc.lo + len;
        pc.done = !(pc.second < pc.hi);
        pieces.push_back(pc);
    }
    typedef EventCalibIni::KeyFrame Frame;
    std::map<double, Frame> frames;  // MapBase keeps key frames ordered by time stamp
    // GPUs: contiguous blocks of pieces (piece k covers [endTime - (k+1) pstep, endTime - k pstep): ascending time = descending k)
    std::vector<int> devices = ecbDevices();
    if ((int) devices.size() > pieceNum) devices.resize((size_t) pieceNum);
    const int G = (int) devices.size();
    std::vector<double> cuts;
    for (int g = 1; g < G; ++g) cuts.push_back(pieces[(size_t) (pieceNum - (int) ((int64_t) g * pieceNum / G))].hi);
    ShardedEventContainer::Ptr container;
    try {
        container = std::make_shared<ShardedEventContainer>(devices, width, height);
        container->load(rec.data() + b, e - b, cuts);
    } catch (const std::exception &ex) {
        std::cerr << "ecb: " << ex.what() << std::endl;
        return 1;
    }
    std::cout << "Events from " << startTime << " second to " << endTime << " second loaded." << std::endl;
    ShardedFrontEnd fe(container, pattern, params);
    TrackingGate gate(pattern->rows, pattern->cols, motionTimeStep);  // EventCalibIni::track; pieces of one round in piece order
    size_t rounds = 0, evaluated = 0;
    for (;;) {
        std::vector<std::pair<double, double>> windows;
        std::vector<int> owner;
        for (int k = 0; k < pieceNum; ++k)
            if (!pieces[(size_t) k].done) {
                windows.emplace_back(pieces[(size_t) k].first, pieces[(size_t) k].second);
                owner.push_back(k);
            }
        if (windows.empty()) break;
        try {
            fe.run(windows);
        } catch (const std::exception &ex) {
            std::cerr << "ecb: " << ex.what() << std::endl;
            return 1;
        }
        ++rounds;
        evaluated += windows.size();
        for (size_t w = 0; w < windows.size(); ++w) {
            Piece &pc = pieces[(size_t) owner[w]];
            const int events_num = fe.eventsNum(w);
            // extractFeatures() (:56): candidate circles found AND ordered by the grid finder (findCirclesGrid, :332-356), then
            // the tracking gate (tracking->process, :60 -> EventCalibIni::track)
            std::vector<CalibCircleLite> c;
            const double ts0 = (pc.first + pc.second) / 2;
            if (CirclesEventFrame::orderFeatures(fe.candidates(w), *pattern, c) && gate.process(ts0, c)) {  // :56-60
                const double ts = (pc.first + pc.second) / 2;  // Bodyframe time stamp (:57)
                Frame f;
                f.timeStamp = ts;
                f.duration = {pc.first, pc.second};
                f.eventsNum = events_num;
                f.features = c;
                frames.emplace(ts, f);  // MapBase::addFrame through TrackingBase (an existing stamp is kept)
                pc.first = pc.second + frameGap;  // :60-62
                pc.second = pc.first + len;
            } else if (events_num > frameEventNumThreshold || (pc.second - pc.first) > 3 * len) {  // :66-68,75-77
                pc.first += motionTimeStep;
                pc.second = pc.first + len;
            } else {
                pc.second += motionTimeStep;  // :70,79
            }
            pc.done = !(pc.second < pc.hi);  // :50
        }
    }
    mkdir(argv[3], 0755);
    std::ofstream out(std::string(argv[3]) + "/candidates.txt");
    out.precision(17);
    std::cout << frames.size() << " frames in Map." << std::endl;
    for (const auto &kv : frames) {
        const Frame &f = kv.second;
        std::cout << "Frame " << f.timeStamp << " contain " << f.eventsNum << " events." << std::endl;
        for (size_t k = 0; k < f.features.size(); ++k)
            out << f.timeStamp << " " << k << " " << f.features[k].center[0] << " " << f.features[k].center[1] << " "
                << f.features[k].radius << "\n";
    }
    out.close();
    std::cerr << evaluated << " windows evaluated on " << G << " GPU(s) in " << rounds << " batched rounds over " << pieceNum
              << " time pieces" << std::endl;

    // EventCalibIni::cvCalibration (eventCameraCalib.cpp:199): intrinsics, frame poses, checkPose, rectifyFeatures
    EventCalibIni ini(setting, motionTimeStep, width, height);
    bool ok = false;
    try {
        ok = ini.cvCalibration(fe, frames, std::cout);
    } catch (const std::exception &ex) {
        std::cerr << "ecb: " << ex.what() << std::endl;
        return 1;
    }
    std::cout << frames.size() << " frames in Map after Initialization." << std::endl;

    // EventCalibSpline (eventCameraCalib.cpp:203-210): the constructor throws std::logic_error like the reference's
    const bool useSO3 = fs.num("useSO3", 0) != 0;
    if (!ok) {
        std::cerr << "initialisation failed" << std::endl;
        return 1;
    }
    std::vector<EventCalibSpline::KeyPose> poses;
    std::vector<EventCalibSpline::KeyFrame> kfs;
    std::vector<double> stamps;
    for (const auto &kv : frames) {
        EventCalibSpline::KeyPose kp;
        kp.timeStamp = kv.second.timeStamp;
        std::copy(kv.second.unitQwb, kv.second.unitQwb + 4, kp.unitQwb);
        std::copy(kv.second.twb, kv.second.twb + 3, kp.twb);
        poses.push_back(kp);
        kfs.push_back(EventCalibSpline::KeyFrame{kv.second.timeStamp, kv.second.circles});
        stamps.push_back(kv.second.timeStamp);
    }
    for (size_t i = 1; i < poses.size(); ++i) {  // one sign per quaternion so the real-valued spline fit sees a continuous curve
        double d = 0;
        for (int a = 0; a < 4; ++a) d += poses[i].unitQwb[a] * poses[i - 1].unitQwb[a];
        if (d < 0)
            for (int a = 0; a < 4; ++a) poses[i].unitQwb[a] = -poses[i].unitQwb[a];
    }
    try {
        std::vector<EventCalibSpline::Segment> segments = EventCalibSpline::segmentsFromKeyframes(poses, motionTimeStep, useSO3);
        // EventCalibSpline.cpp:94-108: radial part of the OpenCV model -> 5-term inverse polynomial
        const ecb::CameraModel &cam = ini.camera;
        const std::array<double, 4> radial = {cam.dist[0], cam.dist[1], cam.dist[4], 0.0};
        const std::array<double, 5> inv = inverseRadialDistortion(radial);
        const std::array<double, 9> intrinsics = {cam.fx, cam.fy, cam.cx, cam.cy, inv[0], inv[1], inv[2], inv[3], inv[4]};
        if (!getenv("ECB_REFERENCE_SIGNATURES")) {  // (the all-in-one constructor below prints them itself, like the reference's)
            std::cout << "OpenCV Distortion before optimization:";
            printEigenLike(std::cout, radial.data(), 1, 4);
            std::cout << std::endl << "Intrinsics before optimization:";
            printEigenLike(std::cout, intrinsics.data(), 1, 9);
            std::cout << std::endl;
        }
        // distinct devices: residuals sharded like the events; the same device listed several times (tests of the sharding
        // logic on a one-GPU box): the optimisation runs on one context holding the whole stream
        bool distinct = true;
        for (int g = 0; g < G; ++g)
            for (int h = 0; h < g; ++h) distinct = distinct && devices[(size_t) g] != devices[(size_t) h];
        ShardedEventContainer::Ptr opt_events = container;
        if (!distinct) {
            opt_events = std::make_shared<ShardedEventContainer>(std::vector<int>(1, devices[0]), width, height);
            opt_events->load(rec.data() + b, e - b, {});
        }
        if (getenv("ECB_REFERENCE_SIGNATURES")) {
            // The same back half through the reference's OWN argument lists (EventCalibSpline.hpp:19, CirclesEventFrame.hpp:43-65;
            // compat types of include/ecb/compat/): a MapBase of Bodyframes + landmarks + camera, the all-in-one constructor, and
            // for the first key frame CirclesEventFrame::rectifyFeatures(outlierIdxs, Rcw, tcw) / findCenter(Eigen::Vector2d).
            EventContainer::Ptr one = opt_events->shards() == 1 ? opt_events->shard[0] : nullptr;
            if (!one) {
                one = std::make_shared<EventContainer>(devices[0], width, height);
                one->load(rec.data() + b, e - b);
            }
            auto map = std::make_shared<MapBase>();
            map->camera = ini.camera;
            std::vector<LandmarkBase::Ptr> lms;
            const std::vector<double> bp = ini.boardPoints();
            for (size_t k = 0; k + 2 < bp.size(); k += 3) {
                lms.push_back(std::make_shared<LandmarkBase>((int) (k / 3), Eigen::Vector3d(bp[k], bp[k + 1], bp[k + 2])));
                map->addLandmark(lms.back());
            }
            for (const auto &kv : frames) {
                const Frame &f = kv.second;
                auto bf = std::make_shared<Bodyframe>(f.timeStamp, Eigen::Quaterniond(f.unitQwb[3], f.unitQwb[0], f.unitQwb[1], f.unitQwb[2]),
                                                      Eigen::Vector3d(f.twb[0], f.twb[1], f.twb[2]));
                bf->circles = f.circles;
                map->addFrame(bf);
            }
            {   // per-frame class with the reference's signatures on the first key frame
                const Frame &f = frames.begin()->second;
                CirclesEventFrame cf(one, f.duration, pattern, params);
                const bool found = cf.extractFeatures();
                cf.setSensor(ini.camera);
                cf.setLandmarks(lms);
                const Eigen::Quaterniond Qwb(f.unitQwb[3], f.unitQwb[0], f.unitQwb[1], f.unitQwb[2]);
                const Eigen::Matrix3d Rwb = Qwb.toRotationMatrix();
                Eigen::Matrix3d Rcw;
                Eigen::Vector3d tcw;
                for (int r = 0; r < 3; ++r) {
                    for (int c = 0; c < 3; ++c) Rcw(r, c) = Rwb(c, r);
                }
                for (int r = 0; r < 3; ++r) tcw[r] = -(Rcw(r, 0) * f.twb[0] + Rcw(r, 1) * f.twb[1] + Rcw(r, 2) * f.twb[2]);
                const bool ok2 = found && cf.rectifyFeatures(std::unordered_set<int>(), Rcw, tcw);
                double worst = 0;
                size_t alive = 0, fi = 0;
                for (const auto &c : f.circles) {
                    if (c[2] < 0) continue;
                    ++alive;
                    if (fi < cf.features().size()) {
                        const CalibCircleLite &g = cf.features()[fi++];
                        worst = std::max(worst, std::max(std::abs(g.center[0] - c[0]), std::max(std::abs(g.center[1] - c[1]), std::abs(g.radius - c[2]))));
                    }
                }
                int hits = 0;
                for (const auto &g : cf.features()) {
                    const LandmarkBase::Ptr lm = cf.findCenter(Eigen::Vector2d(g.center[0] + g.radius, g.center[1]));
                    hits += lm != nullptr;
                }
                std::cerr << "reference signatures: rectifyFeatures(outlierIdxs, Rcw, tcw) " << (ok2 ? "true" : "false") << ", "
                          << cf.features().size() << " of " << alive << " features, max |diff| to the batched result " << worst
                          << ", findCenter(Eigen::Vector2d) -> landmark for " << hits << " rim points" << std::endl;
            }
            EventCalibSpline spline(map, one, useSO3, fs.num("reduceMap", 0) != 0, motionTimeStep, pattern->circleRadius);
            std::ofstream tum(std::string(argv[3]) + "/TrajectoryByEvent.txt");
            tum << std::fixed;
            for (const auto &kv : map->keyframes()) {  // SystemBase::saveKeyFrameTrajectoryTUM on the updated map
                const Eigen::Quaterniond q = kv.second->unitQwb();
                const Eigen::Vector3d t = kv.second->twb();
                tum << std::setprecision(10) << kv.first << " " << t[0] << " " << t[1] << " " << t[2] << " " << q.x() << " " << q.y() << " "
                    << q.z() << " " << q.w() << std::endl;
            }
            std::cout << "press Enter to exit..." << std::endl;
            std::cin.ignore();
            return 0;
        }
        ShardedCalibSpline spline(opt_events, segments, intrinsics, motionTimeStep, pattern->circleRadius, useSO3);
        if (constIntrinsics) {
            static const char *const names[9] = {"fx", "fy", "cx", "cy", "k1", "k2", "k3", "k4", "k5"};
            std::ostringstream line;
            line.precision(17);
            line << "Constant intrinsics:";
            for (int i = 0; i < 9; ++i)
                if ((constIntrinsics >> i) & 1u) line << " " << names[i] << " = " << intrinsics[(size_t) i];
            std::cout << line.str() << std::endl;
            if (spline.setConstantIntrinsics(constIntrinsics) != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
        }
        std::vector<std::array<double, 3>> landmarks;
        const std::vector<double> board = ini.boardPoints();
        for (size_t k = 0; k + 2 < board.size(); k += 3) landmarks.push_back({board[k], board[k + 1], board[k + 2]});
        const int64_t n_res = spline.associate(kfs, landmarks);
        ecb_lm_summary sum;
        if (!spline.optimize(&sum)) {
            std::cerr << "ecb: " << spline.lastError() << std::endl;
            return 1;
        }
        // in place of ceres::Solver::Summary::FullReport() (EventCalibSpline.cpp:248)
        std::cout << "Solver Summary: residuals " << n_res << ", splines " << segments.size() << ", iterations " << sum.iterations
                  << " (successful " << sum.successful_steps << "), cost " << sum.initial_cost << " -> " << sum.final_cost
                  << ", termination " << sum.termination << std::endl;
        for (int round = 1; round <= reassociateRounds; ++round) {  // re-association, then the optimisation again (no reference output)
            EventCalibSpline::ReassociationCounts rc;
            if (spline.reassociate(5.0, 0.0, &rc) != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            std::cout << "Re-association " << round << ": residuals " << rc.residuals << " (same " << rc.same << ", changed "
                      << rc.changed << ", new " << rc.added << ", lost " << rc.lost << ")" << std::endl;
            if (!spline.optimize(&sum)) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            std::cout << "Solver Summary (after re-association " << round << "): residuals " << rc.residuals << ", splines "
                      << segments.size() << ", iterations " << sum.iterations << " (successful " << sum.successful_steps << "), cost "
                      << sum.initial_cost << " -> " << sum.final_cost << ", termination " << sum.termination << std::endl;
        }
        if (rejectK > 0.0) {  // outlier rejection, then the same optimisation again from the first solution (no reference output)
            double s = 0.0, thr = 0.0;
            std::vector<uint8_t> drop;
            int64_t kept = 0, removed = 0;
            if (spline.rejectOutliers(rejectK, &s, &thr, &drop, &kept, &removed) != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            std::ostringstream line;
            line.precision(8);
            int nDrop = 0;
            std::ostringstream dropped;
            dropped << std::fixed << std::setprecision(10);
            for (size_t k = 0; k < drop.size(); ++k)
                if (drop[k]) dropped << (nDrop++ ? " " : "") << kfs[k].timeStamp;
            line << "Outlier rejection: k " << rejectK << ", s " << s << ", threshold " << thr << ", key frames dropped " << nDrop
                 << " [" << dropped.str() << "], records removed " << removed << " of " << kept + removed << " ("
                 << (kept + removed ? 100.0 * (double) removed / (double) (kept + removed) : 0.0) << " %)";
            std::cout << line.str() << std::endl;
            if (!spline.optimize(&sum)) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            std::cout << "Solver Summary (after rejection): residuals " << kept << ", splines " << segments.size() << ", iterations "
                      << sum.iterations << " (successful " << sum.successful_steps << "), cost " << sum.initial_cost << " -> "
                      << sum.final_cost << ", termination " << sum.termination << std::endl;
        }
        std::cout.precision(12);  // updateMap(), EventCalibSpline.cpp:263-264
        std::cout << "Intrinsics after optimization:";
        printEigenLike(std::cout, spline.intrinsics().data(), 1, 9);
        std::cout << std::endl;
        if (getenv("ECB_RESIDUALS") && atoi(getenv("ECB_RESIDUALS")) != 0) {  // how well the model fits (no reference output)
            std::vector<ecb_residual_group> byKf, byCircle, byCell;
            ecb_residual_group tot;
            if (spline.residualGroups(ECB_RESIDUALS_BY_KEYFRAME, residualCell, byKf, &tot) != ECB_OK ||
                spline.residualGroups(ECB_RESIDUALS_BY_CIRCLE, residualCell, byCircle, nullptr) != ECB_OK ||
                spline.residualGroups(ECB_RESIDUALS_BY_SENSOR_CELL, residualCell, byCell, nullptr) != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            const double nan = std::numeric_limits<double>::quiet_NaN();
            auto mean = [&](const ecb_residual_group &g) { return g.count ? g.sum / (double) g.count : nan; };
            auto rms = [&](const ecb_residual_group &g) { return g.count ? std::sqrt(g.sum_sq / (double) g.count) : nan; };
            std::cout << "Residuals: " << tot.count << ", RMS " << rms(tot) << ", mean " << mean(tot) << ", max |r| " << tot.max_abs
                      << ", down-weighted " << tot.n_downweighted << " ("
                      << (tot.count ? 100.0 * (double) tot.n_downweighted / (double) tot.count : 0.0) << " %)" << std::endl;
            auto stats = [&](std::ostream &f, const ecb_residual_group &g) {
                f << std::defaultfloat << std::setprecision(17) << " " << g.count << " " << mean(g) << " " << rms(g) << " " << g.max_abs
                  << " " << g.n_downweighted << " " << g.cost << "\n";
            };
            const char *units = "# r = ||X_w - L|| - circleRadius: distance on the board plane in the units of the board points (not "
                                "pixels), before the Huber loss\n# down-weighted: r^2 > huber_delta^2; cost: sum rho(r^2) / 2\n";
            const std::string dir = std::string(argv[3]) + "/";
            {
                std::ofstream f(dir + "ResidualsByKeyframe.txt");
                f << units << "# stamp count mean RMS max_abs n_downweighted cost (one line per key frame)\n";
                for (size_t k = 0; k < byKf.size(); ++k) {
                    f << std::fixed << std::setprecision(10) << kfs[k].timeStamp;
                    stats(f, byKf[k]);
                }
            }
            {
                std::ofstream f(dir + "ResidualsByCircle.txt");
                f << units << "# id x y z count mean RMS max_abs n_downweighted cost (one line per board circle; x y z: board point)\n";
                for (size_t c = 0; c < byCircle.size(); ++c) {
                    f << c << std::defaultfloat << std::setprecision(17) << " " << landmarks[c][0] << " " << landmarks[c][1] << " "
                      << landmarks[c][2];
                    stats(f, byCircle[c]);
                }
            }
            {
                std::ofstream f(dir + "ResidualMap.txt");
                const int ncx = (width + residualCell - 1) / residualCell;
                f << units << "# cell " << residualCell << " px, " << ncx << " x " << (height + residualCell - 1) / residualCell
                  << " cells of the " << width << " x " << height << " sensor\n"
                  << "# u0 v0 count mean RMS max_abs n_downweighted cost (one line per non-empty cell; u0 v0: its top-left pixel)\n";
                for (size_t c = 0; c < byCell.size(); ++c) {
                    if (byCell[c].count == 0) continue;
                    f << ((int) c % ncx) * residualCell << " " << ((int) c / ncx) * residualCell;
                    stats(f, byCell[c]);
                }
            }
        }
        if (getenv("ECB_REPROJECTION") && atoi(getenv("ECB_REPROJECTION")) != 0) {  // the same fit in pixels (no reference output)
            std::vector<ecb_reprojection_group> byKf, byCircle, byCell;
            ecb_reprojection_group tot, ctot;
            std::vector<double> proj, cerr;
            if (spline.reprojectionGroups(ECB_RESIDUALS_BY_KEYFRAME, residualCell, byKf, &tot) != ECB_OK ||
                spline.reprojectionGroups(ECB_RESIDUALS_BY_CIRCLE, residualCell, byCircle, nullptr) != ECB_OK ||
                spline.reprojectionGroups(ECB_RESIDUALS_BY_SENSOR_CELL, residualCell, byCell, nullptr) != ECB_OK ||
                spline.keyframeReprojection(proj, cerr, &ctot) != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            const std::array<double, 9> &in = spline.intrinsics();
            double fold = 0.0, corner = 0.0;
            ecb_inverse_radial_fold(in.data() + 4, &fold);
            for (int c = 0; c < 4; ++c) {  // distorted radius of the sensor's corner pixels, in pixels of fx
                const double x = ((c & 1) ? width - 1 : 0) - in[2], y = ((c & 2) ? height - 1 : 0) - in[3];
                corner = std::max(corner, in[0] * std::sqrt((x / in[0]) * (x / in[0]) + (y / in[1]) * (y / in[1])));
            }
            const double nan = std::numeric_limits<double>::quiet_NaN();
            auto mean = [&](const ecb_reprojection_group &g) { return g.count ? g.sum / (double) g.count : nan; };
            auto rms = [&](const ecb_reprojection_group &g) { return g.count ? std::sqrt(g.sum_sq / (double) g.count) : nan; };
            // key-frame centres per key frame / per circle: count and sum of squares over the projectable present features
            const size_t K = byKf.size(), nc = byCircle.size();
            std::vector<int64_t> ckN(K, 0), ccN(nc, 0);
            std::vector<double> ckS(K, 0.0), ccS(nc, 0.0);
            for (size_t k = 0; k < K; ++k)
                for (size_t c = 0; c < nc; ++c) {
                    const double e = cerr[k * nc + c];
                    if (std::isnan(e)) continue;
                    ++ckN[k], ++ccN[c];
                    ckS[k] += e * e, ccS[c] += e * e;
                }
            auto crms = [&](int64_t n, double s) { return n ? std::sqrt(s / (double) n) : nan; };
            std::cout << "Reprojection: " << tot.count << " events, RMS " << rms(tot) << " px, mean " << mean(tot) << " px, max |e| "
                      << tot.max_abs << " px, invalid " << tot.n_invalid << "; " << ctot.count << " key-frame centres, RMS " << rms(ctot)
                      << " px; fold at " << fold * in[0] << " px, farthest sensor corner at " << corner << " px" << std::endl;
            auto stats = [&](std::ostream &f, const ecb_reprojection_group &g) {
                f << std::defaultfloat << std::setprecision(17) << " " << g.count << " " << g.n_invalid << " " << mean(g) << " " << rms(g)
                  << " " << g.max_abs;
            };
            const char *units = "# e = sign(|X_w - L| - circleRadius) |q - o| in pixels: o the event pixel, q the projection of the rim "
                                "point L + circleRadius (X_w - L) / |X_w - L| (the residual's correspondence, not the distance to the "
                                "projected ellipse); invalid: not projectable\n# centres: the board point at the key frame's stamp "
                                "projected, against the detected circle centre (pixels)\n";
            const std::string dir = std::string(argv[3]) + "/";
            {
                std::ofstream f(dir + "ReprojectionByKeyframe.txt");
                f << units << "# stamp count n_invalid mean RMS max_abs centre_count centre_RMS (one line per key frame)\n";
                for (size_t k = 0; k < K; ++k) {
                    f << std::fixed << std::setprecision(10) << kfs[k].timeStamp;
                    stats(f, byKf[k]);
                    f << " " << ckN[k] << " " << crms(ckN[k], ckS[k]) << "\n";
                }
            }
            {
                std::ofstream f(dir + "ReprojectionByCircle.txt");
                f << units << "# id x y z count n_invalid mean RMS max_abs centre_count centre_RMS (one line per board circle)\n";
                for (size_t c = 0; c < nc; ++c) {
                    f << c << std::defaultfloat << std::setprecision(17) << " " << landmarks[c][0] << " " << landmarks[c][1] << " "
                      << landmarks[c][2];
                    stats(f, byCircle[c]);
                    f << " " << ccN[c] << " " << crms(ccN[c], ccS[c]) << "\n";
                }
            }
            {
                std::ofstream f(dir + "ReprojectionMap.txt");
                const int ncx = (width + residualCell - 1) / residualCell;
                f << units << "# cell " << residualCell << " px, " << ncx << " x " << (height + residualCell - 1) / residualCell
                  << " cells of the " << width << " x " << height << " sensor\n"
                  << "# u0 v0 count n_invalid mean RMS max_abs (one line per non-empty cell; u0 v0: its top-left pixel)\n";
                for (size_t c = 0; c < byCell.size(); ++c) {
                    if (byCell[c].count + byCell[c].n_invalid == 0) continue;
                    f << ((int) c % ncx) * residualCell << " " << ((int) c / ncx) * residualCell;
                    stats(f, byCell[c]);
                    f << "\n";
                }
            }
        }
        const bool want_cov = getenv("ECB_COVARIANCE") && atoi(getenv("ECB_COVARIANCE")) != 0;
        const bool want_traj_cov = getenv("ECB_TRAJECTORY_COVARIANCE") && atoi(getenv("ECB_TRAJECTORY_COVARIANCE")) != 0;
        if (want_cov || want_traj_cov || motionRate > 0) {  // uncertainty of the result (no reference output)
            EventCalibSpline::Covariance cov;
            const int rc = spline.covariance(cov);
            if (rc == ECB_OK && want_cov) {
                const std::array<double, 9> sd = cov.stdIntrinsics();
                std::cout << "Intrinsics standard deviation:";
                printEigenLike(std::cout, sd.data(), 1, 9);
                std::cout << std::endl;
                std::ofstream f(std::string(argv[3]) + "/IntrinsicsCovariance.txt");
                f.precision(17);
                f << "# sigma2 = 2 cost / (residuals - parameters), " << cov.summary.n_residuals << " residuals, " << cov.summary.dimension
                  << " parameters\n" << cov.summary.sigma2 << "\n# Z = (J^T J)^-1 of fx fy cx cy k1 k2 k3 k4 k5 (covariance = sigma2 Z)\n";
                for (int r = 0; r < 9; ++r)
                    for (int c = 0; c < 9; ++c) f << cov.intrinsics[(size_t) (9 * r + c)] << (c == 8 ? "\n" : " ");
                f << "# standard deviation sqrt(sigma2 Z_ii)\n";
                for (int i = 0; i < 9; ++i) f << sd[(size_t) i] << (i == 8 ? "\n" : " ");
            } else if (rc == ECB_FAILED) {
                std::cerr << "ecb: no covariance: " << spline.lastError() << std::endl;
            } else if (rc != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            }
            if (rc == ECB_OK && want_traj_cov) {  // one line per line of TrajectoryByEvent.txt: its stamp, then sigma2 Sigma row major
                std::vector<double> pose, pc;
                if (spline.poseCovariance(stamps, pose, pc) != ECB_OK) {
                    std::cerr << "ecb: " << spline.lastError() << std::endl;
                    return 1;
                }
                std::ofstream f(std::string(argv[3]) + "/TrajectoryCovariance.txt");
                f << "# covariance sigma2 Sigma of the pose at each stamp of TrajectoryByEvent.txt: stamp, then 36 entries row major\n"
                  << "# tangent: dtheta_x dtheta_y dtheta_z (body frame, R = R^ Exp(dtheta), radians), dp_x dp_y dp_z (t - t^, world "
                     "frame, units of the trajectory)\n"
                  << "# sigma2 = 2 cost / (residuals - parameters) = " << std::setprecision(17) << cov.summary.sigma2 << "\n";
                for (size_t k = 0; k < stamps.size(); ++k) {
                    if (std::isnan(pose[7 * k])) continue;  // outside every segment: TrajectoryByEvent.txt skips the stamp too
                    f << std::fixed << std::setprecision(10) << stamps[k] << std::defaultfloat << std::setprecision(17);
                    for (int e = 0; e < 36; ++e) f << " " << cov.summary.sigma2 * pc[36 * k + (size_t) e];
                    f << "\n";
                }
            }
            if (motionRate > 0) {  // the motion of the final trajectory at t0 + k / rate, with its deviations when rc == ECB_OK
                const auto &seg = spline.segments();
                const double t0 = seg.front().knots.front(), t1 = seg.back().knots.back();
                std::ofstream f(std::string(argv[3]) + "/TrajectoryMotion.txt");
                f << "# motion of the trajectory at t0 + k / rate, rate = " << std::setprecision(17) << motionRate
                  << " Hz, t0 = the first knot; stamps between segments are skipped\n"
                  << "# stamp [s], omega_x omega_y omega_z (body frame, rad/s), v_x v_y v_z (world frame, board units/s), a_x a_y a_z "
                     "(world frame, board units/s^2), then the standard deviations sqrt(sigma2 Sigma_m,ii) of those 9 (NaN without a "
                     "covariance)\n";
                const int64_t total = (int64_t) std::floor((t1 - t0) * motionRate) + 1;
                int64_t samples = 0;
                double maxW = 0.0, maxV = 0.0;
                std::vector<double> times, motion, mc;
                for (int64_t lo = 0; lo < total; lo += (int64_t) 1 << 20) {
                    times.clear();
                    for (int64_t k = lo; k < std::min(total, lo + ((int64_t) 1 << 20)); ++k) times.push_back(t0 + (double) k / motionRate);
                    const int mrc = rc == ECB_OK ? spline.motionCovariance(times, motion, mc) : spline.trajectoryMotion(times, motion);
                    if (mrc != ECB_OK) {
                        std::cerr << "ecb: " << spline.lastError() << std::endl;
                        return 1;
                    }
                    for (size_t k = 0; k < times.size(); ++k) {
                        const double *m = &motion[16 * k];
                        if (std::isnan(m[0])) continue;  // in a gap between segments
                        ++samples;
                        maxW = std::max(maxW, std::sqrt(m[7] * m[7] + m[8] * m[8] + m[9] * m[9]));
                        maxV = std::max(maxV, std::sqrt(m[10] * m[10] + m[11] * m[11] + m[12] * m[12]));
                        f << std::fixed << std::setprecision(10) << times[k] << std::defaultfloat << std::setprecision(17);
                        for (int e = 7; e < 16; ++e) f << " " << m[e];
                        for (int e = 0; e < 9; ++e)
                            f << " " << (rc == ECB_OK ? std::sqrt(cov.summary.sigma2 * mc[81 * k + 10 * (size_t) e]) : NAN);
                        f << "\n";
                    }
                }
                std::cout << "Trajectory motion: " << samples << " samples at " << motionRate << " Hz, max |omega| " << maxW
                          << " rad/s, max |v| " << maxV << " board units/s" << std::endl;
            }
        }
        if (getenv("ECB_GYRO")) {  // camera-gyroscope calibration at the final control points (no reference output)
            const int nOff = gyroMaxOffset > 0.0 ? 1001 : 1;
            ecb_gyro_calibration g;
            std::vector<double> offCost;
            const int grc = spline.calibrateGyroscope(gyro, gyroMaxOffset, nOff, g, &offCost);
            if (grc == ECB_FAILED) {
                std::cerr << "ecb: no camera-gyroscope calibration: " << spline.lastError() << std::endl;
            } else if (grc != ECB_OK) {
                std::cerr << "ecb: " << spline.lastError() << std::endl;
                return 1;
            } else {
                const double x = g.q_gc[0], y = g.q_gc[1], z = g.q_gc[2], w = g.q_gc[3];
                const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)};
                const double angle = 2.0 * std::atan2(std::sqrt(x * x + y * y + z * z), std::fabs(w)) * 180.0 / M_PI;
                std::ofstream f(std::string(argv[3]) + "/CameraGyroscope.txt");
                f << std::setprecision(17)
                  << "# camera-gyroscope calibration: w_g(t) = R_gc w_c(t + offset) + bias + noise\n"
                  << "# w_c: body-frame angular velocity of the calibrated trajectory (camera frame, rad/s); w_g: gyroscope reading "
                     "(gyroscope frame, rad/s); R_gc rotates camera-frame vectors into the gyroscope frame (q_gc x y z w, R_gc row "
                     "major); gyroscope stamp t is event time t + offset; offset, scan_offset in s; bias, rms in rad/s; rotation_std "
                     "in rad (gyroscope frame); sigma2 in (rad/s)^2\n"
                  << "q_gc " << x << " " << y << " " << z << " " << w << "\nR_gc";
                for (double v : R) f << " " << v;
                f << "\nrotation_std " << g.std[0] << " " << g.std[1] << " " << g.std[2] << "\noffset " << g.offset
                  << "\noffset_std " << g.std[3] << "\nbias " << g.bias[0] << " " << g.bias[1] << " " << g.bias[2] << "\nbias_std "
                  << g.std[4] << " " << g.std[5] << " " << g.std[6] << "\nrms " << g.rms << "\nsigma2 " << g.sigma2 << "\nn_used "
                  << g.n_used << "\nn_unused " << g.n_unused << "\nscan_offset " << g.scan_offset << "\niterations " << g.iterations
                  << "\ntermination " << g.termination << "\n# scan: offset d_m (s), mean (|w_c(t + d_m)| - |w_g|)^2 ((rad/s)^2)\n";
                for (int m = 0; m < nOff; ++m)
                    f << (nOff > 1 ? gyroMaxOffset * (double) (2 * m - (nOff - 1)) / (double) (nOff - 1) : 0.0) << " " << offCost[m]
                      << "\n";
                std::cout << "Camera-gyroscope: offset " << 1e3 * g.offset << " ms (+- " << 1e3 * g.std[3] << "), rotation " << angle
                          << " deg, bias " << g.bias[0] << " " << g.bias[1] << " " << g.bias[2] << " rad/s, RMS " << g.rms
                          << " rad/s, " << g.n_used << " samples" << std::endl;
            }
        }
        spline.saveKeyFrameTrajectoryTUM(std::string(argv[3]) + "/TrajectoryByEvent.txt", stamps);  // eventCameraCalib.cpp:212
        if (!getenv("ECB_NO_IMAGES")) {  // :214-227: SavePath/image/<timestamp>.png = cf->image() of every key frame
            const std::string dir = std::string(argv[3]) + "/image/";
            mkdir(dir.c_str(), 0755);
            std::vector<std::pair<double, double>> kw;
            for (const auto &kv : frames) kw.push_back(kv.second.duration);
            fe.run(kw);
            size_t w = 0;
            for (const auto &kv : frames) {
                const ecb::Image8UC3 img = renderFrameImage(fe, w++, &kv.second.circles);
                ecb::write_png(dir + std::to_string(kv.second.timeStamp) + ".png", img);
            }
        }
    } catch (const std::logic_error &ex) {
        std::cerr << "terminate called after throwing an instance of 'std::logic_error'\n  what():  " << ex.what() << std::endl;
        return 134;  // the reference aborts on the uncaught exception
    } catch (const std::exception &ex) {
        std::cerr << "ecb: " << ex.what() << std::endl;
        return 1;
    }
    std::cout << "press Enter to exit..." << std::endl;
    std::cin.ignore();
    return 0;
}
