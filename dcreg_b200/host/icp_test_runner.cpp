// icp_test_runner.cpp - the reference's experiment harness on top of the B200 engine's C ABI.
//
// Same surface as DCReg's `icp_test_runner` executable (DCReg/src/icp_main.cpp:6-52, icp_test_runner.cpp:20-516,
// 603-1510): YAML schema (SURVEY.md Appendix B.1), method table keyed by name, per-method runs, statistics and the
// output file set with the reference's columns (statistics_summary.txt, complete_log.txt, transform_details.csv,
// condition_numbers_detailed.csv, all_results.csv, degeneracy_analysis_{first,last}_iter.txt, iteration_history.csv,
// iteration_details_with_dx.csv).  The whole hot path runs in libdcreg_b200.so (include/dcreg_b200.h); this file is
// host-side orchestration and formatting only.  The config path is argv[1] (default: the reference's hard-coded
// "../config/icp.yaml").
//
// Kept quirks of the reference (SURVEY.md §3.1, Appendix B.4): methods run in alphabetical order (std::map); dispatch is
// by method NAME (only Ours, NONE, ME-SR, FCN-SR, ME-TSVD, ME-TReg reach the SO(3) path; others print the reference's
// "Can not recognize the method" line, since the XICP / SuperLoc / Open3D baselines are out of scope); the per-iteration
// CSV swaps its two error columns (icp_test_runner.cpp:1457-1458); unknown enum strings map to the first enumerator.
// `Time_ms` per iteration is dcreg_iter_log::iter_time_ms, the device's own tic/toc of that iteration (the loop never
// returns to the host between iterations).  Difference: `<method>_error.pcd` (jet-coloured visual artefact) is not written.
//
// Extension (not in the reference, which has no RNG - SURVEY.md §6 C5): an optional `monte_carlo:` block runs a seeded
// perturbation study of every listed method through dcreg_icp_run_batch (all trials advance side by side on the GPU) and
// writes monte_carlo_<method>.csv (ending in the point-to-point metrics of every trial's final pose, one batched
// dcreg_point_to_point_metrics_batch call per method) + monte_carlo_summary.txt.  Absent block = the reference's behaviour, unchanged.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <limits>
#include <map>
#include <random>
#include <string>
#include <sys/stat.h>
#include <vector>

#include "../../include/dcreg_b200.h"
#include "pcd_io.hpp"
#include "yaml_lite.hpp"

namespace {

constexpr double kPi = 3.14159265358979323846;
inline double deg2rad(double d) { return d * kPi / 180.0; }
inline double rad2deg(double r) { return r * 180.0 / kPi; }

struct Pose6D { double x = 0, y = 0, z = 0, roll = 0, pitch = 0, yaw = 0; };

struct IcpParameters {            // DCReg/include/utils.hpp:82-103
    double DEGENERACY_THRES_COND = 10.0, DEGENERACY_THRES_EIG = 120.0, KAPPA_TARGET = 1.0, PCG_TOLERANCE = 1e-6;
    int PCG_MAX_ITER = 10;
    double ADAPTIVE_REG_ALPHA = 10.0, STD_REG_GAMMA = 0.01, LOAM_EIGEN_THRESH = 120.0, TSVD_SINGULAR_THRESH = 120.0;
};

struct Mat4 { double m[16]; };    // row-major

Mat4 identity4() { Mat4 T{}; for (int i = 0; i < 4; ++i) T.m[i * 5] = 1.0; return T; }

Mat4 pose6d_to_matrix(const Pose6D& p) {          // utils.hpp:452-460: Trans * Rz * Ry * Rx
    const double cr = std::cos(p.roll), sr = std::sin(p.roll), cp = std::cos(p.pitch), sp = std::sin(p.pitch);
    const double cy = std::cos(p.yaw), sy = std::sin(p.yaw);
    Mat4 T = identity4();
    T.m[0] = cy * cp; T.m[1] = cy * sp * sr - sy * cr; T.m[2] = cy * sp * cr + sy * sr; T.m[3] = p.x;
    T.m[4] = sy * cp; T.m[5] = sy * sp * sr + cy * cr; T.m[6] = sy * sp * cr - cy * sr; T.m[7] = p.y;
    T.m[8] = -sp;     T.m[9] = cp * sr;                T.m[10] = cp * cr;               T.m[11] = p.z;
    return T;
}

struct Config {                    // DCReg/include/utils.hpp:132-171
    int num_runs = 1;
    bool save_pcd = true, save_error_pcd = true, visualize = false;
    double CONVERGENCE_THRESH_ROT = 1e-5, CONVERGENCE_THRESH_TRANS = 1e-3;
    std::string folder_path, source_pcd, target_pcd, output_folder;
    double search_radius = 1.0;
    int max_iterations = 30, normal_nn = 5;
    double error_threshold = 0.05;
    Pose6D initial_noise, gt_pose;
    Mat4 gt_matrix = identity4(), initial_matrix = identity4();
    IcpParameters icp_params;
    std::map<std::string, std::pair<std::string, std::string>> test_methods;
    bool use_so3_parameterization = true;
    bool use_weight_derivative = false;     // USE_WEIGHT_DERIVATIVE (icp_test_runner.cpp:1691), optional key icp.use_weight_derivative
    // optional block monte_carlo: (extension, BASELINE.json configs[4]): trials initial poses drawn uniformly in
    // [-max_trans_m, max_trans_m]^3 x [-max_rot_deg, max_rot_deg]^3 (roll, pitch, yaw), std::mt19937_64(seed)
    int mc_trials = 0;
    unsigned long long mc_seed = 45;
    double mc_max_trans = 1.0, mc_max_rot_deg = 3.0;
};

bool loadConfig(const std::string& filename, Config& c) {      // icp_test_runner.cpp:20-153
    try {
        const yaml_lite::Node y = yaml_lite::load_file(filename);
        if (y["test"]) {
            c.num_runs = y["test"]["num_runs"].as<int>();
            c.save_pcd = y["test"]["save_pcd"].as<bool>();
            c.save_error_pcd = y["test"]["save_error_pcd"].as<bool>();
            c.visualize = y["test"]["visualize"].as<bool>();
        }
        if (y["paths"]) {
            c.folder_path = y["paths"]["folder_path"].as<std::string>();
            c.source_pcd = y["paths"]["source_pcd"].as<std::string>();
            c.target_pcd = y["paths"]["target_pcd"].as<std::string>();
            c.output_folder = y["paths"]["output_folder"].as<std::string>();
        }
        if (y["icp"]) {
            c.search_radius = y["icp"]["search_radius"].as<double>();
            c.max_iterations = y["icp"]["max_iterations"].as<int>();
            c.normal_nn = y["icp"]["normal_nn"].as<int>();
            c.error_threshold = y["icp"]["error_threshold"].as<double>();
            c.CONVERGENCE_THRESH_TRANS = y["icp"]["CONVERGENCE_THRESH_TRANS"].as<double>();
            c.CONVERGENCE_THRESH_ROT = y["icp"]["CONVERGENCE_THRESH_ROT"].as<double>();
            if (y["icp"]["use_weight_derivative"]) c.use_weight_derivative = y["icp"]["use_weight_derivative"].as<bool>();
            std::cout << "CONVERGENCE_THRESH_TRANS: " << c.CONVERGENCE_THRESH_TRANS << std::endl;
            std::cout << "CONVERGENCE_THRESH_ROT: " << c.CONVERGENCE_THRESH_ROT << std::endl;
        }
        auto pose = [](const yaml_lite::Node& n, Pose6D& p) {
            p.x = n["x"].as<double>(); p.y = n["y"].as<double>(); p.z = n["z"].as<double>();
            p.roll = deg2rad(n["roll_deg"].as<double>()); p.pitch = deg2rad(n["pitch_deg"].as<double>());
            p.yaw = deg2rad(n["yaw_deg"].as<double>());
        };
        if (y["initial_noise"]) { pose(y["initial_noise"], c.initial_noise); c.initial_matrix = pose6d_to_matrix(c.initial_noise); }
        if (y["gt_pose"]) { pose(y["gt_pose"], c.gt_pose); c.gt_matrix = pose6d_to_matrix(c.gt_pose); }
        if (y["degeneracy"]) {
            c.icp_params.DEGENERACY_THRES_COND = y["degeneracy"]["condition_threshold"].as<double>();
            c.icp_params.DEGENERACY_THRES_EIG = y["degeneracy"]["eigenvalue_threshold"].as<double>();
        }
        if (y["method_params"]) {
            const auto& mp = y["method_params"];
            if (mp["adaptive_reg"]) c.icp_params.ADAPTIVE_REG_ALPHA = mp["adaptive_reg"]["alpha"].as<double>();
            if (mp["standard_reg"]) c.icp_params.STD_REG_GAMMA = mp["standard_reg"]["gamma"].as<double>();
            if (mp["pcg"]) {
                c.icp_params.KAPPA_TARGET = mp["pcg"]["kappa_target"].as<double>();
                c.icp_params.PCG_TOLERANCE = mp["pcg"]["tolerance"].as<double>();
                c.icp_params.PCG_MAX_ITER = mp["pcg"]["max_iter"].as<int>();
            }
            if (mp["tsvd"]) c.icp_params.TSVD_SINGULAR_THRESH = mp["tsvd"]["singular_threshold"].as<double>();
            if (mp["solution_remapping"]) c.icp_params.LOAM_EIGEN_THRESH = mp["solution_remapping"]["eigen_threshold"].as<double>();
        }
        if (y["monte_carlo"]) {
            const auto& mc = y["monte_carlo"];
            c.mc_trials = mc["trials"].as<int>();
            if (mc["seed"]) c.mc_seed = (unsigned long long)mc["seed"].as<double>();
            if (mc["max_trans_m"]) c.mc_max_trans = mc["max_trans_m"].as<double>();
            if (mc["max_rot_deg"]) c.mc_max_rot_deg = mc["max_rot_deg"].as<double>();
            if (c.mc_trials < 0 || c.mc_trials > 65535) throw yaml_lite::ParseError("monte_carlo.trials must be in [0, 65535]");
        }
        // icp_params.XICP_*: parsed by the reference for the (out-of-scope) XICP baseline; accepted and ignored here
        if (y["test_methods"])
            for (const auto& kv : y["test_methods"].map) {
                const auto v = kv.second->as<std::vector<std::string>>();
                if (v.size() < 2) throw yaml_lite::ParseError("test_methods." + kv.first + " needs [detection, handling]");
                c.test_methods[kv.first] = {v[0], v[1]};
            }
        std::cout << "\n=== Loaded Configuration ===" << std::endl;
        std::cout << "STD_REG_GAMMA: " << c.icp_params.STD_REG_GAMMA << std::endl;
        std::cout << "ADAPTIVE_REG_ALPHA: " << c.icp_params.ADAPTIVE_REG_ALPHA << std::endl;
        std::cout << "KAPPA_TARGET: " << c.icp_params.KAPPA_TARGET << std::endl;
        std::cout << "DEGENERACY_THRES_COND: " << c.icp_params.DEGENERACY_THRES_COND << std::endl;
        std::cout << "DEGENERACY_THRES_EIG: " << c.icp_params.DEGENERACY_THRES_EIG << std::endl;
        std::cout << "USE_SO3 ICP: " << c.use_so3_parameterization << std::endl;
        std::cout << "==========================\n" << std::endl;
        return true;
    } catch (const std::exception& e) {
        std::cerr << "Error loading YAML config: " << e.what() << std::endl;
        return false;
    }
}

int detection_from_string(const std::string& s) {     // icp_test_runner.cpp:178-195 (unknown -> first enumerator)
    static const std::map<std::string, int> m = {{"NONE_DETE", 0}, {"SCHUR_CONDITION_NUMBER", 1}, {"FULL_EVD_MIN_EIGENVALUE", 2},
                                                 {"EVD_SUB_CONDITION", 3}, {"FULL_SVD_CONDITION", 4}};
    const auto it = m.find(s);
    return it == m.end() ? 0 : it->second;
}
int handling_from_string(const std::string& s) {      // icp_test_runner.cpp:197-220
    static const std::map<std::string, int> m = {{"NONE_HAND", 0}, {"STANDARD_REGULARIZATION", 1}, {"ADAPTIVE_REGULARIZATION", 2},
                                                 {"PRECONDITIONED_CG", 3}, {"SOLUTION_REMAPPING", 4}, {"TRUNCATED_SVD", 5}};
    const auto it = m.find(s);
    if (it == m.end()) { std::cerr << "Unknown handling method: " << s << std::endl; return 0; }
    return it->second;
}

struct PoseError { double translation_error = 0, rotation_error = 0; };

PoseError calculatePoseError(const Mat4& gt, const Mat4& fin) {      // utils.hpp:497-535, degrees
    // E = gt^-1 * fin for rigid gt: R_e = Rg^T Rf, t_e = Rg^T (tf - tg)
    double R[9], t[3];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            double s = 0;
            for (int k = 0; k < 3; ++k) s += gt.m[k * 4 + i] * fin.m[k * 4 + j];
            R[i * 3 + j] = s;
        }
        double s = 0;
        for (int k = 0; k < 3; ++k) s += gt.m[k * 4 + i] * (fin.m[k * 4 + 3] - gt.m[k * 4 + 3]);
        t[i] = s;
    }
    PoseError e;
    e.translation_error = std::sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
    // Eigen::AngleAxisd(R).angle(): through the quaternion, angle = 2 atan2(|vec|, |w|)
    const double tr = R[0] + R[4] + R[8];
    double w, x, y, z;
    if (tr > 0) { double s = std::sqrt(tr + 1.0); w = 0.5 * s; s = 0.5 / s; x = (R[7] - R[5]) * s; y = (R[2] - R[6]) * s; z = (R[3] - R[1]) * s; }
    else {
        int i = 0; if (R[4] > R[0]) i = 1; if (R[8] > R[i * 4]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        double s = std::sqrt(R[i * 4] - R[j * 4] - R[k * 4] + 1.0);
        double q[3]; q[i] = 0.5 * s; s = 0.5 / s;
        w = (R[k * 3 + j] - R[j * 3 + k]) * s; q[j] = (R[j * 3 + i] + R[i * 3 + j]) * s; q[k] = (R[k * 3 + i] + R[i * 3 + k]) * s;
        x = q[0]; y = q[1]; z = q[2];
    }
    const double n = std::sqrt(x * x + y * y + z * z);
    const double ang = n < std::numeric_limits<double>::epsilon() ? 0.0 : 2.0 * std::atan2(n, std::fabs(w));
    e.rotation_error = rad2deg(std::fabs(ang));
    return e;
}

struct IterData { dcreg_iter_log g; double iter_time_ms = 0, trans_error_vs_gt = 0, rot_error_vs_gt = 0; };

struct TestResult {               // DCReg/include/utils.hpp TestResult
    std::string method_name;
    bool converged = false;
    int iterations = 0, corr_num = 0;
    double time_ms = 0, trans_error_m = 0, rot_error_deg = 0, final_rmse = 0, final_fitness = 0;
    double p2p_rmse = 0, p2p_fitness = 0, chamfer_distance = 0;
    Mat4 final_transform = identity4();
    std::vector<double> condition_numbers, eigenvalues;
    std::vector<int> degenerate_mask;
    std::vector<IterData> iteration_data;
};

struct MethodStatistics {
    int total_runs = 0, converged_runs = 0;
    double mean_trans_error = 0, mean_rot_error = 0, mean_time_ms = 0, mean_iterations = 0, mean_rmse = 0, mean_fitness = 0;
    double mean_p2p_rmse = 0, mean_p2p_fitness = 0, mean_chamfer = 0, corr_num = 0, success_rate = 0;
    double std_trans_error = 0, std_rot_error = 0, std_time_ms = 0;
    double min_trans_error = std::numeric_limits<double>::max(), max_trans_error = 0;
    double min_rot_error = std::numeric_limits<double>::max(), max_rot_error = 0;
};

class TestRunner {
public:
    explicit TestRunner(const Config& c) : config_(c) {}
    ~TestRunner() { if (ctx_) dcreg_destroy(ctx_); }

    bool runAllTests() {                                   // icp_test_runner.cpp:299-328
        if (!loadPointClouds()) return false;
        const int rc = dcreg_create(0, &ctx_);
        if (rc != DCREG_OK) { std::cerr << "[ICP Error] " << (ctx_ ? dcreg_last_error(ctx_) : "no CUDA device") << " (status " << rc << ")" << std::endl; return false; }
        if (!check(dcreg_set_source(ctx_, source_.xyzi.data(), (int64_t)source_.size(), 4), "set_source")) return false;
        if (!check(dcreg_set_target(ctx_, target_.xyzi.data(), (int64_t)target_.size(), 4, config_.search_radius), "set_target")) return false;
        for (const auto& kv : config_.test_methods) {
            const int det = detection_from_string(kv.second.first), hand = handling_from_string(kv.second.second);
            std::cout << "\n--- Testing method: " << kv.first << " ---" << std::endl;
            std::cout << "\n=== Method: " << kv.first << " ===\nDetection: " << kv.second.first << "\nHandling: " << kv.second.second << std::endl;
            if (!runMethod(kv.first, det, hand)) { std::cerr << "Failed to run method: " << kv.first << std::endl; return false; }
        }
        if (config_.mc_trials > 0 && !runMonteCarlo()) return false;
        finalizeStatistics();
        saveStatistics();
        saveDetailedResults();
        return true;
    }

private:
    Config config_;
    dcreg_ctx* ctx_ = nullptr;
    pcd::Cloud source_, target_;
    std::map<std::string, MethodStatistics> statistics_;
    std::map<std::string, std::vector<TestResult>> detailed_results_;

    bool check(int rc, const char* what) {
        if (rc == DCREG_OK) return true;
        std::cerr << "[ICP Error] " << what << ": " << dcreg_last_error(ctx_) << " (status " << rc << ")" << std::endl;
        return false;
    }

    bool loadPointClouds() {                                // icp_test_runner.cpp:156-176
        const std::string sp = config_.folder_path + config_.source_pcd, tp = config_.folder_path + config_.target_pcd;
        std::string err;
        if (!pcd::load(sp, source_, &err)) { std::cerr << "Failed to load source cloud: " << sp << " (" << err << ")" << std::endl; return false; }
        if (!pcd::load(tp, target_, &err)) { std::cerr << "Failed to load target cloud: " << tp << " (" << err << ")" << std::endl; return false; }
        if (source_.empty() || target_.empty()) { std::cerr << "Error: Loaded point cloud is empty: " << sp << std::endl; return false; }
        std::cout << "Loaded point clouds - Source: " << source_.size() << " points, Target: " << target_.size() << " points" << std::endl;
        return true;
    }

    void p2p(const Mat4& T, double& rmse, double& fitness, double& chamfer, int& corr) {
        double out[4] = {0, 0, 0, 0};
        if (check(dcreg_point_to_point_metrics(ctx_, T.m, config_.error_threshold, out), "point_to_point_metrics")) {
            rmse = out[0]; fitness = out[1]; chamfer = out[2]; corr = (int)out[3];
        }
    }

    // dcreg_point_to_point_metrics for every pose of T (n x 16) in one call: out = n x {rmse, fitness, chamfer, n_valid},
    // zeros when the call fails (as p2p leaves them)
    void p2pBatch(const std::vector<double>& T, std::vector<double>& out) {
        const int n = (int)(T.size() / 16);
        out.assign((size_t)n * 4, 0.0);
        if (n > 0 && !check(dcreg_point_to_point_metrics_batch(ctx_, n, T.data(), config_.error_threshold, out.data()), "point_to_point_metrics_batch"))
            out.assign((size_t)n * 4, 0.0);
    }

    static bool isSo3Method(const std::string& name) {
        static const char* so3_names[] = {"Ours", "NONE", "ME-SR", "FCN-SR", "ME-TSVD", "ME-TReg"};
        return std::find_if(std::begin(so3_names), std::end(so3_names), [&](const char* s) { return name == s; }) != std::end(so3_names);
    }

    dcreg_icp_params engineParams(int det, int hand) const {
        dcreg_icp_params p;
        dcreg_default_params(&p);
        p.search_radius = config_.search_radius; p.max_iterations = config_.max_iterations;
        p.detection = det; p.handling = hand; p.use_weight_derivative = config_.use_weight_derivative ? 1 : 0;
        p.conv_thresh_rot = config_.CONVERGENCE_THRESH_ROT; p.conv_thresh_trans = config_.CONVERGENCE_THRESH_TRANS;
        p.cond_thresh = config_.icp_params.DEGENERACY_THRES_COND; p.eig_thresh = config_.icp_params.DEGENERACY_THRES_EIG;
        p.kappa_target = config_.icp_params.KAPPA_TARGET; p.pcg_tol = config_.icp_params.PCG_TOLERANCE;
        p.pcg_max_iter = config_.icp_params.PCG_MAX_ITER; p.std_reg_gamma = config_.icp_params.STD_REG_GAMMA;
        return p;
    }

    // The perturbation study (extension, see the file header): one dcreg_icp_run_batch call per method.
    bool runMonteCarlo() {
        const int n = config_.mc_trials;
        std::mt19937_64 gen(config_.mc_seed);
        auto uni = [&](double a) { return ((double)(gen() >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0) * a; };   // [-a, a)
        std::vector<Pose6D> init((size_t)n);
        std::vector<double> T0((size_t)n * 16), T1((size_t)n * 16);
        for (int i = 0; i < n; ++i) {
            Pose6D& q = init[i];
            q.x = uni(config_.mc_max_trans); q.y = uni(config_.mc_max_trans); q.z = uni(config_.mc_max_trans);
            q.roll = deg2rad(uni(config_.mc_max_rot_deg)); q.pitch = deg2rad(uni(config_.mc_max_rot_deg)); q.yaw = deg2rad(uni(config_.mc_max_rot_deg));
            const Mat4 T = pose6d_to_matrix(q);
            std::memcpy(&T0[(size_t)i * 16], T.m, sizeof(T.m));
        }
        std::ofstream summary(config_.output_folder + "monte_carlo_summary.txt");
        summary << "Perturbation Monte-Carlo: " << n << " trials, seed " << config_.mc_seed << ", |t| <= " << config_.mc_max_trans
                << " m per axis, |rpy| <= " << config_.mc_max_rot_deg << " deg per axis\n\n";
        summary << std::setw(15) << "Method" << std::setw(12) << "Converged%" << std::setw(12) << "Failed" << std::setw(14) << "MeanTrans(m)"
                << std::setw(14) << "MedTrans(m)" << std::setw(14) << "MeanRot(deg)" << std::setw(14) << "MedRot(deg)" << std::setw(12) << "Avg_Iters"
                << std::setw(12) << "Time(ms)" << std::setw(12) << "Trials/s\n";
        for (const auto& kv : config_.test_methods) {
            if (!isSo3Method(kv.first)) continue;
            const dcreg_icp_params p = engineParams(detection_from_string(kv.second.first), handling_from_string(kv.second.second));
            std::vector<int> iters((size_t)n), conv((size_t)n), status((size_t)n);
            const auto t0 = std::chrono::high_resolution_clock::now();
            if (!check(dcreg_icp_run_batch(ctx_, &p, n, T0.data(), T1.data(), iters.data(), conv.data(), status.data(), nullptr, 0), "icp_run_batch")) return false;
            const double ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
            std::ofstream f(config_.output_folder + "monte_carlo_" + kv.first + ".csv");
            f << "Trial,Init_x,Init_y,Init_z,Init_roll_deg,Init_pitch_deg,Init_yaw_deg,Converged,Iterations,Status,Trans_Error_m,Rot_Error_deg";
            for (int k = 0; k < 12; ++k) f << ",T" << k / 4 << k % 4;
            f << ",P2P_RMSE,P2P_Fitness,Chamfer_Distance";
            f << "\n" << std::setprecision(17);
            std::vector<double> p2p_out;
            p2pBatch(T1, p2p_out);
            std::vector<double> te, re;
            long long it_sum = 0; int n_conv = 0, n_fail = 0;
            for (int i = 0; i < n; ++i) {
                Mat4 Tf; std::memcpy(Tf.m, &T1[(size_t)i * 16], sizeof(Tf.m));
                const PoseError e = calculatePoseError(config_.gt_matrix, Tf);
                f << i << ',' << init[i].x << ',' << init[i].y << ',' << init[i].z << ',' << rad2deg(init[i].roll) << ',' << rad2deg(init[i].pitch) << ','
                  << rad2deg(init[i].yaw) << ',' << conv[i] << ',' << iters[i] << ',' << status[i] << ',' << e.translation_error << ',' << e.rotation_error;
                for (int k = 0; k < 12; ++k) f << ',' << Tf.m[k];
                f << ',' << p2p_out[(size_t)i * 4] << ',' << p2p_out[(size_t)i * 4 + 1] << ',' << p2p_out[(size_t)i * 4 + 2];
                f << "\n";
                if (status[i] != DCREG_OK) { ++n_fail; continue; }
                te.push_back(e.translation_error); re.push_back(e.rotation_error);
                it_sum += iters[i]; n_conv += conv[i] != 0;
            }
            auto mean = [](const std::vector<double>& v) { double s = 0; for (double x : v) s += x; return v.empty() ? 0.0 : s / (double)v.size(); };
            auto median = [](std::vector<double> v) { if (v.empty()) return 0.0; std::sort(v.begin(), v.end()); return v[v.size() / 2]; };
            const double ok = (double)std::max<size_t>(1, te.size());
            summary << std::setw(15) << kv.first << std::fixed << std::setw(12) << std::setprecision(1) << 100.0 * n_conv / (double)n << std::setw(12) << n_fail
                    << std::setw(14) << std::setprecision(6) << mean(te) << std::setw(14) << median(te) << std::setw(14) << mean(re) << std::setw(14) << median(re)
                    << std::setw(12) << std::setprecision(1) << (double)it_sum / ok << std::setw(12) << std::setprecision(2) << ms
                    << std::setw(12) << std::setprecision(0) << 1000.0 * n / ms << "\n";
            std::cout << "Monte-Carlo " << kv.first << ": " << n << " trials in " << ms << " ms, " << n_conv << " converged, " << n_fail << " aborted" << std::endl;
        }
        std::cout << "Monte-Carlo results saved to " << config_.output_folder << "monte_carlo_summary.txt" << std::endl;
        return true;
    }

    TestResult runSingleTest(const std::string& name, int det, int hand) {      // icp_test_runner.cpp:393-516
        TestResult r;
        r.method_name = name;
        if (!isSo3Method(name)) {
            std::cout << "Can not recognize the method!!!!! pls check your yaml!!!" << std::endl;
            return r;
        }
        dcreg_icp_params p = engineParams(det, hand);
        std::vector<dcreg_iter_log> log((size_t)std::max(1, config_.max_iterations));
        int n_iter = 0, converged = 0;
        const auto t0 = std::chrono::high_resolution_clock::now();
        const int st = dcreg_icp_run(ctx_, &p, config_.initial_matrix.m, r.final_transform.m, log.data(), config_.max_iterations, &n_iter, &converged);
        const auto t1 = std::chrono::high_resolution_clock::now();
        if (st == DCREG_NOT_ENOUGH_POINTS) std::cerr << "[ICP Warn Iter " << n_iter - 1 << "] Not enough effective points. Aborting." << std::endl;
        else if (st == DCREG_NONFINITE_UPDATE) std::cerr << "[ICP Error Iter " << n_iter << "] Solver returned non-finite values!" << std::endl;
        else if (st != DCREG_OK) std::cerr << "[ICP Error] " << dcreg_last_error(ctx_) << " (status " << st << ")" << std::endl;
        r.converged = converged != 0;
        r.time_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
        r.iterations = n_iter;
        const int nrec = st == DCREG_NOT_ENOUGH_POINTS ? std::max(0, n_iter - 1) : std::min(n_iter, config_.max_iterations);
        for (int i = 0; i < nrec; ++i) {
            IterData d;
            d.g = log[i];
            d.iter_time_ms = log[i].iter_time_ms;   // device-measured tic/toc of this iteration (icp_test_runner.cpp:1695, 1973)
            Mat4 Ti; std::memcpy(Ti.m, log[i].T, sizeof(Ti.m));
            const PoseError e = calculatePoseError(config_.gt_matrix, Ti);
            d.rot_error_vs_gt = e.rotation_error; d.trans_error_vs_gt = e.translation_error;
            r.iteration_data.push_back(d);
        }
        if (!r.iteration_data.empty()) {
            const IterData& last = r.iteration_data.back();
            r.final_rmse = last.g.rmse; r.final_fitness = last.g.fitness; r.corr_num = last.g.n_effective;
            std::memcpy(r.final_transform.m, last.g.T, sizeof(r.final_transform.m));
            r.condition_numbers = {last.g.analysis.cond_schur_rot, last.g.analysis.cond_schur_trans, last.g.analysis.cond_full};
            r.eigenvalues.assign(last.g.analysis.eigenvalues_full, last.g.analysis.eigenvalues_full + 6);
            r.degenerate_mask.assign(last.g.analysis.degenerate_mask, last.g.analysis.degenerate_mask + 6);
        }
        const PoseError e = calculatePoseError(config_.gt_matrix, r.final_transform);
        r.trans_error_m = e.translation_error; r.rot_error_deg = e.rotation_error;
        p2p(r.final_transform, r.p2p_rmse, r.p2p_fitness, r.chamfer_distance, r.corr_num);
        std::cout << "--- ICP SO(3) Final State (Iter " << n_iter << ") ---\nConverged: " << (r.converged ? "Yes" : "No") << " | RMSE: "
                  << r.final_rmse << " | Fitness: " << r.final_fitness << "\nWeight Derivative: " << (config_.use_weight_derivative ? "Enabled" : "Disabled") << std::endl;
        std::cout << "Translation error: " << r.trans_error_m << " m, Rotation error: " << r.rot_error_deg << " deg" << std::endl;
        std::cout << "P2P RMSE: " << r.p2p_rmse << ", Chamfer: " << r.chamfer_distance << std::endl;
        return r;
    }

    bool runMethod(const std::string& name, int det, int hand) {                 // icp_test_runner.cpp:331-391
        statistics_[name] = MethodStatistics();
        for (int run = 0; run < config_.num_runs; ++run) {
            if (config_.num_runs > 1 && run % 10 == 0) std::cout << "  Run " << run + 1 << "/" << config_.num_runs << std::endl;
            TestResult r = runSingleTest(name, det, hand);
            detailed_results_[name].push_back(r);
            updateStatistics(name, r);
            if (run == 0 && config_.save_pcd) savePcds(name, r);
            if (run == 0 && config_.save_error_pcd) std::cout << "(<method>_error.pcd is a visual artefact and is not written by this build)" << std::endl;
        }
        return true;
    }

    void transformCloud(const Mat4& T, std::vector<float>& out) const {
        out.resize(source_.xyzi.size());
        for (size_t i = 0; i < source_.size(); ++i) {
            const double x = source_.xyzi[4 * i], y = source_.xyzi[4 * i + 1], z = source_.xyzi[4 * i + 2];
            for (int k = 0; k < 3; ++k) out[4 * i + k] = (float)(T.m[k * 4] * x + T.m[k * 4 + 1] * y + T.m[k * 4 + 2] * z + T.m[k * 4 + 3]);
            out[4 * i + 3] = source_.xyzi[4 * i + 3];
        }
    }

    void savePcds(const std::string& name, const TestResult& r) {                // icp_test_runner.cpp:347-381, 520-552
        std::vector<float> aligned, initial;
        transformCloud(r.final_transform, aligned);
        transformCloud(config_.initial_matrix, initial);
        std::vector<float> xyz; std::vector<uint32_t> rgb;
        auto push = [&](const std::vector<float>& c, uint32_t col) {
            for (size_t i = 0; i < c.size() / 4; ++i) { xyz.insert(xyz.end(), {c[4 * i], c[4 * i + 1], c[4 * i + 2]}); rgb.push_back(col); }
        };
        push(aligned, (245u << 16) | (121u << 8) | 0u);
        push(target_.xyzi, (144u << 16) | (159u << 8) | 207u);
        pcd::save_xyzrgb_binary(config_.output_folder + name + "_aligned_clouds.pcd", xyz, rgb);
        pcd::save_xyzi_binary(config_.output_folder + name + "_aligned_clouds_sig.pcd", aligned.data(), aligned.size() / 4);
        pcd::save_xyzi_binary(config_.output_folder + "initial_clouds.pcd", initial.data(), initial.size() / 4);
        pcd::save_xyzi_binary(config_.output_folder + "target_clouds.pcd", source_.xyzi.data(), source_.size());   // sic: the reference saves the SOURCE cloud here
        std::cout << "Saved aligned clouds for " << name << " to " << config_.output_folder + name + "_aligned_clouds.pcd" << std::endl;
    }

    void updateStatistics(const std::string& name, const TestResult& r) {        // icp_test_runner.cpp:603-630
        auto& s = statistics_[name];
        s.total_runs++;
        if (r.converged) s.converged_runs++;
        s.mean_trans_error += r.trans_error_m; s.mean_rot_error += r.rot_error_deg; s.mean_time_ms += r.time_ms;
        s.mean_iterations += r.iterations; s.mean_rmse += r.final_rmse; s.mean_fitness += r.final_fitness;
        s.mean_p2p_rmse += r.p2p_rmse; s.mean_p2p_fitness += r.p2p_fitness; s.mean_chamfer += r.chamfer_distance; s.corr_num += r.corr_num;
        s.min_trans_error = std::min(s.min_trans_error, r.trans_error_m); s.max_trans_error = std::max(s.max_trans_error, r.trans_error_m);
        s.min_rot_error = std::min(s.min_rot_error, r.rot_error_deg); s.max_rot_error = std::max(s.max_rot_error, r.rot_error_deg);
    }

    void finalizeStatistics() {                                                   // icp_test_runner.cpp:633-665
        for (auto& kv : statistics_) {
            auto& s = kv.second;
            if (s.total_runs == 0) continue;
            const double n = s.total_runs;
            s.mean_trans_error /= n; s.mean_rot_error /= n; s.mean_time_ms /= n; s.mean_iterations /= n; s.mean_rmse /= n;
            s.mean_fitness /= n; s.mean_p2p_rmse /= n; s.mean_p2p_fitness /= n; s.mean_chamfer /= n;
            s.success_rate = s.converged_runs / n;
            double a = 0, b = 0, c = 0;
            for (const auto& r : detailed_results_[kv.first]) {
                a += std::pow(r.trans_error_m - s.mean_trans_error, 2); b += std::pow(r.rot_error_deg - s.mean_rot_error, 2);
                c += std::pow(r.time_ms - s.mean_time_ms, 2);
            }
            s.std_trans_error = std::sqrt(a / n); s.std_rot_error = std::sqrt(b / n); s.std_time_ms = std::sqrt(c / n);
        }
    }

    void saveStatistics() {                                                       // icp_test_runner.cpp:668-796
        const std::string filename = config_.output_folder + "statistics_summary.txt";
        std::ofstream file(filename);
        if (!file.is_open()) { std::cerr << "Failed to open statistics file: " << filename << std::endl; return; }
        file << "ICP Test Statistics Summary\n===========================\n\nConfiguration:\n";
        file << "  Source: " << config_.source_pcd << "\n  Target: " << config_.target_pcd << "\n";
        file << "  Cloud size: " << source_.size() << " " << target_.size() << "\n  Runs per method: " << config_.num_runs << "\n\n";
        file << std::fixed << std::setprecision(6);
        file << std::setw(15) << "Method" << std::setw(12) << "Success%" << std::setw(12) << "Trans(m)" << std::setw(12) << "Rot(deg)"
             << std::setw(12) << "ICP_RMSE" << std::setw(12) << "Avg_Iters" << std::setw(12) << "P2PDis" << std::setw(12) << "ChamferDis"
             << std::setw(12) << "P2P_Fit%" << std::setw(12) << "P2P_Corr" << std::setw(12) << "Time(ms)\n";
        file << std::string(135, '-') << "\n";
        for (const auto& kv : statistics_) {
            const auto& s = kv.second;
            file << std::setw(15) << kv.first << std::setw(12) << std::fixed << std::setprecision(1) << (s.success_rate * 100)
                 << std::setw(12) << std::setprecision(4) << s.mean_trans_error << std::setw(12) << s.mean_rot_error
                 << std::setw(12) << s.mean_rmse << std::setw(12) << std::setprecision(1) << s.mean_iterations
                 << std::setw(12) << std::setprecision(4) << s.mean_p2p_rmse << std::setw(12) << s.mean_chamfer
                 << std::setw(12) << std::setprecision(2) << (s.mean_p2p_fitness * 100) << std::setw(12) << std::setprecision(1) << s.corr_num
                 << std::setw(12) << std::setprecision(2) << s.mean_time_ms << "\n";
        }
        file << "\n\nDetailed Statistics:\n===================\n\n";
        for (const auto& kv : statistics_) {
            const auto& s = kv.second;
            file << "Method: " << kv.first << "\n";
            file << "  Converged: " << s.converged_runs << "/" << s.total_runs << " (Success Rate: " << std::fixed << std::setprecision(1)
                 << (s.success_rate * 100) << "%)\n";
            file << "  Iterations: " << std::setprecision(1) << s.mean_iterations << "\n";
            file << "  Translation Error (m): " << std::setprecision(6) << s.mean_trans_error << " ± " << s.std_trans_error << " ["
                 << s.min_trans_error << ", " << s.max_trans_error << "]\n";
            file << "  Rotation Error (deg): " << s.mean_rot_error << " ± " << s.std_rot_error << " [" << s.min_rot_error << ", "
                 << s.max_rot_error << "]\n";
            file << "  Time (ms): " << std::setprecision(2) << s.mean_time_ms << " ± " << s.std_time_ms << "\n";
            file << "  ICP RMSE: " << std::setprecision(6) << s.mean_rmse << "\n  ICP Fitness: " << std::setprecision(4) << s.mean_fitness << "\n";
            file << "  ICP Correspondence: " << s.corr_num << "\n  Point-to-Point RMSE: " << std::setprecision(6) << s.mean_p2p_rmse << "\n";
            file << "  Point-to-Point Fitness: " << std::setprecision(4) << s.mean_p2p_fitness << "\n  Chamfer Distance: " << std::setprecision(6)
                 << s.mean_chamfer << "\n\n";
        }
        file.close();
        std::cout << "Statistics saved to: " << filename << std::endl;

        std::ofstream lg(config_.output_folder + "complete_log.txt");
        if (lg.is_open()) {
            lg << std::fixed << std::setprecision(6) << "Complete ICP Test Log\n====================\n\nConfiguration:\n";
            lg << "  Source: " << config_.source_pcd << "\n  Target: " << config_.target_pcd << "\n  Runs: " << config_.num_runs << "\n";
            lg << "  Initial noise: x=" << config_.initial_noise.x << ", y=" << config_.initial_noise.y << ", z=" << config_.initial_noise.z
               << ", roll=" << rad2deg(config_.initial_noise.roll) << ", pitch=" << rad2deg(config_.initial_noise.pitch)
               << ", yaw=" << rad2deg(config_.initial_noise.yaw) << " deg\n\n";
            lg << "ICP Parameters:\n  DEGENERACY_THRES_COND: " << config_.icp_params.DEGENERACY_THRES_COND
               << "\n  DEGENERACY_THRES_EIG: " << config_.icp_params.DEGENERACY_THRES_EIG << "\n  STD_REG_GAMMA: " << config_.icp_params.STD_REG_GAMMA
               << "\n  ADAPTIVE_REG_ALPHA: " << config_.icp_params.ADAPTIVE_REG_ALPHA << "\n  KAPPA_TARGET: " << config_.icp_params.KAPPA_TARGET
               << "\n  PCG_TOLERANCE: " << config_.icp_params.PCG_TOLERANCE << "\n  PCG_MAX_ITER: " << config_.icp_params.PCG_MAX_ITER << "\n\n";
            lg << "Results Summary:\n================\n";
            for (const auto& kv : statistics_) {
                const auto& s = kv.second;
                lg << "\nMethod: " << kv.first << "\n  Success rate: " << (s.success_rate * 100) << "%\n  Trans error: " << s.mean_trans_error << " ± "
                   << s.std_trans_error << " m\n  Rot error: " << s.mean_rot_error << " ± " << s.std_rot_error << " deg\n  P2P RMSE: "
                   << s.mean_p2p_rmse << " m\n  Chamfer: " << s.mean_chamfer << " m\n  Time: " << s.mean_time_ms << " ± " << s.std_time_ms << " ms\n";
            }
            std::cout << "Complete log saved to: " << config_.output_folder + "complete_log.txt" << std::endl;
        }
    }

    static void writeAlignment(std::ofstream& f, const dcreg_analysis& a) {      // icp_test_runner.cpp:1143-1187 (paper Alg. 2 report)
        f << "  Alignment Analysis:\n";
        for (int blk = 0; blk < 2; ++blk) {
            f << (blk == 0 ? "    Rotation Axes:\n" : "    Translation Axes:\n");
            const double* V = blk == 0 ? a.aligned_V_rot : a.aligned_V_trans;
            const int* idx = blk == 0 ? a.rot_indices : a.trans_indices;
            const double* lam = blk == 0 ? a.lambda_schur_rot : a.lambda_schur_trans;
            const char* nm = blk == 0 ? "RPY" : "XYZ";
            for (int i = 0; i < 3; ++i) {
                const double v[3] = {V[0 * 3 + i], V[1 * 3 + i], V[2 * 3 + i]};
                const double dot = std::fabs(v[i]);
                const double ang = std::acos(std::min(1.0, std::max(0.0, dot))) * 180.0 / kPi;
                const double sabs = std::max(1e-9, std::fabs(v[0]) + std::fabs(v[1]) + std::fabs(v[2]));
                const double l = (idx[i] >= 0 && idx[i] < 3) ? lam[idx[i]] : NAN;
                f << "      [" << i << "]~" << nm[i] << " (orig_idx=" << idx[i] << "): λ=" << l << ", Angle=" << ang << "°, "
                  << 100 * std::fabs(v[0]) / sabs << "%" << nm[0] << "+" << 100 * std::fabs(v[1]) / sabs << "%" << nm[1] << "+"
                  << 100 * std::fabs(v[2]) / sabs << "%" << nm[2] << "\n";
            }
        }
        f << " \n";
    }

    static void writeP(std::ofstream& f, const double* P) {
        f << "  Preconditioner Matrix P:\n";
        for (int i = 0; i < 6; ++i) {
            f << "    ";
            for (int j = 0; j < 6; ++j) f << std::setw(12) << P[i * 6 + j] << " ";
            f << "\n";
        }
        f << "\n";
    }

    void saveDetailedResults() {                                                  // icp_test_runner.cpp:799-1510
        {   // transform_details.csv
            std::ofstream tf(config_.output_folder + "transform_details.csv");
            tf << "Method,Run,Converged,Iterations,Time_ms,Trans_Error_m,Rot_Error_deg,Final_RMSE,Final_Fitness,Corr_Number,";
            for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) tf << "Transform_" << i << j << ",";
            tf << "SVD_Sigma_0,SVD_Sigma_1,SVD_Sigma_2,SVD_Sigma_3,SVD_Sigma_4,SVD_Sigma_5,";
            tf << "EVD_Lambda_0,EVD_Lambda_1,EVD_Lambda_2,EVD_Lambda_3,EVD_Lambda_4,EVD_Lambda_5,";
            tf << "Schur_Rot_Lambda_0,Schur_Rot_Lambda_1,Schur_Rot_Lambda_2,Schur_Trans_Lambda_0,Schur_Trans_Lambda_1,Schur_Trans_Lambda_2,";
            tf << "Cond_Full_SVD,Cond_Sub_Rot,Cond_Sub_Trans,Cond_Schur_Rot,Cond_Schur_Trans,";
            tf << "Degenerate_Mask_0,Degenerate_Mask_1,Degenerate_Mask_2,Degenerate_Mask_3,Degenerate_Mask_4,Degenerate_Mask_5";
            tf << "SuperLoc_Has_Data,SuperLoc_Uncertainty_X,SuperLoc_Uncertainty_Y,SuperLoc_Uncertainty_Z,";
            tf << "SuperLoc_Uncertainty_Roll,SuperLoc_Uncertainty_Pitch,SuperLoc_Uncertainty_Yaw,";
            tf << "SuperLoc_Cond_Full,SuperLoc_Cond_Rot,SuperLoc_Cond_Trans,SuperLoc_Is_Degenerate\n";
            for (const auto& kv : detailed_results_) {
                int run = 0;
                for (const auto& r : kv.second) {
                    tf << kv.first << "," << run++ << "," << (r.converged ? 1 : 0) << "," << r.iterations << "," << r.time_ms << ","
                       << r.trans_error_m << "," << r.rot_error_deg << "," << r.final_rmse << "," << r.final_fitness << "," << r.corr_num << ",";
                    for (int i = 0; i < 16; ++i) { tf << r.final_transform.m[i]; if (i < 15) tf << ","; }
                    if (r.eigenvalues.size() >= 6) { for (int rep = 0; rep < 2; ++rep) for (int i = 0; i < 6; ++i) tf << r.eigenvalues[i] << ","; }
                    else for (int i = 0; i < 12; ++i) tf << "0.0,";
                    for (int i = 0; i < 6; ++i) tf << "0.0,";
                    for (size_t i = 0; i < r.condition_numbers.size() && i < 5; ++i) tf << r.condition_numbers[i] << ",";
                    for (size_t i = r.condition_numbers.size(); i < 5; ++i) tf << "0.0,";
                    for (int i = 0; i < 6; ++i) { tf << (i < (int)r.degenerate_mask.size() ? (r.degenerate_mask[i] ? 1 : 0) : 0); if (i < 5) tf << ","; }
                    tf << "0,NaN,NaN,NaN,NaN,NaN,NaN,NaN,NaN,NaN,0\n";
                }
            }
        }
        if (config_.num_runs == 1) {   // condition_numbers_detailed.csv
            std::ofstream cf(config_.output_folder + "condition_numbers_detailed.csv");
            cf << "Method,Iteration,Effective_Points,RMSE,Fitness,Cond_Schur_Rot,Cond_Schur_Trans,Cond_Diag_Rot,Cond_Diag_Trans,"
               << "Cond_Full_EVD_Sub_Rot,Cond_Full_EVD_Sub_Trans,Cond_Full_SVD,Lambda_Schur_Rot_0,Lambda_Schur_Rot_1,Lambda_Schur_Rot_2,"
               << "Lambda_Schur_Trans_0,Lambda_Schur_Trans_1,Lambda_Schur_Trans_2,Eigenvalues_Full_0,Eigenvalues_Full_1,Eigenvalues_Full_2,"
               << "Eigenvalues_Full_3,Eigenvalues_Full_4,Eigenvalues_Full_5,Singular_Values_0,Singular_Values_1,Singular_Values_2,"
               << "Singular_Values_3,Singular_Values_4,Singular_Values_5,Is_Degenerate,Degenerate_Mask_0,Degenerate_Mask_1,Degenerate_Mask_2,"
               << "Degenerate_Mask_3,Degenerate_Mask_4,Degenerate_Mask_5\n";
            for (const auto& kv : detailed_results_) {
                if (kv.second.empty()) continue;
                for (const auto& d : kv.second[0].iteration_data) {
                    const dcreg_analysis& a = d.g.analysis;
                    cf << kv.first << "," << d.g.iter << "," << d.g.n_effective << "," << d.g.rmse << "," << d.g.fitness << ","
                       << a.cond_schur_rot << "," << a.cond_schur_trans << "," << a.cond_diag_rot << "," << a.cond_diag_trans << ","
                       << a.cond_full_sub_rot << "," << a.cond_full_sub_trans << "," << a.cond_full << ",";
                    for (int i = 0; i < 3; ++i) cf << a.lambda_schur_rot[i] << ",";
                    for (int i = 0; i < 3; ++i) cf << a.lambda_schur_trans[i] << ",";
                    for (int i = 0; i < 6; ++i) cf << a.eigenvalues_full[i] << ",";
                    for (int i = 0; i < 6; ++i) cf << a.singular_values[i] << ",";
                    cf << (a.is_degenerate ? 1 : 0) << ",";
                    for (int i = 0; i < 6; ++i) { cf << (a.degenerate_mask[i] ? 1 : 0); if (i < 5) cf << ","; }
                    cf << "\n";
                }
            }
        }
        {   // all_results.csv
            std::ofstream csv(config_.output_folder + "all_results.csv");
            csv << "Method,Run,Converged,Iterations,Time_ms,Trans_Error_m,Rot_Error_deg,ICP_RMSE,ICP_Fitness,P2P_RMSE,P2P_Fitness,Chamfer_Distance\n";
            for (const auto& kv : detailed_results_) {
                int run = 0;
                for (const auto& r : kv.second)
                    csv << kv.first << "," << run++ << "," << (r.converged ? 1 : 0) << "," << r.iterations << "," << r.time_ms << "," << r.trans_error_m
                        << "," << r.rot_error_deg << "," << r.final_rmse << "," << r.final_fitness << "," << r.p2p_rmse << "," << r.p2p_fitness << ","
                        << r.chamfer_distance << "\n";
            }
        }
        if (config_.num_runs == 1) {   // degeneracy_analysis_first_iter.txt
            std::ofstream dn(config_.output_folder + "degeneracy_analysis_first_iter.txt");
            dn << "Degeneracy Analysis Results (First Iteration)\n============================================\n\n";
            for (const auto& kv : detailed_results_) {
                if (kv.second.empty()) continue;
                const auto& r = kv.second[0];
                if (r.iteration_data.empty()) { dn << "Method: " << kv.first << " - No iteration data available\n\n"; continue; }
                const dcreg_analysis& a = r.iteration_data[0].g.analysis;
                dn << "Method: " << kv.first << "\n  Condition Numbers:\n" << std::fixed << std::setprecision(2);
                dn << "    Schur Rot: " << a.cond_schur_rot << "\n    Schur Trans: " << a.cond_schur_trans << "\n    Diag Rot: " << a.cond_diag_rot
                   << "\n    Diag Trans: " << a.cond_diag_trans << "\n    SVD Diag Rot: " << a.cond_full_sub_rot << "\n    SVD Diag Trans: "
                   << a.cond_full_sub_trans << "\n    Full SVD: " << a.cond_full << "\n";
                dn << "  Eigenvalues (Full): " << std::setprecision(3);
                for (int i = 0; i < 6; ++i) dn << a.eigenvalues_full[i] << " ";
                dn << "\n  Degenerate Mask (wxwywz xyz): ";
                for (int i = 0; i < 6; ++i) dn << (a.degenerate_mask[i] ? "1" : "0") << " ";
                dn << "\n  Is Degenerate: " << (a.is_degenerate ? "Yes" : "No") << "\n\n" << std::setprecision(6);
                if (kv.first.find("PCG") != std::string::npos || kv.first == "Ours") writeP(dn, a.P_preconditioner);
                if ((kv.first == "Ours" || kv.first.find("SCHUR") != std::string::npos) && a.is_degenerate) writeAlignment(dn, a);
            }
            dn << "\n\n";
        }
        {   // degeneracy_analysis_last_iter.txt
            std::ofstream dg(config_.output_folder + "degeneracy_analysis_last_iter.txt");
            dg << std::fixed << std::setprecision(6) << "Degeneracy Analysis Results\n==========================\n\n";
            for (const auto& kv : detailed_results_) {
                if (kv.second.empty()) continue;
                const auto& r = kv.second[0];
                dg << "Method: " << kv.first << "\nFinal Transform Matrix:\n";
                for (int i = 0; i < 4; ++i) { for (int j = 0; j < 4; ++j) dg << std::setw(12) << r.final_transform.m[i * 4 + j] << " "; dg << "\n"; }
                dg << "\n";
                if (!r.iteration_data.empty()) {
                    const dcreg_analysis& a = r.iteration_data.back().g.analysis;
                    dg << "  Condition Numbers:\n    Schur Rot: " << a.cond_schur_rot << "\n    Schur Trans: " << a.cond_schur_trans << "\n    Diag Rot: "
                       << a.cond_diag_rot << "\n    Diag Trans: " << a.cond_diag_trans << "\n    SVD Diag Rot: " << a.cond_full_sub_rot
                       << "\n    SVD Diag Trans: " << a.cond_full_sub_trans << "\n    Full SVD: " << a.cond_full << "\n\n";
                    dg << "  EVD Eigenvalues (Full):\n";
                    for (int i = 0; i < 6; ++i) dg << "    λ" << i << ": " << a.eigenvalues_full[i] << "\n";
                    dg << "\n  SVD Singular Values:\n";
                    for (int i = 0; i < 6; ++i) dg << "    σ" << i << ": " << a.singular_values[i] << "\n";
                    dg << "\n  Diagonal Block Eigenvalues:\n    Rotation: [" << a.lambda_sub_rot[0] << " " << a.lambda_sub_rot[1] << " " << a.lambda_sub_rot[2]
                       << "]\n    Translation: [" << a.lambda_sub_trans[0] << " " << a.lambda_sub_trans[1] << " " << a.lambda_sub_trans[2] << "]\n\n";
                    dg << "  Schur Complement Eigenvalues:\n    Rotation: [" << a.lambda_schur_rot[0] << " " << a.lambda_schur_rot[1] << " " << a.lambda_schur_rot[2]
                       << "]\n    Translation: [" << a.lambda_schur_trans[0] << " " << a.lambda_schur_trans[1] << " " << a.lambda_schur_trans[2] << "]\n\n";
                    dg << "  Degenerate Mask (ωxωyωz xyz): ";
                    for (int i = 0; i < 6; ++i) dg << (a.degenerate_mask[i] ? "1" : "0") << " ";
                    dg << "\n\n";
                    if (kv.first.find("PCG") != std::string::npos || kv.first == "Ours") writeP(dg, a.P_preconditioner);
                    if ((kv.first == "Ours" || kv.first.find("SCHUR") != std::string::npos) && a.is_degenerate) writeAlignment(dg, a);
                }
                dg << "\n" << std::string(60, '-') << "\n\n";
            }
        }
        {   // iteration_history.csv
            std::ofstream ih(config_.output_folder + "iteration_history.csv");
            ih << "Method,Iteration,RMSE,Fitness,TransError,RotError,CorrNum\n" << std::fixed << std::setprecision(8);
            for (const auto& kv : detailed_results_) {
                if (kv.second.empty()) continue;
                for (const auto& d : kv.second[0].iteration_data)
                    ih << kv.first << "," << d.g.iter << "," << d.g.rmse << "," << d.g.fitness << "," << d.trans_error_vs_gt << "," << d.rot_error_vs_gt
                       << "," << d.g.n_effective << "\n";
            }
        }
        {   // iteration_details_with_dx.csv (SURVEY.md Appendix B.4)
            std::ofstream ic(config_.output_folder + "iteration_details_with_dx.csv");
            ic << std::fixed << std::setprecision(8);
            ic << "Method,Run,Iteration,RMSE,Fitness,Time_ms,Trans_Error_m,Rot_Error_deg,P2P_RMSE,Chamfer_Distance,"
               << "dx_wx,dx_wy,dx_wz,dx_x,dx_y,dx_z,grad_wx,grad_wy,grad_wz,grad_x,grad_y,grad_z,objective_value,";
            for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) ic << "T_" << i << j << ",";
            ic << "Cond_Schur_Rot,Cond_Schur_Trans,Cond_Sub_Rot,Cond_Sub_Trans,Cond_Full_SVD,";
            for (int i = 0; i < 6; ++i) ic << "Degenerate_" << i << ",";
            ic << "Is_Degenerate\n";
            for (const auto& kv : detailed_results_)
                for (size_t run = 0; run < kv.second.size(); ++run) {
                    // the reference evaluates every row's pose (icp_test_runner.cpp:1460-1468); one batched call per run
                    const std::vector<IterData>& iters = kv.second[run].iteration_data;
                    std::vector<double> poses(iters.size() * 16), p2p_out;
                    for (size_t it = 0; it < iters.size(); ++it) std::memcpy(&poses[it * 16], iters[it].g.T, 16 * sizeof(double));
                    p2pBatch(poses, p2p_out);
                    for (size_t it = 0; it < iters.size(); ++it) {
                        const IterData& d = iters[it];
                        Mat4 Ti; std::memcpy(Ti.m, d.g.T, sizeof(Ti.m));
                        const PoseError e = calculatePoseError(config_.gt_matrix, Ti);
                        const double trans_error = e.rotation_error, rot_error = e.translation_error;   // sic (icp_test_runner.cpp:1457-1458)
                        const double p2p_rmse = p2p_out[it * 4], chamfer = p2p_out[it * 4 + 2];
                        ic << kv.first << "," << run << "," << it << "," << d.g.rmse << "," << d.g.fitness << "," << d.iter_time_ms << ","
                           << trans_error << "," << rot_error << "," << p2p_rmse << "," << chamfer << ",";
                        for (int i = 0; i < 6; ++i) ic << d.g.dx[i] << ",";
                        for (int i = 0; i < 6; ++i) ic << d.g.gradient[i] << ",";
                        ic << d.g.objective << ",";
                        for (int i = 0; i < 16; ++i) ic << d.g.T[i] << ",";
                        const dcreg_analysis& a = d.g.analysis;
                        ic << a.cond_schur_rot << "," << a.cond_schur_trans << "," << a.cond_diag_rot << "," << a.cond_diag_trans << "," << a.cond_full << ",";
                        for (int i = 0; i < 6; ++i) ic << (a.degenerate_mask[i] ? 1 : 0) << ",";
                        ic << (a.is_degenerate ? 1 : 0) << "\n";
                    }
                }
            std::cout << "Iteration details with dx saved to: " << config_.output_folder + "iteration_details_with_dx.csv" << std::endl;
        }
    }
};

void make_dirs(const std::string& path) {
    std::string cur;
    for (size_t i = 0; i < path.size(); ++i) {
        cur.push_back(path[i]);
        if (path[i] == '/' || i + 1 == path.size()) ::mkdir(cur.c_str(), 0755);
    }
}

// Host-only self checks used by the CPU test-suite (no device needed).
int dumpConfig(const std::string& config_file) {
    Config c;
    if (!loadConfig(config_file, c)) return 1;
    std::cout << std::setprecision(17);
    std::cout << "num_runs=" << c.num_runs << "\nsave_pcd=" << c.save_pcd << "\nsave_error_pcd=" << c.save_error_pcd << "\nvisualize=" << c.visualize
              << "\nfolder_path=" << c.folder_path << "\nsource_pcd=" << c.source_pcd << "\ntarget_pcd=" << c.target_pcd << "\noutput_folder="
              << c.output_folder << "\nsearch_radius=" << c.search_radius << "\nmax_iterations=" << c.max_iterations << "\nnormal_nn=" << c.normal_nn
              << "\nerror_threshold=" << c.error_threshold << "\nCONVERGENCE_THRESH_TRANS=" << c.CONVERGENCE_THRESH_TRANS
              << "\nCONVERGENCE_THRESH_ROT=" << c.CONVERGENCE_THRESH_ROT << "\nuse_weight_derivative=" << c.use_weight_derivative
              << "\nDEGENERACY_THRES_COND=" << c.icp_params.DEGENERACY_THRES_COND << "\nDEGENERACY_THRES_EIG=" << c.icp_params.DEGENERACY_THRES_EIG
              << "\nSTD_REG_GAMMA=" << c.icp_params.STD_REG_GAMMA << "\nKAPPA_TARGET=" << c.icp_params.KAPPA_TARGET << "\nPCG_TOLERANCE="
              << c.icp_params.PCG_TOLERANCE << "\nPCG_MAX_ITER=" << c.icp_params.PCG_MAX_ITER << "\nTSVD_SINGULAR_THRESH="
              << c.icp_params.TSVD_SINGULAR_THRESH << "\nLOAM_EIGEN_THRESH=" << c.icp_params.LOAM_EIGEN_THRESH << "\nmc_trials=" << c.mc_trials
              << "\nmc_seed=" << c.mc_seed << "\nmc_max_trans=" << c.mc_max_trans << "\nmc_max_rot_deg=" << c.mc_max_rot_deg << "\n";
    std::cout << "initial_matrix=";
    for (int i = 0; i < 16; ++i) std::cout << c.initial_matrix.m[i] << (i < 15 ? "," : "\n");
    std::cout << "gt_matrix=";
    for (int i = 0; i < 16; ++i) std::cout << c.gt_matrix.m[i] << (i < 15 ? "," : "\n");
    for (const auto& kv : c.test_methods)
        std::cout << "method=" << kv.first << "|" << kv.second.first << "|" << kv.second.second << "|" << detection_from_string(kv.second.first) << "|"
                  << handling_from_string(kv.second.second) << "\n";
    return 0;
}

int pcdRoundtrip(const std::string& in, const std::string& out) {
    pcd::Cloud c;
    std::string err;
    if (!pcd::load(in, c, &err)) { std::cerr << err << std::endl; return 1; }
    if (!pcd::save_xyzi_binary(out, c.xyzi.data(), c.size())) { std::cerr << "cannot write " << out << std::endl; return 1; }
    std::cout << "points=" << c.size() << std::endl;
    return 0;
}

int poseError(char** v) {           // 32 doubles: gt (row-major 4x4) then final
    Mat4 a, b;
    for (int i = 0; i < 16; ++i) { a.m[i] = std::atof(v[i]); b.m[i] = std::atof(v[16 + i]); }
    const PoseError e = calculatePoseError(a, b);
    std::cout << std::setprecision(17) << e.translation_error << " " << e.rotation_error << std::endl;
    return 0;
}

}  // namespace

int main(int argc, char** argv) {                                 // DCReg/src/icp_main.cpp:6-52
    if (argc == 3 && std::string(argv[1]) == "--dump-config") return dumpConfig(argv[2]);
    if (argc == 4 && std::string(argv[1]) == "--pcd-roundtrip") return pcdRoundtrip(argv[2], argv[3]);
    if (argc == 34 && std::string(argv[1]) == "--pose-error") return poseError(argv + 2);
    std::cout << "=== ICP Test Runner ===" << std::endl;
    const std::string config_file = argc > 1 ? argv[1] : "../config/icp.yaml";
    Config config;
    if (!loadConfig(config_file, config)) { std::cerr << "Failed to load configuration file: " << config_file << std::endl; return -1; }
    make_dirs(config.output_folder);
    std::cout << "\nConfiguration loaded successfully!" << std::endl;
    std::cout << "Number of runs: " << config.num_runs << std::endl;
    std::cout << "Source PCD: " << config.source_pcd << std::endl;
    std::cout << "Target PCD: " << config.target_pcd << std::endl;
    std::cout << "Output folder: " << config.output_folder << std::endl;
    TestRunner runner(config);
    if (!runner.runAllTests()) { std::cerr << "Test run failed!" << std::endl; return -1; }
    std::cout << "\n=== All tests completed successfully! ===" << std::endl;
    return 0;
}
