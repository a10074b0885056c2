// calc_grasppoints_b200.hpp -- ROS-free C++ host mirror of the hot-path-facing part of the reference's
// CCalc_Grasppoints (src/calc_grasppoints_action_server.cpp), sitting directly on the C ABI (include/hafgpu.h).
// Same member names, same argument meaning, same result fields, so a maintainer can lift the bodies into the ROS
// node (INTEGRATION.md) and the tests read like the reference's flow:
//     read_pc_cb (goal -> members, :250-329)  ->  loop_control (:335-402)  ->  transform_gp_in_wcs_and_publish (:1274-1401)
// Everything numeric on the hot path happens in libhafgpu (CUDA), the grasp poses included; this file only keeps the
// reference's bookkeeping.
#pragma once
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../../include/hafgpu.h"
#include "pcd_io.hpp"

namespace haf_b200 {

struct Point3 { double x = 0, y = 0, z = 0; };

// hot-path fields of haf_grasping/GraspInput (msg/GraspInput.msg:3-15)
struct GraspInput {
    Point3 grasp_area_center;
    float grasp_area_length_x = 32, grasp_area_length_y = 44;   // client default 18x30 + 14 (client.cpp:183-184)
    Point3 approach_vector{};                                     // default (0,0,1) set below
    int gripper_opening_width = 1;
    bool show_only_best_grasp = false;
    double max_calculation_time = 50;                             // seconds; mapped to roll_limit by the caller
    GraspInput() { approach_vector.z = 1; }
};

// haf_grasping/GraspOutput (msg/GraspOutput.msg:1-7)
struct GraspOutput {
    int eval = -20;
    Point3 graspPoint1, graspPoint2, averagedGraspPoint, approachVector;
    float roll = 0;
};

class CCalc_Grasppoints_B200 {
public:
    // members named like the reference's (server.cpp:130-163)
    Point3 graspsearchcenter;
    int grasp_search_area_size_x_dir = 32, grasp_search_area_size_y_dir = 44;
    Point3 approach_vector;
    int gripper_opening_width = 1;
    bool return_only_best_gp = false;
    int graspval_th = 70, graspval_top = 119;
    int id_row_top_overall = -1, id_col_top_overall = -1, nr_roll_top_overall = -1, nr_tilt_top_overall = -1, topval_gp_overall = -1000;
    float av_trans_mat[16];
    float trans_z_after_pc_transform = 0.15f;
    GraspOutput gp_result;
    int G, R;
    std::vector<float> heightsgridroll;          // [R][G][G]
    std::vector<unsigned char> point_inside_box_grid;  // [R][G][G]
    std::vector<float> graspseval;               // [R][G][G]
    std::vector<int> per_roll_top;               // [R][3]
    haf_best best;
    std::vector<GraspOutput> published_per_roll; // what :962-972 would publish when !return_only_best_gp

    CCalc_Grasppoints_B200(const std::string& feature_file_path, const std::string& range_file_path,
                           const std::string& svmmodel_file_path, int nr_features_without_shaf = 302, int grid = 56,
                           int roll_steps_degree = 15, int roll_max_degree = 190, int device = 0, int svm_mode = HAF_SVM_TENSOR_GUARD)
        : G(grid), R(roll_max_degree / roll_steps_degree), step_deg_(roll_steps_degree) {
        haf_config cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.features_path = feature_file_path.c_str();
        cfg.range_path = range_file_path.c_str();
        cfg.model_path = svmmodel_file_path.c_str();
        cfg.nr_features_without_shaf = nr_features_without_shaf;
        cfg.grid = grid; cfg.roll_step_deg = roll_steps_degree; cfg.roll_max_deg = roll_max_degree;
        cfg.device = device; cfg.emulate_text_roundtrip = 1; cfg.svm_mode = svm_mode;
        if (haf_create(&ctx_, &cfg) != HAF_OK) throw std::runtime_error(std::string("hafgpu: ") + haf_last_error(NULL));
        approach_vector.z = 1;
        memset(av_trans_mat, 0, sizeof av_trans_mat);
        heightsgridroll.assign((size_t)R * G * G, 0.0f);
        point_inside_box_grid.assign((size_t)R * G * G, 0);
        graspseval.assign((size_t)R * G * G, 0.0f);
        per_roll_top.assign((size_t)R * 3, -1);
        grasp_per_roll_.resize(R);
    }
    ~CCalc_Grasppoints_B200() { haf_destroy(ctx_); }
    CCalc_Grasppoints_B200(const CCalc_Grasppoints_B200&) = delete;
    CCalc_Grasppoints_B200& operator=(const CCalc_Grasppoints_B200&) = delete;

    // The client's open_pcd_and_trig_get_grasp_cb (src/calc_grasppoints_action_client.cpp:137-157: pcl::io::loadPCDFile, toROSMsg)
    // followed by the server's pcl::fromROSMsg (:313-316), as ONE device-side ingest: the file's bytes are decoded by kernels
    // (haf_pcd_decode) and the goal runs on the decoded cloud without the points ever existing in host memory.
    size_t open_pcd_and_trig_get_grasp_cb(const GraspInput& goal, const void* file_bytes, size_t n_bytes) {
        const float* d_xyz = NULL;
        size_t n = 0;
        if (haf_pcd_decode(ctx_, file_bytes, n_bytes, &d_xyz, &n) != HAF_OK) throw std::runtime_error(std::string("hafgpu: ") + haf_last_error(ctx_));
        read_pc_cb(goal, d_xyz, n, 12);
        return n;
    }

    // read_pc_cb (:250-329): goal -> members (the tf transform of the cloud is the caller's business), then loop_control
    void read_pc_cb(const GraspInput& goal, const float* xyz, size_t n_points, size_t stride_bytes) {
        set_goal(goal);
        loop_control(xyz, n_points, stride_bytes);
    }

    // One goal on every cloud of a batch: what loop_control leaves behind for each cloud when it runs on that cloud alone
    struct CloudResult {
        size_t n_points;
        haf_best best;                          // row, col, roll, tilt, topval, rolls_done, n_windows_scored as loop_control reads them
        GraspOutput gp_result;
        std::vector<int> per_roll_top;          // [R][3]
        std::vector<GraspOutput> published_per_roll;
    };
    // PCD files back to back in host memory (file f = bytes [file_offsets[f], file_offsets[f+1])), decoded on the device in one
    // call (haf_search_batch_pcd)
    std::vector<CloudResult> open_pcds_and_trig_get_grasps_cb(const GraspInput& goal, const void* files, const size_t* file_offsets, int n_files) {
        return batch_control(goal, files, file_offsets, NULL, NULL, n_files);
    }
    // clouds already decoded on the host: packed xyz, cloud c = points [point_offsets[c], point_offsets[c+1]) (haf_search_batch_requests)
    std::vector<CloudResult> read_pcs_cb(const GraspInput& goal, const float* xyz_all, const size_t* point_offsets, int n_clouds) {
        return batch_control(goal, NULL, NULL, xyz_all, point_offsets, n_clouds);
    }

    // goal -> members (:258-326)
    void set_goal(const GraspInput& goal) {
        graspsearchcenter = goal.grasp_area_center;                              // :258-260
        grasp_search_area_size_x_dir = (int)goal.grasp_area_length_x;             // :266-267
        grasp_search_area_size_y_dir = (int)goal.grasp_area_length_y;
        raw_approach_ = goal.approach_vector;
        float vector_length = (float)std::sqrt(goal.approach_vector.x * goal.approach_vector.x + goal.approach_vector.y * goal.approach_vector.y +
                                               goal.approach_vector.z * goal.approach_vector.z);   // :270
        approach_vector.x = goal.approach_vector.x / vector_length;               // :271-273
        approach_vector.y = goal.approach_vector.y / vector_length;
        approach_vector.z = goal.approach_vector.z / vector_length;
        gripper_opening_width = goal.gripper_opening_width;                       // :281
        return_only_best_gp = goal.show_only_best_grasp;                          // :284
        id_row_top_overall = id_col_top_overall = nr_roll_top_overall = nr_tilt_top_overall = -1;  // :322-326
        topval_gp_overall = -1000;
    }

    // loop_control (:335-402): the five per-roll calls (:376-385) and the grasp poses of transform_gp_in_wcs_and_publish
    // (:1274-1401) are ONE haf_search_grasps call; the poses are computed on the device (haf_grasp records)
    void loop_control(const float* xyz, size_t n_points, size_t stride_bytes, int roll_limit = 0) {
        haf_request rq = request(roll_limit);
        haf_grasp grasp;
        int rc = haf_search_grasps(ctx_, xyz, n_points, stride_bytes, &rq, 1, &best, NULL, graspseval.data(), point_inside_box_grid.data(),
                                   heightsgridroll.data(), per_roll_top.data(), &grasp, NULL, grasp_per_roll_.data());
        if (rc != HAF_OK) throw std::runtime_error(std::string("hafgpu: ") + haf_last_error(ctx_));
        published_per_roll = published(per_roll_top.data(), grasp_per_roll_.data(), best.rolls_done);
        // av_trans_mat (:484) = generate_grid's matrix of the roll just evaluated; only its third row is read (:1370-1374), and
        // that row is the same for every roll (S * Rroll leaves it untouched)
        haf_build_transform(&rq, best.roll >= 0 ? best.roll : 0, step_deg_, av_trans_mat);
        id_row_top_overall = best.row; id_col_top_overall = best.col; nr_roll_top_overall = best.roll;       // :953-960
        nr_tilt_top_overall = best.tilt; topval_gp_overall = best.topval;
        gp_result = to_grasp_output(grasp);                                       // :390 (eval = topval_gp_overall - 20)
    }

    // the GraspOutput message transform_gp_in_wcs_and_publish fills (:1384-1401) from the library's record
    static GraspOutput to_grasp_output(const haf_grasp& g) {
        GraspOutput out;
        out.eval = g.eval;
        out.graspPoint1.x = g.graspPoint1[0]; out.graspPoint1.y = g.graspPoint1[1]; out.graspPoint1.z = g.graspPoint1[2];
        out.graspPoint2.x = g.graspPoint2[0]; out.graspPoint2.y = g.graspPoint2[1]; out.graspPoint2.z = g.graspPoint2[2];
        out.averagedGraspPoint.x = g.averagedGraspPoint[0]; out.averagedGraspPoint.y = g.averagedGraspPoint[1];
        out.averagedGraspPoint.z = g.averagedGraspPoint[2];
        out.approachVector.x = g.approachVector[0]; out.approachVector.y = g.approachVector[1]; out.approachVector.z = g.approachVector[2];
        out.roll = g.roll;
        return out;
    }

    haf_ctx* ctx() { return ctx_; }

private:
    // the request loop_control sends for the current members
    haf_request request(int roll_limit) const {
        haf_request rq;
        memset(&rq, 0, sizeof rq);
        rq.center[0] = graspsearchcenter.x; rq.center[1] = graspsearchcenter.y; rq.center[2] = graspsearchcenter.z;
        rq.area_len_x = (float)grasp_search_area_size_x_dir; rq.area_len_y = (float)grasp_search_area_size_y_dir;
        rq.approach[0] = raw_approach_.x; rq.approach[1] = raw_approach_.y; rq.approach[2] = raw_approach_.z;
        rq.gripper_opening_width = gripper_opening_width;
        rq.return_only_best = return_only_best_gp ? 1 : 0;
        rq.graspval_top = graspval_top;
        rq.roll_limit = roll_limit;
        return rq;
    }
    // what show_predicted_gps published per evaluated roll (:962-972; eval = max(top - 20, 10) in the record)
    std::vector<GraspOutput> published(const int* top, const haf_grasp* grasp_per_roll, int rolls_done) const {
        std::vector<GraspOutput> out;
        for (int roll = 0; roll < rolls_done; roll++)
            if (!return_only_best_gp && top[roll * 3 + 2] > graspval_th) out.push_back(to_grasp_output(grasp_per_roll[roll]));
        return out;
    }
    // one haf_search_batch_pcd (files) or haf_search_batch_requests (xyz_all) call with the goal's request for every cloud
    std::vector<CloudResult> batch_control(const GraspInput& goal, const void* files, const size_t* file_offsets, const float* xyz_all,
                                           const size_t* point_offsets, int n) {
        set_goal(goal);
        const std::vector<haf_request> reqs(n, request(0));
        std::vector<haf_best> best_c(n);
        std::vector<int> top((size_t)n * R * 3, -1);
        std::vector<haf_grasp> grasp_c(n), grasp_r((size_t)n * R);
        const int rc = files ? haf_search_batch_pcd(ctx_, files, file_offsets, n, reqs.data(), NULL, best_c.data(), NULL, top.data(), grasp_c.data(),
                                                    NULL, grasp_r.data())
                             : haf_search_batch_requests(ctx_, xyz_all, point_offsets, n, reqs.data(), NULL, best_c.data(), NULL, top.data(),
                                                         grasp_c.data(), NULL, grasp_r.data());
        if (rc != HAF_OK) throw std::runtime_error(std::string("hafgpu: ") + haf_last_error(ctx_));
        std::vector<size_t> pts(n + 1, 0);
        if (files) {   // the clouds' sizes: the headers' POINTS (the call above has parsed every header)
            for (int c = 0; c < n; c++) {
                hafpcd::PcdHeader hd;
                hafpcd::parse_pcd_header(static_cast<const unsigned char*>(files) + file_offsets[c], file_offsets[c + 1] - file_offsets[c], hd, NULL);
                pts[c + 1] = pts[c] + (size_t)hd.npts;
            }
        } else {
            pts.assign(point_offsets, point_offsets + n + 1);
        }
        std::vector<CloudResult> out(n);
        for (int c = 0; c < n; c++) {
            CloudResult& r = out[c];
            r.n_points = pts[c + 1] - pts[c];
            r.best = best_c[c];
            r.gp_result = to_grasp_output(grasp_c[c]);
            r.per_roll_top.assign(top.begin() + (size_t)c * R * 3, top.begin() + (size_t)(c + 1) * R * 3);
            r.published_per_roll = published(r.per_roll_top.data(), grasp_r.data() + (size_t)c * R, best_c[c].rolls_done);
        }
        return out;
    }

public:

private:
    haf_ctx* ctx_ = nullptr;
    int step_deg_;
    Point3 raw_approach_{};
    std::vector<haf_grasp> grasp_per_roll_;   // [R] records of the evaluated rolls (haf_search_grasps)
};

}  // namespace haf_b200
