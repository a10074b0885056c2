// haf_cli -- ROS-free harness: PCD + the GraspInput fields in, the GraspOutput fields (+ per-roll tops) out.
//   haf_cli --features F --range R --model M --pcd cloud.pcd [--center x y z] [--area lx ly] [--approach x y z]
//           [--width n] [--only-best] [--grid G] [--svm-mode 0|1|2] [--json] [--host-pcd]
// The PCD file is decoded ON THE DEVICE (haf_pcd_decode) unless --host-pcd asks for the host reader (pcd_io.hpp).
// --pcd may be repeated: the files are searched with the same goal in ONE batch call (haf_search_batch_pcd, or with --host-pcd
// haf_search_batch_requests on the host-decoded clouds), one output line per file in argument order, each what a run on that
// file alone prints.
//   haf_cli --pcd cloud.pcd --dump-pcd          (parse only, no GPU)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "calc_grasppoints_b200.hpp"
#include "pcd_io.hpp"

static bool read_file(const std::string& path, std::vector<unsigned char>& out) {
    FILE* fp = fopen(path.c_str(), "rb");
    if (!fp) return false;
    unsigned char buf[1 << 16];
    size_t nr;
    while ((nr = fread(buf, 1, sizeof buf, fp)) > 0) out.insert(out.end(), buf, buf + nr);
    fclose(fp);
    return true;
}

static void print_result(bool json, size_t n_points, const haf_best& best, const haf_b200::GraspOutput& g, const int* per_roll_top, int R,
                         size_t n_published) {
    if (json) {
        printf("{\"points\": %zu, \"row\": %d, \"col\": %d, \"roll_index\": %d, \"topval\": %d, \"eval\": %d, \"rolls_done\": %d, \"windows\": %d, "
               "\"graspPoint1\": [%.9g, %.9g, %.9g], \"graspPoint2\": [%.9g, %.9g, %.9g], \"averagedGraspPoint\": [%.9g, %.9g, %.9g], "
               "\"approachVector\": [%.9g, %.9g, %.9g], \"roll\": %.9g, \"per_roll_top\": [",
               n_points, best.row, best.col, best.roll, best.topval, g.eval,
               best.rolls_done, best.n_windows_scored, g.graspPoint1.x, g.graspPoint1.y, g.graspPoint1.z, g.graspPoint2.x,
               g.graspPoint2.y, g.graspPoint2.z, g.averagedGraspPoint.x, g.averagedGraspPoint.y, g.averagedGraspPoint.z, g.approachVector.x,
               g.approachVector.y, g.approachVector.z, (double)g.roll);
        for (int r = 0; r < R; r++) printf("%s[%d, %d, %d]", r ? ", " : "", per_roll_top[r * 3], per_roll_top[r * 3 + 1], per_roll_top[r * 3 + 2]);
        printf("], \"published_per_roll\": %zu}\n", n_published);
    } else {
        // same field order as the string the reference publishes on /haf_grasping/grasp_hypothesis_with_eval (:1384)
        printf("%d %g %g %g %g %g %g %g %g %g %g %g %g %d\n", g.eval, g.graspPoint1.x, g.graspPoint1.y, g.graspPoint1.z, g.graspPoint2.x,
               g.graspPoint2.y, g.graspPoint2.z, g.approachVector.x, g.approachVector.y, g.approachVector.z, g.averagedGraspPoint.x,
               g.averagedGraspPoint.y, g.averagedGraspPoint.z, best.roll * 15);
    }
}

int main(int argc, char** argv) {
    std::string features, range, model, pcd;
    std::vector<std::string> pcds;
    haf_b200::GraspInput goal;
    int grid = 56, svm_mode = HAF_SVM_TENSOR_GUARD;
    bool json = false, dump_pcd = false, host_pcd = false;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto need = [&](int n) { if (i + n >= argc) { fprintf(stderr, "haf_cli: %s needs %d value(s)\n", a.c_str(), n); exit(2); } };
        if (a == "--features") { need(1); features = argv[++i]; }
        else if (a == "--range") { need(1); range = argv[++i]; }
        else if (a == "--model") { need(1); model = argv[++i]; }
        else if (a == "--pcd") { need(1); pcd = argv[++i]; pcds.push_back(pcd); }
        else if (a == "--center") { need(3); goal.grasp_area_center.x = atof(argv[++i]); goal.grasp_area_center.y = atof(argv[++i]); goal.grasp_area_center.z = atof(argv[++i]); }
        else if (a == "--area") { need(2); goal.grasp_area_length_x = (float)atof(argv[++i]); goal.grasp_area_length_y = (float)atof(argv[++i]); }
        else if (a == "--approach") { need(3); goal.approach_vector.x = atof(argv[++i]); goal.approach_vector.y = atof(argv[++i]); goal.approach_vector.z = atof(argv[++i]); }
        else if (a == "--width") { need(1); goal.gripper_opening_width = atoi(argv[++i]); }
        else if (a == "--only-best") goal.show_only_best_grasp = true;
        else if (a == "--grid") { need(1); grid = atoi(argv[++i]); }
        else if (a == "--svm-mode") { need(1); svm_mode = atoi(argv[++i]); }
        else if (a == "--json") json = true;
        else if (a == "--dump-pcd") dump_pcd = true;
        else if (a == "--host-pcd") host_pcd = true;
        else { fprintf(stderr, "haf_cli: unknown argument %s\n", a.c_str()); return 2; }
    }
    if (dump_pcd && !pcd.empty()) {  // parse only (no GPU): point count + FNV-1a of the packed xyz bytes
        std::vector<float> pts;
        std::string e;
        if (!hafpcd::read_pcd(pcd, pts, &e)) { fprintf(stderr, "haf_cli: %s\n", e.c_str()); return 1; }
        unsigned long long h = 1469598103934665603ull;
        const unsigned char* b = reinterpret_cast<const unsigned char*>(pts.data());
        for (size_t k = 0; k < pts.size() * 4; k++) { h ^= b[k]; h *= 1099511628211ull; }
        printf("%zu %llu\n", pts.size() / 3, h);
        return 0;
    }
    if (features.empty() || range.empty() || model.empty() || pcd.empty()) {
        fprintf(stderr, "usage: haf_cli --features F --range R --model M --pcd cloud.pcd [--center x y z] [--area lx ly] [--approach x y z] [--width n] [--only-best] [--grid G] [--svm-mode m] [--json]\n");
        return 2;
    }
    if (pcds.size() > 1) {   // one batch call for all files
        std::vector<float> xyz_all;
        std::vector<unsigned char> files;
        std::vector<size_t> offsets(1, 0);
        for (size_t f = 0; f < pcds.size(); f++) {
            std::string err;
            if (host_pcd) {
                std::vector<float> xyz;
                if (!hafpcd::read_pcd(pcds[f], xyz, &err)) { fprintf(stderr, "haf_cli: %s\n", err.c_str()); return 1; }
                xyz_all.insert(xyz_all.end(), xyz.begin(), xyz.end());
                offsets.push_back(xyz_all.size() / 3);
            } else {
                if (!read_file(pcds[f], files)) { fprintf(stderr, "haf_cli: cannot open %s\n", pcds[f].c_str()); return 1; }
                offsets.push_back(files.size());
            }
        }
        try {
            haf_b200::CCalc_Grasppoints_B200 server(features, range, model, 302, grid, 15, 190, 0, svm_mode);
            const int n = (int)pcds.size();
            const std::vector<haf_b200::CCalc_Grasppoints_B200::CloudResult> res =
                host_pcd ? server.read_pcs_cb(goal, xyz_all.data(), offsets.data(), n) : server.open_pcds_and_trig_get_grasps_cb(goal, files.data(), offsets.data(), n);
            for (int f = 0; f < n; f++)
                print_result(json, res[f].n_points, res[f].best, res[f].gp_result, res[f].per_roll_top.data(), server.R, res[f].published_per_roll.size());
        } catch (const std::exception& e) {
            fprintf(stderr, "haf_cli: %s\n", e.what());
            return 1;
        }
        return 0;
    }
    std::vector<float> xyz;
    std::vector<unsigned char> file_bytes;
    std::string err;
    if (host_pcd) {
        if (!hafpcd::read_pcd(pcd, xyz, &err)) { fprintf(stderr, "haf_cli: %s\n", err.c_str()); return 1; }
    } else {
        if (!read_file(pcd, file_bytes)) { fprintf(stderr, "haf_cli: cannot open %s\n", pcd.c_str()); return 1; }
    }
    try {
        haf_b200::CCalc_Grasppoints_B200 server(features, range, model, 302, grid, 15, 190, 0, svm_mode);
        size_t n_points = xyz.size() / 3;
        if (host_pcd) server.read_pc_cb(goal, xyz.data(), n_points, 12);
        else n_points = server.open_pcd_and_trig_get_grasp_cb(goal, file_bytes.data(), file_bytes.size());
        print_result(json, n_points, server.best, server.gp_result, server.per_roll_top.data(), server.R, server.published_per_roll.size());
    } catch (const std::exception& e) {
        fprintf(stderr, "haf_cli: %s\n", e.what());
        return 1;
    }
    return 0;
}
