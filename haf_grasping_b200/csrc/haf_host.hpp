// haf_host.hpp -- host-side pieces of libhafgpu: byte-compatible loaders for the reference's three input
// files and the per-roll transform / mask constants that must be computed with the HOST libm (glibc
// cosf/sinf/atan2f are not bitwise equal to CUDA's; SURVEY 8a row a1).
#pragma once
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>

#include "../../include/hafgpu.h"

namespace hafhost {

static const double kPI = 3.141592653;  // the reference's own PI (server.cpp:94), NOT M_PI

// ---------------------------------------------------------------------------------------------------
// Feature table: data/Features.txt as CIntImage_to_Featurevec::read_features parses it
// (reference II2FV.cpp:47-84) and CHaarFeature's 4-region constructor stores it (Haar.cpp:54-78).
// ---------------------------------------------------------------------------------------------------
struct Feature {
    int reg[16];  // 4 regions x (x1, x2, y1, y2); x indexes the FIRST (row) index of the 15x15 patch
    float w[4];   // weights as calc_featurevalue sees them; w[3] is always 0 (Haar.cpp:55-60 never assigns it)
};

inline bool load_features(const char* path, std::vector<Feature>& out, std::string& err) {
    std::ifstream in(path);
    if (!in) { err = std::string("cannot open feature file ") + path; return false; }
    std::string line;
    std::getline(in, line);
    // `while (file.good())` (II2FV.cpp:61): a trailing blank line is still "good" and yields one more,
    // all-zero, feature -- F = 324 for the shipped file.
    while (in.good()) {
        Feature ft;
        size_t start = 0;
        for (int k = 0; k < 20; k++) {
            // token = [start, next tab); when no tab is left the token is the rest of the line and the
            // cursor wraps to 0, exactly like `end = line.find("\t", start); start = end + 1` with int end
            size_t tab = line.find('\t', start);
            std::string tok = (start <= line.size()) ? line.substr(start, tab == std::string::npos ? std::string::npos : tab - start) : std::string();
            if (k < 16) ft.reg[k] = atoi(tok.c_str());
            else ft.w[k - 16] = (float)atof(tok.c_str());
            start = (tab == std::string::npos) ? 0 : tab + 1;
        }
        ft.w[3] = 0.0f;
        out.push_back(ft);
        std::getline(in, line);
    }
    if (out.empty()) { err = std::string("no features parsed from ") + path; return false; }
    return true;
}

// region skipped by calc_featurevalue (II2FV.cpp:155-159)
inline bool region_skipped(const Feature& f, int r) {
    int x1 = f.reg[4 * r], x2 = f.reg[4 * r + 1], y1 = f.reg[4 * r + 2], y2 = f.reg[4 * r + 3];
    return (f.w[r] == 0.0f) || (x2 < x1) || (y2 < y1) || (x2 == 0 && y2 == 0);
}

// ---------------------------------------------------------------------------------------------------
// Range file as `svm-scale -r` restores it (svm-scale.c:108-132, :204-231).
// ---------------------------------------------------------------------------------------------------
struct Range {
    double lower = -1.0, upper = 1.0;
    int max_index = 0;
    std::vector<double> fmin, fmax;
    std::vector<char> has;
};

inline bool load_range(const char* path, Range& R, std::string& err) {
    FILE* fp = fopen(path, "r");
    if (!fp) { err = std::string("cannot open range file ") + path; return false; }
    int c = fgetc(fp);
    if (c == 'y') {
        double a, b;
        if (fscanf(fp, "%lf %lf\n", &a, &b) != 2 || fscanf(fp, "%lf %lf\n", &a, &b) != 2) { fclose(fp); err = "bad y block in range file"; return false; }
    } else {
        ungetc(c, fp);
    }
    if (fgetc(fp) != 'x') { fclose(fp); err = std::string("range file has no x block: ") + path; return false; }
    if (fscanf(fp, "%lf %lf\n", &R.lower, &R.upper) != 2) { fclose(fp); err = "bad lower/upper in range file"; return false; }
    int idx;
    double mn, mx;
    while (fscanf(fp, "%d %lf %lf\n", &idx, &mn, &mx) == 3) {
        if (idx < 1 || idx > (1 << 20)) continue;
        if (idx > R.max_index) R.max_index = idx;
        if ((int)R.has.size() <= idx) { R.fmin.resize(idx + 1, 0.0); R.fmax.resize(idx + 1, 0.0); R.has.resize(idx + 1, 0); }
        R.fmin[idx] = mn; R.fmax[idx] = mx; R.has[idx] = 1;
    }
    fclose(fp);
    if (!(R.upper > R.lower)) { err = "range file: upper <= lower"; return false; }
    return true;
}

// ---------------------------------------------------------------------------------------------------
// libsvm 3.12 text model as svm_load_model reads it (svm.cpp:2714-2927); 2-class RBF C-SVC only.
// ---------------------------------------------------------------------------------------------------
struct Model {
    double gamma = 0, rho = 0;
    int l = 0, nr_class = 0, label[2] = {0, 0}, nSV[2] = {0, 0};
    int max_index = 0;
    bool has_probA = false, has_probB = false;   // svm_check_probability_model (svm.cpp:3098-3104): both present
    double probA = 0, probB = 0;                 // sigmoid of the one class pair (svm.cpp:2811-2824)
    std::vector<double> coef;  // [l] file order
    std::vector<std::vector<std::pair<int, double> > > sv;
};

inline bool load_model(const char* path, Model& m, std::string& err, bool& unsupported) {
    unsupported = false;
    FILE* fp = fopen(path, "rb");
    if (!fp) { err = std::string("cannot open model file ") + path; return false; }
    char cmd[81];
    bool have_sv = false;
    while (fscanf(fp, "%80s", cmd) == 1) {
        if (!strcmp(cmd, "svm_type")) {
            if (fscanf(fp, "%80s", cmd) != 1) break;
            if (strcmp(cmd, "c_svc")) { unsupported = true; err = std::string("model svm_type ") + cmd + " (only c_svc is on the path)"; fclose(fp); return false; }
        } else if (!strcmp(cmd, "kernel_type")) {
            if (fscanf(fp, "%80s", cmd) != 1) break;
            if (strcmp(cmd, "rbf")) { unsupported = true; err = std::string("model kernel_type ") + cmd + " (only rbf is on the path)"; fclose(fp); return false; }
        } else if (!strcmp(cmd, "gamma")) { if (fscanf(fp, "%lf", &m.gamma) != 1) break; }
        else if (!strcmp(cmd, "degree")) { int d; if (fscanf(fp, "%d", &d) != 1) break; }
        else if (!strcmp(cmd, "coef0")) { double d; if (fscanf(fp, "%lf", &d) != 1) break; }
        else if (!strcmp(cmd, "nr_class")) {
            if (fscanf(fp, "%d", &m.nr_class) != 1) break;
            if (m.nr_class != 2) { unsupported = true; err = "model nr_class != 2"; fclose(fp); return false; }
        } else if (!strcmp(cmd, "total_sv")) { if (fscanf(fp, "%d", &m.l) != 1) break; }
        else if (!strcmp(cmd, "rho")) { if (fscanf(fp, "%lf", &m.rho) != 1) break; }
        else if (!strcmp(cmd, "label")) { if (fscanf(fp, "%d %d", &m.label[0], &m.label[1]) != 2) break; }
        else if (!strcmp(cmd, "probA")) { if (fscanf(fp, "%lf", &m.probA) != 1) break; m.has_probA = true; }
        else if (!strcmp(cmd, "probB")) { if (fscanf(fp, "%lf", &m.probB) != 1) break; m.has_probB = true; }
        else if (!strcmp(cmd, "nr_sv")) { if (fscanf(fp, "%d %d", &m.nSV[0], &m.nSV[1]) != 2) break; }
        else if (!strcmp(cmd, "SV")) {
            int ch;
            while ((ch = getc(fp)) != EOF && ch != '\n') {}
            have_sv = true;
            break;
        } else { err = std::string("unknown text in model file: [") + cmd + "]"; fclose(fp); return false; }
    }
    if (!have_sv || m.l <= 0 || m.nr_class != 2) { fclose(fp); err = std::string("malformed libsvm model ") + path; return false; }
    std::vector<char> buf(1 << 16);
    std::string line;
    for (int i = 0; i < m.l; i++) {
        line.clear();
        while (fgets(buf.data(), (int)buf.size(), fp)) {
            line += buf.data();
            if (!line.empty() && line[line.size() - 1] == '\n') break;
        }
        if (line.empty()) { fclose(fp); err = "model file ends before total_sv lines"; return false; }
        char* s = &line[0];
        char* save = NULL;
        char* p = strtok_r(s, " \t", &save);
        if (!p) { fclose(fp); err = "empty SV line in model"; return false; }
        m.coef.push_back(strtod(p, NULL));
        std::vector<std::pair<int, double> > row;
        while (true) {
            char* idx = strtok_r(NULL, ":", &save);
            char* val = strtok_r(NULL, " \t", &save);
            if (val == NULL) break;
            int id = (int)strtol(idx, NULL, 10);
            double v = strtod(val, NULL);
            if (id < 1 || id > (1 << 20)) { fclose(fp); err = "SV index out of range in model"; return false; }
            if (!row.empty() && id <= row.back().first) { unsupported = true; fclose(fp); err = "SV indices not ascending in model"; return false; }
            row.push_back(std::make_pair(id, v));
            if (id > m.max_index) m.max_index = id;
        }
        m.sv.push_back(row);
    }
    fclose(fp);
    return true;
}

// graspsgrid value of a predicted label: svm-predict prints "%g\n" (svm-predict.c:127), the server takes
// atoi of the first two characters (server.cpp:843).
inline int label_to_gridvalue(int label) {
    char buf[64];
    snprintf(buf, sizeof buf, "%g", (double)label);
    buf[2] = 0;
    return atoi(buf);
}

// ---------------------------------------------------------------------------------------------------
// a1: mat_transform = S * Rroll * T2 * Rx * Rz * T1 (server.cpp:406-484), float, left to right, each
// product entry ((a0*b0 + a1*b1) + a2*b2) + a3*b3 (Eigen's fixed-size coefficient product, no FMA).
//
// The libm calls (atan2f / atan2, cosf / sinf, sin / cos) depend on the approach vector and the roll alone and are the
// only operations whose results differ between glibc and CUDA: approach_trig / roll_trig evaluate them on the host.
// Everything else (centre, gripper width, area, the five products, the inverse) is plain IEEE arithmetic in a fixed
// order: compose_transform / compose_mask / invert4 are HAF_HD, and the device build of haf_search_batch_requests
// (kernels.cuh, expand_units_kernel) runs the same source.  The device code is compiled with -fmad=false, the host
// code with -ffp-contract=off, so both round every product and sum on its own.
// ---------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
#define HAF_HD __host__ __device__
#else
#define HAF_HD
#endif
#if defined(__CUDA_ARCH__)
#define HAF_NOFMA_FLOAT float            // -fmad=false
#else
#define HAF_NOFMA_FLOAT volatile float   // forbid the host compiler from contracting to FMA
#endif

HAF_HD inline void mul4(const float* A, const float* B, float* C) {
    float T[16];
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) {
            HAF_NOFMA_FLOAT s = A[i * 4] * B[j];
            s = s + A[i * 4 + 1] * B[4 + j];
            s = s + A[i * 4 + 2] * B[8 + j];
            s = s + A[i * 4 + 3] * B[12 + j];
            T[i * 4 + j] = s;
        }
    for (int k = 0; k < 16; k++) C[k] = T[k];
}
HAF_HD inline void eye4(float* A) {
    for (int k = 0; k < 16; k++) A[k] = 0.0f;
    A[0] = A[5] = A[10] = A[15] = 1.0f;
}

inline void normalize_approach(const double in[3], double out[3]) {  // server.cpp:270-273
    float len = (float)std::sqrt(in[0] * in[0] + in[1] * in[1] + in[2] * in[2]);
    out[0] = in[0] / len; out[1] = in[1] / len; out[2] = in[2] / len;
}

// cos / sin of the two angles of an approach vector, trig = {cos rot_z, sin rot_z, cos rot_x, sin rot_x}.  wcs = false: as
// generate_grid builds them (:444-453; the angles from the float PointXYZ copy of the approach vector, :418-420).  wcs = true:
// as transform_gp_in_wcs_and_publish rebuilds them (:1293-1303; the angles from the DOUBLE members this->approach_vector) --
// the two differ in the last bits for a tilted approach vector.
inline void approach_trig(const double approach[3], bool wcs, float trig[4]) {
    double av[3];
    normalize_approach(approach, av);
    const float ax = (float)av[0], ay = (float)av[1], az = (float)av[2];  // PointXYZ floats (:418-420)
    float rot_z, rot_x = 0;
    if (wcs) {                                                                 // :1293-1303
        if (av[1] == 0 && av[0] == 0) {
            rot_z = 0;
            rot_x = (av[2] >= 0) ? 0.0f : (float)kPI;
        } else {
            rot_z = (float)(90 * kPI / 180.0 - std::atan2(av[1], av[0]));
            rot_x = (float)(90 * kPI / 180.0 - std::atan2(av[2], std::sqrt(av[1] * av[1] + av[0] * av[0])));
        }
    } else if (ay == 0 && ax == 0) {                                           // :444-450
        rot_z = 0;
        rot_x = (az >= 0) ? 0.0f : (float)kPI;
    } else {                                                                   // :452-453
        rot_z = (float)(90 * kPI / 180.0 - (double)atan2f(ay, ax));
        rot_x = (float)(90 * kPI / 180.0 - (double)atan2f(az, sqrtf(ay * ay + ax * ax)));
    }
    trig[0] = cosf(rot_z); trig[1] = sinf(rot_z); trig[2] = cosf(rot_x); trig[3] = sinf(rot_x);
}
struct ApproachTrig {   // one approach vector of haf_search_batch_requests' table
    float grid[4], wcs[4];
};

// the libm part of one roll: the roll matrix (:462-466) and the box rotation of pnt_in_box (:679-696); boxrot_angle_init
// is an uninitialised member in the reference (:131) that reads as 0.0 in practice -- treated as 0 (SURVEY 8a row a5)
struct RollTrig {
    float cos_roll, sin_roll;   // cosf / sinf of the roll angle
    float sa, ca;               // sinf / cosf(alpha)
    double s90, c90;            // sin / cos(alpha + PI / 2)
};
inline RollTrig roll_trig(int roll, int roll_step_deg) {
    RollTrig t;
    const float angle = (float)(roll * roll_step_deg * kPI / 180);             // :462
    t.cos_roll = cosf(angle); t.sin_roll = sinf(angle);
    const float boxrot_angle_init = 0.0f;
    float alpha_deg = (float)(-roll * roll_step_deg - boxrot_angle_init * 180 / kPI);
    float alpha = (float)(alpha_deg * kPI / 180);
    t.sa = sinf(alpha);
    t.ca = cosf(alpha);
    t.s90 = sin(alpha + kPI / 2);
    t.c90 = cos(alpha + kPI / 2);
    return t;
}

// trig: approach_trig of the request's approach vector
HAF_HD inline void compose_transform(const float trig[4], const RollTrig& rt, int gripper_opening_width, const double center[3], float M[16]) {
    float S[16], Rr[16], T2[16], Rx[16], Rz[16], T1[16];
    eye4(S); eye4(Rr); eye4(T2); eye4(Rx); eye4(Rz); eye4(T1);
    S[0] = (float)gripper_opening_width;                                       // :433
    T1[3] = (float)(-center[0]); T1[7] = (float)(-center[1]); T1[11] = (float)(-center[2]);  // :435-437
    T2[11] = 0 + 0.15f;                                                        // :441, trans_z_after_pc_transform (:214)
    Rr[0] = rt.cos_roll; Rr[1] = -rt.sin_roll; Rr[4] = rt.sin_roll; Rr[5] = rt.cos_roll;   // :463-466
    Rz[0] = trig[0]; Rz[1] = -trig[1]; Rz[4] = trig[1]; Rz[5] = trig[0];       // :469-472
    Rx[5] = trig[2]; Rx[6] = -trig[3]; Rx[9] = trig[3]; Rx[10] = trig[2];      // :476-479
    float P[16];
    mul4(S, Rr, P); mul4(P, T2, P); mul4(P, Rx, P); mul4(P, Rz, P); mul4(P, T1, P);            // :483
    for (int k = 0; k < 16; k++) M[k] = P[k];
}

// wcs = false: mat_transform as generate_grid builds it; wcs = true: as transform_gp_in_wcs_and_publish rebuilds it
inline void build_transform(const haf_request& rq, int roll, int roll_step_deg, float M[16], bool wcs = false) {
    float trig[4];
    approach_trig(rq.approach, wcs, trig);
    compose_transform(trig, roll_trig(roll, roll_step_deg), rq.gripper_opening_width, rq.center, M);
}
inline void build_transform_wcs(const haf_request& rq, int roll, int roll_step_deg, float M[16]) { build_transform(rq, roll, roll_step_deg, M, true); }

// a16: general 4x4 float inverse by cofactors (adjugate / determinant).  transform_gp_in_wcs_and_publish calls Eigen's
// Matrix4f::inverse() (:1376), which the reference does not vendor (unpinned); this is the restatement the oracle uses too.
// Every product and sum rounds on its own (see above).
HAF_HD inline void invert4(const float* m, float* inv) {
    float a[16];
    a[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    a[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    a[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    a[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    a[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    a[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    a[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    a[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    a[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    a[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    a[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    a[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    a[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    a[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    a[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    a[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const float det = m[0] * a[0] + m[1] * a[4] + m[2] * a[8] + m[3] * a[12];
    const float inv_det = 1.0f / det;
    for (int i = 0; i < 16; i++) inv[i] = a[i] * inv_det;
}

// a5 constants of pnt_in_box (server.cpp:679-696) for one roll
struct MaskConsts {
    float sa, ca;  // sinf(alpha), cosf(alpha)
    float cx1, cy1, cx2, cy2, cx3, cy3, cx4, cy4;
};
HAF_HD inline MaskConsts compose_mask(int G, const RollTrig& rt, int area_x, int area_y) {
    float cx = (float)(G / 2), cy = (float)(G / 2);
    float boarder = 7.0f;
    float height_r = area_x / 2 - boarder;
    float width_r = area_y / 2 - boarder;
    MaskConsts m;
    m.sa = rt.sa;
    m.ca = rt.ca;
    HAF_NOFMA_FLOAT t;
    t = m.sa * height_r; m.cx1 = cx - t;  m.cx2 = cx + t;
    t = m.ca * height_r; m.cy1 = cy + t;  m.cy2 = cy - t;
    m.cx3 = (float)(cx - rt.s90 * width_r);
    m.cy3 = (float)(cy + rt.c90 * width_r);
    m.cx4 = (float)(cx + rt.s90 * width_r);
    m.cy4 = (float)(cy - rt.c90 * width_r);
    return m;
}
inline MaskConsts mask_consts(int G, int roll, int roll_step_deg, int area_x, int area_y) {
    return compose_mask(G, roll_trig(roll, roll_step_deg), area_x, area_y);
}

}  // namespace hafhost
