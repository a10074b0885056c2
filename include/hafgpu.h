/* hafgpu.h -- C ABI of libhafgpu.so: the B200-native (sm_100a) grasp-search hot path of haf_grasping.
 *
 * The reference has no plugin / FFI interface: the hot path is private members of the ROS node class
 * CCalc_Grasppoints plus two child processes (svm-scale, svm-predict).  This ABI is the narrowest seam that
 * leaves every ROS contract (CalcGraspPointsServer.action, GraspInput / GraspOutput, the parameter services)
 * untouched: inside CCalc_Grasppoints::loop_control (reference src/calc_grasppoints_action_server.cpp:335-402)
 * the five per-roll calls at :376-385
 *      generate_grid        (:406-529)   calc_intimage          (:577-613)
 *      calc_featurevectors  (:616-656)   [pnt_in_box            (:666-749)]
 *      predict_bestgp_withsvm (:754-800) show_predicted_gps     (:803-973)
 * and with them CIntImage_to_Featurevec::calc_featurevalue / write_featurevector (src/CIntImage_to_Featurevec.cpp
 * :122-199), svm-scale (libsvm-3.12/svm-scale.c) and svm-predict (libsvm-3.12/svm-predict.c, svm.cpp:2459-2533)
 * are replaced by ONE call, haf_search().  See INTEGRATION.md for the patch a maintainer applies.
 *
 * Conventions: 0 = OK, negative = error (haf_last_error gives text); no C++ exceptions, ROS or torch types
 * cross the boundary; the caller owns every output buffer; pointers named *_hostdev may be host or device
 * memory (detected with cudaPointerGetAttributes); there is NO CPU fallback -- without a usable sm_100
 * device haf_create fails with HAF_ERR_NO_DEVICE.  A context is entered from one thread at a time (the
 * action server runs one goal at a time on its execute thread, server.cpp:182, :227).
 */
#ifndef HAFGPU_H_
#define HAFGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HAF_OK 0
#define HAF_ERR_ARG (-1)         /* bad argument */
#define HAF_ERR_IO (-2)          /* features / range / model file missing or unparsable */
#define HAF_ERR_CUDA (-3)        /* CUDA runtime error */
#define HAF_ERR_NO_DEVICE (-4)   /* no sm_100 device: no fallback exists */
#define HAF_ERR_UNSUPPORTED (-5) /* input outside what the path reproduces exactly (see haf_last_error) */
#define HAF_ERR_NOMEM (-6)

typedef struct haf_ctx haf_ctx;

/* svm_mode (0 = what a zero-initialised config gets = the production path) */
#define HAF_SVM_TENSOR_GUARD 0 /* tcgen05 split-fp16 contraction in TMEM (1-3 products per k-slice, calibrated per model) + FP64
                                  re-evaluation inside the guard band (FMA tier, then exact order) */
#define HAF_SVM_FP64_EXACT 1   /* every window in FP64, libsvm's summation order (svm.cpp:326-365, :2500-2514) */
#define HAF_SVM_FP32_GUARD 2   /* FP32 SIMT contraction (CUDA cores) + the same FP64 guard band; conservative mode */

typedef struct {
    const char* features_path; /* data/Features.txt               (server param feature_file_path, :218-219) */
    const char* range_path;    /* data/range21062012_allfeatures  (range_file_path, :220-221)                */
    const char* model_path;    /* libsvm text model               (svmmodel_file_path, :222-223)             */
    int nr_features_without_shaf; /* 302 (server.cpp:224)                                                   */
    int grid;                  /* G: 56 = reference HEIGHT/WIDTH (server.cpp:92-93); even, 16..1024          */
    int roll_step_deg;         /* 15  (ROLL_STEPS_DEGREE, :95)                                               */
    int roll_max_deg;          /* 190 (ROLL_MAX_DEGREE, :101) -> R = 190/15 = 12 rolls                        */
    int device;                /* CUDA ordinal; one context (and one process) per GPU                         */
    int emulate_text_roundtrip; /* 0 (a zero-initialised config) or 1 = reproduce the "%.4g" / "%g" text round
                                   trips (reference-exact); -1 = skip them (NOT the reference's numbers)        */
    int svm_mode;              /* HAF_SVM_*                                                                   */
    float guard_rel;           /* guard band half-width as a fraction of E + |rho|,
                                  E = sum_i |coef_i| K_i (1 + gamma log2(e) (|x|^2 + |sv_i|^2)); <=0 -> default:
                                  FP32 SIMT 2e-6 (measured error <= 1.3e-7 E); tensor max(4e-6, 15 x (calibrated operand
                                  error of the chosen number of products + 2.5e-7)) -- 8.3e-6 for the 2048-SV bench model
                                  with one product; haf_get_info reports the value in use (reserved[1], units of 1e-9).
                                  Every tensor-mode call audits the band against its own windows (haf_timing)   */
    int reserved[4];           /* [0]: bits 0-1: tensor-path kernel, 0 = auto (X-resident CTA pair where one product is in use, else the
                                       streaming CTA pair; both cta_group::2), 2 = streaming CTA pair always;
                                       bits 4-5: tensor-core products per k-slice, 0 = calibrated per model (default), 1 / 2 / 3 forced;
                                       bit 8: audit sample off; bits 16+: audit every n-th window (default 4096; see haf_timing);
                                  [1]: bits 0-3: 1 = always use the point-parallel binning kernel (no whole-cloud CTAs), 2 = whole-cloud
                                       kernel with scalar loads; bit 4: 1 = CUDA graphs: a call that fits one pass and repeats the
                                       previous call's shape -- unit and window bounds, 64 k-point bucket of the cloud, buffers -- is
                                       captured once and replayed (one goal is ~25 dependent stream operations; not while haf_set_profiling
                                       is on).  Measured on B200: one table1 goal 0.224 ms launched, 0.189 ms replayed;
                                  [2]: bits 0-1: guard band tier 2 (FP64 re-evaluation by contraction): 0 = on, 1 = off (every guard
                                       window goes to the exact-order kernels), 2 = on, but every window escalates as well (tests);
                                       bits 2-3: its kernel: 0 / 1 = FP64 tensor cores (DMMA), 2 = DFMA register tiles (round 1's kernel);
                                  [3]: 1 = tensor kernels read the coef table from global memory even when it fits in
                                       shared memory (the path models with > 4096 support vectors take) */
    int n_devices;             /* > 1: one context drives several GPUs of the box (SURVEY 8b / 8e): haf_search shards its units
                                  (request, roll) and haf_search_batch* its clouds over them, one host thread and one stream per
                                  GPU; the per-unit tops / per-cloud records are merged on the host with the reference's own
                                  rules (strict >, earliest unit wins, early exit), so the result equals the one-GPU result.
                                  0 or 1: `device` alone                                                              */
    const int* devices;        /* [n_devices] CUDA ordinals (read at haf_create); NULL = 0 .. n_devices-1              */
} haf_config;

/* One grasp goal = the hot-path fields of GraspInput (msg/GraspInput.msg:3-15). */
typedef struct {
    double center[3];          /* grasp_area_center (server.cpp:258-260)                                      */
    float area_len_x, area_len_y; /* grasp_area_length_x/y in cm incl. the client's +14 (client.cpp:183-184);
                                     truncated to int like server.cpp:266-267                                 */
    double approach[3];        /* approach_vector, un-normalised; normalised like server.cpp:270-273          */
    int gripper_opening_width; /* :281, :433                                                                  */
    int return_only_best;      /* show_only_best_grasp: enables the early exit at graspval_top (:362-365)     */
    int graspval_top;          /* 119 (:203)                                                                  */
    int roll_limit;            /* evaluate only rolls [roll_begin, roll_limit); <=0 = up to R.  Stand-in for the
                                  caller's time budget / preempt checks (:350-357, :367-374)                   */
    int roll_begin;            /* first roll to evaluate (0 normally); > 0 only when one goal's rolls are sharded
                                  over several GPUs (SURVEY 8e) -- the caller merges the per-roll tops          */
    int svm_with_probability;  /* the `svm_with_probability` switch of loop_control (server.cpp:383-385; hard-wired false there):
                                  1 = classify with probability estimates (svm-predict -b 1 on a model carrying probA / probB) and
                                  score the float grid res * prob exactly as show_predicted_gps does (:831-841), one-line shift
                                  included; every request of a call must agree.  0 = labels only (the reference as shipped) */
} haf_request;

typedef struct {
    int row, col, roll, tilt;  /* id_row_top_overall, id_col_top_overall, nr_roll_top_overall, nr_tilt (=0)   */
    int approach_idx;          /* index of the winning request (approach vector); earliest wins ties          */
    int topval;                /* topval_gp_overall (:953-960); -1000 when no roll was evaluated              */
    int eval;                  /* topval - 20 (:390)                                                          */
    float roll_rad;            /* roll * step * PI / 180 (:1401)                                              */
    float M[16];               /* mat_transform of the winning roll, row-major (:483); av_trans_mat           */
    int rolls_done;            /* rolls the reference loop would have evaluated (early exit / roll_limit)     */
    int n_windows_scored;      /* feature vectors classified in those rolls                                   */
    int n_guard;               /* windows re-evaluated in FP64 because |dec| fell inside the guard band       */
    int reserved;
} haf_best;

typedef struct {
    int n_features;   /* F: features parsed (324 for data/Features.txt: 323 lines + the trailing blank line)  */
    int n_dims;       /* D: dimensions fed to the SVM (323)                                                   */
    int n_sv;         /* S: support vectors                                                                   */
    int n_rolls;      /* R                                                                                    */
    int grid;         /* G                                                                                    */
    int label0, label1; /* model label order (svm.cpp:2516-2531)                                              */
    int sm_count;
    double gamma, rho;
    int reserved[4];  /* [0]: tensor-core products per k-slice in use (1-3; 0 outside tensor mode); [1]: guard_rel * 1e9;
                         [2]: contraction kernel of the context's last decision-value launch (haf_search* / haf_svm_predict*):
                              0 none / FP64 exact order, 1 svm_rbf_tc3_kernel (X-resident pair), 2 svm_rbf_tc2_kernel (streaming
                              pair), 3 FP32 SIMT -- tc3 falls back to tc2 where the X tile, ring and table do not fit;
                         [3]: that launch's split of the support-vector tiles per work item (tensor kernels; 0 otherwise) */
} haf_info;

typedef struct {
    float ms_total;   /* device time of the last haf_search / haf_search_batch* call (CUDA events on its stream) */
    float ms_bin, ms_integral, ms_mask, ms_features, ms_svm, ms_guard, ms_score;
    long long n_points, n_units, n_windows, n_guard, launches;
    long long n_chunks; /* passes over the stage sequence (each launches every stage kernel once) */
    long long n_exact;  /* guard windows that went on to the exact-order FP64 kernels (tier 3); svm_mode 1: 0 */
    long long n_audit;  /* windows OUTSIDE the guard band re-evaluated in FP64 as the audit sample (tensor mode)  */
    float audit_max_rel; /* max |dec_tensor - dec_fp64| / (E + |rho|) over guard + audit windows of the call      */
    int tc_passes;      /* tensor-core products per k-slice the call ended with (0 outside tensor mode)           */
    int escalations;    /* times this context repeated a call with more products because the audit left < 4x     */
    int graph_replays;  /* calls of this context served by replaying its captured CUDA graph (reserved[1] bit 4)      */
    long long n_clamped; /* points of the call inside the box whose cell index floor(100 (t + r)) reached G and was clamped
                            to G - 1 (summed over units; the reference clamps and counts them the same way).  0 at G = 56;
                            a point a few ulps inside +r reaches it at many other grid sides */
} haf_timing;

/* ---- lifetime --------------------------------------------------------------------------------------------- */
int haf_create(haf_ctx** out, const haf_config* cfg);       /* parses + uploads features / range / model ONCE */
void haf_destroy(haf_ctx* ctx);
const char* haf_last_error(const haf_ctx* ctx);              /* ctx may be NULL (error of a failed haf_create) */
int haf_get_info(const haf_ctx* ctx, haf_info* info);
int haf_set_stream(haf_ctx* ctx, void* cuda_stream);         /* cudaStream_t; default: the legacy default stream */
int haf_set_profiling(haf_ctx* ctx, int per_stage_events);   /* 1: haf_timing carries per-stage ms (adds events) */
int haf_get_timing(const haf_ctx* ctx, haf_timing* t);
long long haf_launch_count(const haf_ctx* ctx);              /* kernels launched by this context so far         */

/* ---- the hot path ------------------------------------------------------------------------------------------ */
/* One cloud, n_requests goals that differ in approach vector / centre / area (the reference has one approach
 * vector per goal; units (request, roll) are independent, SURVEY 8e).  xyz: n_points records of 3 floats with a
 * byte stride (12 = packed, 16 = pcl::PointXYZ).  `best` = overall winner over requests in order (strict >,
 * earliest request wins ties -- the rule of server.cpp:953 extended); best_per_request [n_requests] optional.
 * Optional per-roll outputs (NULL to skip), host or device memory, R = n_rolls, G = grid:
 *   graspseval [n_requests][R][G][G] float  (graspseval of show_predicted_gps, :823-880)
 *   mask       [n_requests][R][G][G] uint8  (point_inside_box_grid, :138)
 *   heights    [n_requests][R][G][G] float  (heightsgridroll, :136)
 *   per_roll_top [n_requests][R][3] int     (id_row_top_all, id_col_top_all, topval_gp_all per roll, :811-815);
 *                                           rolls not evaluated (roll_begin / roll_limit) get (-1, -1, -1000)
 * In graspseval / mask / heights the rolls not evaluated are left untouched. */
int haf_search(haf_ctx* ctx, const float* xyz_hostdev, size_t n_points, size_t stride_bytes,
               const haf_request* reqs, int n_requests, haf_best* best, haf_best* best_per_request,
               float* graspseval, unsigned char* mask, float* heights, int* per_roll_top);

/* Throughput mode: n_clouds independent clouds, one request applied to each.  clouds[i] host or device
 * pointers to packed xyz (stride 12). */
int haf_search_batch(haf_ctx* ctx, const float* const* clouds, const size_t* n_points, int n_clouds,
                     const haf_request* req, haf_best* best_per_cloud);
/* Same, clouds concatenated in one packed buffer (host or device); point_offsets has n_clouds+1 entries.
 * A HOST buffer is staged piece by piece while the compute follows in chunks of 16, 24, 32, 48, 56, 56, ... clouds that
 * alternate between three streams of the library's own (the call still returns complete results, ordered after prior
 * work on the context's stream).  Pinned memory is read by the copy engine directly; pageable memory of 4 MB and more is
 * copied into a ring of pinned slots by up to 8 host threads of the library first (512 clouds of 100 k points: 12.6 ms
 * from pinned, 22 ms from pageable memory, 75 ms through the driver's pageable path).
 * Environment switches (operations / experiments; read per call unless noted):
 *   HAF_STAGE_THREADS=n   host threads staging a pageable batch, 0 = leave it to the driver (read at haf_create)
 *   HAF_DUAL_STREAM=0|2|3|4  streams the chunks of a host-staged batch alternate between (0 = one; default 3)
 *   HAF_STAGE_SCHED=a,b,c,...  clouds per chunk of a host-staged batch (the last value repeats)
 *   HAF_RESIDENT_SPLIT=k  split a device-resident batch into k chunks on the streams as well (default 1)
 *   HAF_X_BUDGET_GIB=g    cap of the per-chunk SVM input matrix
 *   HAF_GRAPH=1           CUDA graphs as with reserved[1] bit 4 (read at haf_create) */
int haf_search_batch_packed(haf_ctx* ctx, const float* xyz_all_hostdev, const size_t* point_offsets, int n_clouds,
                            const haf_request* req, haf_best* best_per_cloud);

/* ---- grasp poses (transform_gp_in_wcs_and_publish, server.cpp:1274-1401) ---------------------------------------------
 * msg/GraspOutput.msg plus the indices the pose was built from.  The pose is computed on the device from the winning roll's
 * height grid while that grid is still resident: the maximum over the 9 x 8 neighbourhood of the cell (:1343-1351), minus
 * 0.01 in double (:1354), the two grasp points (+-0.03 m along the row axis, :1360) mapped through the inverse of the
 * transform rebuilt from the double approach vector (:1276-1334, inverted on the host by adjugate / determinant), float
 * sums in the order ((a x + b y) + c z) + d w.  Bit-equal to the reference's arithmetic (oracle/haf_oracle.cpp). */
typedef struct {
    int eval;                    /* topval - 20 for a best grasp (:390); max(topval - 20, 10) for a per-roll record (:962-972) */
    float roll;                  /* radians, (float)((roll * step * 3.141592653) / 180) (:1401) */
    double graspPoint1[3], graspPoint2[3], averagedGraspPoint[3];   /* world frame (:1339-1397) */
    double approachVector[3];    /* third row of generate_grid's matrix (:1370-1374) */
    int row, col, roll_index;    /* the cell and roll the pose was built from (-1 when no roll was evaluated) */
    int reserved;
} haf_grasp;

/* haf_search plus the grasp poses, in one call.  grasp: the pose of `best`; grasp_per_request [n_requests] (optional): the
 * pose of each best_per_request; grasp_per_roll [n_requests][R] (optional): the pose of every evaluated roll's top cell
 * (per_roll_top), eval = max(top - 20, 10) -- rolls not evaluated (roll_begin / roll_limit) are left untouched.  When no
 * roll was evaluated the record is the reference's pose for roll -1: roll 0's transforms and no height (h = -10 - 0.01).
 * Records are written to host memory.  The caller applies graspval_th (70, server.cpp:962) before publishing. */
int haf_search_grasps(haf_ctx* ctx, const float* xyz_hostdev, size_t n_points, size_t stride_bytes,
                      const haf_request* reqs, int n_requests, haf_best* best, haf_best* best_per_request,
                      float* graspseval, unsigned char* mask, float* heights, int* per_roll_top,
                      haf_grasp* grasp, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll);
/* haf_search_batch_packed plus one pose per cloud (grasp_per_cloud [n_clouds]) and optionally per evaluated roll of every
 * cloud (grasp_per_roll [n_clouds][R]); the same staging, chunking and streams as haf_search_batch_packed. */
int haf_search_batch_packed_grasps(haf_ctx* ctx, const float* xyz_all_hostdev, const size_t* point_offsets, int n_clouds,
                                   const haf_request* req, haf_best* best_per_cloud,
                                   haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_roll);
/* Batched goals with their own requests: cloud c is searched with reqs[request_offsets[c] .. request_offsets[c+1]) (at least one
 * request per cloud; request_offsets [n_clouds+1] starts at 0; NULL = one request per cloud), each request with its own centre,
 * area, approach vector, gripper width, roll range and return_only_best.  For every cloud, every output equals what
 * haf_search_grasps returns for that cloud with that request list, field for field (n_guard aside: 0, as in the other batch
 * calls): best_per_cloud [n_clouds] is the winner over the cloud's requests (strict >, earliest request wins ties, approach_idx =
 * index within the cloud's list, n_windows_scored / rolls_done summed over them); best_per_request [n_reqs], per_roll_top
 * [n_reqs][R][3], grasp_per_request [n_reqs] and grasp_per_roll [n_reqs][R] (evaluated rolls only) are optional, n_reqs =
 * request_offsets[n_clouds].  grasp_per_cloud NULL: no pose kernel runs (and the other two grasp outputs must be NULL too).
 * Every request of a call must agree on svm_with_probability.  The same staging, chunking (on request boundaries: a cloud's
 * requests may span two chunks), streams, CUDA graphs and multi-GPU sharding (blocks of clouds with all their requests) as
 * haf_search_batch_packed.  The unit parameters (transforms, mask constants, inverse WCS matrices) are built on the device by one
 * kernel per call; the host evaluates only the libm calls, once per distinct approach vector (bitwise) and per roll, so its
 * work per call grows with the requests, not with the units.  Bit-equal to the host build of haf_search. */
int haf_search_batch_requests(haf_ctx* ctx, const float* xyz_all_hostdev, const size_t* point_offsets, int n_clouds,
                              const haf_request* reqs, const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request,
                              int* per_roll_top, haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll);

/* ---- ranked grasp candidates: the k best distinct grasps of every cloud ----------------------------------------------------
 * What a pick pipeline asks for when IK or collision checking rejects the best grasp.  For cloud c, a cell (request q, roll r, row,
 * col) is eligible when r is one of the rolls the reference loop evaluated for q ([roll_begin, roll_begin + rolls_done), the early
 * exit of return_only_best included) and mask == 1 there; its score is its graspseval value.  Cells are ordered by score descending,
 * then q, r, row, col ascending.  Each unit (q, r) contributes its first per_unit eligible cells in that order (its list).  Rank 0 is
 * the cloud's best grasp, exactly grasp_per_cloud (tie rule cell, eval = topval - 20); its cell leaves the lists.  The union of the
 * lists is then walked in order, and a cell is accepted unless an accepted candidate of the cloud lies within min_distance:
 * d2 = (dx dx + dy dy) + dz dz between averagedGraspPoints in double, suppressed iff d2 < min_distance^2 (min_distance <= 0: no
 * suppression), up to k candidates.  With min_distance <= 0 and per_unit >= k the list is the global top k of the eligible cells
 * after rank 0.  Every candidate carries a full haf_grasp record, eval = (int)score - 20: transform_gp_in_wcs_and_publish of its cell
 * with its roll's heights, bit-equal to the reference's arithmetic. */
typedef struct {
    int k;                 /* candidates per cloud, 1..256 */
    int per_unit;          /* eligible cells each (request, roll) contributes, k..1024; 0 = max(k, 64) */
    double min_distance;   /* metres between averagedGraspPoints of two candidates of one cloud; <= 0: no suppression */
    int reserved[4];       /* must be 0 */
} haf_rank_params;
typedef struct {
    haf_grasp grasp;       /* eval = (int)score - 20; row / col / roll_index = the cell */
    float score;           /* graspseval value of the cell */
    int request;           /* index within the cloud's request list */
} haf_candidate;           /* 128 bytes */
/* haf_search_batch_requests (same inputs, staging, chunking, streams, CUDA graphs, multi-GPU sharding; a single goal is n_clouds = 1)
 * plus the ranked candidates: candidates [n_clouds][k], n_candidates [n_clouds] (<= k; the slots after them are zeroed).  A cloud with
 * no evaluated roll gets 0 candidates (its grasp_per_cloud is the roll -1 record); one whose evaluated rolls have no eligible cell gets
 * 1 (the best).  best_per_cloud / grasp_per_cloud as in haf_search_batch_requests.  All outputs in host memory.  Each chunk's units
 * select their lists on the device with a radix select on the score and an ordered compaction (rank_unit_kernel; rank_tile_kernel
 * first where G > 90); one CTA per cloud walks them (rank_cloud_kernel).  HAF_ERR_ARG: k, per_unit out of range, NaN min_distance,
 * nonzero reserved, requests x R x per_unit above 2^31. */
int haf_search_batch_candidates(haf_ctx* ctx, const float* xyz_all_hostdev, const size_t* point_offsets, int n_clouds,
                                const haf_request* reqs, const int* request_offsets, const haf_rank_params* rp,
                                haf_best* best_per_cloud, haf_grasp* grasp_per_cloud,
                                haf_candidate* candidates /* [n_clouds][k] */, int* n_candidates /* [n_clouds] */);

/* ---- PCD / PointCloud2 ingest on the device (SURVEY 8f-2) -----------------------------------------------------------
 * What the reference does on the CPU before the hot path starts: the client's pcl::io::loadPCDFile<pcl::PointXYZ>
 * (src/calc_grasppoints_action_client.cpp:137-157) and the server's pcl::fromROSMsg (src/calc_grasppoints_action_server.cpp
 * :313-316).  file_bytes: the whole .pcd file in host memory (v0.7; DATA ascii, binary or binary_compressed; x / y / z
 * float32).  The text header is parsed on the host; the data section is decoded by kernels: ASCII records (correctly
 * rounded decimal -> float, exactly POINTS records, further lines ignored), binary records, or the LZF stream + the
 * struct-of-arrays -> xyz gather.  *d_xyz: packed xyz in DEVICE memory owned by the context (valid until the next ingest
 * call), accepted by haf_search / haf_debug_cell_indices as xyz_hostdev.  Errors: HAF_ERR_IO (malformed / truncated file,
 * fewer records than POINTS), HAF_ERR_UNSUPPORTED (other field types; a > 19-digit token next to a rounding boundary). */
int haf_pcd_decode(haf_ctx* ctx, const void* file_bytes, size_t n_bytes, const float** d_xyz, size_t* n_points);
/* haf_pcd_decode + haf_search in one call */
int haf_search_pcd(haf_ctx* ctx, const void* file_bytes, size_t n_bytes, const haf_request* reqs, int n_requests, haf_best* best,
                   haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top);
/* sensor_msgs/PointCloud2 -> packed xyz on the device (pcl::fromROSMsg for PointXYZ): n_points records of point_step bytes
 * (host or device memory), x / y / z float32 at byte offsets off_x / off_y / off_z (any alignment).  The batch of one of
 * haf_pointcloud2_batch_to_xyz. */
int haf_pointcloud2_to_xyz(haf_ctx* ctx, const void* data_hostdev, size_t n_points, size_t point_step, int off_x, int off_y, int off_z,
                           const float** d_xyz);

/* ---- batches of PCD files and PointCloud2 buffers --------------------------------------------------------------------
 * files: n_files PCD files concatenated in HOST memory (pinned or pageable); file f = bytes [file_offsets[f], file_offsets[f+1]).
 * Kinds may be mixed; POINTS 0 is an empty cloud.  *d_xyz: packed xyz of every cloud in DEVICE memory owned by the context
 * (valid until the next ingest call); point_offsets [n_files+1] (out) from the headers' POINTS.  Every cloud is decoded as
 * haf_pcd_decode decodes one file (haf_pcd_decode is this call with one file); the number of kernel launches does not grow
 * with the number of files: per data kind present one sequence over all its files (ASCII: count, scan, parse; binary_compressed:
 * one LZF launch with one CTA per file; binary and binary_compressed: one gather), then one stream sync.  Pinned input is copied
 * in one cudaMemcpyAsync; pageable input of 4 MB and more goes through the library's staging thread in pieces cut on file
 * boundaries.  Errors: the single-file code and text, prefixed "PCD file <i>: ".  Header and size checks run on the host
 * before any device work (the lowest such file is named); otherwise the lowest file the decode flags is named.  On error
 * nothing is written.  ASCII data of a batch is limited to 2^32 records and 2^31 tiles of 4 KB (HAF_ERR_UNSUPPORTED).
 * Multi-GPU context: the decode runs on its first GPU. */
int haf_pcd_decode_batch(haf_ctx* ctx, const void* files, const size_t* file_offsets, int n_files,
                         const float** d_xyz, size_t* point_offsets);
/* haf_pcd_decode_batch + haf_search_batch_requests on the decoded clouds; arguments and outputs as there */
int haf_search_batch_pcd(haf_ctx* ctx, const void* files, const size_t* file_offsets, int n_files,
                         const haf_request* reqs, const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request,
                         int* per_roll_top, haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll);
/* PointCloud2 data of n_clouds clouds (host or device): cloud c = bytes [byte_offsets[c], byte_offsets[c+1]), a whole number of
 * records of layouts[c][0] bytes with x / y / z float32 at byte offsets layouts[c][1..3]; rows without padding
 * (row_step = width * point_step).  One gather launch for the whole batch.  *d_xyz and point_offsets [n_clouds+1] (out) as
 * in haf_pcd_decode_batch; HAF_ERR_ARG naming the cloud for an offset + 4 > step or a span that is not a multiple of the step. */
int haf_pointcloud2_batch_to_xyz(haf_ctx* ctx, const void* data_hostdev, const size_t* byte_offsets, int n_clouds,
                                 const int* layouts, const float** d_xyz, size_t* point_offsets);

/* ---- batches of depth images: back-projection (and the camera -> base transform) on the device -----------------------
 * What a camera-fed server otherwise does on the CPU before a search: depth_image_proc's point_cloud_xyz (convert() of
 * depth_conversions.h for 16UC1 and 32FC1, range_max = 0, no lens distortion), then pcl_ros::transformPointCloud into the base
 * frame (server.cpp:316).  Image i = height rows of step bytes, little-endian, bytes [byte_offsets[i], byte_offsets[i+1]) of
 * data (host, pinned or pageable, or device); its cloud is the organized cloud of width x height points in row-major pixel
 * order, invalid pixels kept as NaN points.
 * Per image, on the host in double, stored as float: s = depth_scale (0: 0.001f for U16, 1.0f for F32), kx = s / fx,
 * ky = s / fy, cxf = cx, cyf = cy.  Pixel (u, v) with raw value d is valid when d != 0 (U16) or isfinite(d) (F32, negative
 * depths included); then D = (float)d and, one float rounding per operation, left to right, no FMA:
 *     x = ((float)u - cxf) * D * kx,   y = ((float)v - cyf) * D * ky,   z = D * s.
 * An invalid pixel is x = y = z = quiet NaN 0x7fc00000.  has_pose = 1: a point whose three coordinates are finite becomes
 * x' = ((m00 x + m01 y) + m02 z) + m03 (and so on per row; float, left to right, no FMA), any other point stays as it is (PCL
 * 1.7's transformPointCloud of a non-dense cloud).  has_pose = 0: no arithmetic at all (an identity pose would turn -0 into +0).
 * With depth_scale <= 1 every valid pixel has a finite z, so a point with a non-finite coordinate has a non-finite x or y and
 * fails the search's box test whatever its pose.
 * HAF_ERR_ARG "depth image <i>: ..." names the lowest bad image, checked on the host before any device work (nothing is
 * written): width or height outside [0, 2^24), unknown encoding, step not a multiple of the element size or below width x
 * element size, byte span != height x step, non-finite fx / fy / cx / cy or fx / fy = 0, depth_scale outside [0, 1] or NaN,
 * has_pose not 0 / 1, a non-finite camera_to_base entry with has_pose = 1, nonzero reserved. */
#define HAF_DEPTH_U16 1        /* 16UC1 / mono16; 0 = no return */
#define HAF_DEPTH_F32 2        /* 32FC1 metres; non-finite = no return */
typedef struct {
    int width, height, encoding, has_pose;
    long long step;            /* sensor_msgs/Image.step */
    double fx, fy, cx, cy;     /* CameraInfo K[0], K[4], K[2], K[5] */
    float depth_scale;         /* metres per unit, 0 = per-encoding default, <= 1 */
    float camera_to_base[16];  /* row-major, what pcl_ros::transformAsMatrix gives */
    int reserved[3];           /* must be 0 */
} haf_depth_image;             /* 136 bytes */
/* n_images images -> packed xyz of every cloud in ctx's ingest buffer: *d_xyz and point_offsets [n_images+1] (out) as in
 * haf_pcd_decode_batch (valid until the next ingest call; accepted by every search entry point as xyz_hostdev).  One kernel
 * launch covers every non-empty image (none when all are empty); no stream sync.  Device input is read in place, pinned input
 * is copied with one cudaMemcpyAsync, pageable input of 4 MB and more goes through the staging thread in pieces cut on image
 * boundaries.  Multi-GPU context: runs on its first GPU. */
int haf_depth_to_xyz_batch(haf_ctx* ctx, const void* data_hostdev, const size_t* byte_offsets, int n_images,
                           const haf_depth_image* images, const float** d_xyz, size_t* point_offsets);
/* haf_depth_to_xyz_batch + haf_search_batch_requests on the clouds, on the same stream; arguments and outputs as there */
int haf_search_batch_depth(haf_ctx* ctx, const void* data_hostdev, const size_t* byte_offsets, int n_images,
                           const haf_depth_image* images, const haf_request* reqs, const int* request_offsets,
                           haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                           haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll);

/* ---- libsvm-compatible front ends (SURVEY 8f-3) ----------------------------------------------------------------
 * The reference classifies by running two child processes per roll on text files (server.cpp:775-776, :786-792):
 *     svm-scale -r <range> /tmp/features.txt > /tmp/features.txt.scale      (libsvm-3.12/svm-scale.c)
 *     svm-predict /tmp/features.txt.scale <model> /tmp/output_calc_gp.txt   (libsvm-3.12/svm-predict.c)
 * These entry points are what CLI-compatible replacements of the two programs bind (csrc/host/svm_predict_b200.cpp,
 * svm_scale_b200.cpp): a second drop-in seam that needs no server patch.  Rows are given in CSR form with libsvm's
 * 1-based, ascending feature indices; row_ptr has n_rows + 1 entries indexing `index` / `value` (host memory).
 * No CPU fallback: all arithmetic runs on the device; text parsing / printing stays with the caller. */
typedef struct haf_ctx haf_svm;
/* model only (C-SVC, RBF, 2 classes: what svm_load_model reads for this path, svm.cpp:2714-2927).  min_dims: largest
 * feature index the data will carry (the distance loop covers max(model, data) dimensions, svm.cpp:328-364). */
int haf_svm_create(haf_svm** out, const char* model_path, int device, int svm_mode, int min_dims, float guard_rel);
/* the same, with every knob of the config: model_path, device, svm_mode, guard_rel and the reserved[] switches: tensor kernel,
 * products per k-slice, audit, guard tier 2 and its kernel, global coef table.  features_path, range_path, n_devices and
 * devices are ignored.  haf_svm_create(...) is haf_svm_create_config with a zeroed config carrying its four arguments. */
int haf_svm_create_config(haf_svm** out, const haf_config* cfg, int min_dims);
void haf_svm_destroy(haf_svm* s);
/* svm_predict for every row (svm.cpp:2535-2548): labels [n_rows] (as doubles, what svm-predict prints with %g) and,
 * optionally, the decision values [n_rows] (svm_predict_values, svm.cpp:2459-2533).  Labels equal libsvm's; decision
 * values carry the tolerance of the chosen svm_mode.  haf_last_error / haf_get_timing / haf_get_info take the handle. */
int haf_svm_predict(haf_svm* s, const long long* row_ptr, const int* index, const double* value, int n_rows,
                    double* labels, double* dec_values);
/* svm-predict -b 1 (svm-predict.c:111-118): svm_predict_probability for every row (svm.cpp:2550-2590: sigmoid_predict :1818,
 * clamp to [1e-7, 1 - 1e-7], multiclass_probability :1829-1890).  prob_estimates [n_rows][2] in the order of the model's
 * labels (haf_get_info: label0, label1), labels [n_rows] = the label with the larger estimate (first on ties).  Every row is
 * evaluated on the FP64 exact-order path whatever svm_mode the handle was made with (the estimates are printed with six
 * digits).  HAF_ERR_UNSUPPORTED with libsvm's own message when the model carries no probA / probB.
 * haf_svm_check_probability_model: svm_check_probability_model (svm.cpp:3098-3104), 1 / 0. */
int haf_svm_predict_probability(haf_svm* s, const long long* row_ptr, const int* index, const double* value, int n_rows,
                                double* labels, double* prob_estimates);
int haf_svm_check_probability_model(const haf_svm* s);
/* svm-scale pass 2 (svm-scale.c:165-198): per-feature min / max over the rows, absent entries counting as 0.
 * fmin / fmax: [max_index + 1], entry 0 unused, IN/OUT (start from +DBL_MAX / -DBL_MAX; call per piece of a file). */
int haf_scale_minmax(int device, const long long* row_ptr, const int* index, const double* value, int n_rows, int max_index,
                     double* fmin, double* fmax);
/* svm-scale pass 3 (output(), svm-scale.c:333-353) for every feature 1..max_index of every row (absent = 0):
 * dense_out [n_rows][max_index]; single-valued features (max == min) give 0 = "not printed". */
int haf_scale_apply(int device, const long long* row_ptr, const int* index, const double* value, int n_rows, int max_index,
                    const double* fmin, const double* fmax, double lower, double upper, double* dense_out);

/* Host-only helpers (no GPU work): the transform of one roll exactly as generate_grid builds it (:406-484),
 * and the ordered key that turns "strictly greater wins, earliest unit wins ties" into a max-reduction, for the
 * cross-GPU best-grasp exchange (SURVEY 8e). */
int haf_build_transform(const haf_request* req, int roll, int roll_step_deg, float M_rowmajor[16]);
/* the same chain as transform_gp_in_wcs_and_publish rebuilds it for the grasp points (:1276-1334): there the two angles come
 * from the double members approach_vector.{x,y,z} (:1293-1303), not from the float copy generate_grid uses (:418-420) */
int haf_build_transform_wcs(const haf_request* req, int roll, int roll_step_deg, float M_rowmajor[16]);
uint64_t haf_best_key(int topval, uint32_t unit_order);
/* records [n][8] int32 = {topval, row, col, roll, tilt, approach_idx, n_windows_scored, rolls_done}: the 32-byte record
 * of the cross-GPU best-grasp exchange (SURVEY 8e), e.g. straight into a pinned buffer an NCCL all-gather reads */
int haf_pack_best_records(const haf_best* best, int n, int32_t* records);

/* ---- parity / inspection entry points (used by tests; they re-run stages on the state of the LAST haf_search) */
/* 1: haf_search_batch* calls keep their per-window state for the accessors below as well; such a call must then fit one
 * pass over the stage sequence (<= ~2.4 M windows), else it fails with HAF_ERR_UNSUPPORTED */
int haf_set_debug(haf_ctx* ctx, int keep_batch_state);
int haf_debug_window_count(const haf_ctx* ctx);
/* windows of the last search: win_unit_cell [W][2] = (unit = request*R + roll, cell = row*G + col) */
int haf_debug_windows(haf_ctx* ctx, int* win_unit_cell, int cap_windows);
/* raw features [W][F] float (calc_featurevalue), scaled SVM inputs [W][D] double (after both text round trips) */
int haf_debug_features(haf_ctx* ctx, float* raw, double* scaled, int cap_windows);
/* tensor mode: SVM inputs as the tensor-core contraction sees them (fp16 hi + lo, as float) [W][D] */
int haf_debug_tensor_inputs(haf_ctx* ctx, float* x, int cap_windows);
/* decision values, libsvm labels and guard flags [W] of the last search */
int haf_debug_decisions(haf_ctx* ctx, double* dec, int* labels, unsigned char* guard, int cap_windows);
/* integral images [n_units][G+1][G+1] float of the last search */
int haf_debug_integral(haf_ctx* ctx, float* integral, size_t cap_floats);
/* unit parameters of the last search, whichever path built them (host: haf_search* / haf_search_batch_packed*; device:
 * haf_search_batch_requests), unit u = job * R + roll: M [U][16] mat_transform (row-major), mask [U][10] pnt_in_box constants
 * (sinf / cosf(alpha), then cx1 cy1 cx2 cy2 cx3 cy3 cx4 cy4), Minv [U][16] the inverse WCS matrix of the unit's pose (only after a
 * call that built poses: the *_grasps entry points, or haf_search_batch_requests with grasp_per_cloud).  Any of the three may be
 * NULL.  Returns the number of units written (<= cap_units).  On a multi-GPU context: the share of the first GPU. */
int haf_debug_unit_params(haf_ctx* ctx, float* M, float* mask, float* Minv, int cap_units);
/* chunks of the last search, out [n][HAF_CHUNK_RECORD = 10] = {first cloud, end cloud, stream set (0 = the call's stream), copy
 * piece of a host-staged batch the chunk's stream waited for (-1: input in device memory), end cloud of that piece, binning kernel
 * (0 point-parallel, 1 whole-cloud with 16-byte loads, 2 whole-cloud with scalar loads), unit groups per cloud, units per group,
 * slices per cloud (the last three: the whole-cloud kernel's grid; 0 for the point-parallel kernel), integral image (0 one kernel
 * per unit with the tile in shared memory, 1 row pass + column pass)}.  Pieces are copied in order on one stream, so a chunk's
 * clouds are all on the device once its piece is: end cloud of the piece >= end cloud of the chunk.
 * Returns the number of chunks written (<= cap_chunks). */
#define HAF_CHUNK_RECORD 10
int haf_debug_chunk_copy_waits(const haf_ctx* ctx, int* out, int cap_chunks);
/* decoded height grids [n_units][G][G] float of the last search (unit u = job * R + roll; batches under haf_set_debug(1)).  Only
 * the units of active rolls are defined: inactive ones (outside [roll_begin, roll_limit)) are never decoded and hold bin keys.
 * Returns the number of units written. */
int haf_debug_heights(haf_ctx* ctx, float* heights, size_t cap_floats);
/* cell index (idx_x*G+idx_y, or -1 outside the box) of every point for one request / roll */
int haf_debug_cell_indices(haf_ctx* ctx, const float* xyz_hostdev, size_t n_points, size_t stride_bytes,
                           const haf_request* req, int roll, int* cell_idx_host);
/* device evaluation of text4 (float -> "%.4g" -> double) and text6 (double -> "%g" -> double) */
int haf_debug_text_roundtrip(haf_ctx* ctx, const float* in4, int n4, double* out4, const double* in6, int n6,
                             double* out6);

/* packed xyz of the last ingest call (haf_pcd_decode[_batch], haf_pointcloud2[_batch]_to_xyz, haf_depth_to_xyz_batch; all clouds of a batch: total
 * points), copied to host memory (n_points records) */
int haf_debug_pcd_xyz(haf_ctx* ctx, float* xyz_host, size_t n_points);

/* cycle counters of the role threads of the last X-resident tensor kernel launch made under HAF_TC_DEBUG=32 (timing
 * experiments, tools/tc_pipeline_probe.py; layout in csrc/svm_tc.cuh, g_tc_probe): out [n_ctas][16] */
int haf_debug_tc_probe(haf_ctx* ctx, unsigned long long* out, int n_ctas);

const char* haf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HAFGPU_H_ */
