// hafgpu.cu -- C ABI of libhafgpu.so (include/hafgpu.h): context, buffers, launch sequence.
// One context = one GPU = one stream.  No CPU fallback: every stage below is a CUDA kernel from kernels.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <string>
#include <thread>
#include <vector>

#include "../../include/hafgpu.h"
#include "haf_host.hpp"
#include "host/pcd_io.hpp"
#include "kernels.cuh"
#include "pcd_ingest.cuh"
#include "svm_tc.cuh"

using namespace hafk;

static thread_local std::string g_create_error;

#define HAF_VERSION_STRING "hafgpu 0.1 (sm_100a)"

namespace {

// (Re)allocations done at creation time (outside ENSURE) move this on; the ENSURE macro moves the owning context's alloc_epoch on.
// A captured CUDA graph bakes the buffers' addresses in and is only replayed while both stand.
static unsigned long long g_alloc_epoch = 0;
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    int ensure(size_t n) {
        if (n <= cap) return 0;
        g_alloc_epoch++;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 256;
        if (cudaMalloc(&p, want * sizeof(T)) != cudaSuccess) { cudaGetLastError(); if (cudaMalloc(&p, n * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return -1; } want = n; }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
template <typename T>
struct PinBuf {
    T* p = nullptr;
    size_t cap = 0;
    int ensure(size_t n) {
        if (n <= cap) return 0;
        g_alloc_epoch++;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 64;
        if (cudaMallocHost(&p, want * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return -1; }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct Job {  // one (cloud, request)
    int cloud;
    haf_request rq;
    int roll_begin;
    int n_rolls_active;   // rolls [roll_begin, n_rolls_active) are evaluated
    long long wbound;  // upper bound on valid windows of this job (all active rolls)
};

}  // namespace

struct haf_ctx {
    haf_config cfg;
    std::string err;
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = 0;
    bool profiling = false;
    long long launches = 0;
    haf_timing timing;
    cudaEvent_t ev[10];               // [8] start, [9] end of a call
    bool ev_ok = false;
    std::vector<cudaEvent_t> ev_pool; // 8 per chunk when per-stage profiling is on (no host sync inside a call)
    // host -> device staging of a batch overlapped with compute: pieces copied on copy_stream, one event per piece
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> copy_ev;
    std::vector<int> copy_cloud_end;  // piece k covers clouds [copy_cloud_end[k-1], copy_cloud_end[k])
    int copy_pieces = 0;              // > 0 while a plan is active

    // model-side constants
    int F = 0, D = 0, Dsv = 0, Kpad = 0, S = 0, Spad = 0, R = 0, G = 0;
    double lower = -1, upper = 1, gamma = 0, rho = 0;
    int label[2] = {0, 0}, gv[2] = {0, 0};
    float guard_rel = 4e-6f;
    DevBuf<FeatDev> d_feats;
    DevBuf<DimDev> d_dims;
    DevBuf<float> d_svT, d_svn, d_coef;
    DevBuf<double> d_sv64T, d_coef64;
    // tensor-core path (HAF_SVM_TENSOR_GUARD): fp16 hi/lo operands, K-major, k-block tiled (kernels.cuh, kt_off):
    // Krow = columns in use (dimensions + 6 extra columns, rounded up to 16), KB = k-blocks of 64 columns stored
    int Krow = 0, KB = 0, SpadT = 0;
    float c_log2 = 0.0f;
    float csvn_max = 0.0f;      // |c| * max_n ||sv_n||^2 (guard scale of the tensor kernels)
    float e_floor = 0.0f;       // sum|coef| * 2^-100: windows whose guard scale E is below it lose terms to FP32 underflow -> FP64
    DevBuf<__half> d_SVh, d_SVl, d_Xh, d_Xl;   // d_Xl only with three products per k-slice
    DevBuf<float> d_svcoef;     // coef in the tensor path's order (sorted by sign, sign groups padded to whole tiles)
    DevBuf<double> d_dec_tc;    // audit: the contraction's decision value of every window on the guard list
    int audit_every = 4096;     // every audit_every-th window joins the guard list as an unbiased error sample (0 = off)
    float audit_max_rel = 0.0f; // last call: max |dec_tc - dec_fp64| / (E + |rho|) over guard + sample windows
    int escalations = 0;        // times a call was repeated with more tensor-core products because the audit left < 4x margin
    DevBuf<DimFeat> d_dimfeat;
    DevBuf<Round4Tab> d_round4;   // "%.4g" tables of the fast tier
    DevBuf<float> d_asum;
    CUtensorMap tmSh2, tmSl2;   // 128-row boxes: one per CTA of a pair
    int tc_variant = 0;         // 0: auto (X-resident CTA-pair kernel where eligible, else streaming CTA pair), 2: streaming CTA pair always
    int tc_passes = 3;          // tensor-core products per k-slice: 3, 2 or 1 (calibrate_tensor_passes)
    double tc_operand_err = 0;  // calibrated operand error of the chosen scheme, as a fraction of the guard scale E
    int last_svm_kernel = 0;    // contraction kernel of the last stage-5 launch (haf_info.reserved[2]): 0 none / FP64 exact, 1 tc3, 2 tc2, 3 SIMT
    int last_nsplit2 = 0;       // its SV-tile split (haf_info.reserved[3]; 0 outside the tensor kernels)
    int smem_optin = 0;         // the device's opt-in shared memory per block

    // per-call state
    DevBuf<unsigned char> d_xyz;       // staging for host clouds
    DevBuf<unsigned char> d_params;    // per-call parameter block (units, jobs, point offsets, unit ranges)
    DevBuf<long long> d_ptoff;
    DevBuf<int> d_cloud_ubegin;
    DevBuf<UnitParams> d_units;
    DevBuf<JobParams> d_jobs;
    DevBuf<JobResult> d_results;
    DevBuf<int> d_per_roll_top;
    DevBuf<unsigned> d_keys;            // [Uc][G][G] keys -> heights
    DevBuf<float> d_integral;           // [Uc][G+1][G+1]
    DevBuf<double> d_rowscan;           // large-G scratch
    DevBuf<unsigned char> d_mask;
    DevBuf<signed char> d_labelgrid;
    DevBuf<float> d_evals;
    DevBuf<unsigned long long> d_unit_block;            // one allocation, one memset per call: unit_top [U], unit_run [U] (u64), unit_windows [U] (u32)
    DevBuf<int2> d_win;
    DevBuf<float> d_X, d_xn;
    DevBuf<double> d_dec;
    DevBuf<unsigned char> d_guardflag;
    DevBuf<int> d_guardlist;
    DevBuf<double> d_kscratch;
    // guard band tier 2 (FP64 FMA contraction on the exact inputs, kernels.cuh guard_fma_kernel)
    int tier2_mode = 0;                 // cfg.reserved[2] & 3: 0 on, 1 off (guard list straight to the exact-order kernels), 2 on but everything escalates (tests)
    int tier2_kernel = 0;               // cfg.reserved[2] >> 2: 0 auto (DMMA for batches, DFMA for a single goal's handful), 1 DMMA always, 2 DFMA always
    DevBuf<double> d_svn64, d_Xg, d_g2accum, d_xn64;
    DevBuf<unsigned> d_g2tickets;
    DevBuf<int> d_guardlist2;
    DevBuf<unsigned> d_counters;        // [0]=win_count [1]=guard_count [2]=overflow [3]=unsupported ; [4..5] clamp (u64)
    // Host-staged batches run their chunks ALTERNATELY on two streams with two sets of the per-chunk buffers (swap_chunk_ws):
    // a chunk is a chain of ~18 dependent kernels, half of them latency-sized (integral prefix chains, guard tiers, score,
    // tie rule) -- the next chunk's big kernels fill the SMs those leave idle.  Set B's counters are d_counters[16..32).
    struct ChunkWs {
        DevBuf<__half> d_Xh, d_Xl;
        DevBuf<float> d_asum, d_integral, d_evals, d_X, d_xn, d_probgrid;
        DevBuf<double> d_dec_tc, d_rowscan, d_dec, d_kscratch, d_Xg, d_g2accum, d_xn64;
        DevBuf<unsigned> d_keys, d_g2tickets;
        DevBuf<unsigned char> d_mask, d_guardflag;
        DevBuf<signed char> d_labelgrid;
        DevBuf<int2> d_win;
        DevBuf<int> d_guardlist, d_guardlist2;
        DevBuf<uint2> d_rank_tiles;
    } alt[3];
    cudaStream_t chunk_stream2[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_dual[4];             // [0] head of the call done on the main stream, [1 + k] extra stream k drained
    bool ev_dual_ok = false;
    // PAGEABLE host clouds (what the action server holds: a pcl::PointCloud, INTEGRATION.md): cudaMemcpyAsync from pageable
    // memory goes through the driver's own staging at ~9 GB/s and blocks the calling thread.  Batches of 4 MB and more are
    // staged by the library instead: a helper thread copies each piece into a ring of pinned slots with a few host threads
    // (stage_threads, HAF_STAGE_THREADS; 0 = leave it to the driver) and issues the piece's H2D copy and event; the enqueuing
    // thread waits (host side) until the pieces a chunk needs have been ISSUED before it makes the chunk's stream wait for them.
    struct Stager {
        std::thread th;
        std::mutex mu;
        std::condition_variable cv;
        int issued = 0;        // pieces whose copy + event have been issued on copy_stream
        bool failed = false, active = false;
    } stager;
    PinBuf<unsigned char> h_ring;       // kRingSlots pinned slots of one piece each
    static constexpr int kRingSlots = 4;
    int stage_threads = 8;
    PinBuf<unsigned char> h_stage;      // pinned staging for params / results
    PinBuf<JobResult> h_results;
    PinBuf<int> h_per_roll_top;
    PinBuf<unsigned> h_counters;

    // ONE CUDA GRAPH PER REQUEST SHAPE (SURVEY 7 "hard parts"; server.cpp:335-402 is one goal = ~25 dependent stream operations of a
    // few microseconds each).  A call that fits one pass and repeats the shape of the previous one (same unit / window bounds,
    // same buffers, same kernel choices -- GraphKey) is captured once and then replayed with cudaGraphLaunch; the request itself
    // travels through the pinned parameter block, which the graph's first node reads afresh.  graph_mode: 0 on, 1 off (the default of a zero-initialised config).
    struct GraphKey {
        unsigned long long epoch; const void* xyz; size_t stride, wcap; long long pts_bucket; int n_jobs, n_clouds, flags, tc_passes;
        const void *o_evals, *o_mask, *o_heights; unsigned long long rolls_hash; cudaStream_t st;
        int rank_k, rank_p; double rank_md2;   // candidate ranking (0 when off)
        bool operator==(const GraphKey& o) const { return memcmp(this, &o, sizeof *this) == 0; }
    };
    // a few graphs per context, least recently used out: a goal sharded over ranks alternates between two or three shapes
    // (roll ranges of 12, 12 and 6 units, say), and one graph slot made every other call re-capture (instantiation costs more
    // than the launches it saves: configs[2] on two GPUs took 1.20 ms per step that way)
    struct GraphEntry { GraphKey key; cudaGraphExec_t exec; long long nodes; unsigned long long last_use; };
    std::vector<GraphEntry> graphs;       // <= kMaxGraphs instantiated graphs
    std::vector<GraphKey> graph_seen;     // shapes met once (a ring of kMaxGraphs): the second call of a shape captures
    size_t graph_seen_next = 0;
    unsigned long long graph_clock = 0;
    static constexpr size_t kMaxGraphs = 8;
    long long graph_replays = 0;
    unsigned long long alloc_epoch = 0;   // moved on by every ENSURE that (re)allocates one of this context's buffers
    int graph_mode = 0;
    cudaStream_t own_stream = nullptr;     // capture is not allowed on the legacy default stream: a blocking stream of our own stands in
    PinBuf<float> h_out_evals, h_out_heights;   // per-roll outputs asked for in HOST memory go through pinned staging (graph-capturable)
    PinBuf<unsigned char> h_out_mask;

    // grasp poses (haf_search_grasps / haf_search_batch_packed_grasps, kernels.cuh a16): 0 = not asked for (no pose kernel runs),
    // 1 = one record per job, 2 = the record of every unit comes back to the host as well.  Set for one call by GraspScope.
    int grasp_mode = 0;
    DevBuf<GraspRec> d_unit_grasp;       // [U] written chunk by chunk (outlives the per-chunk buffers)
    PinBuf<GraspRec> h_unit_grasp, h_job_grasp;   // h_job_grasp [n_jobs] is written by grasp_gather_kernel itself (UVA)

    // unit parameters built on the device (haf_search_batch_requests, kernels.cuh expand_units_kernel); set for one call by
    // DeviceUnitsScope.  The host part: the libm values per roll (built at haf_create) and per distinct approach vector.
    bool device_units = false;
    std::vector<hafhost::RollTrig> roll_trig;            // [R]
    std::vector<hafhost::ApproachTrig> approach_trig;    // distinct approach vectors of the call, first occurrence order
    std::vector<int> job_approach;                       // [n_jobs] index into approach_trig
    struct ApproachKey {
        uint64_t b[3];
        bool operator==(const ApproachKey& o) const { return b[0] == o.b[0] && b[1] == o.b[1] && b[2] == o.b[2]; }
    };
    struct ApproachHash {
        size_t operator()(const ApproachKey& k) const { return (size_t)((k.b[0] * 0x9E3779B97F4A7C15ull) ^ (k.b[1] * 0xC2B2AE3D27D4EB4Full) ^ (k.b[2] * 0x165667B19E3779F9ull)); }
    };
    std::unordered_map<ApproachKey, int, ApproachHash> approach_index;
    DevBuf<UnitParams> d_dev_units;      // [U]
    DevBuf<UnitPose> d_dev_pose;         // [U] one pose per unit
    PinBuf<float> h_best_M;              // [n_jobs][16] matrix of each job's winning roll (written by reduce_rolls_kernel, UVA)

    // ranked candidates (haf_search_batch_candidates, kernels.cuh rank_*_kernel); set for one call by RankScope.  rank_k 0 = off.
    int rank_k = 0, rank_p = 0;          // candidates per cloud, list depth per unit
    double rank_md2 = -1.0;              // min_distance^2; -1 = no suppression
    DevBuf<CandRec> d_rank_entries;      // [U][P] unit lists (call-wide, written chunk by chunk)
    DevBuf<RankCompact> d_rank_compact;  // [U][P]
    DevBuf<float> d_rank_top_score;      // [U] graspseval value of each unit's top cell
    DevBuf<uint2> d_rank_tiles;          // [Uc][tiles][P] per-tile selections (G > 90)
    PinBuf<CandRec> h_cand;              // [n_clouds][k], written by rank_cloud_kernel (UVA)
    PinBuf<int> h_ncand;                 // [n_clouds]
    // where the unit parameters of the last call live, whichever path built them (haf_debug_unit_params); units 0 = none
    const UnitParams* last_up_units = nullptr;
    const UnitPose* last_up_pose = nullptr;   // NULL: the call built no poses
    const int* last_up_jpose = nullptr;       // [n_jobs] pose set of each job
    int last_up_n = 0, last_up_jobs = 0;
    // per chunk of the last call: first cloud, end cloud, stream set, copy piece its stream waited for (-1: none), that piece's
    // end cloud, then binning kernel, unit groups, units per group, slices and integral variant (haf_debug_chunk_copy_waits)
    std::vector<int> last_chunk_waits;

    // probability estimates (SURVEY 8f-4): the model's sigmoid (svm.cpp:2811-2824); probability calls evaluate EVERY row /
    // window on the FP64 exact-order path (force_exact), whatever svm_mode the context was made with
    bool has_prob = false, force_exact = false;
    double probA = 0, probB = 0;
    int prob_res[2] = {0, 0};        // (int)atof(first two characters of "%g"(label)): server.cpp:833
    float prob_header_val = 0.0f;    // the "labels l0 l1" line parsed as a prediction: 0 * (float)l0 (server.cpp:817, :833-841)
    DevBuf<float> d_probgrid;        // [Uc][G][G] graspsgrid as floats (probability mode)

    // PCD / PointCloud2 ingest on the device (pcd_ingest.cuh)
    DevBuf<unsigned char> d_pcd_raw, d_pcd_blob;
    DevBuf<float> d_pcd_xyz;
    DevBuf<unsigned> d_pcd_tiles;
    DevBuf<unsigned long long> d_pcd_status;  // per call: [0] ASCII record total, then record counts, flags and LZF status per file
    DevBuf<unsigned char> d_pcd_params;       // per call: the file / segment tables (pcd_ingest.cuh), sent from h_pcd_params
    PinBuf<unsigned char> h_pcd_params;
    PinBuf<unsigned long long> h_pcd_status;
    cudaEvent_t pcd_params_ev = nullptr;      // the last H2D copy of h_pcd_params (the next call refills it after that copy)

    // libsvm front end (haf_svm_*): inputs given by the caller
    bool svm_only = false;
    const double* cur_xdense = nullptr;   // non-null while haf_svm_predict runs: exact_scaled_input reads it
    DevBuf<double> d_xdense, d_labels, d_probs;
    DevBuf<long long> d_csr_ptr;
    DevBuf<int> d_csr_idx;
    DevBuf<double> d_csr_val;

    // state of the last search kept for the debug entry points
    // several GPUs behind one context (haf_config.n_devices > 1): group[0] is this context itself, the others are member
    // contexts, one per further device, driven by one host thread each (group_search / group_batch below)
    std::vector<haf_ctx*> group;
    PinBuf<unsigned> h_unit_windows;   // windows per unit of the last call (the group merge replays the early exit with them)
    bool debug_keep_batch = false;   // haf_set_debug: keep the per-window state of single-chunk batch calls too
    int last_units = 0, last_unit_base = 0;
    unsigned last_W = 0;
    size_t last_ldx = 0;
    bool last_valid = false;

    int fail(int code, const char* fmt, ...) {
        char buf[1024];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return code;
    }
};

// exchanges the per-chunk buffers of the context with its second set (pointers and capacities only)
static void swap_chunk_ws(haf_ctx* c, int k = 0) {
#define HAF_SWAP(m) std::swap(c->m, c->alt[k].m)
    HAF_SWAP(d_Xh); HAF_SWAP(d_Xl); HAF_SWAP(d_asum); HAF_SWAP(d_integral); HAF_SWAP(d_evals); HAF_SWAP(d_X); HAF_SWAP(d_xn); HAF_SWAP(d_probgrid);
    HAF_SWAP(d_dec_tc); HAF_SWAP(d_rowscan); HAF_SWAP(d_dec); HAF_SWAP(d_kscratch); HAF_SWAP(d_Xg); HAF_SWAP(d_g2accum); HAF_SWAP(d_xn64);
    HAF_SWAP(d_keys); HAF_SWAP(d_g2tickets); HAF_SWAP(d_mask); HAF_SWAP(d_guardflag); HAF_SWAP(d_labelgrid); HAF_SWAP(d_win);
    HAF_SWAP(d_guardlist); HAF_SWAP(d_guardlist2); HAF_SWAP(d_rank_tiles);
#undef HAF_SWAP
}

#define CUDA_TRY(ctx, expr)                                                                                   \
    do {                                                                                                      \
        cudaError_t _e = (expr);                                                                              \
        if (_e != cudaSuccess) return (ctx)->fail(HAF_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define ENSURE(ctx, buf, n)                                                                                   \
    do {                                                                                                      \
        const void* _p0 = (const void*)(buf).p;                                                               \
        const unsigned long long _g0 = g_alloc_epoch;                                                         \
        const int _rc = (buf).ensure(n);                                                                      \
        g_alloc_epoch = _g0; /* this context's buffer: only this context's graph goes stale */                \
        if ((const void*)(buf).p != _p0) (ctx)->alloc_epoch++;                                                \
        if (_rc != 0) return (ctx)->fail(HAF_ERR_NOMEM, "out of device/pinned memory for %s (%zu elements)", #buf, (size_t)(n)); \
    } while (0)
#define LAUNCHED(ctx)                                                                                         \
    do {                                                                                                      \
        (ctx)->launches++;                                                                                    \
        cudaError_t _e = cudaGetLastError();                                                                  \
        if (_e != cudaSuccess) return (ctx)->fail(HAF_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

static size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

// ------------------------------------------------------------------------------------------------------------
// context creation: parse the three files once, derive the per-dimension scaling table, upload everything
// ------------------------------------------------------------------------------------------------------------
extern "C" const char* haf_version(void) { return HAF_VERSION_STRING; }

extern "C" const char* haf_last_error(const haf_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

static int create_fail(int code, const std::string& msg) {
    g_create_error = msg;
    return code;
}

// ---- tensor-core path helpers -------------------------------------------------------------------------------
// IEEE binary16 <-> float on the host (round to nearest even, subnormals kept): the operand format of the contraction
static uint16_t f2h16(float f) { return __half_as_ushort(__float2half_rn(f)); }
static float h16f(uint16_t h) { return __half2float(__ushort_as_half(h)); }
typedef CUresult (*haf_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static haf_encode_tiled_fn get_encode_tiled() {
    static haf_encode_tiled_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (haf_encode_tiled_fn)p;
        else
            cudaGetLastError();
    }
    return fn;
}
// How many of the three split products does this model need?  The operand error of the cheaper schemes -- 2 passes:
// x rounded to fp16, sv kept as a pair; 1 pass: both rounded to fp16 -- scales with gamma and is measured here in the
// unit the guard band uses (E = sum_i |coef_i| K_i (1 + gamma log2e (|x|^2 + |sv_i|^2)) + |rho|), with up to 48 of the
// model's own support vectors standing in for the windows (they ARE scaled feature vectors of training windows).
// rel[p] = max over probes of |dec_p - dec| / E.  The caller accepts the cheapest scheme whose error, together with the
// measured FP32 epilogue error (2.5e-7 E), keeps the default 15x margin inside a guard band of at most 1.2e-5.
static void calibrate_tensor_passes(const hafhost::Model& model, int Dsv, double rel[4]) {
    const int S = model.l;
    std::vector<double> sv((size_t)S * Dsv, 0.0), sh((size_t)S * Dsv, 0.0), sn(S, 0.0);
    for (int i = 0; i < S; i++)
        for (size_t e = 0; e < model.sv[i].size(); e++) {
            const int d = model.sv[i][e].first - 1;
            const double v = model.sv[i][e].second;
            sv[(size_t)i * Dsv + d] = v;
            sh[(size_t)i * Dsv + d] = (double)h16f(f2h16((float)v));
            sn[i] += v * v;
        }
    rel[1] = rel[2] = rel[3] = 0.0;
    const int nprobe = std::min(S, 48);
    const double g2 = model.gamma * 1.4426950408889634;
    for (int k = 0; k < nprobe; k++) {
        const int j = (int)((long long)k * S / nprobe);
        const double* x = &sv[(size_t)j * Dsv];
        const double* xh = &sh[(size_t)j * Dsv];
        double dec = 0, dec1 = 0, dec2 = 0, E = fabs(model.rho);
        for (int i = 0; i < S; i++) {
            const double* s = &sv[(size_t)i * Dsv];
            const double* s16 = &sh[(size_t)i * Dsv];
            double dot = 0, dot1 = 0, dot2 = 0;   // exact, x_hi.sv_hi, x_hi.sv
            for (int d = 0; d < Dsv; d++) { dot += x[d] * s[d]; dot1 += xh[d] * s16[d]; dot2 += xh[d] * s[d]; }
            const double base = sn[j] + sn[i];
            const double K = exp(-model.gamma * std::max(base - 2.0 * dot, 0.0));
            dec += model.coef[i] * K;
            dec1 += model.coef[i] * exp(-model.gamma * std::max(base - 2.0 * dot1, 0.0));
            dec2 += model.coef[i] * exp(-model.gamma * std::max(base - 2.0 * dot2, 0.0));
            E += fabs(model.coef[i]) * K * (1.0 + g2 * base);
        }
        rel[1] = std::max(rel[1], fabs(dec1 - dec) / E);
        rel[2] = std::max(rel[2], fabs(dec2 - dec) / E);
    }
}
// Operand tensor in the k-block tiled layout (kernels.cuh, kt_off): seen by TMA as [n_tiles * 128 rows][64 fp16], pitch 128 B
// = fully contiguous; one box = 64 x 128 = one 16 KB tile (row tile, k-block), 128B swizzle.  rows is a multiple of 128.
static bool make_tensor_map(CUtensorMap* m, void* base, int KB, uint64_t rows) {
    haf_encode_tiled_fn fn = get_encode_tiled();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)haftc::BK, rows / 128 * (cuuint64_t)KB * 128};
    cuuint64_t strides[1] = {(cuuint64_t)haftc::BK * 2};
    cuuint32_t box[2] = {(cuuint32_t)haftc::BK, (cuuint32_t)haftc::BM};
    cuuint32_t es[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// svm_only: context of the libsvm front end (haf_svm_create): model only, the SVM inputs are given by the caller, at
// least min_dims dimensions wide.
static int create_impl(haf_ctx** out, const haf_config* cfg, bool svm_only, int min_dims) {
    if (!out || !cfg) return create_fail(HAF_ERR_ARG, "haf_create: null argument");
    *out = nullptr;
    if (!cfg->model_path || (!svm_only && (!cfg->features_path || !cfg->range_path)))
        return create_fail(HAF_ERR_ARG, "haf_create: features_path, range_path and model_path are required");
    const int emu = cfg->emulate_text_roundtrip >= 0 ? 1 : 0;   // 0 (a zeroed config) and 1 = reference-exact; -1 = skip the text round trips
    const int G = cfg->grid > 0 ? cfg->grid : 56;
    if (G < 16 || G > 1024 || (G & 1)) return create_fail(HAF_ERR_ARG, "haf_create: grid must be even and within 16..1024");
    const int step = cfg->roll_step_deg > 0 ? cfg->roll_step_deg : 15;
    const int rmax = cfg->roll_max_deg > 0 ? cfg->roll_max_deg : 190;
    const int R = rmax / step;
    if (R < 1 || R > 360) return create_fail(HAF_ERR_ARG, "haf_create: roll_max_deg / roll_step_deg must give 1..360 rolls");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return create_fail(HAF_ERR_NO_DEVICE, "no CUDA device visible: libhafgpu has no CPU fallback"); }
    if (cfg->device < 0 || cfg->device >= ndev) return create_fail(HAF_ERR_ARG, "haf_create: device ordinal out of range");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) { cudaGetLastError(); return create_fail(HAF_ERR_CUDA, "cudaGetDeviceProperties failed"); }
    if (prop.major != 10) {
        char b[256];
        snprintf(b, sizeof b, "device %d is sm_%d%d; libhafgpu is built for sm_100a only and has no fallback", cfg->device, prop.major, prop.minor);
        return create_fail(HAF_ERR_NO_DEVICE, b);
    }

    std::string err;
    std::vector<hafhost::Feature> feats;
    if (!svm_only && !hafhost::load_features(cfg->features_path, feats, err)) return create_fail(HAF_ERR_IO, err);
    hafhost::Range range;
    if (!svm_only && !hafhost::load_range(cfg->range_path, range, err)) return create_fail(HAF_ERR_IO, err);
    hafhost::Model model;
    bool unsupported = false;
    if (!hafhost::load_model(cfg->model_path, model, err, unsupported)) return create_fail(unsupported ? HAF_ERR_UNSUPPORTED : HAF_ERR_IO, err);

    const int F = (int)feats.size();
    const int nshaf = cfg->nr_features_without_shaf > 0 ? cfg->nr_features_without_shaf : 302;
    // region corners index the 15x15 patch: x2+1, y2+1 must stay <= 14 (the reference would read out of bounds)
    for (int k = 0; k < F; k++)
        for (int r = 0; r < 3; r++) {
            if (hafhost::region_skipped(feats[k], r)) continue;
            for (int q = 0; q < 4; q++)
                if (feats[k].reg[4 * r + q] < 0 || feats[k].reg[4 * r + q] > 13) {
                    char b[256];
                    snprintf(b, sizeof b, "feature %d region %d has a corner outside 0..13: outside the reference's 15x15 patch", k + 1, r + 1);
                    return create_fail(HAF_ERR_UNSUPPORTED, b);
                }
        }

    // svm-scale's dimension table.  max_index = max(range file, data) (svm-scale.c:106-146); features without a
    // range entry would be scaled by the min/max of each roll's own data (:165-198): reproduced only when the
    // feature is structurally constant (all regions skipped -> single-valued -> dropped, :336-337).
    const int max_index = svm_only ? 0 : std::max(range.max_index, F);
    std::vector<DimDev> dims(max_index);
    int D_eff = 0;
    for (int i = 1; i <= max_index; i++) {
        DimDev d;
        memset(&d, 0, sizeof d);
        const bool has = i < (int)range.has.size() && range.has[i];
        if (i <= F) {
            d.feat = i - 1;
            if (has) {
                d.fmin = range.fmin[i]; d.fmax = range.fmax[i]; d.den = d.fmax - d.fmin;
                d.drop = (d.fmax == d.fmin) ? 1 : 0;
            } else {
                bool constant = true;
                for (int r = 0; r < 3; r++) if (!hafhost::region_skipped(feats[i - 1], r)) constant = false;
                if (!constant) {
                    char b[320];
                    snprintf(b, sizeof b, "feature %d has no entry in the range file: svm-scale -r would scale it with the min/max of each roll's own data, which this path does not reproduce", i);
                    return create_fail(HAF_ERR_UNSUPPORTED, b);
                }
                d.drop = 1;
            }
        } else {  // index only in the range file: the data never carries it -> value 0 every time (svm-scale.c:281-282)
            d.feat = -1;
            d.fmin = range.fmin[i]; d.fmax = range.fmax[i]; d.den = d.fmax - d.fmin;
            d.drop = (d.fmax == d.fmin) ? 1 : 0;
            double val = 0.0;
            if (!d.drop) {
                double v = 0.0;
                if (v == d.fmin) val = range.lower;
                else if (v == d.fmax) val = range.upper;
                else val = range.lower + (range.upper - range.lower) * (v - d.fmin) / (d.fmax - d.fmin);
                if (val != 0.0 && emu) val = hafdec::text6(val);
            }
            d.cval = val;
        }
        d.slope = d.drop ? 0.0 : (range.upper - range.lower) / d.den;
        dims[i - 1] = d;
        if (!d.drop) D_eff = i;
    }
    if (svm_only) {   // inputs are given: every dimension up to the widest of model / data takes part (svm.cpp:328-364)
        D_eff = std::max(std::max(model.max_index, min_dims), 1);
        DimDev dz;
        memset(&dz, 0, sizeof dz);
        dz.feat = -1;
        dims.assign(D_eff, dz);
    }
    if (D_eff == 0) return create_fail(HAF_ERR_UNSUPPORTED, "no feature survives scaling");
    const int D = D_eff;                              // trailing dropped dimensions are always 0: not stored
    const int Dsv = std::max(D, model.max_index);     // distance loop length of the exact path
    const int Kpad = (int)round_up((size_t)Dsv, SVM_BK);
    const int S = model.l;
    const int Spad = (int)round_up((size_t)S, SVM_BN);

    haf_ctx* ctx = new haf_ctx();
    ctx->cfg = *cfg;
    ctx->cfg.emulate_text_roundtrip = emu;
    ctx->cfg.grid = G; ctx->cfg.roll_step_deg = step; ctx->cfg.roll_max_deg = rmax; ctx->cfg.nr_features_without_shaf = nshaf;
    ctx->device = cfg->device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    ctx->F = F; ctx->D = D; ctx->Dsv = Dsv; ctx->Kpad = Kpad; ctx->S = S; ctx->Spad = Spad; ctx->R = R; ctx->G = G;
    for (int roll = 0; roll < R; roll++) ctx->roll_trig.push_back(hafhost::roll_trig(roll, step));
    ctx->lower = range.lower; ctx->upper = range.upper; ctx->gamma = model.gamma; ctx->rho = model.rho;
    ctx->label[0] = model.label[0]; ctx->label[1] = model.label[1];
    ctx->gv[0] = hafhost::label_to_gridvalue(model.label[0]);
    ctx->gv[1] = hafhost::label_to_gridvalue(model.label[1]);
    {
        double sac = 0.0;
        for (int i = 0; i < model.l; i++) sac += fabs(model.coef[i]);
        ctx->e_floor = (float)(sac * 7.888609052210118e-31);   // 2^-100
    }
    ctx->has_prob = model.has_probA && model.has_probB;   // svm_check_probability_model (svm.cpp:3098-3104)
    ctx->probA = model.probA; ctx->probB = model.probB;
    for (int k = 0; k < 2; k++) {
        char b[64];
        snprintf(b, sizeof b, "%g", (double)model.label[k]);   // svm-predict.c:114
        b[2] = 0;
        ctx->prob_res[k] = (int)atof(b);                         // int res = atof(line.substr(0,2)) (server.cpp:833)
    }
    ctx->prob_header_val = (float)0 * (float)(double)model.label[0];
    ctx->guard_rel = cfg->guard_rel > 0 ? cfg->guard_rel : 2e-6f;   // of E = sum|coef|K(1+|c|(xn+svn)) + |rho|; measured FP32 SIMT error <= 1.3e-7 E (tools/dec_error_probe.py)
    memset(&ctx->timing, 0, sizeof ctx->timing);
    if (ctx->gv[0] < -128 || ctx->gv[0] > 127 || ctx->gv[1] < -128 || ctx->gv[1] > 127) { delete ctx; return create_fail(HAF_ERR_UNSUPPORTED, "model labels do not fit the grasp grid"); }

#define CREATE_TRY(expr)                                                                     \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            std::string m = std::string(#expr) + " failed: " + cudaGetErrorString(_e);       \
            haf_destroy(ctx);                                                                \
            return create_fail(HAF_ERR_CUDA, m);                                             \
        }                                                                                    \
    } while (0)
    CREATE_TRY(cudaSetDevice(ctx->device));

    // device feature table (corner offsets for row stride G+1)
    std::vector<FeatDev> fd(F);
    const int ld = G + 1;
    for (int k = 0; k < F; k++) {
        FeatDev f;
        memset(&f, 0, sizeof f);
        for (int r = 0; r < 3; r++) {
            if (hafhost::region_skipped(feats[k], r)) continue;
            const int x1 = feats[k].reg[4 * r], x2 = feats[k].reg[4 * r + 1], y1 = feats[k].reg[4 * r + 2], y2 = feats[k].reg[4 * r + 3];
            f.off[4 * r + 0] = (x2 + 1) * ld + (y2 + 1);
            f.off[4 * r + 1] = x1 * ld + (y2 + 1);
            f.off[4 * r + 2] = (x2 + 1) * ld + y1;
            f.off[4 * r + 3] = x1 * ld + y1;
            f.w[r] = feats[k].w[r];
            f.flags |= (1 << r);
        }
        if (!(k < nshaf)) f.flags |= 0x100;
        fd[k] = f;
    }
    std::vector<float> svT((size_t)Kpad * Spad, 0.0f), svn(Spad, 0.0f), coef(Spad, 0.0f);
    const int Dsv16 = (int)round_up((size_t)Dsv, 16);   // the DMMA guard tier walks k-chunks of 16 dimensions: zero rows behind Dsv
    std::vector<double> sv64T((size_t)Dsv16 * Spad, 0.0), coef64(Spad, 0.0), svn64(Spad, 0.0);
    for (int i = 0; i < S; i++) {
        coef[i] = (float)model.coef[i];
        coef64[i] = model.coef[i];
        for (size_t e = 0; e < model.sv[i].size(); e++) svn64[i] = fma(model.sv[i][e].second, model.sv[i][e].second, svn64[i]);
        float nrm = 0.0f;
        for (size_t e = 0; e < model.sv[i].size(); e++) {
            const int d = model.sv[i][e].first - 1;
            const double v = model.sv[i][e].second;
            sv64T[(size_t)d * Spad + i] = v;
            const float fv = (float)v;
            svT[(size_t)d * Spad + i] = fv;
            nrm = fmaf(fv, fv, nrm);
        }
        svn[i] = nrm;
    }
    bool okb = ctx->d_feats.ensure(F) == 0 && ctx->d_dims.ensure(D) == 0 && ctx->d_svT.ensure(svT.size()) == 0 &&
               ctx->d_svn.ensure(Spad) == 0 && ctx->d_coef.ensure(Spad) == 0 && ctx->d_sv64T.ensure(sv64T.size()) == 0 &&
               ctx->d_coef64.ensure(Spad) == 0 && ctx->d_svn64.ensure(Spad) == 0 && ctx->d_counters.ensure(64) == 0 && ctx->h_counters.ensure(16) == 0;
    if (!okb) { haf_destroy(ctx); return create_fail(HAF_ERR_NOMEM, "out of device memory uploading the model"); }
    CREATE_TRY(cudaMemcpy(ctx->d_feats.p, fd.data(), F * sizeof(FeatDev), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_dims.p, dims.data(), D * sizeof(DimDev), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_svT.p, svT.data(), svT.size() * sizeof(float), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_svn.p, svn.data(), Spad * sizeof(float), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_coef.p, coef.data(), Spad * sizeof(float), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_sv64T.p, sv64T.data(), sv64T.size() * sizeof(double), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_coef64.p, coef64.data(), Spad * sizeof(double), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMemcpy(ctx->d_svn64.p, svn64.data(), Spad * sizeof(double), cudaMemcpyHostToDevice));
    // CUDA graphs are opt-in (cfg.reserved[1] bit 4 or HAF_GRAPH=1; a zero-initialised config launches plainly).  Measured on B200
    // WITHOUT per-stage timing events (profiling on disables graphs, and every timing event between two kernels costs ~20 us):
    // one table1 goal 0.224 ms launched, 0.189 ms replayed; the 512-grid 1 M-point goal 4.34 vs 4.31 ms (profiles/r2_final_*).
    ctx->graph_mode = ((cfg->reserved[1] & 16) || (getenv("HAF_GRAPH") && atoi(getenv("HAF_GRAPH")))) ? 0 : 1;
    // host threads that copy a pageable batch into the pinned ring: half the cores, at most 8 (measured, 614 MB per call, 16 cores:
    // the driver's pageable path 75 ms; 2 threads 45, 4: 28, 8: 24.8, 12: 23.3 ms -- against 12.6 ms from pinned memory)
    ctx->stage_threads = (int)std::max(1u, std::min(8u, std::thread::hardware_concurrency() / 2));
    if (const char* e = getenv("HAF_STAGE_THREADS")) ctx->stage_threads = std::max(0, std::min(16, atoi(e)));
    ctx->tier2_mode = cfg->reserved[2] & 3;
    ctx->tier2_kernel = (cfg->reserved[2] >> 2) & 3;
    CREATE_TRY(cudaFuncSetAttribute(guard_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HAF_GD_SMEM_BYTES));
    CREATE_TRY(cudaFuncSetAttribute(guard_fma_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CREATE_TRY(cudaFuncSetAttribute(guard_fma_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CREATE_TRY(cudaFuncSetAttribute(svm_rbf_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SVM_STAGES * SVM_BK * (SVM_BM + SVM_BN) * 4));
    CREATE_TRY(cudaFuncSetAttribute(integral_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    {   // the exact-order kernel stages the inputs of HAF_EXACT_WB windows (Dsv doubles each) in shared memory; a model too wide
        // for the device's opt-in maximum reads them from global memory instead (launch_exact).  The limit is only ever raised:
        // it is per function, and a context made earlier may need more than this one.
        const size_t need = (size_t)HAF_EXACT_WB * Dsv * sizeof(double);
        cudaFuncAttributes fa;
        CREATE_TRY(cudaFuncGetAttributes(&fa, svm_exact_terms_kernel));
        const int want = (int)std::max<size_t>(100 * 1024, need <= (size_t)ctx->smem_optin ? need : 0);
        if (want > fa.maxDynamicSharedSizeBytes) CREATE_TRY(cudaFuncSetAttribute(svm_exact_terms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, want));
    }
    CREATE_TRY(cudaFuncSetAttribute(bin_maxz_cloud_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CREATE_TRY(cudaFuncSetAttribute(bin_maxz_cloud_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    if (cfg->svm_mode == HAF_SVM_TENSOR_GUARD) {
        const int Krow = (int)round_up((size_t)Dsv + haftc::NAUG, 16);   // dimensions + the six extra operand columns (svm_tc.cuh)
        ctx->c_log2 = (float)(-model.gamma * 1.4426950408889634);
        if (cfg->guard_rel <= 0) ctx->guard_rel = 4e-6f;  // of E (see svm_tc.cuh); measured split-fp16 + fast-tier error <= 3.3e-7 E (tools/dec_error_probe.py)
        // tensor-path order of the support vectors: coef > 0 first, then coef <= 0, each group padded to whole tiles of BN,
        // so that every tile is uniform in sign (the guard scale is then sum over tiles of |tile sum|)
        std::vector<int> order;
        for (int pass = 0; pass < 2; pass++) {
            for (int i = 0; i < S; i++)
                if ((model.coef[i] > 0) == (pass == 0)) order.push_back(i);
            while (order.size() % haftc::BN) order.push_back(-1);
        }
        if (order.empty()) order.assign(haftc::BN, -1);
        const int SpadT = (int)order.size();
        const int KB = (Krow + haftc::BK - 1) / haftc::BK;
        ctx->Krow = Krow; ctx->KB = KB; ctx->SpadT = SpadT;
        std::vector<uint16_t> svh((size_t)SpadT * KB * haftc::BK, 0), svl((size_t)SpadT * KB * haftc::BK, 0);
        std::vector<float> tab(SpadT, 0.0f);
        const uint16_t one16 = f2h16(1.0f);
        for (int r = 0; r < SpadT; r++) {
            const int i = order[r];
            if (i < 0) continue;   // padding: all-zero row, coef 0
            float nrm = 0.0f;
            for (size_t e = 0; e < model.sv[i].size(); e++) {
                const int d = model.sv[i][e].first - 1;
                const float fv = (float)model.sv[i][e].second;
                if (!(fabsf(fv) <= 65504.0f)) {
                    haf_destroy(ctx);
                    return create_fail(HAF_ERR_UNSUPPORTED, "a support-vector component exceeds the fp16 range of the tensor path (use svm_mode HAF_SVM_FP32_GUARD)");
                }
                const uint16_t h = f2h16(fv);
                const uint16_t l = f2h16(fv - h16f(h));
                svh[kt_off((size_t)r, d, KB)] = h;
                svl[kt_off((size_t)r, d, KB)] = l;
                const float rep = h16f(h) + h16f(l);
                nrm = fmaf(rep, rep, nrm);
            }
            if (!(nrm < 1.3e5f)) {
                haf_destroy(ctx);
                return create_fail(HAF_ERR_UNSUPPORTED, "a support vector's squared norm exceeds the fp16 range of the tensor path (use svm_mode HAF_SVM_FP32_GUARD)");
            }
            // extra operand columns: 1 1 1 (against the window's -|x|^2 / 2 terms), then -|sv|^2 / 2 as three fp16 terms
            const float b = -0.5f * nrm;
            const uint16_t bh = f2h16(b);
            const float r1 = b - h16f(bh);
            const uint16_t bm = f2h16(r1);
            const uint16_t aug[6] = {one16, one16, one16, bh, bm, f2h16(r1 - h16f(bm))};
            for (int q = 0; q < 6; q++) svh[kt_off((size_t)r, Dsv + q, KB)] = aug[q];
            tab[r] = (float)model.coef[i];
            ctx->csvn_max = std::max(ctx->csvn_max, fabsf(ctx->c_log2 * nrm));
        }
        bool okt = ctx->d_SVh.ensure(svh.size()) == 0 && ctx->d_SVl.ensure(svl.size()) == 0 && ctx->d_svcoef.ensure(SpadT) == 0;
        if (!okt) { haf_destroy(ctx); return create_fail(HAF_ERR_NOMEM, "out of device memory uploading the fp16 model"); }
        CREATE_TRY(cudaMemcpy(ctx->d_SVh.p, svh.data(), svh.size() * 2, cudaMemcpyHostToDevice));
        CREATE_TRY(cudaMemcpy(ctx->d_SVl.p, svl.data(), svl.size() * 2, cudaMemcpyHostToDevice));
        CREATE_TRY(cudaMemcpy(ctx->d_svcoef.p, tab.data(), SpadT * sizeof(float), cudaMemcpyHostToDevice));
        ctx->tc_variant = cfg->reserved[0] & 3;
        if (cfg->reserved[0] & 0x100) ctx->audit_every = 0;                       // bit 8: audit sample off (guard-band windows are still compared)
        else if (cfg->reserved[0] >> 16) ctx->audit_every = cfg->reserved[0] >> 16;   // bits 16+: sample every n-th window (tests)
        {   // number of tensor-core products per k-slice: forced by cfg.reserved[0] bits 4-5, else calibrated per model
            const int forced = (cfg->reserved[0] >> 4) & 3;
            double rel[4] = {0, 0, 0, 0};
            if (!forced || cfg->guard_rel <= 0) calibrate_tensor_passes(model, Dsv, rel);
            int passes = 3;
            if (forced) passes = forced;
            else if (rel[1] <= 5.5e-7) passes = 1;
            else if (rel[2] <= 5.5e-7) passes = 2;
            ctx->tc_passes = passes;
            ctx->tc_operand_err = passes < 3 ? rel[passes] : 0.0;
            if (cfg->guard_rel <= 0) ctx->guard_rel = std::max(4e-6f, (float)(15.0 * (ctx->tc_operand_err + 2.5e-7)));
        }
        if (!make_tensor_map(&ctx->tmSh2, ctx->d_SVh.p, KB, SpadT) || !make_tensor_map(&ctx->tmSl2, ctx->d_SVl.p, KB, SpadT)) {
            haf_destroy(ctx);
            return create_fail(HAF_ERR_CUDA, "cuTensorMapEncodeTiled failed for the support-vector operands");
        }
        // one table per row-stride class of the staged integral rows (features_tc_kernel: bank-conflict-free staging)
        std::vector<DimFeat> joined((size_t)32 * D);
        for (int cls = 0; cls < 32; cls++)
        for (int d = 0; d < D; d++) {
            DimFeat j;
            memset(&j, 0, sizeof j);
            const DimDev& dd = dims[d];
            if (dd.feat >= 0) {
                const FeatDev& ff = fd[dd.feat];
                for (int r = 0; r < 3; r++) {
                    if (ff.flags & (1 << r)) {
                        for (int q = 0; q < 4; q++) {   // ff.off = x * ld + y  ->  (x * (ld + cls) + y) bytes
                            const int x = ff.off[4 * r + q] / ld, y = ff.off[4 * r + q] % ld;
                            j.off[4 * r + q] = (x * (ld + cls) + y) * 4;
                        }
                        j.w[r] = ff.w[r];
                    } else {  // skipped region: identical corners, weight +0.0 -> contributes exactly +0.0
                        for (int q = 0; q < 4; q++) j.off[4 * r + q] = 0;
                        j.w[r] = 0.0f;
                    }
                }
                j.flags = ff.flags & 0x104;   // SHAF, third region present
            } else {
                j.flags = 0x200;
            }
            if (dd.drop) j.flags |= 0x400;
            j.fmin = (float)dd.fmin; j.slope = (float)dd.slope; j.cval = (float)dd.cval;
            joined[(size_t)cls * D + d] = j;
        }
        Round4Tab r4;
        make_round4_table(r4);
        if (ctx->d_round4.ensure(1) != 0) { haf_destroy(ctx); return create_fail(HAF_ERR_NOMEM, "out of device memory uploading the rounding table"); }
        CREATE_TRY(cudaMemcpy(ctx->d_round4.p, &r4, sizeof(Round4Tab), cudaMemcpyHostToDevice));
        if (ctx->d_dimfeat.ensure(joined.size()) != 0) { haf_destroy(ctx); return create_fail(HAF_ERR_NOMEM, "out of device memory uploading the joined feature table"); }
        CREATE_TRY(cudaMemcpy(ctx->d_dimfeat.p, joined.data(), joined.size() * sizeof(DimFeat), cudaMemcpyHostToDevice));
        CREATE_TRY(cudaFuncSetAttribute(haftc::svm_rbf_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, haftc::SMEM2_BYTES + haftc::TAB_SMEM_MAX * 4));
        CREATE_TRY(cudaFuncSetAttribute(haftc::svm_rbf_tc3_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, haftc::TC3_SMEM_LIMIT));
        CREATE_TRY(cudaFuncSetAttribute(haftc::svm_rbf_tc3_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, haftc::TC3_SMEM_LIMIT));
        CREATE_TRY(cudaFuncSetAttribute(features_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ft_smem_layout(G, 1)));
        CREATE_TRY(cudaFuncSetAttribute(features_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ft_smem_layout(G, 2)));
        // 4 CTAs x ~49 KB: ask for just that much shared memory so that the rest of the SM's 256 KB stays L1 (the corner-offset table)
        CREATE_TRY(cudaFuncSetAttribute(features_tc_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 90));
        CREATE_TRY(cudaFuncSetAttribute(features_tc_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 90));
    }
    for (int i = 0; i < 10; i++) CREATE_TRY(cudaEventCreate(&ctx->ev[i]));
    ctx->ev_ok = true;
#undef CREATE_TRY
    *out = ctx;
    return HAF_OK;
}

extern "C" int haf_create(haf_ctx** out, const haf_config* cfg) {
    if (!out || !cfg) return create_fail(HAF_ERR_ARG, "haf_create: null argument");
    if (cfg->n_devices <= 1) {
        haf_config one = *cfg;
        if (cfg->n_devices == 1 && cfg->devices) one.device = cfg->devices[0];
        one.n_devices = 0; one.devices = nullptr;
        return create_impl(out, &one, false, 0);
    }
    // one context per device; the first one owns the group
    *out = nullptr;
    if (cfg->n_devices > 64) return create_fail(HAF_ERR_ARG, "haf_create: n_devices out of range");
    std::vector<haf_ctx*> members;
    for (int k = 0; k < cfg->n_devices; k++) {
        haf_config one = *cfg;
        one.device = cfg->devices ? cfg->devices[k] : k;
        one.n_devices = 0; one.devices = nullptr;
        for (size_t j = 0; j < members.size(); j++)
            if (members[j]->device == one.device) {
                for (size_t i = 0; i < members.size(); i++) haf_destroy(members[i]);
                return create_fail(HAF_ERR_ARG, "haf_create: devices[] names the same GPU twice");
            }
        haf_ctx* c = nullptr;
        const int rc = create_impl(&c, &one, false, 0);
        if (rc != HAF_OK) {
            for (size_t i = 0; i < members.size(); i++) haf_destroy(members[i]);
            return rc;   // g_create_error is set
        }
        members.push_back(c);
    }
    members[0]->group = members;
    *out = members[0];
    return HAF_OK;
}

// ---- libsvm front ends (SURVEY 8f-3) -------------------------------------------------------------------------
static int svm_stage(haf_ctx* ctx, unsigned* cnt, size_t Wcap, size_t ldx, int G, int ubase, cudaStream_t st, cudaEvent_t ev_guard);
extern "C" int haf_svm_create_config(haf_svm** out, const haf_config* cfg, int min_dims) {
    if (!out || !cfg) return create_fail(HAF_ERR_ARG, "haf_svm_create_config: null argument");
    haf_config one = *cfg;
    one.features_path = one.range_path = nullptr;
    one.n_devices = 0; one.devices = nullptr;
    const int rc = create_impl(out, &one, true, min_dims);
    if (rc == HAF_OK) (*out)->svm_only = true;
    return rc;
}
extern "C" int haf_svm_create(haf_svm** out, const char* model_path, int device, int svm_mode, int min_dims, float guard_rel) {
    haf_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.model_path = model_path;
    cfg.device = device;
    cfg.svm_mode = svm_mode;
    cfg.guard_rel = guard_rel;
    return haf_svm_create_config(out, &cfg, min_dims);
}
extern "C" void haf_svm_destroy(haf_svm* s) { haf_destroy(s); }

static int check_csr(haf_ctx* ctx, const long long* row_ptr, const int* index, const double* value, int n_rows) {
    if (!row_ptr || n_rows < 0) return ctx->fail(HAF_ERR_ARG, "null row_ptr / negative row count");
    for (int r = 0; r < n_rows; r++)
        if (row_ptr[r + 1] < row_ptr[r]) return ctx->fail(HAF_ERR_ARG, "row_ptr is not non-decreasing at row %d", r);
    if (n_rows && row_ptr[n_rows] > row_ptr[0] && (!index || !value)) return ctx->fail(HAF_ERR_ARG, "null index / value arrays");
    return HAF_OK;
}

// prob_estimates != NULL: svm_predict_probability for every row (svm.cpp:2550-2590) -- decision values on the FP64 exact-order
// path for EVERY row (the estimates are printed with six digits: they need the reference's own decision values, not a sign),
// then sigmoid + pairwise coupling on the device (prob_from_dec_kernel)
static int svm_predict_impl(haf_svm* ctx, const long long* row_ptr, const int* index, const double* value, int n_rows,
                            double* labels, double* dec_values, double* prob_estimates);
extern "C" int haf_svm_predict(haf_svm* ctx, const long long* row_ptr, const int* index, const double* value, int n_rows,
                               double* labels, double* dec_values) {
    if (!ctx) return HAF_ERR_ARG;
    return svm_predict_impl(ctx, row_ptr, index, value, n_rows, labels, dec_values, nullptr);
}
extern "C" int haf_svm_check_probability_model(const haf_svm* ctx) { return (ctx && ctx->has_prob) ? 1 : 0; }
extern "C" int haf_svm_predict_probability(haf_svm* ctx, const long long* row_ptr, const int* index, const double* value, int n_rows,
                                           double* labels, double* prob_estimates) {
    if (!ctx) return HAF_ERR_ARG;
    if (!prob_estimates) return ctx->fail(HAF_ERR_ARG, "haf_svm_predict_probability: prob_estimates is null");
    if (!ctx->has_prob) return ctx->fail(HAF_ERR_UNSUPPORTED, "Model does not support probabiliy estimates");   // svm-predict.c:213 (sic)
    ctx->force_exact = true;
    const int rc = svm_predict_impl(ctx, row_ptr, index, value, n_rows, labels, nullptr, prob_estimates);
    ctx->force_exact = false;
    return rc;
}
static int svm_predict_impl(haf_svm* ctx, const long long* row_ptr, const int* index, const double* value, int n_rows,
                            double* labels, double* dec_values, double* prob_estimates) {
    if (!ctx->svm_only) return ctx->fail(HAF_ERR_ARG, "haf_svm_predict needs a context made by haf_svm_create");
    const bool prob = prob_estimates != nullptr;
    { int rc = check_csr(ctx, row_ptr, index, value, n_rows); if (rc) return rc; }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const long long launches0 = ctx->launches;
    const int W = ctx->Dsv;
    for (int r = 0; r < n_rows; r++)   // svm-predict would index past the model's width: the caller sizes the context (min_dims)
        for (long long e = row_ptr[r]; e < row_ptr[r + 1]; e++)
            if (index[e] < 1 || index[e] > W) return ctx->fail(HAF_ERR_ARG, "row %d carries index %d outside 1..%d (create the context with min_dims >= the data's largest index)", r, index[e], W);
    memset(&ctx->timing, 0, sizeof ctx->timing);
    ctx->last_valid = false;
    if (n_rows == 0) return HAF_OK;
    const bool tc = ctx->cfg.svm_mode == HAF_SVM_TENSOR_GUARD && !prob;
    const size_t chunk_rows = std::max<size_t>(256, std::min<size_t>((size_t)n_rows, ((size_t)512 << 20) / ((size_t)W * sizeof(double))));
    ENSURE(ctx, ctx->h_stage, 64);
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[8], st));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, 16 * 4, st));
    long long total_guard = 0;
    for (size_t r0 = 0; r0 < (size_t)n_rows; r0 += chunk_rows) {
        const size_t rows = std::min(chunk_rows, (size_t)n_rows - r0);
        const size_t ldx = round_up(rows, 2 * haftc::BM);
        const long long e0 = row_ptr[r0], e1 = row_ptr[r0 + rows];
        ENSURE(ctx, ctx->d_csr_ptr, rows + 1); ENSURE(ctx, ctx->d_csr_idx, (size_t)std::max<long long>(e1 - e0, 1)); ENSURE(ctx, ctx->d_csr_val, (size_t)std::max<long long>(e1 - e0, 1));
        ENSURE(ctx, ctx->d_xdense, rows * W); ENSURE(ctx, ctx->d_labels, rows);
        ENSURE(ctx, ctx->d_xn, ldx); ENSURE(ctx, ctx->d_dec, ldx); ENSURE(ctx, ctx->d_guardflag, ldx); ENSURE(ctx, ctx->d_guardlist, ldx);
        if (tc) { ENSURE(ctx, ctx->d_Xh, ldx * ctx->KB * haftc::BK); if (ctx->tc_passes >= 3) ENSURE(ctx, ctx->d_Xl, ldx * ctx->KB * haftc::BK); ENSURE(ctx, ctx->d_asum, ldx); }
        else if (ctx->cfg.svm_mode == HAF_SVM_FP32_GUARD && !prob) ENSURE(ctx, ctx->d_X, (size_t)ctx->Kpad * ldx);
        if (prob) ENSURE(ctx, ctx->d_probs, rows * 2);
        const size_t exact_cap = std::min<size_t>(ldx, std::max<size_t>(4096, ((size_t)1 << 30) / ((size_t)ctx->Spad * 8)));
        ENSURE(ctx, ctx->d_kscratch, exact_cap * ctx->Spad);
        unsigned* cnt = ctx->d_counters.p;
        // the pinned word must not be rewritten while an earlier chunk's copy may still be in flight
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        *reinterpret_cast<unsigned*>(ctx->h_stage.p) = (unsigned)rows;
        if (r0 > 0) CUDA_TRY(ctx, cudaMemsetAsync(cnt, 0, 2 * 4, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(cnt, ctx->h_stage.p, 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_csr_ptr.p, row_ptr + r0, (rows + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
        if (e1 > e0) {
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_csr_idx.p, index + e0, (size_t)(e1 - e0) * sizeof(int), cudaMemcpyHostToDevice, st));
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_csr_val.p, value + e0, (size_t)(e1 - e0) * sizeof(double), cudaMemcpyHostToDevice, st));
        }
        CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_xdense.p, 0, rows * W * sizeof(double), st));
        csr_to_dense_kernel<<<(unsigned)rows, 128, 0, st>>>(ctx->d_csr_ptr.p, ctx->d_csr_idx.p, ctx->d_csr_val.p, (int)rows, W, ctx->d_xdense.p);
        LAUNCHED(ctx);
        if (ctx->cfg.svm_mode != HAF_SVM_FP64_EXACT && !prob) {
            pack_svm_inputs_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(ctx->d_xdense.p, (int)rows, W, ctx->Krow, ctx->KB, tc ? ctx->d_Xh.p : nullptr,
                                                                              (tc && ctx->tc_passes >= 3) ? ctx->d_Xl.p : nullptr, tc ? nullptr : ctx->d_X.p, ldx, ctx->Kpad, ctx->d_xn.p,
                                                                              tc ? ctx->d_dec.p : nullptr, tc ? ctx->d_asum.p : nullptr);
            LAUNCHED(ctx);
        }
        ctx->cur_xdense = ctx->d_xdense.p;
        const int rcs = svm_stage(ctx, cnt, rows, ldx, ctx->G, 0, st, nullptr);
        ctx->cur_xdense = nullptr;
        if (rcs) return rcs;
        if (prob) prob_from_dec_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(ctx->d_dec.p, (int)rows, ctx->probA, ctx->probB, (double)ctx->label[0], (double)ctx->label[1],
                                                                                      ctx->d_labels.p, ctx->d_probs.p);
        else labels_from_dec_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(ctx->d_dec.p, (int)rows, (double)ctx->label[0], (double)ctx->label[1], ctx->d_labels.p);
        LAUNCHED(ctx);
        if (prob) CUDA_TRY(ctx, cudaMemcpyAsync(prob_estimates + 2 * r0, ctx->d_probs.p, rows * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
        accumulate_counts_kernel<<<1, 1, 0, st>>>(cnt);
        LAUNCHED(ctx);
        if (labels) CUDA_TRY(ctx, cudaMemcpyAsync(labels + r0, ctx->d_labels.p, rows * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (dec_values) CUDA_TRY(ctx, cudaMemcpyAsync(dec_values + r0, ctx->d_dec.p, rows * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_counters.p, ctx->d_counters.p, 16 * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[9], st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (ctx->h_counters.p[10]) return ctx->fail(HAF_ERR_UNSUPPORTED, "the guard band holds more rows than the exact path is provisioned for (guard_rel too wide for this model)");
    total_guard = ctx->h_counters.p[9];
    memcpy(&ctx->audit_max_rel, &ctx->h_counters.p[12], sizeof(float));
    if (tc && ctx->tier2_mode != 1 && ctx->audit_max_rel > 0.25f * ctx->guard_rel) {   // audit (see run_jobs): repeat with one more product
        if (ctx->tc_passes >= 3)
            return ctx->fail(HAF_ERR_UNSUPPORTED, "audit: the tensor contraction is off by %.3g E on these rows, guard_rel = %.3g leaves less than a 4x margin",
                             (double)ctx->audit_max_rel, (double)ctx->guard_rel);
        ctx->tc_passes++;
        ctx->escalations++;
        return svm_predict_impl(ctx, row_ptr, index, value, n_rows, labels, dec_values, prob_estimates);
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[8], ctx->ev[9]);
    ctx->timing.ms_total = ms;
    ctx->timing.n_audit = ctx->h_counters.p[14];
    ctx->timing.audit_max_rel = ctx->audit_max_rel;
    ctx->timing.tc_passes = tc ? ctx->tc_passes : 0;
    ctx->timing.escalations = ctx->escalations;
    ctx->timing.n_windows = n_rows;
    ctx->timing.n_guard = total_guard;
    ctx->timing.n_exact = (ctx->tier2_mode == 1 && ctx->cfg.svm_mode != HAF_SVM_FP64_EXACT) ? total_guard : ctx->h_counters.p[11];
    ctx->timing.launches = ctx->launches - launches0;
    ctx->timing.n_chunks = (long long)((n_rows + chunk_rows - 1) / chunk_rows);
    return HAF_OK;
}

// svm-scale on the device.  fmin / fmax: [max_index + 1] (entry 0 unused), in/out for haf_scale_minmax so that a file can
// be walked in pieces (initialise with +DBL_MAX / -DBL_MAX like svm-scale.c:158-162).
struct ScaleBufs {
    long long* ptr = nullptr; int* idx = nullptr; double* val = nullptr; double* dense = nullptr;
    ~ScaleBufs() { cudaFree(ptr); cudaFree(idx); cudaFree(val); cudaFree(dense); }
};
static int scale_upload(int device, const long long* row_ptr, const int* index, const double* value, int n_rows, int max_index, ScaleBufs& b) {
    if (!row_ptr || n_rows < 0 || max_index < 1) return create_fail(HAF_ERR_ARG, "haf_scale: bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return create_fail(HAF_ERR_NO_DEVICE, "no CUDA device visible: libhafgpu has no CPU fallback"); }
    if (device < 0 || device >= ndev) return create_fail(HAF_ERR_ARG, "haf_scale: device ordinal out of range");
    const long long e0 = row_ptr[0], e1 = row_ptr[n_rows];
    for (long long e = e0; e < e1; e++)
        if (index[e - 0] < 1 || index[e] > max_index) return create_fail(HAF_ERR_ARG, "haf_scale: index outside 1..max_index");
#define SC_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return create_fail(HAF_ERR_CUDA, std::string(#expr) + " failed: " + cudaGetErrorString(_e)); } while (0)
    SC_TRY(cudaSetDevice(device));
    const size_t nnz = (size_t)std::max<long long>(e1 - e0, 1);
    SC_TRY(cudaMalloc(&b.ptr, ((size_t)n_rows + 1) * sizeof(long long)));
    SC_TRY(cudaMalloc(&b.idx, nnz * sizeof(int)));
    SC_TRY(cudaMalloc(&b.val, nnz * sizeof(double)));
    SC_TRY(cudaMalloc(&b.dense, std::max<size_t>((size_t)n_rows * max_index, 1) * sizeof(double)));
    SC_TRY(cudaMemcpy(b.ptr, row_ptr, ((size_t)n_rows + 1) * sizeof(long long), cudaMemcpyHostToDevice));
    if (e1 > e0) {
        SC_TRY(cudaMemcpy(b.idx, index + e0, (size_t)(e1 - e0) * sizeof(int), cudaMemcpyHostToDevice));
        SC_TRY(cudaMemcpy(b.val, value + e0, (size_t)(e1 - e0) * sizeof(double), cudaMemcpyHostToDevice));
    }
    SC_TRY(cudaMemset(b.dense, 0, std::max<size_t>((size_t)n_rows * max_index, 1) * sizeof(double)));
    if (n_rows) csr_to_dense_kernel<<<(unsigned)n_rows, 128>>>(b.ptr, b.idx, b.val, n_rows, max_index, b.dense);
    SC_TRY(cudaGetLastError());
    return HAF_OK;
}
static unsigned long long host_dkey(double v) {
    unsigned long long u;
    memcpy(&u, &v, 8);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
extern "C" int haf_scale_minmax(int device, const long long* row_ptr, const int* index, const double* value, int n_rows, int max_index,
                                double* fmin, double* fmax) {
    if (!fmin || !fmax) return create_fail(HAF_ERR_ARG, "haf_scale_minmax: null output");
    if (n_rows == 0) return HAF_OK;
    ScaleBufs b;
    { int rc = scale_upload(device, row_ptr, index, value, n_rows, max_index, b); if (rc) return rc; }
    std::vector<unsigned long long> kmin(max_index), kmax(max_index);
    for (int d = 0; d < max_index; d++) { kmin[d] = host_dkey(fmin[d + 1]); kmax[d] = host_dkey(fmax[d + 1]); }
    unsigned long long *dmin = nullptr, *dmax = nullptr; double* dout = nullptr; int* dflag = nullptr;
    struct Free { unsigned long long*& a; unsigned long long*& b; double*& c; int*& d; ~Free() { cudaFree(a); cudaFree(b); cudaFree(c); cudaFree(d); } } fr{dmin, dmax, dout, dflag};
    SC_TRY(cudaMalloc(&dmin, max_index * 8)); SC_TRY(cudaMalloc(&dmax, max_index * 8)); SC_TRY(cudaMalloc(&dout, 2 * (size_t)max_index * 8)); SC_TRY(cudaMalloc(&dflag, 4));
    SC_TRY(cudaMemcpy(dmin, kmin.data(), max_index * 8, cudaMemcpyHostToDevice));
    SC_TRY(cudaMemcpy(dmax, kmax.data(), max_index * 8, cudaMemcpyHostToDevice));
    SC_TRY(cudaMemset(dflag, 0, 4));
    const int rpb = 256;
    scale_minmax_kernel<<<dim3((max_index + 127) / 128, (n_rows + rpb - 1) / rpb), 128>>>(b.dense, n_rows, max_index, rpb, dmin, dmax, dflag);
    scale_minmax_decode_kernel<<<(max_index + 127) / 128, 128>>>(dmin, dmax, max_index, dout, dout + max_index);
    SC_TRY(cudaGetLastError());
    int flag = 0;
    SC_TRY(cudaMemcpy(&flag, dflag, 4, cudaMemcpyDeviceToHost));
    if (flag) return create_fail(HAF_ERR_UNSUPPORTED, "haf_scale_minmax: NaN in the data (svm-scale's max/min macros are order-dependent for NaN)");
    SC_TRY(cudaMemcpy(fmin + 1, dout, (size_t)max_index * 8, cudaMemcpyDeviceToHost));
    SC_TRY(cudaMemcpy(fmax + 1, dout + max_index, (size_t)max_index * 8, cudaMemcpyDeviceToHost));
    return HAF_OK;
}
extern "C" int haf_scale_apply(int device, const long long* row_ptr, const int* index, const double* value, int n_rows, int max_index,
                               const double* fmin, const double* fmax, double lower, double upper, double* dense_out) {
    if (!fmin || !fmax || !dense_out) return create_fail(HAF_ERR_ARG, "haf_scale_apply: null argument");
    if (n_rows == 0) return HAF_OK;
    ScaleBufs b;
    { int rc = scale_upload(device, row_ptr, index, value, n_rows, max_index, b); if (rc) return rc; }
    double* dmm = nullptr;
    struct Free { double*& a; ~Free() { cudaFree(a); } } fr{dmm};
    SC_TRY(cudaMalloc(&dmm, 2 * (size_t)max_index * 8));
    SC_TRY(cudaMemcpy(dmm, fmin + 1, (size_t)max_index * 8, cudaMemcpyHostToDevice));
    SC_TRY(cudaMemcpy(dmm + max_index, fmax + 1, (size_t)max_index * 8, cudaMemcpyHostToDevice));
    const size_t n = (size_t)n_rows * max_index;
    scale_apply_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 32), 256>>>(b.dense, n, max_index, dmm, dmm + max_index, lower, upper);
    SC_TRY(cudaGetLastError());
    SC_TRY(cudaMemcpy(dense_out, b.dense, n * sizeof(double), cudaMemcpyDeviceToHost));
    return HAF_OK;
#undef SC_TRY
}

extern "C" void haf_destroy(haf_ctx* ctx) {
    if (!ctx) return;
    for (size_t k = 1; k < ctx->group.size(); k++) haf_destroy(ctx->group[k]);   // member contexts of a multi-GPU group
    ctx->group.clear();
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    ctx->d_feats.release(); ctx->d_dims.release(); ctx->d_svT.release(); ctx->d_svn.release(); ctx->d_coef.release();
    ctx->d_sv64T.release(); ctx->d_coef64.release(); ctx->d_xyz.release(); ctx->d_ptoff.release(); ctx->d_cloud_ubegin.release();
    ctx->d_units.release(); ctx->d_jobs.release(); ctx->d_results.release(); ctx->d_per_roll_top.release(); ctx->d_keys.release();
    ctx->d_integral.release(); ctx->d_rowscan.release(); ctx->d_mask.release(); ctx->d_labelgrid.release(); ctx->d_evals.release();
    ctx->d_unit_block.release(); ctx->d_win.release(); ctx->d_X.release();
    ctx->d_xn.release(); ctx->d_dec.release(); ctx->d_guardflag.release(); ctx->d_guardlist.release(); ctx->d_kscratch.release();
    ctx->d_xdense.release(); ctx->d_labels.release(); ctx->d_probs.release(); ctx->d_probgrid.release(); ctx->d_pcd_raw.release(); ctx->d_pcd_blob.release(); ctx->d_pcd_xyz.release(); ctx->d_pcd_tiles.release(); ctx->d_pcd_status.release(); ctx->d_pcd_params.release(); ctx->h_pcd_params.release(); ctx->h_pcd_status.release(); ctx->d_csr_ptr.release(); ctx->d_csr_idx.release(); ctx->d_csr_val.release();
    ctx->d_svn64.release(); ctx->d_Xg.release(); ctx->d_xn64.release(); ctx->d_g2accum.release(); ctx->d_g2tickets.release(); ctx->d_guardlist2.release();
    ctx->d_SVh.release(); ctx->d_SVl.release(); ctx->d_Xh.release(); ctx->d_Xl.release(); ctx->d_svcoef.release(); ctx->d_dec_tc.release(); ctx->d_asum.release(); ctx->d_dimfeat.release(); ctx->d_round4.release();
    ctx->d_params.release(); ctx->d_counters.release(); ctx->h_stage.release(); ctx->h_results.release(); ctx->h_per_roll_top.release(); ctx->h_counters.release(); ctx->h_unit_windows.release();
    ctx->d_rank_tiles.release();
    for (int k = 0; k < 3; k++) {
    swap_chunk_ws(ctx, k);   // the further sets of per-chunk buffers (host-staged batches, one per extra stream)
    ctx->d_keys.release(); ctx->d_integral.release(); ctx->d_rowscan.release(); ctx->d_mask.release(); ctx->d_labelgrid.release(); ctx->d_evals.release();
    ctx->d_win.release(); ctx->d_X.release(); ctx->d_xn.release(); ctx->d_dec.release(); ctx->d_guardflag.release(); ctx->d_guardlist.release(); ctx->d_kscratch.release();
    ctx->d_probgrid.release(); ctx->d_Xg.release(); ctx->d_xn64.release(); ctx->d_g2accum.release(); ctx->d_g2tickets.release(); ctx->d_guardlist2.release();
    ctx->d_Xh.release(); ctx->d_Xl.release(); ctx->d_dec_tc.release(); ctx->d_asum.release(); ctx->d_rank_tiles.release();
    if (ctx->chunk_stream2[k]) cudaStreamDestroy(ctx->chunk_stream2[k]);
    }
    if (ctx->ev_dual_ok) for (int k = 0; k < 4; k++) cudaEventDestroy(ctx->ev_dual[k]);
    for (size_t i = 0; i < ctx->graphs.size(); i++) cudaGraphExecDestroy(ctx->graphs[i].exec);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    ctx->h_out_evals.release(); ctx->h_out_heights.release(); ctx->h_out_mask.release(); ctx->h_ring.release();
    ctx->d_unit_grasp.release(); ctx->h_unit_grasp.release(); ctx->h_job_grasp.release();
    ctx->d_rank_entries.release(); ctx->d_rank_compact.release(); ctx->d_rank_top_score.release(); ctx->h_cand.release(); ctx->h_ncand.release();
    if (ctx->ev_ok) for (int i = 0; i < 10; i++) cudaEventDestroy(ctx->ev[i]);
    for (size_t i = 0; i < ctx->ev_pool.size(); i++) cudaEventDestroy(ctx->ev_pool[i]);
    for (size_t i = 0; i < ctx->copy_ev.size(); i++) cudaEventDestroy(ctx->copy_ev[i]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->pcd_params_ev) cudaEventDestroy(ctx->pcd_params_ev);
    cudaGetLastError();
    delete ctx;
}

extern "C" int haf_get_info(const haf_ctx* ctx, haf_info* info) {
    if (!ctx || !info) return HAF_ERR_ARG;
    memset(info, 0, sizeof *info);
    info->n_features = ctx->F; info->n_dims = ctx->D; info->n_sv = ctx->S; info->n_rolls = ctx->R; info->grid = ctx->G;
    info->label0 = ctx->label[0]; info->label1 = ctx->label[1]; info->sm_count = ctx->sm_count;
    info->gamma = ctx->gamma; info->rho = ctx->rho;
    info->reserved[0] = ctx->cfg.svm_mode == HAF_SVM_TENSOR_GUARD ? ctx->tc_passes : 0;   // tensor-core products per k-slice
    info->reserved[1] = (int)lrint(ctx->guard_rel * 1e9);                                  // guard_rel in units of 1e-9
    info->reserved[2] = ctx->last_svm_kernel;                                              // what the last stage-5 launch ran
    info->reserved[3] = ctx->last_nsplit2;
    return HAF_OK;
}
extern "C" int haf_set_stream(haf_ctx* ctx, void* s) { if (!ctx) return HAF_ERR_ARG; ctx->stream = (cudaStream_t)s; return HAF_OK; }
extern "C" int haf_set_debug(haf_ctx* ctx, int keep_batch_state) { if (!ctx) return HAF_ERR_ARG; ctx->debug_keep_batch = keep_batch_state != 0; return HAF_OK; }
extern "C" int haf_set_profiling(haf_ctx* ctx, int on) {
    if (!ctx) return HAF_ERR_ARG;
    ctx->profiling = on != 0;
    for (size_t k = 1; k < ctx->group.size(); k++) ctx->group[k]->profiling = on != 0;
    return HAF_OK;
}
extern "C" int haf_get_timing(const haf_ctx* ctx, haf_timing* t) { if (!ctx || !t) return HAF_ERR_ARG; *t = ctx->timing; return HAF_OK; }
extern "C" long long haf_launch_count(const haf_ctx* ctx) {
    if (!ctx) return 0;
    long long n = ctx->launches;
    for (size_t k = 1; k < ctx->group.size(); k++) n += ctx->group[k]->launches;
    return n;
}

extern "C" int haf_build_transform(const haf_request* req, int roll, int roll_step_deg, float M[16]) {
    if (!req || !M) return HAF_ERR_ARG;
    hafhost::build_transform(*req, roll, roll_step_deg > 0 ? roll_step_deg : 15, M);
    return HAF_OK;
}
extern "C" int haf_build_transform_wcs(const haf_request* req, int roll, int roll_step_deg, float M[16]) {
    if (!req || !M) return HAF_ERR_ARG;
    hafhost::build_transform_wcs(*req, roll, roll_step_deg > 0 ? roll_step_deg : 15, M);
    return HAF_OK;
}
// the 32-byte record of the cross-GPU best-grasp exchange (SURVEY 8e), straight from the haf_best structs of a batch
extern "C" int haf_pack_best_records(const haf_best* best, int n, int32_t* records) {
    if (!best || !records || n < 0) return HAF_ERR_ARG;
    for (int i = 0; i < n; i++) {
        int32_t* r = records + (size_t)i * 8;
        r[0] = best[i].topval; r[1] = best[i].row; r[2] = best[i].col; r[3] = best[i].roll; r[4] = best[i].tilt;
        r[5] = best[i].approach_idx; r[6] = best[i].n_windows_scored; r[7] = best[i].rolls_done;
    }
    return HAF_OK;
}
extern "C" uint64_t haf_best_key(int topval, uint32_t unit_order) {
    return ((uint64_t)(uint32_t)(topval + (1 << 30)) << 32) | (uint64_t)(0xFFFFFFFFu - unit_order);
}

// ------------------------------------------------------------------------------------------------------------
// the launch sequence
// ------------------------------------------------------------------------------------------------------------
namespace {

struct CloudSet {
    const unsigned char* d_xyz;  // device base
    size_t stride;
    std::vector<long long> off;  // [n_clouds+1] point offsets
};

long long window_bound(int G, const haf_request& rq) {
    const long long full = (long long)(G - 14) * (G - 14);
    const int ax = (int)rq.area_len_x, ay = (int)rq.area_len_y;
    const long long hr = std::llabs((long long)(ax / 2) - 7), wr = std::llabs((long long)(ay / 2) - 7);
    const long long geo = (2 * hr + 3) * (2 * wr + 3);
    return std::min(full, geo);
}

// host memory the copy engine can read directly (cudaMallocHost / cudaHostRegister)
bool is_pinned_host_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

}  // namespace

static size_t ft_smem_bytes(const haf_ctx* ctx) { return ft_smem_layout(ctx->G, ctx->tc_passes >= 3 ? 2 : 1); }
// launches the two phases of the FP64 exact-order path on stream st
static int launch_exact(haf_ctx* ctx, ExactArgs a, cudaStream_t st, size_t max_windows) {
    const int slices = (ctx->S + HAF_EXACT_SLICE - 1) / HAF_EXACT_SLICE;
    // inputs of HAF_EXACT_WB windows in shared memory where they fit (create_impl raised the kernel's limit), else from global memory
    const size_t smem = (size_t)HAF_EXACT_WB * ctx->Dsv * sizeof(double);
    a.x_global = smem > (size_t)ctx->smem_optin ? 1 : 0;
    // all-windows mode (list == NULL) walks the windows in passes of max_entries; guard mode is a single pass
    const size_t passes = a.list ? 1 : (max_windows + a.max_entries - 1) / (size_t)a.max_entries;
    for (size_t p = 0; p < passes; p++) {
        a.entry_begin = (int)(p * (size_t)a.max_entries);
        const dim3 grid((unsigned)(ctx->sm_count * 2), (unsigned)slices);
        if (a.x_global) svm_exact_terms_xglobal_kernel<<<grid, 256, 0, st>>>(a);
        else svm_exact_terms_kernel<<<grid, 256, smem, st>>>(a);
        LAUNCHED(ctx);
        svm_exact_sum_kernel<<<ctx->sm_count * 4, 128, 0, st>>>(a);
        LAUNCHED(ctx);
    }
    return HAF_OK;
}
// Guard band after the FP32 / tensor contraction: tier 2 (FP64 FMA contraction on the bit-exact inputs) settles every
// window whose sign it can guarantee; the rest (list 2, counter cnt[6]) and -- with tier 2 switched off -- the whole
// guard list go through the exact-order kernels.
static ExactArgs make_exact_args(haf_ctx* ctx, const int* list, const unsigned* list_count, unsigned* cnt, int G, int ubase);
static int launch_guard(haf_ctx* ctx, unsigned* cnt, int G, int ubase, cudaStream_t st, size_t Wcap, size_t ldx) {
    if (ctx->tier2_mode == 1) return launch_exact(ctx, make_exact_args(ctx, ctx->d_guardlist.p, cnt + 1, cnt, G, ubase), st, Wcap);
    const size_t cap = std::min<size_t>(ldx, 32768);
    const size_t acc_cap0 = ctx->d_g2accum.cap, tk_cap0 = ctx->d_g2tickets.cap;
    const int ldxg = (int)round_up((size_t)ctx->Dsv, 16);
    ENSURE(ctx, ctx->d_Xg, cap * ldxg); ENSURE(ctx, ctx->d_g2accum, cap * 2); ENSURE(ctx, ctx->d_g2tickets, cap / HAF_G2_WB + 1); ENSURE(ctx, ctx->d_xn64, cap);
    ENSURE(ctx, ctx->d_guardlist2, ldx);
    if (ctx->d_g2accum.cap != acc_cap0) CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_g2accum.p, 0, ctx->d_g2accum.cap * sizeof(double), st));
    if (ctx->d_g2tickets.cap != tk_cap0) CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_g2tickets.p, 0, ctx->d_g2tickets.cap * sizeof(unsigned), st));
    ExactArgs a = make_exact_args(ctx, ctx->d_guardlist.p, cnt + 1, cnt, G, ubase);
    Guard2Args q;
    q.list = ctx->d_guardlist.p; q.list_count = cnt + 1; q.cap = (int)cap; q.Xg = ctx->d_Xg.p; q.svn64 = ctx->d_svn64.p;
    q.ldx = ldxg; q.xn64 = ctx->d_xn64.p;
    q.accum = ctx->d_g2accum.p; q.tickets = ctx->d_g2tickets.p; q.tol2 = ctx->tier2_mode == 2 ? 1e30 : 1e-10;
    q.list2 = ctx->d_guardlist2.p; q.list2_count = cnt + 6;
    const bool audit = ctx->cfg.svm_mode == HAF_SVM_TENSOR_GUARD && ctx->d_dec_tc.p;
    q.dec_tc = audit ? ctx->d_dec_tc.p : nullptr; q.audit_max = cnt + 12; q.guard_flag = audit ? ctx->d_guardflag.p : nullptr;
    const size_t smem = ((size_t)ctx->Dsv * HAF_G2_WB + HAF_G2_WB + 8 * HAF_G2_WB * 2) * sizeof(double);
    const bool few = Wcap < 65536;   // a single goal: a handful of guard windows -> spread the support vectors over more CTAs
    // FP64 tensor cores (DMMA) unless the DFMA register-tile kernel is asked for (tests; it cannot hold models wider than ~780
    // dimensions).  Measured: 2x on the bench batch; also ahead on the 13 guard windows of a single table1 goal (64 vs 71 us),
    // although three quarters of its 64-window tile are padding there.
    const bool dmma = ctx->tier2_kernel != 2 || smem > 100 * 1024;
    if (few) {
        guard_inputs_flat_kernel<<<32, 256, 0, st>>>(a, q);
        LAUNCHED(ctx);
        if (dmma) { guard_norms_kernel<<<8, 256, 0, st>>>(q); LAUNCHED(ctx); }
    } else {
        guard_inputs_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(a, q);
        LAUNCHED(ctx);
    }
    if (dmma) {
        guard_dmma_kernel<<<(unsigned)ctx->sm_count * 2, 256, HAF_GD_SMEM_BYTES, st>>>(a, q, ctx->Spad / HAF_GD_SB);
    }
    // one CTA per SM walks (window group, SV slice) items; a single goal's handful of windows: slices of 256 SVs over more CTAs
    else if (few) guard_fma_kernel<1><<<(unsigned)ctx->sm_count, 256, smem, st>>>(a, q, (ctx->Spad + 255) / 256);
    else guard_fma_kernel<2><<<(unsigned)ctx->sm_count, 256, smem, st>>>(a, q, (ctx->Spad + 511) / 512);
    LAUNCHED(ctx);
    return launch_exact(ctx, make_exact_args(ctx, ctx->d_guardlist2.p, cnt + 6, cnt, G, ubase), st, Wcap);
}
static ExactArgs make_exact_args(haf_ctx* ctx, const int* list, const unsigned* list_count, unsigned* cnt, int G, int ubase) {
    ExactArgs a;
    a.list = list; a.list_count = list_count; a.win_count = cnt + 0; a.integral = ctx->d_integral.p; a.win = ctx->d_win.p;
    a.G = G; a.unit_base = ubase; a.feats = ctx->d_feats.p; a.dims = ctx->d_dims.p; a.D = ctx->D; a.lower = ctx->lower; a.upper = ctx->upper;
    a.emulate_text = ctx->cfg.emulate_text_roundtrip; a.sv64T = ctx->d_sv64T.p; a.Spad = ctx->Spad; a.S = ctx->S; a.Dsv = ctx->Dsv;
    a.coef64 = ctx->d_coef64.p; a.gamma = ctx->gamma; a.rho = ctx->rho; a.terms = ctx->d_kscratch.p; a.dec = ctx->d_dec.p;
    a.unsupported_flag = (int*)(cnt + 3);
    a.max_entries = (int)std::min<size_t>(ctx->d_kscratch.cap / (size_t)ctx->Spad, 0x7fffffff);
    a.entry_begin = 0;
    a.overflow_flag = list ? (int*)(cnt + 10) : nullptr;   // guard mode: one launch must cover the whole list
    a.xdense = ctx->cur_xdense;
    a.x_global = 0;   // launch_exact decides
    return a;
}

// timing experiments on the tensor kernel's pipeline (tools/tc_pipeline_probe.py); results are garbage when set
static int tc_debug_flags() {
    const char* e = getenv("HAF_TC_DEBUG");
    return e ? atoi(e) : 0;
}
// Stage 5 of the path, also the whole of haf_svm_predict: decision values of the windows [0, *cnt[0]) whose SVM inputs
// are in ctx->d_Xh/d_Xl (tensor mode), ctx->d_X (SIMT mode) or re-derivable by exact_scaled_input (FP64 mode / guard
// band), then the guard band.  ev_guard (optional) is recorded between the contraction and the guard-band kernels.
static int svm_stage(haf_ctx* ctx, unsigned* cnt, size_t Wcap, size_t ldx, int G, int ubase, cudaStream_t st, cudaEvent_t ev_guard) {
    const bool tc = ctx->cfg.svm_mode == HAF_SVM_TENSOR_GUARD && !ctx->force_exact;
    const float neg_gamma_log2e = (float)(-ctx->gamma * 1.4426950408889634);
    ctx->last_svm_kernel = 0;
    ctx->last_nsplit2 = 0;
    if (ctx->cfg.svm_mode == HAF_SVM_FP64_EXACT || ctx->force_exact) {
        CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_guardflag.p, 0, ldx, st));
        { int rce = launch_exact(ctx, make_exact_args(ctx, nullptr, nullptr, cnt, G, ubase), st, Wcap); if (rce) return rce; }
        if (ev_guard) CUDA_TRY(ctx, cudaEventRecord(ev_guard, st));
    } else if (tc) {
        CUtensorMap tmXh, tmXl;
        const bool need_lo = ctx->tc_passes >= 3;   // X_lo takes part in the third product only
        if (!make_tensor_map(&tmXh, ctx->d_Xh.p, ctx->KB, ldx) || !make_tensor_map(&tmXl, need_lo ? ctx->d_Xl.p : ctx->d_Xh.p, ctx->KB, ldx))
            return ctx->fail(HAF_ERR_CUDA, "cuTensorMapEncodeTiled failed for the window operands");
        // (the accumulators d_dec / d_asum were zeroed by the kernel that wrote the operand rows: features_tc_kernel / pack_svm_inputs_kernel)
        const int n_ntiles = ctx->SpadT / haftc::BN;
        const int mt_cap = (int)(ldx / haftc::BM);
        int nsplit = 1;
        if (mt_cap < ctx->sm_count) nsplit = std::min(n_ntiles, (2 * ctx->sm_count + mt_cap - 1) / mt_cap);
        const int kblocks = ctx->KB;
        const int last_slices = (ctx->Krow - haftc::BK * (kblocks - 1)) / 16;
        const int tab_smem = (ctx->SpadT <= haftc::TAB_SMEM_MAX && !ctx->cfg.reserved[3]) ? 1 : 0;   // coef table staged in shared memory
        const size_t tab_bytes = tab_smem ? (size_t)ctx->SpadT * 4 : 0;
        (void)nsplit;
        {
            const int pairs_cap = (mt_cap + 1) / 2;
            int nsplit2 = 1;
            if (pairs_cap < ctx->sm_count / 2) nsplit2 = std::min(n_ntiles, (ctx->sm_count + pairs_cap - 1) / pairs_cap);
            else {   // mid-sized launches (the chunks of a host-staged batch): split the SV tiles of an item when that fills the last round better
                const double clusters = ctx->sm_count / 2;
                double best_eff = 0.0;
                for (int ns = 1; ns <= n_ntiles && ns <= 8; ns *= 2) {
                    if (n_ntiles % ns) continue;
                    const double rounds = (double)pairs_cap * ns / clusters;
                    const double eff = rounds / std::ceil(rounds);
                    if (eff > best_eff + 0.02) { best_eff = eff; nsplit2 = ns; }
                }
            }
            int grid2 = (int)std::min<long long>((long long)pairs_cap * nsplit2 * 2, ctx->sm_count);
            grid2 &= ~1;  // whole clusters
            // X-resident kernel: one product, the X tile (kblocks x 16 KB) + at least 3 ring stages + the table must fit
            int stages3 = 0;
            if (ctx->tc_variant == 0 && ctx->tc_passes == 1 && kblocks <= haftc::XK_MAX)
                stages3 = std::min(8, (haftc::TC3_SMEM_LIMIT - haftc::tc3_smem_bytes(kblocks, 0, (int)(tab_bytes / 4))) / (haftc::KBS * haftc::B2_TILE_BYTES));
            ctx->last_svm_kernel = stages3 >= 2 ? 1 : 2;
            ctx->last_nsplit2 = nsplit2;
            if (stages3 >= 2 && (tc_debug_flags() & 64))   // experiment: four epilogue warps per TMEM lane quarter
                haftc::svm_rbf_tc3_kernel<4><<<grid2, 64 + 128 * 4, haftc::tc3_smem_bytes(kblocks, stages3, (int)(tab_bytes / 4)), st>>>(
                    tmXh, ctx->tmSh2, ctx->d_xn.p, ctx->d_svcoef.p, ctx->c_log2, cnt + 0, n_ntiles, nsplit2, kblocks, last_slices, stages3, ctx->d_dec.p,
                    ctx->d_asum.p, tab_smem, ctx->csvn_max, tc_debug_flags() & ~64);
            else if (stages3 >= 2)
                haftc::svm_rbf_tc3_kernel<2><<<grid2, haftc::THREADS3, haftc::tc3_smem_bytes(kblocks, stages3, (int)(tab_bytes / 4)), st>>>(
                    tmXh, ctx->tmSh2, ctx->d_xn.p, ctx->d_svcoef.p, ctx->c_log2, cnt + 0, n_ntiles, nsplit2, kblocks, last_slices, stages3, ctx->d_dec.p,
                    ctx->d_asum.p, tab_smem, ctx->csvn_max, tc_debug_flags());
            else
                haftc::svm_rbf_tc2_kernel<<<grid2, haftc::THREADS, haftc::SMEM2_BYTES + tab_bytes, st>>>(tmXh, tmXl, ctx->tmSh2, ctx->tmSl2, ctx->d_xn.p, ctx->d_svcoef.p,
                                                                                                 ctx->c_log2, cnt + 0, n_ntiles, nsplit2, kblocks, last_slices,
                                                                                                 ctx->d_dec.p, ctx->d_asum.p, tab_smem, ctx->csvn_max, ctx->tc_passes);
        }
        LAUNCHED(ctx);
        // audit (svm_tc.cuh): with the FP64 FMA tier on, every listed window's contraction value is kept and a sample of all windows joins the list
        const bool audit = ctx->tier2_mode != 1 && !tc_debug_flags();
        if (audit) ENSURE(ctx, ctx->d_dec_tc, ldx);
        haftc::svm_finalize_kernel<<<(unsigned)((Wcap + 255) / 256), 256, 0, st>>>(ctx->d_dec.p, ctx->d_asum.p, ctx->d_xn.p, cnt + 0, ctx->rho,
                                                                                   tc_debug_flags() ? -1.0f : ctx->guard_rel,   // timing experiments: empty guard band
                                                                                   ctx->d_guardflag.p, ctx->d_guardlist.p, cnt + 1, audit ? ctx->audit_every : 0,
                                                                                   audit ? ctx->d_dec_tc.p : nullptr, cnt + 13, ctx->e_floor);
        LAUNCHED(ctx);
        if (ev_guard) CUDA_TRY(ctx, cudaEventRecord(ev_guard, st));
        { int rce = launch_guard(ctx, cnt, G, ubase, st, Wcap, ldx); if (rce) return rce; }
    } else {
        ctx->last_svm_kernel = 3;
        svm_rbf_simt_kernel<<<(unsigned)(ldx / SVM_BM), 256, SVM_STAGES * SVM_BK * (SVM_BM + SVM_BN) * 4, st>>>(
            ctx->d_X.p, ldx, ctx->d_svT.p, ctx->Spad, ctx->Kpad, ctx->d_xn.p, ctx->d_svn.p, ctx->d_coef.p, neg_gamma_log2e, ctx->rho,
            ctx->guard_rel, ctx->e_floor, cnt + 0, ctx->d_dec.p, ctx->d_guardflag.p, ctx->d_guardlist.p, cnt + 1);
        LAUNCHED(ctx);
        if (ev_guard) CUDA_TRY(ctx, cudaEventRecord(ev_guard, st));
        { int rce = launch_guard(ctx, cnt, G, ubase, st, Wcap, ldx); if (rce) return rce; }
    }
    return HAF_OK;
}

// Runs the whole path for `jobs` (sorted by cloud).  Outputs land in ctx->h_results / h_per_roll_top (pinned) and,
// when out_* are given (single-chunk calls only), in the caller's buffers.
static int run_jobs_once(haf_ctx* ctx, const CloudSet& cs, std::vector<Job>& jobs, float* out_evals, unsigned char* out_mask,
                         float* out_heights, bool keep_debug_state) {
    const int G = ctx->G, R = ctx->R, GG = G * G, ld = G + 1;
    const int n_jobs = (int)jobs.size();
    const int n_clouds = (int)cs.off.size() - 1;
    cudaStream_t st = ctx->stream;   // (replaced by a stream of our own when the call may be captured into a graph and this is the legacy stream)
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const long long launches0 = ctx->launches;

    // probability mode (server.cpp:383-385 with svm_with_probability = true): all requests of a call agree
    bool prob = false;
    for (int j = 0; j < n_jobs; j++) {
        const bool pj = jobs[j].rq.svm_with_probability != 0;
        if (j == 0) prob = pj;
        else if (pj != prob) return ctx->fail(HAF_ERR_ARG, "svm_with_probability must be the same for every request of a call");
    }
    if (prob && !ctx->has_prob) return ctx->fail(HAF_ERR_UNSUPPORTED, "Model does not support probabiliy estimates");   // svm-predict.c:213 (sic)
    struct ForceExact { haf_ctx* c; bool on; ~ForceExact() { if (on) c->force_exact = false; } } force_exact_scope{ctx, prob};
    if (prob) ctx->force_exact = true;

    // ---- host: unit parameters (transforms and mask constants use the HOST libm, see haf_host.hpp).  With device_units the
    // host writes one JobSpec per job and the libm tables instead, and expand_units_kernel builds the units, JobParams and poses.
    const bool dev_units = ctx->device_units;
    const int U = n_jobs * R;
    ctx->last_up_n = 0;
    ctx->last_chunk_waits.clear();
    const bool grasp = ctx->grasp_mode > 0;
    const bool rank = ctx->rank_k > 0;   // (RankScope: only with grasp poses)
    if (dev_units) {   // distinct approach vectors (bitwise), in order of first occurrence
        ctx->approach_trig.clear(); ctx->approach_index.clear(); ctx->job_approach.resize(n_jobs);
        for (int j = 0; j < n_jobs; j++) {
            haf_ctx::ApproachKey k;
            memcpy(k.b, jobs[j].rq.approach, sizeof k.b);
            if (j > 0 && memcmp(jobs[j - 1].rq.approach, k.b, sizeof k.b) == 0) { ctx->job_approach[j] = ctx->job_approach[j - 1]; continue; }
            const auto ins = ctx->approach_index.emplace(k, (int)ctx->approach_trig.size());
            if (ins.second) {
                hafhost::ApproachTrig t;
                hafhost::approach_trig(jobs[j].rq.approach, false, t.grid);
                if (grasp) hafhost::approach_trig(jobs[j].rq.approach, true, t.wcs);
                else memset(t.wcs, 0, sizeof t.wcs);
                ctx->approach_trig.push_back(t);
            }
            ctx->job_approach[j] = ins.first->second;
        }
    }
    const int n_approach = dev_units ? (int)ctx->approach_trig.size() : 0;
    const size_t bytes_units = dev_units ? 0 : (size_t)U * sizeof(UnitParams), bytes_jobs = (size_t)n_jobs * sizeof(JobParams);
    const size_t bytes_off = (size_t)(n_clouds + 1) * sizeof(long long), bytes_ub = (size_t)(n_clouds + 1) * sizeof(int);
    const size_t o_units = 0, o_jobs = round_up(o_units + bytes_units, 256), o_off = round_up(o_jobs + bytes_jobs, 256), o_ub = round_up(o_off + bytes_off, 256);
    // grasp poses: the inverse WCS matrices per (distinct request, roll) and each job's request index, after the block above
    // (device_units: one pose per unit outside the block, each job its own set)
    int n_pose_sets = 0;
    if (grasp && !dev_units)
        for (int j = 0; j < n_jobs; j++)
            if (j == 0 || memcmp(&jobs[j - 1].rq, &jobs[j].rq, sizeof(haf_request)) != 0) n_pose_sets++;
    const size_t o_jpose = round_up(o_ub + bytes_ub, 256), o_pose = round_up(o_jpose + (grasp ? (size_t)n_jobs * sizeof(int) : 0), 256);
    const size_t bytes_host_units = grasp ? o_pose + (size_t)n_pose_sets * R * sizeof(UnitPose) : o_ub + bytes_ub;
    // device_units: the job records and the libm tables
    const size_t o_spec = round_up(bytes_host_units, 256), o_rtrig = round_up(o_spec + (size_t)n_jobs * sizeof(JobSpec), 256),
                 o_atrig = round_up(o_rtrig + (size_t)R * sizeof(hafhost::RollTrig), 256);
    const size_t bytes_block = dev_units ? o_atrig + (size_t)n_approach * sizeof(hafhost::ApproachTrig) : bytes_host_units;
    ENSURE(ctx, ctx->h_stage, bytes_block + 16);
    UnitParams* hu = reinterpret_cast<UnitParams*>(ctx->h_stage.p + o_units);
    JobParams* hj = reinterpret_cast<JobParams*>(ctx->h_stage.p + o_jobs);
    long long* hoff = reinterpret_cast<long long*>(ctx->h_stage.p + o_off);
    int* hub = reinterpret_cast<int*>(ctx->h_stage.p + o_ub);
    int* hjpose = reinterpret_cast<int*>(ctx->h_stage.p + o_jpose);
    UnitPose* hpose = reinterpret_cast<UnitPose*>(ctx->h_stage.p + o_pose);
    JobSpec* hspec = reinterpret_cast<JobSpec*>(ctx->h_stage.p + o_spec);
    if (dev_units) {
        memcpy(ctx->h_stage.p + o_rtrig, ctx->roll_trig.data(), (size_t)R * sizeof(hafhost::RollTrig));
        memcpy(ctx->h_stage.p + o_atrig, ctx->approach_trig.data(), (size_t)n_approach * sizeof(hafhost::ApproachTrig));
    }
    long long max_points = 0;
    for (int c = 0; c <= n_clouds; c++) hoff[c] = cs.off[c];
    for (int c = 0; c < n_clouds; c++) max_points = std::max(max_points, cs.off[c + 1] - cs.off[c]);
    {
        int j = 0;
        for (int c = 0; c < n_clouds; c++) {
            hub[c] = j * R;
            while (j < n_jobs && jobs[j].cloud == c) j++;
        }
        hub[n_clouds] = n_jobs * R;
        if (j != n_jobs) return ctx->fail(HAF_ERR_ARG, "internal: jobs not sorted by cloud");
    }
    for (int j = 0; j < n_jobs; j++) {
        Job& jb = jobs[j];
        const int ax = (int)jb.rq.area_len_x, ay = (int)jb.rq.area_len_y;  // server.cpp:266-267
        jb.n_rolls_active = (jb.rq.roll_limit > 0) ? std::min(R, jb.rq.roll_limit) : R;
        jb.roll_begin = std::max(0, std::min(jb.rq.roll_begin, jb.n_rolls_active));
        jb.wbound = window_bound(G, jb.rq) * (jb.n_rolls_active - jb.roll_begin);
        if (dev_units) {
            JobSpec& sp = hspec[j];
            memcpy(sp.center, jb.rq.center, sizeof sp.center);
            sp.cloud = jb.cloud; sp.approach = ctx->job_approach[j];
            sp.gripper_opening_width = jb.rq.gripper_opening_width; sp.area_x = ax; sp.area_y = ay;
            sp.roll_begin = jb.roll_begin; sp.n_rolls_active = jb.n_rolls_active;
            sp.return_only_best = jb.rq.return_only_best; sp.graspval_top = jb.rq.graspval_top; sp.pad = 0;
            if (grasp) hjpose[j] = j;
            continue;
        }
        hj[j].return_only_best = jb.rq.return_only_best; hj[j].graspval_top = jb.rq.graspval_top;
        hj[j].n_rolls_active = jb.n_rolls_active; hj[j].roll_begin = jb.roll_begin;
        // a batch applies ONE request to every cloud: the transforms and mask constants (host libm, ~1 us per unit) are built
        // once and copied -- at 6144 units per bench step they were ~1 ms of GPU idle time at the head of every call
        const bool same_rq = j > 0 && memcmp(&jobs[j - 1].rq, &jb.rq, sizeof(haf_request)) == 0;
        if (grasp) {   // transform_gp_in_wcs_and_publish's matrix (:1276-1334), inverted -- once per distinct request as well
            const int p = same_rq ? hjpose[j - 1] : (j == 0 ? 0 : hjpose[j - 1] + 1);
            hjpose[j] = p;
            if (!same_rq)
                for (int roll = 0; roll < R; roll++) {
                    float Mw[16];
                    hafhost::build_transform_wcs(jb.rq, roll, ctx->cfg.roll_step_deg, Mw);
                    hafhost::invert4(Mw, hpose[(size_t)p * R + roll].Minv);
                }
        }
        for (int roll = 0; roll < R; roll++) {
            UnitParams& up = hu[j * R + roll];
            if (same_rq) {
                up = hu[(j - 1) * R + roll];
            } else {
                memset(&up, 0, sizeof up);
                float M[16];
                hafhost::build_transform(jb.rq, roll, ctx->cfg.roll_step_deg, M);
                memcpy(up.M, M, sizeof M);
                const hafhost::MaskConsts mc = hafhost::mask_consts(G, roll, ctx->cfg.roll_step_deg, ax, ay);
                up.sa = mc.sa; up.ca = mc.ca; up.cx1 = mc.cx1; up.cy1 = mc.cy1; up.cx2 = mc.cx2; up.cy2 = mc.cy2;
                up.cx3 = mc.cx3; up.cy3 = mc.cy3; up.cx4 = mc.cx4; up.cy4 = mc.cy4;
            }
            up.cloud = (roll >= jb.roll_begin && roll < jb.n_rolls_active) ? jb.cloud : -1;
            up.job = j; up.roll = roll;
        }
    }
    // ---- chunking: bound the feature matrix X (Kpad x windows) per pass
    size_t x_budget_floats = (size_t)8 << 28;  // 8 GiB of FP32 SVM inputs per chunk at most (fp16 operands: a quarter of that): the 512-cloud bench batch is ONE pass
    if (const char* e = getenv("HAF_X_BUDGET_GIB")) { const long g = atol(e); if (g >= 1 && g <= 64) x_budget_floats = (size_t)g << 28; }   // experiments
    std::vector<std::pair<int, int> > chunks;   // [job_begin, job_end)
    bool split_resident = false;
    {
        int jb0 = 0, stage_limit = 16;
        std::vector<int> sched;   // experiments: HAF_STAGE_SCHED="16,24,36,..." = clouds per chunk of a host-staged batch (last value repeats)
        if (const char* e = getenv("HAF_STAGE_SCHED")) {
            for (const char* q = e; *q;) { const int v = atoi(q); if (v > 0) sched.push_back(v); while (*q && *q != ',') q++; if (*q == ',') q++; }
            if (!sched.empty()) stage_limit = sched[0];
        }
        // device-resident batches: optionally split into equal chunks that alternate between the streams as well (experiments)
        int resident_split = 1;
        if (const char* e = getenv("HAF_RESIDENT_SPLIT")) resident_split = std::max(1, std::min(16, atoi(e)));
        if (ctx->copy_pieces > 0 || out_evals || out_mask || out_heights || keep_debug_state || n_jobs < 32 * resident_split) resident_split = 1;
        split_resident = resident_split > 1;
        const int split_jobs = (n_jobs + resident_split - 1) / resident_split;
        while (jb0 < n_jobs) {
            long long wsum = 0;
            int je = jb0;
            while (je < n_jobs) {
                const long long w = jobs[je].wbound;
                if (split_resident && (je - jb0) >= split_jobs) break;
                if (je > jb0 && (size_t)(wsum + w) * ctx->Kpad > x_budget_floats) break;
                if (je > jb0 && (je - jb0) * R >= 16384) break;
                // clouds being staged from host memory: the first chunk is small so that compute starts after ~0.35 ms of
                // copying; later chunks grow so that the bulk of the work runs in large launches
                if (je > jb0 && ctx->copy_pieces > 0 && (je - jb0) >= stage_limit) break;
                wsum += w;
                je++;
            }
            chunks.push_back(std::make_pair(jb0, je));
            jb0 = je;
            // ... up to 56 clouds: the host -> device copy (PCIe, ~22 us per 100 k-point cloud) is slower than the compute (~19 us),
            // so what follows the last copy -- the LAST chunk's chain of ~15 dependent kernels -- has to be short, while every chunk
            // pays ~0.2 ms of launch gaps and fixed kernel latencies.  Measured with the chunks alternating between three streams
            // (bench e2e, 512 clouds): 16, 24, 32, 48, 56, 56, ... 12.9 ms; 16, 24, 36, 54, 64, ... 13.2; at most 48: 13.0; at most
            // 32: 13.5.  (One stream, round 1: a cap of 256 left 180 clouds behind the copy, 15.1 ms; a cap of 64: 14.3 ms.)
            static const int kSched[5] = {16, 24, 32, 48, 56};
            stage_limit = kSched[std::min<size_t>(chunks.size(), 4)];
            if (!sched.empty()) stage_limit = sched[std::min(chunks.size(), sched.size() - 1)];
        }
    }
    if ((out_evals || out_mask || out_heights || keep_debug_state) && chunks.size() != 1)
        return ctx->fail(HAF_ERR_UNSUPPORTED, "per-roll outputs need the whole request in one chunk (windows x dims too large)");

    ENSURE(ctx, ctx->d_params, bytes_block + 16); ENSURE(ctx, ctx->d_results, n_jobs); ENSURE(ctx, ctx->d_per_roll_top, (size_t)U * 3);
    if (dev_units) {
        ENSURE(ctx, ctx->d_dev_units, U); ENSURE(ctx, ctx->h_best_M, (size_t)n_jobs * 16);
        if (grasp) ENSURE(ctx, ctx->d_dev_pose, U);
    }
    if (grasp) {
        ENSURE(ctx, ctx->d_unit_grasp, U); ENSURE(ctx, ctx->h_job_grasp, n_jobs);
        if (ctx->grasp_mode > 1) ENSURE(ctx, ctx->h_unit_grasp, U);
    }
    const int rank_P = ctx->rank_p;
    // one CTA per unit selects from the grid itself up to HAF_RANK_TILE cells, tiles of that many cells above
    const int rank_tiles = rank && G * G > HAF_RANK_TILE ? (G * G + HAF_RANK_TILE - 1) / HAF_RANK_TILE : 0;
    int rank_cap = 0;   // entries of the largest cloud's lists walked in shared memory (larger clouds: in place)
    if (rank) {
        ENSURE(ctx, ctx->d_rank_entries, (size_t)U * rank_P); ENSURE(ctx, ctx->d_rank_compact, (size_t)U * rank_P);
        ENSURE(ctx, ctx->d_rank_top_score, U); ENSURE(ctx, ctx->h_cand, (size_t)n_clouds * ctx->rank_k); ENSURE(ctx, ctx->h_ncand, n_clouds);
        for (int c = 0; c < n_clouds; c++) rank_cap = std::max(rank_cap, (hub[c + 1] - hub[c]) * rank_P);
        rank_cap = std::min(rank_cap, (int)((46 * 1024) / sizeof(RankCompact)));
    }
    ENSURE(ctx, ctx->d_unit_block, (size_t)2 * U + (U + 1) / 2);
    unsigned long long* const d_unit_top = ctx->d_unit_block.p;
    unsigned long long* const d_unit_run = d_unit_top + U;
    unsigned* const d_unit_windows = reinterpret_cast<unsigned*>(d_unit_run + U);
    ENSURE(ctx, ctx->h_results, n_jobs); ENSURE(ctx, ctx->h_per_roll_top, (size_t)U * 3);
    ENSURE(ctx, ctx->h_unit_windows, U);
    // per-roll outputs asked for in HOST memory: pinned staging (an async copy into pageable memory cannot be captured), copied on after the sync
    const bool host_evals = out_evals && !is_device_ptr(out_evals), host_mask = out_mask && !is_device_ptr(out_mask),
               host_heights = out_heights && !is_device_ptr(out_heights);
    float* dst_evals = out_evals; unsigned char* dst_mask = out_mask; float* dst_heights = out_heights;
    if (host_evals) { ENSURE(ctx, ctx->h_out_evals, (size_t)U * GG); dst_evals = ctx->h_out_evals.p; }
    if (host_mask) { ENSURE(ctx, ctx->h_out_mask, (size_t)U * GG); dst_mask = ctx->h_out_mask.p; }
    if (host_heights) { ENSURE(ctx, ctx->h_out_heights, (size_t)U * GG); dst_heights = ctx->h_out_heights.p; }
    const bool prof = ctx->profiling;
    if (prof) {
        while (ctx->ev_pool.size() < chunks.size() * 8) {
            cudaEvent_t e;
            CUDA_TRY(ctx, cudaEventCreate(&e));
            ctx->ev_pool.push_back(e);
        }
    }
    // ---- one CUDA graph per request shape (see haf_ctx::GraphKey): 0 = enqueue as usual, 1 = capture while enqueuing, 2 = replay
    int gmode = 0, graph_slot = -1, seen_slot = -1;
    haf_ctx::GraphKey gkey;
    memset(&gkey, 0, sizeof gkey);
    const long long pts_bucket = (long long)round_up((size_t)std::max<long long>(max_points, 1), 65536);
    const bool graph_ok = ctx->graph_mode != 1 && chunks.size() == 1 && !ctx->profiling && ctx->copy_pieces == 0 && !tc_debug_flags();
    if (graph_ok) {
        if (!ctx->stream) {   // the legacy default stream cannot be captured: a blocking stream of our own (it orders with legacy-stream work)
            if (!ctx->own_stream) CUDA_TRY(ctx, cudaStreamCreate(&ctx->own_stream));
            st = ctx->own_stream;
        }
        cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cst) == cudaSuccess && cst != cudaStreamCaptureStatusNone) {   // an earlier call failed mid-capture
            cudaGraph_t stale = nullptr;
            cudaStreamEndCapture(st, &stale);
            if (stale) cudaGraphDestroy(stale);
            cudaGetLastError();
        }
        unsigned long long hsh = 1469598103934665603ull;
        for (int j = 0; j < n_jobs; j++) {
            const unsigned long long v[3] = {(unsigned long long)jobs[j].roll_begin, (unsigned long long)jobs[j].n_rolls_active, (unsigned long long)jobs[j].wbound};
            for (int q = 0; q < 3; q++) { hsh ^= v[q]; hsh *= 1099511628211ull; }
        }
        const long long avg_points_all = (cs.off[n_clouds] - cs.off[0]) / std::max(1, n_clouds);
        gkey.epoch = g_alloc_epoch + ctx->alloc_epoch; gkey.xyz = cs.d_xyz; gkey.stride = cs.stride; gkey.wcap = (size_t)std::max<long long>(jobs.empty() ? 0 : 0, 0);
        long long wsum_all = 0;
        for (int j = 0; j < n_jobs; j++) wsum_all += jobs[j].wbound;
        gkey.wcap = (size_t)wsum_all; gkey.pts_bucket = pts_bucket; gkey.n_jobs = n_jobs; gkey.n_clouds = n_clouds;
        // (grasp poses: the two pose kernels, the record copies and the size of the parameter block belong to the graph too)
        gkey.flags = (prob ? 1 : 0) | (keep_debug_state ? 2 : 0) | (avg_points_all >= 8 * (long long)GG ? 4 : 0) | (ctx->cfg.emulate_text_roundtrip ? 8 : 0) |
                     (ctx->grasp_mode << 4) | (dev_units ? 64 : 0) | ((dev_units ? n_approach : n_pose_sets) << 8);
        if (rank) { gkey.rank_k = ctx->rank_k; gkey.rank_p = rank_P; gkey.rank_md2 = ctx->rank_md2; }
        gkey.tc_passes = ctx->tc_passes; gkey.o_evals = dst_evals; gkey.o_mask = dst_mask; gkey.o_heights = dst_heights; gkey.rolls_hash = hsh; gkey.st = st;
        for (size_t i = 0; i < ctx->graphs.size() && gmode == 0; i++)
            if (ctx->graphs[i].key == gkey) { gmode = 2; graph_slot = (int)i; }
        for (size_t i = 0; i < ctx->graph_seen.size() && gmode == 0; i++)
            if (ctx->graph_seen[i] == gkey) { gmode = 1; seen_slot = (int)i; }
        if (gmode == 0) {   // first call of this shape: remember it (its key is completed after the call's own allocations, below)
            if (ctx->graph_seen.size() < haf_ctx::kMaxGraphs) { ctx->graph_seen.push_back(gkey); seen_slot = (int)ctx->graph_seen.size() - 1; }
            else { seen_slot = (int)(ctx->graph_seen_next++ % haf_ctx::kMaxGraphs); ctx->graph_seen[seen_slot] = gkey; }
        }
    }
    UnitParams* const d_units = dev_units ? ctx->d_dev_units.p : reinterpret_cast<UnitParams*>(ctx->d_params.p + o_units);
    JobParams* const d_jobs = reinterpret_cast<JobParams*>(ctx->d_params.p + o_jobs);
    long long* const d_ptoff = reinterpret_cast<long long*>(ctx->d_params.p + o_off);
    int* const d_cloud_ubegin = reinterpret_cast<int*>(ctx->d_params.p + o_ub);
    const int* const d_jpose = reinterpret_cast<const int*>(ctx->d_params.p + o_jpose);
    const UnitPose* const d_pose = dev_units ? ctx->d_dev_pose.p : reinterpret_cast<const UnitPose*>(ctx->d_params.p + o_pose);
    float ms_stage[7] = {0, 0, 0, 0, 0, 0, 0};
    long long total_windows = 0, total_guard = 0;
    if (gmode == 2) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[8], st));
        ctx->graphs[graph_slot].last_use = ++ctx->graph_clock;
        CUDA_TRY(ctx, cudaGraphLaunch(ctx->graphs[graph_slot].exec, st));
        ctx->launches += ctx->graphs[graph_slot].nodes;
        ctx->graph_replays++;
        if (keep_debug_state) { ctx->last_units = U; ctx->last_unit_base = 0; ctx->last_ldx = round_up((size_t)std::max<long long>((long long)gkey.wcap, 1), 2 * haftc::BM); }
    } else {
    if (gmode == 1) CUDA_TRY(ctx, cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
    else CUDA_TRY(ctx, cudaEventRecord(ctx->ev[8], st));
    const long long launches_cap0 = ctx->launches;
    // The parameter block goes up with a tiny kernel that reads the pinned staging buffer directly (UVA), NOT with a
    // copy-engine memcpy: the H2D engine is a FIFO, and behind a large staging copy of clouds (this call's, or any other
    // stream's) a small memcpy would stall every kernel of the call until that copy has finished.
    {
        const size_t n16 = (bytes_block + 15) / 16;
        copy_params_kernel<<<(unsigned)std::min<size_t>((n16 + 255) / 256, 1024), 256, 0, st>>>(reinterpret_cast<const uint4*>(ctx->h_stage.p),
                                                                                              reinterpret_cast<uint4*>(ctx->d_params.p), n16);
        LAUNCHED(ctx);
    }
    if (dev_units) {
        expand_units_kernel<<<(U + 127) / 128, 128, 0, st>>>(reinterpret_cast<const JobSpec*>(ctx->d_params.p + o_spec),
                                                            reinterpret_cast<const hafhost::ApproachTrig*>(ctx->d_params.p + o_atrig),
                                                            reinterpret_cast<const hafhost::RollTrig*>(ctx->d_params.p + o_rtrig), n_jobs, R, G,
                                                            d_units, d_jobs, grasp ? ctx->d_dev_pose.p : nullptr);
        LAUNCHED(ctx);
    }
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_unit_block.p, 0, ((size_t)2 * U + (U + 1) / 2) * 8, st));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, 64 * 4, st));
    // host-staged batch in several chunks: chunks alternate between the call's stream and a second one (see haf_ctx::ChunkWs)
    int nsets = ((ctx->copy_pieces > 0 || split_resident) && chunks.size() >= 2 && !graph_ok) ? 3 : 1;
    if (const char* e = getenv("HAF_DUAL_STREAM")) { const int v = atoi(e); if (nsets > 1) nsets = v <= 0 ? 1 : std::min(4, std::max(2, v)); }   // 0 = one stream, 2..4 streams
    nsets = (int)std::min<size_t>((size_t)nsets, chunks.size());
    const bool dual = nsets > 1;
    if (dual) {
        if (!ctx->ev_dual_ok) {
            for (int k = 0; k < 4; k++) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_dual[k], cudaEventDisableTiming));
            ctx->ev_dual_ok = true;
        }
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_dual[0], st));
        for (int k = 0; k + 1 < nsets; k++) {
            if (!ctx->chunk_stream2[k]) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->chunk_stream2[k], cudaStreamNonBlocking));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->chunk_stream2[k], ctx->ev_dual[0], 0));
        }
    }
    cudaStream_t const st_main = st;
    struct WsSwapBack { haf_ctx* c; int set; ~WsSwapBack() { if (set > 0) swap_chunk_ws(c, set - 1); } } ws_scope{ctx, 0};   // (error returns inside a chunk)

    const float r = (float)((0.5 * (float)G) / 100.0);  // server.cpp:410-411
    const bool smallG = (size_t)G * ld * sizeof(double) <= 200 * 1024;
    const float neg_gamma_log2e = (float)(-ctx->gamma * 1.4426950408889634);

    int last_piece = 0;   // copy piece that holds the last cloud of the current chunk
    for (size_t ci = 0; ci < chunks.size(); ci++) {
        const int j0 = chunks[ci].first, j1 = chunks[ci].second;
        const int Uc = (j1 - j0) * R, ubase = j0 * R;
        const int set = dual ? (int)(ci % (size_t)nsets) : 0;   // 0: the call's stream and the context's own buffers
        if (set) { swap_chunk_ws(ctx, set - 1); ws_scope.set = set; }
        st = set ? ctx->chunk_stream2[set - 1] : st_main;
        long long wcap_ll = 0;
        for (int j = j0; j < j1; j++) wcap_ll += jobs[j].wbound;
        const size_t Wcap = (size_t)std::max<long long>(wcap_ll, 1);
        const size_t ldx = round_up(Wcap, 2 * haftc::BM);  // whole window-tile pairs (CTA-pair kernel); also a multiple of SVM_BM
        const int c0 = jobs[j0].cloud, c1 = jobs[j1 - 1].cloud + 1;  // clouds touched by this chunk
        ENSURE(ctx, ctx->d_keys, (size_t)Uc * GG); ENSURE(ctx, ctx->d_integral, (size_t)Uc * ld * ld);
        ENSURE(ctx, ctx->d_mask, (size_t)Uc * GG); ENSURE(ctx, ctx->d_labelgrid, (size_t)Uc * GG); ENSURE(ctx, ctx->d_evals, (size_t)Uc * GG);
        const bool tc = ctx->cfg.svm_mode == HAF_SVM_TENSOR_GUARD && !prob;
        if (prob) ENSURE(ctx, ctx->d_probgrid, (size_t)Uc * GG);
        ENSURE(ctx, ctx->d_win, ldx); ENSURE(ctx, ctx->d_xn, ldx);
        if (tc) { ENSURE(ctx, ctx->d_Xh, ldx * ctx->KB * haftc::BK); if (ctx->tc_passes >= 3) ENSURE(ctx, ctx->d_Xl, ldx * ctx->KB * haftc::BK); ENSURE(ctx, ctx->d_asum, ldx); }
        else if (ctx->cfg.svm_mode == HAF_SVM_FP32_GUARD && !prob) ENSURE(ctx, ctx->d_X, (size_t)ctx->Kpad * ldx);
        ENSURE(ctx, ctx->d_dec, ldx); ENSURE(ctx, ctx->d_guardflag, ldx); ENSURE(ctx, ctx->d_guardlist, ldx);
        if (!smallG) ENSURE(ctx, ctx->d_rowscan, (size_t)Uc * GG);
        // terms scratch of the exact path: one row of Spad doubles per entry; the guard list is bounded by what fits in 1 GiB
        // (a guard band wider than that means a mis-configured guard_rel: the call then fails loudly below)
        const size_t exact_cap = std::min<size_t>(ldx, std::max<size_t>(4096, ((size_t)1 << 30) / ((size_t)ctx->Spad * 8)));
        ENSURE(ctx, ctx->d_kscratch, exact_cap * ctx->Spad);
        unsigned* cnt = ctx->d_counters.p + 16 * set;
        if (ci >= (size_t)nsets) CUDA_TRY(ctx, cudaMemsetAsync(cnt, 0, 2 * 4, st));  // win_count, guard_count
        const UnitParams* units_c = d_units + ubase;

        // staged host clouds: this chunk's stream waits for the copy piece that holds the chunk's last cloud.  The pieces are
        // copied in order on one stream, so that event covers every earlier piece as well.  The wait is made on this chunk's own
        // stream even when a chunk on another stream has waited for the same piece: a wait orders only the stream it is made on
        // (chunks split on request boundaries, so several chunks of a call may end inside one piece).
        if (ctx->copy_pieces > 0) {
            while (ctx->copy_cloud_end[last_piece] < c1) last_piece++;   // c1 never decreases; the last piece ends at n_clouds
            if (ctx->stager.active) {   // pageable source: the helper thread records the event -- wait until it has (an unrecorded event does not block)
                std::unique_lock<std::mutex> lk(ctx->stager.mu);
                ctx->stager.cv.wait(lk, [&] { return ctx->stager.issued > last_piece; });
                if (ctx->stager.failed) return ctx->fail(HAF_ERR_CUDA, "staging a pageable host batch failed (pinned ring copy / cudaMemcpyAsync)");
            }
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->copy_ev[last_piece], 0));
        }
        // the chunk's record (haf_debug_chunk_copy_waits): its clouds and copy wait, then the binning and integral launches it made
        int rec[HAF_CHUNK_RECORD] = {c0, c1, set, ctx->copy_pieces > 0 ? last_piece : -1, ctx->copy_pieces > 0 ? ctx->copy_cloud_end[last_piece] : -1,
                                     0, 0, 0, 0, smallG ? 0 : 1};
        // 1. binning
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 0], st));
        {
            const size_t n = (size_t)Uc * GG;
            fill_u32_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 16), 256, 0, st>>>(ctx->d_keys.p, n, HAF_KEY_MINUS_ONE);
            LAUNCHED(ctx);
            // small grids with enough points per cloud: whole-cloud CTAs with shared-memory lower bounds (fewer REDs)
            const int upg = std::min(16, (int)((200 * 1024) / ((size_t)GG * 4)));
            const long long avg_points = (cs.off[c1] - cs.off[c0]) / std::max(1, c1 - c0);
            if (upg >= 1 && avg_points >= 8 * (long long)GG && (c1 - c0) * 8 >= ctx->sm_count && (ctx->cfg.reserved[1] & 15) != 1) {
                int max_units_per_cloud = 0;
                for (int c = c0; c < c1; c++) max_units_per_cloud = std::max(max_units_per_cloud, std::min(hub[c + 1], ubase + Uc) - std::max(hub[c], ubase));
                const int ug = std::min(upg, std::max(1, max_units_per_cloud));
                // The kernel is instruction-bound once the REDs are filtered, one 1024-thread CTA per SM.  A CTA costs a fixed part
                // (150 KB of shared-memory bounds initialised and flushed, launch) plus its slice of the cloud's points; the CTAs
                // (clouds x unit groups x slices) run in rounds of one per SM.  Slice count <= 12 that minimises
                //     rounds x (1 / slices + fixed / whole-cloud time),   fixed / whole-cloud time ~ 4.2 G^2 / points
                // fitted to the ncu launch list of a host-staged bench step (profiles/r2_final_launches_e2e.md: 144 CTAs of 1/6 cloud 86 us,
                // of 1/4 cloud 108 us).  512 clouds: 2 slices = 7 rounds (round 2 found that by wave efficiency alone); the
                // 64-cloud chunks of a staged batch: 2 slices = one round of 128 CTAs (167 us) where wave efficiency picked 9 (210 us).
                int slices = 1;
                {
                    const long long groups = (long long)(c1 - c0) * ((max_units_per_cloud + ug - 1) / ug);
                    const double fixed = std::min(1.0, 4.2 * (double)GG / (double)std::max<long long>(avg_points, 1));
                    double best_cost = 0.0;
                    for (int sl = 1; sl <= 12; sl++) {
                        const double cost = std::ceil((double)(groups * sl) / ctx->sm_count) * (1.0 / sl + fixed);
                        if (sl == 1 || cost < best_cost) { best_cost = cost; slices = sl; }
                    }
                }
                dim3 gridc((unsigned)(c1 - c0), (unsigned)((max_units_per_cloud + ug - 1) / ug), (unsigned)slices);
                const bool vec4 = cs.stride == 12 && (ctx->cfg.reserved[1] & 15) != 2;
                rec[5] = vec4 ? 1 : 2; rec[6] = (int)gridc.y; rec[7] = ug; rec[8] = slices;
                if (vec4)
                    bin_maxz_cloud_kernel<4><<<gridc, 1024, (size_t)ug * GG * 4, st>>>(cs.d_xyz, cs.stride, d_ptoff + c0, d_cloud_ubegin + c0, d_units,
                                                                                     ctx->d_keys.p - (size_t)ubase * GG, G, r, ug,
                                                                                     reinterpret_cast<unsigned long long*>(cnt + 4), ubase, ubase + Uc);
                else
                    bin_maxz_cloud_kernel<1><<<gridc, 1024, (size_t)ug * GG * 4, st>>>(cs.d_xyz, cs.stride, d_ptoff + c0, d_cloud_ubegin + c0, d_units,
                                                                                     ctx->d_keys.p - (size_t)ubase * GG, G, r, ug,
                                                                                     reinterpret_cast<unsigned long long*>(cnt + 4), ubase, ubase + Uc);
                LAUNCHED(ctx);
            } else {
                const int PPT = 4;
                // (a graph-eligible call sizes the grid for the 64 k-point bucket of the cloud: surplus CTAs return at once)
                const long long grid_points = graph_ok ? pts_bucket : max_points;
                dim3 grid((unsigned)((grid_points + 256 * PPT - 1) / (256 * PPT)), (unsigned)(c1 - c0));
                if (grid.x > 0) {
                    // cloud_unit_begin is relative to unit 0 of the call: shift the key base so unit u lands at keys[u - ubase]
                    bin_maxz_kernel<PPT><<<grid, 256, 0, st>>>(cs.d_xyz, cs.stride, d_ptoff + c0, d_cloud_ubegin + c0, d_units,
                                                               ctx->d_keys.p - (size_t)ubase * GG, G, r, nullptr,
                                                               reinterpret_cast<unsigned long long*>(cnt + 4), ubase, ubase + Uc);
                    LAUNCHED(ctx);
                }
            }
        }
        ctx->last_chunk_waits.insert(ctx->last_chunk_waits.end(), rec, rec + HAF_CHUNK_RECORD);
        // 2. integral image
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 1], st));
        if (smallG) {
            integral_small_kernel<<<Uc, 128, (size_t)G * ld * sizeof(double), st>>>(ctx->d_keys.p, ctx->d_integral.p, G, units_c);
            LAUNCHED(ctx);
        } else {
            integral_rows_kernel<<<dim3((G + 31) / 32, Uc), 32, 0, st>>>(ctx->d_keys.p, ctx->d_rowscan.p, G, units_c);
            LAUNCHED(ctx);
            integral_cols_kernel<<<dim3((G + 1 + 127) / 128, Uc), 128, 0, st>>>(ctx->d_rowscan.p, ctx->d_integral.p, G, units_c);
            LAUNCHED(ctx);
        }
        // 3. mask + window compaction
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 2], st));
        mask_windows_kernel<<<dim3((GG + 4095) / 4096, Uc), 256, 0, st>>>(ctx->d_integral.p, units_c, G, ctx->d_mask.p, ctx->d_labelgrid.p,
                                                                         ctx->d_win.p, cnt + 0, (unsigned)Wcap, (int*)(cnt + 2), ubase, d_unit_windows + ubase);
        LAUNCHED(ctx);
        // 4. features -> scaled SVM inputs
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 3], st));
        const unsigned wblocks32 = (unsigned)((Wcap + 31) / 32);
        if (tc) {
            const unsigned fblocks = (unsigned)((Wcap + 32 * HAF_FT_WT - 1) / (32 * HAF_FT_WT));
            (ctx->tc_passes >= 3 ? features_tc_kernel<true> : features_tc_kernel<false>)<<<fblocks, 256, ft_smem_bytes(ctx), st>>>(
                ctx->d_integral.p, ctx->d_win.p, cnt + 0, G, ubase, ctx->d_dimfeat.p, ctx->D, ctx->Krow, (float)ctx->lower,
                ctx->cfg.emulate_text_roundtrip, ctx->d_round4.p, ctx->d_Xh.p, ctx->tc_passes >= 3 ? ctx->d_Xl.p : nullptr, ctx->d_xn.p,
                ctx->Dsv, ctx->KB, ctx->d_dec.p, ctx->d_asum.p);
            LAUNCHED(ctx);
        } else if (ctx->cfg.svm_mode != HAF_SVM_FP64_EXACT && !prob) {
            features_kernel<false><<<wblocks32, 256, 0, st>>>(ctx->d_integral.p, ctx->d_win.p, cnt + 0, G, ubase, ctx->d_feats.p, ctx->d_dims.p,
                                                              ctx->D, ctx->Kpad, ctx->lower, ctx->upper, ctx->cfg.emulate_text_roundtrip,
                                                              ctx->d_X.p, ldx, ctx->F, nullptr, nullptr, (int*)(cnt + 3));
            LAUNCHED(ctx);
            xnorm_kernel<<<(unsigned)((Wcap + 255) / 256), 256, 0, st>>>(ctx->d_X.p, ldx, ctx->Kpad, cnt + 0, ctx->d_xn.p);
            LAUNCHED(ctx);
        }
        // 5. SVM decision values (+ guard band)
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 4], st));
        { int rcs = svm_stage(ctx, cnt, Wcap, ldx, G, ubase, st, prof ? ctx->ev_pool[ci * 8 + 5] : nullptr); if (rcs) return rcs; }
        // 6. labels -> grids, score stencil, argmax, tie rule
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 6], st));
        if (prob) {   // float grid res * prob with the reference's one-line shift, then the same stencil in float (kernels.cuh)
            prob_value_kernel<<<(unsigned)((Wcap + 127) / 128), 128, 0, st>>>(ctx->d_dec.p, ctx->d_win.p, cnt + 0, G, ubase, ctx->probA, ctx->probB,
                                                                             ctx->prob_res[0], ctx->prob_res[1], ctx->d_evals.p, (int*)(cnt + 3));
            LAUNCHED(ctx);
            prob_shift_grid_kernel<<<Uc, 1024, 0, st>>>(ctx->d_mask.p, ctx->d_evals.p, G, units_c, ctx->prob_header_val, ctx->d_probgrid.p);
            LAUNCHED(ctx);
            score_prob_kernel<<<dim3((GG + 255) / 256, Uc), 256, 0, st>>>(ctx->d_probgrid.p, G, units_c, ctx->d_evals.p, d_unit_top + ubase);
            LAUNCHED(ctx);
        } else {
            label_scatter_kernel<<<(unsigned)((Wcap + 255) / 256), 256, 0, st>>>(ctx->d_dec.p, ctx->d_win.p, cnt + 0, G, ubase, ctx->gv[0], ctx->gv[1],
                                                                                ctx->d_labelgrid.p);
            LAUNCHED(ctx);
            score_kernel<<<dim3((GG + 255) / 256, Uc), 256, 0, st>>>(ctx->d_labelgrid.p, G, units_c, ctx->d_evals.p, d_unit_top + ubase);
            LAUNCHED(ctx);
        }
        tie_rule_kernel<<<dim3((G + 7) / 8, Uc), 256, 0, st>>>(ctx->d_evals.p, G, units_c, d_unit_top + ubase, d_unit_run + ubase);
        LAUNCHED(ctx);
        if (grasp) {   // a16 per unit while this chunk's heights are still in d_keys (the next chunk of this set overwrites them)
            grasp_unit_kernel<<<(Uc + 127) / 128, 128, 0, st>>>(ctx->d_keys.p, G, units_c, Uc, d_unit_top + ubase, d_unit_run + ubase, d_pose, d_jpose,
                                                               R, ctx->cfg.roll_step_deg, ctx->d_unit_grasp.p + ubase);
            LAUNCHED(ctx);
        }
        if (rank) {   // each unit's candidate list, while evals / mask / heights of the chunk are resident
            if (rank_tiles) {
                ENSURE(ctx, ctx->d_rank_tiles, (size_t)Uc * rank_tiles * rank_P);
                rank_tile_kernel<<<dim3(rank_tiles, Uc), HAF_RANK_THREADS, 0, st>>>(ctx->d_evals.p, ctx->d_mask.p, G, units_c, d_jobs, d_unit_top, R,
                                                                                   rank_P, ctx->d_rank_tiles.p);
                LAUNCHED(ctx);
                rank_unit_kernel<true><<<Uc, HAF_RANK_THREADS, 0, st>>>(ctx->d_evals.p, ctx->d_mask.p, ctx->d_keys.p, G, units_c, d_jobs, d_unit_top, d_unit_run,
                                                                        ubase, R, d_pose, d_jpose, ctx->cfg.roll_step_deg, rank_P, ctx->d_rank_tiles.p,
                                                                        rank_tiles, ctx->d_rank_entries.p, ctx->d_rank_compact.p, ctx->d_rank_top_score.p);
            } else {
                rank_unit_kernel<false><<<Uc, HAF_RANK_THREADS, 0, st>>>(ctx->d_evals.p, ctx->d_mask.p, ctx->d_keys.p, G, units_c, d_jobs, d_unit_top, d_unit_run,
                                                                         ubase, R, d_pose, d_jpose, ctx->cfg.roll_step_deg, rank_P, nullptr, 0,
                                                                         ctx->d_rank_entries.p, ctx->d_rank_compact.p, ctx->d_rank_top_score.p);
            }
            LAUNCHED(ctx);
        }
        if (prof) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[ci * 8 + 7], st));

        // bookkeeping per chunk: window / guard counts accumulate on the device ([8] windows, [9] guard), no host sync
        accumulate_counts_kernel<<<1, 1, 0, st>>>(cnt);
        LAUNCHED(ctx);
        if (keep_debug_state) { ctx->last_units = Uc; ctx->last_unit_base = ubase; ctx->last_ldx = ldx; }

        // optional per-roll outputs (single chunk): active units only
        if (out_evals || out_mask || out_heights) {
            for (int j = j0; j < j1; j++) {
                const int na = jobs[j].n_rolls_active - jobs[j].roll_begin;
                if (na <= 0) continue;
                const size_t uo = (size_t)(j * R + jobs[j].roll_begin - ubase) * GG, go = ((size_t)j * R + jobs[j].roll_begin) * GG, nel = (size_t)na * GG;
                if (out_evals) CUDA_TRY(ctx, cudaMemcpyAsync(dst_evals + go, ctx->d_evals.p + uo, nel * 4, cudaMemcpyDefault, st));
                if (out_mask) CUDA_TRY(ctx, cudaMemcpyAsync(dst_mask + go, ctx->d_mask.p + uo, nel, cudaMemcpyDefault, st));
                if (out_heights) CUDA_TRY(ctx, cudaMemcpyAsync(dst_heights + go, ctx->d_keys.p + uo, nel * 4, cudaMemcpyDefault, st));
            }
        }
        if (set) { swap_chunk_ws(ctx, set - 1); ws_scope.set = 0; }
    }
    st = st_main;
    if (dual) {   // join: the other streams' chunks, then their counters into the first set's
        for (int k = 0; k + 1 < nsets; k++) {
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_dual[1 + k], ctx->chunk_stream2[k]));
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_dual[1 + k], 0));
        }
        merge_counts_kernel<<<1, 1, 0, st>>>(ctx->d_counters.p, nsets - 1);
        LAUNCHED(ctx);
    }
    // 7. cross-roll reduction per job, results to pinned host memory
    reduce_rolls_kernel<<<(n_jobs + 127) / 128, 128, 0, st>>>(d_unit_top, d_unit_run, d_unit_windows, d_jobs, n_jobs, R, G,
                                                             ctx->d_per_roll_top.p, ctx->d_results.p, d_units, dev_units ? ctx->h_best_M.p : nullptr);
    LAUNCHED(ctx);
    if (grasp) {   // a16 per job: the winning unit's record (or the roll -1 pose), written straight into pinned host memory (a
                   // copy node less on a single goal's critical path; the stream synchronise below makes it visible)
        grasp_gather_kernel<<<(n_jobs + 127) / 128, 128, 0, st>>>(ctx->d_results.p, n_jobs, d_units, d_pose, d_jpose, R, G, ctx->cfg.roll_step_deg,
                                                                 ctx->d_unit_grasp.p, ctx->h_job_grasp.p);
        LAUNCHED(ctx);
        if (rank) {   // the ranked candidates of every cloud, straight into pinned host memory as well
            rank_cloud_kernel<<<n_clouds, 256, (size_t)rank_cap * sizeof(RankCompact), st>>>(ctx->d_results.p, d_cloud_ubegin, R, G, ctx->d_unit_grasp.p,
                                                                                            ctx->d_rank_top_score.p, ctx->d_rank_entries.p,
                                                                                            ctx->d_rank_compact.p, rank_P, ctx->rank_k, ctx->rank_md2,
                                                                                            rank_cap, ctx->h_cand.p, ctx->h_ncand.p);
            LAUNCHED(ctx);
        }
        if (ctx->grasp_mode > 1)
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_unit_grasp.p, ctx->d_unit_grasp.p, (size_t)U * sizeof(GraspRec), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_results.p, ctx->d_results.p, (size_t)n_jobs * sizeof(JobResult), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_per_roll_top.p, ctx->d_per_roll_top.p, (size_t)U * 3 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_counters.p, ctx->d_counters.p, 16 * 4, cudaMemcpyDeviceToHost, st));
    if (keep_debug_state)   // single goals: windows per unit, for the multi-GPU merge
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_unit_windows.p, d_unit_windows, (size_t)U * 4, cudaMemcpyDeviceToHost, st));
    if (gmode == 1) {   // everything above was recorded, not run: instantiate, keep, run
        cudaGraph_t graph = nullptr;
        CUDA_TRY(ctx, cudaStreamEndCapture(st, &graph));
        cudaGraphExec_t gexec = nullptr;
        const cudaError_t ie = cudaGraphInstantiate(&gexec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) return ctx->fail(HAF_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
        if (ctx->graphs.size() >= haf_ctx::kMaxGraphs) {   // evict the least recently used one (stale keys -- an older allocation epoch -- age out this way)
            size_t lru = 0;
            for (size_t i = 1; i < ctx->graphs.size(); i++) if (ctx->graphs[i].last_use < ctx->graphs[lru].last_use) lru = i;
            cudaGraphExecDestroy(ctx->graphs[lru].exec);
            ctx->graphs.erase(ctx->graphs.begin() + lru);
        }
        gkey.epoch = g_alloc_epoch + ctx->alloc_epoch;   // (unchanged unless a buffer grew while capturing: then the next call re-captures)
        ctx->graphs.push_back(haf_ctx::GraphEntry{gkey, gexec, ctx->launches - launches_cap0, ++ctx->graph_clock});
        if (seen_slot >= 0) memset(&ctx->graph_seen[seen_slot], 0xff, sizeof(haf_ctx::GraphKey));   // (no longer "seen once")
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[8], st));
        CUDA_TRY(ctx, cudaGraphLaunch(gexec, st));
    } else if (graph_ok) {
        if (seen_slot >= 0) ctx->graph_seen[seen_slot].epoch = g_alloc_epoch + ctx->alloc_epoch;   // buffers this first call of the shape grew: the second call captures
    }
    }   // gmode != 2
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[9], st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    for (int j = 0; j < n_jobs && (host_evals || host_mask || host_heights); j++) {   // pinned staging -> the caller's host buffers
        const int na = jobs[j].n_rolls_active - jobs[j].roll_begin;
        if (na <= 0) continue;
        const size_t go = ((size_t)j * R + jobs[j].roll_begin) * GG, nel = (size_t)na * GG;
        if (host_evals) memcpy(out_evals + go, dst_evals + go, nel * 4);
        if (host_mask) memcpy(out_mask + go, dst_mask + go, nel);
        if (host_heights) memcpy(out_heights + go, dst_heights + go, nel * 4);
    }
    total_windows = ctx->h_counters.p[8];
    total_guard = ctx->h_counters.p[9];
    if (ctx->h_counters.p[2]) return ctx->fail(HAF_ERR_UNSUPPORTED, "window list overflow (internal bound too small)");
    if (ctx->h_counters.p[10]) return ctx->fail(HAF_ERR_UNSUPPORTED, "the guard band holds more windows than the exact path is provisioned for (guard_rel too wide for this model)");
    if (ctx->h_counters.p[3]) return ctx->fail(HAF_ERR_UNSUPPORTED, "a feature value fell outside the range the decimal text emulation reproduces exactly");
    float ms_total = 0;
    cudaEventElapsedTime(&ms_total, ctx->ev[8], ctx->ev[9]);
    if (prof)
        for (size_t ci = 0; ci < chunks.size(); ci++)
            for (int s = 0; s < 7; s++) { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev_pool[ci * 8 + s], ctx->ev_pool[ci * 8 + s + 1]); ms_stage[s] += ms; }
    haf_timing& t = ctx->timing;
    memset(&t, 0, sizeof t);
    t.ms_total = ms_total;
    t.ms_bin = ms_stage[0]; t.ms_integral = ms_stage[1]; t.ms_mask = ms_stage[2]; t.ms_features = ms_stage[3];
    t.ms_svm = ms_stage[4]; t.ms_guard = ms_stage[5]; t.ms_score = ms_stage[6];
    t.n_points = cs.off[n_clouds] - cs.off[0]; t.n_units = 0;
    for (int j = 0; j < n_jobs; j++) t.n_units += jobs[j].n_rolls_active - jobs[j].roll_begin;
    t.n_windows = total_windows; t.n_guard = total_guard; t.launches = ctx->launches - launches0;
    t.n_chunks = (long long)chunks.size();
    t.n_exact = (ctx->tier2_mode == 1 && ctx->cfg.svm_mode != HAF_SVM_FP64_EXACT) ? total_guard : ctx->h_counters.p[11];
    t.n_audit = ctx->h_counters.p[14];
    memcpy(&ctx->audit_max_rel, &ctx->h_counters.p[12], sizeof(float));
    t.audit_max_rel = ctx->audit_max_rel;
    t.tc_passes = ctx->cfg.svm_mode == HAF_SVM_TENSOR_GUARD ? ctx->tc_passes : 0;
    t.escalations = ctx->escalations;
    t.graph_replays = (int)std::min<long long>(ctx->graph_replays, 0x7fffffff);
    {   // d_counters[4..5]: points clamped into row / column G - 1 (both binning kernels; zeroed above, merged across streams)
        unsigned long long clamped;
        memcpy(&clamped, &ctx->h_counters.p[4], sizeof clamped);
        t.n_clamped = (long long)clamped;
    }
    if (keep_debug_state) { ctx->last_W = (unsigned)total_windows; ctx->last_valid = true; }
    ctx->last_up_units = d_units; ctx->last_up_pose = grasp ? d_pose : nullptr; ctx->last_up_jpose = d_jpose;
    ctx->last_up_n = U; ctx->last_up_jobs = n_jobs;
    return HAF_OK;
}

// AUDIT.  The number of tensor-core products per k-slice is calibrated at haf_create on stand-in windows; every call then
// MEASURES the contraction's error on its own windows: the guard band's windows and a 1-in-audit_every sample of all
// windows are re-evaluated in FP64 anyway / as well, and guard_fma_kernel records max |dec_tc - dec_fp64| / (E + |rho|).
// A window outside the band keeps the contraction's sign, which is the reference's as long as the error stays below
// guard_rel; if the measured maximum leaves less than a 4x margin, the call is repeated with one more product (and stays
// there for the life of the context); with all three products in use it fails loudly instead of returning labels it
// cannot vouch for.
static int run_jobs(haf_ctx* ctx, const CloudSet& cs, std::vector<Job>& jobs, float* out_evals, unsigned char* out_mask,
                    float* out_heights, bool keep_debug_state) {
    for (;;) {
        const int rc = run_jobs_once(ctx, cs, jobs, out_evals, out_mask, out_heights, keep_debug_state);
        if (rc != HAF_OK || ctx->cfg.svm_mode != HAF_SVM_TENSOR_GUARD || ctx->tier2_mode == 1 || tc_debug_flags()) return rc;
        if (!(ctx->audit_max_rel > 0.25f * ctx->guard_rel)) return rc;
        if (ctx->tc_passes >= 3)
            return ctx->fail(HAF_ERR_UNSUPPORTED, "audit: the tensor contraction is off by %.3g E on this call's windows, guard_rel = %.3g leaves less than a 4x margin "
                             "(widen guard_rel, or use svm_mode HAF_SVM_FP32_GUARD / HAF_SVM_FP64_EXACT)", (double)ctx->audit_max_rel, (double)ctx->guard_rel);
        ctx->tc_passes++;
        ctx->escalations++;
        ctx->copy_pieces = 0;   // a host-staged batch is on the device by now
    }
}

// M: the winning roll's matrix as the device built it (haf_search_batch_requests); NULL = build it on the host
static void fill_best(const haf_ctx* ctx, const Job& jb, const JobResult& r, int approach_idx, long long n_guard, haf_best* b,
                      const float* M = nullptr) {
    memset(b, 0, sizeof *b);
    b->row = r.row; b->col = r.col; b->roll = r.roll; b->tilt = (r.roll >= 0) ? 0 : -1; b->approach_idx = approach_idx;
    b->topval = r.topval; b->eval = r.topval - 20;                                          // server.cpp:390
    b->roll_rad = (float)((r.roll * ctx->cfg.roll_step_deg * hafhost::kPI) / 180);           // :1401
    if (r.roll >= 0) {
        if (M) memcpy(b->M, M, sizeof b->M);
        else hafhost::build_transform(jb.rq, r.roll, ctx->cfg.roll_step_deg, b->M);
    }
    b->rolls_done = r.rolls_done; b->n_windows_scored = r.n_windows; b->n_guard = (int)n_guard;
}

// helper thread of a pageable host batch (haf_ctx::Stager): piece by piece, src -> pinned ring slot (stage_threads host threads),
// then the slot -> dst (device) copy and the piece's event on copy_stream.  A slot is reused once the copy that read it has finished.
static void stager_main(haf_ctx* ctx, unsigned char* dst, const unsigned char* src, std::vector<std::pair<size_t, size_t> > pieces, size_t slot_bytes) {
    bool ok = cudaSetDevice(ctx->device) == cudaSuccess;
    const int T = std::max(1, std::min(16, ctx->stage_threads));
    for (size_t k = 0; k < pieces.size(); k++) {
        const size_t b0 = pieces[k].first, n = pieces[k].second - pieces[k].first;
        unsigned char* slot = ctx->h_ring.p + (k % haf_ctx::kRingSlots) * slot_bytes;
        if (ok && k >= (size_t)haf_ctx::kRingSlots) ok = cudaEventSynchronize(ctx->copy_ev[k - haf_ctx::kRingSlots]) == cudaSuccess;
        if (ok && n) {
            std::vector<std::thread> helpers;
            const size_t per = round_up((n + T - 1) / T, 4096);
            // slice t of T goes to helper thread t (t >= 1); this thread copies slice 0 and whatever could not get a thread
            size_t covered = std::min(per, n);   // bytes [0, covered) are this thread's or a started helper's
            for (int t = 1; t < T && covered < n; t++) {
                const size_t o = covered, len = std::min(per, n - o);
                try { helpers.emplace_back([=] { memcpy(slot + o, src + b0 + o, len); }); }
                catch (...) { break; }
                covered = o + len;
            }
            memcpy(slot, src + b0, std::min(per, n));
            if (covered < n) memcpy(slot + covered, src + b0 + covered, n - covered);
            for (size_t t = 0; t < helpers.size(); t++) helpers[t].join();
            ok = cudaMemcpyAsync(dst + b0, slot, n, cudaMemcpyHostToDevice, ctx->copy_stream) == cudaSuccess;
        }
        if (cudaEventRecord(ctx->copy_ev[k], ctx->copy_stream) != cudaSuccess) ok = false;
        {
            std::lock_guard<std::mutex> lk(ctx->stager.mu);
            if (!ok) ctx->stager.failed = true;
            ctx->stager.issued = (int)k + 1;
        }
        ctx->stager.cv.notify_all();
    }
}

// stage a host cloud set on the device (or use device pointers in place)
static int stage_points(haf_ctx* ctx, const void* src, size_t bytes, bool* is_dev) {
    *is_dev = is_device_ptr(src);
    if (*is_dev) return HAF_OK;
    ENSURE(ctx, ctx->d_xyz, bytes + 16);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_xyz.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return HAF_OK;
}

// grasp poses asked for by haf_search_grasps / haf_search_batch_packed_grasps: where the records go (host memory, NULL = not
// wanted).  best: the overall winner's (single goals only); per_job [n_jobs]; per_roll [n_jobs][R], evaluated rolls only.
// units: the per-unit records stay readable in ctx->h_unit_grasp after the call (members of a multi-GPU group).
struct GraspOut {
    haf_grasp* best = nullptr;
    haf_grasp* per_job = nullptr;
    haf_grasp* per_roll = nullptr;
    bool units = false;
};
static_assert(sizeof(haf_grasp) == sizeof(GraspRec) && offsetof(haf_grasp, graspPoint1) == offsetof(GraspRec, gp1) &&
              offsetof(haf_grasp, approachVector) == offsetof(GraspRec, approach) && offsetof(haf_grasp, row) == offsetof(GraspRec, row) &&
              offsetof(haf_grasp, reserved) == offsetof(GraspRec, reserved), "haf_grasp and GraspRec must share their layout");
// grasp_mode of the context for the length of one call
struct GraspScope {
    haf_ctx* c;
    GraspScope(haf_ctx* ctx, const GraspOut* go) : c(ctx) { c->grasp_mode = go ? ((go->per_roll || go->units) ? 2 : 1) : 0; }
    ~GraspScope() { c->grasp_mode = 0; }
};
// unit parameters built on the device for the length of one call (haf_search_batch_requests)
struct DeviceUnitsScope {
    haf_ctx* c;
    explicit DeviceUnitsScope(haf_ctx* ctx) : c(ctx) { c->device_units = true; }
    ~DeviceUnitsScope() { c->device_units = false; }
};
// ranked candidates for the length of one call (haf_search_batch_candidates): the parameters, checked, and where the records go
struct RankOut {
    int k, per_unit;
    double md2;                       // min_distance^2, -1 = no suppression
    haf_candidate* candidates;        // [n_clouds][k]
    int* n_candidates;                // [n_clouds]
};
static_assert(sizeof(haf_candidate) == sizeof(CandRec) && offsetof(haf_candidate, score) == offsetof(CandRec, score) &&
              offsetof(haf_candidate, request) == offsetof(CandRec, request), "haf_candidate and CandRec must share their layout");
struct RankScope {
    haf_ctx* c;
    RankScope(haf_ctx* ctx, const RankOut* ro) : c(ctx) {
        c->rank_k = ro ? ro->k : 0; c->rank_p = ro ? ro->per_unit : 0; c->rank_md2 = ro ? ro->md2 : -1.0;
    }
    ~RankScope() { c->rank_k = 0; c->rank_p = 0; c->rank_md2 = -1.0; }
};
// per-roll records of the evaluated rolls of each job: h_unit_grasp -> out [n_jobs][R] (the other rolls are left untouched)
static void copy_roll_grasps(const haf_ctx* ctx, const std::vector<Job>& jobs, haf_grasp* out) {
    const int R = ctx->R;
    for (size_t j = 0; j < jobs.size(); j++)
        if (jobs[j].n_rolls_active > jobs[j].roll_begin)
            memcpy(out + j * R + jobs[j].roll_begin, ctx->h_unit_grasp.p + j * R + jobs[j].roll_begin,
                   (size_t)(jobs[j].n_rolls_active - jobs[j].roll_begin) * sizeof(haf_grasp));
}

static int group_search(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* reqs, int n_requests,
                        haf_best* best, haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top,
                        const GraspOut* go = nullptr);
static int group_batch_packed(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* req,
                              haf_best* best_per_cloud, const GraspOut* go = nullptr);
static int group_batch_requests(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll, const RankOut* rank = nullptr);
static void group_timing(haf_ctx* ctx);

// one GPU: the context itself (also what each member of a multi-GPU group runs -- group[0] IS the head context, so the
// group entry points must never be re-entered from a member thread)
static int search_single(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* reqs, int n_requests,
                         haf_best* best, haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top,
                         const GraspOut* go = nullptr);
static int batch_packed_single(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* req,
                               haf_best* best_per_cloud, const GraspOut* go = nullptr);
static int batch_requests_single(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                 const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                 haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll, const RankOut* rank = nullptr);
static int batch_single(haf_ctx* ctx, const float* const* clouds, const size_t* n_points, int n_clouds, const haf_request* req,
                        haf_best* best_per_cloud);

extern "C" int haf_search(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* reqs, int n_requests,
                          haf_best* best, haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top) {
    if (!ctx) return HAF_ERR_ARG;
    if (ctx->group.size() > 1)
        return group_search(ctx, xyz, n_points, stride_bytes, reqs, n_requests, best, best_per_request, graspseval, mask, heights, per_roll_top);
    return search_single(ctx, xyz, n_points, stride_bytes, reqs, n_requests, best, best_per_request, graspseval, mask, heights, per_roll_top);
}
extern "C" int haf_search_grasps(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* reqs, int n_requests,
                                 haf_best* best, haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights,
                                 int* per_roll_top, haf_grasp* grasp, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll) {
    if (!ctx) return HAF_ERR_ARG;
    if (!grasp) return ctx->fail(HAF_ERR_ARG, "haf_search_grasps: grasp is required");
    GraspOut go;
    go.best = grasp; go.per_job = grasp_per_request; go.per_roll = grasp_per_roll;
    if (ctx->group.size() > 1)
        return group_search(ctx, xyz, n_points, stride_bytes, reqs, n_requests, best, best_per_request, graspseval, mask, heights, per_roll_top, &go);
    return search_single(ctx, xyz, n_points, stride_bytes, reqs, n_requests, best, best_per_request, graspseval, mask, heights, per_roll_top, &go);
}
static int search_single(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* reqs, int n_requests,
                         haf_best* best, haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top,
                         const GraspOut* go) {
    if (!reqs || n_requests < 1 || !best) return ctx->fail(HAF_ERR_ARG, "haf_search: reqs, n_requests >= 1 and best are required");
    if (n_points > 0 && !xyz) return ctx->fail(HAF_ERR_ARG, "haf_search: xyz is null");
    if (stride_bytes == 0) stride_bytes = 12;
    if (stride_bytes < 12 || (stride_bytes & 3)) return ctx->fail(HAF_ERR_ARG, "haf_search: stride_bytes must be >= 12 and a multiple of 4");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    ctx->last_valid = false;
    CloudSet cs;
    cs.stride = stride_bytes;
    cs.off.push_back(0);
    cs.off.push_back((long long)n_points);
    bool dev = false;
    if (n_points > 0) {
        int rc = stage_points(ctx, xyz, n_points * stride_bytes, &dev);
        if (rc) return rc;
    }
    cs.d_xyz = n_points == 0 ? nullptr : (dev ? reinterpret_cast<const unsigned char*>(xyz) : ctx->d_xyz.p);
    std::vector<Job> jobs(n_requests);
    for (int a = 0; a < n_requests; a++) { jobs[a].cloud = 0; jobs[a].rq = reqs[a]; }
    int rc;
    {
        GraspScope gs(ctx, go);
        rc = run_jobs(ctx, cs, jobs, graspseval, mask, heights, true);
    }
    if (rc) return rc;
    const int R = ctx->R;
    // overall winner over requests: strict >, earliest request wins ties (server.cpp:953 extended over approach vectors)
    int win = -1, wtop = -1000;
    for (int a = 0; a < n_requests; a++) {
        const JobResult& r = ctx->h_results.p[a];
        if (best_per_request) fill_best(ctx, jobs[a], r, a, ctx->timing.n_guard, &best_per_request[a]);
        if (r.topval > wtop) { wtop = r.topval; win = a; }
        if (per_roll_top)   // every roll: the ones not evaluated (roll_begin / roll_limit) carry (-1, -1, -1000)
            memcpy(per_roll_top + (size_t)a * R * 3, ctx->h_per_roll_top.p + (size_t)a * R * 3, (size_t)R * 3 * sizeof(int));
    }
    if (win < 0) {
        JobResult none; memset(&none, 0, sizeof none);
        none.row = none.col = none.roll = -1; none.topval = -1000;
        fill_best(ctx, jobs[0], none, -1, ctx->timing.n_guard, best);
    } else {
        fill_best(ctx, jobs[win], ctx->h_results.p[win], win, ctx->timing.n_guard, best);
        long long nw = 0; int rd = 0;
        for (int a = 0; a < n_requests; a++) { nw += ctx->h_results.p[a].n_windows; rd += ctx->h_results.p[a].rolls_done; }
        best->n_windows_scored = (int)nw; best->rolls_done = rd;
    }
    if (go) {   // no winner at all: request 0's roll -1 pose, like `best`
        if (go->best) memcpy(go->best, ctx->h_job_grasp.p + (win < 0 ? 0 : win), sizeof(haf_grasp));
        if (go->per_job) memcpy(go->per_job, ctx->h_job_grasp.p, (size_t)n_requests * sizeof(haf_grasp));
        if (go->per_roll) copy_roll_grasps(ctx, jobs, go->per_roll);
    }
    return HAF_OK;
}

extern "C" int haf_search_batch_packed(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* req,
                                       haf_best* best_per_cloud) {
    if (!ctx) return HAF_ERR_ARG;
    if (ctx->group.size() > 1) return group_batch_packed(ctx, xyz_all, point_offsets, n_clouds, req, best_per_cloud);
    return batch_packed_single(ctx, xyz_all, point_offsets, n_clouds, req, best_per_cloud);
}
extern "C" int haf_search_batch_packed_grasps(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* req,
                                              haf_best* best_per_cloud, haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_roll) {
    if (!ctx) return HAF_ERR_ARG;
    if (!grasp_per_cloud) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_packed_grasps: grasp_per_cloud is required");
    GraspOut go;
    go.per_job = grasp_per_cloud; go.per_roll = grasp_per_roll;
    if (ctx->group.size() > 1) return group_batch_packed(ctx, xyz_all, point_offsets, n_clouds, req, best_per_cloud, &go);
    return batch_packed_single(ctx, xyz_all, point_offsets, n_clouds, req, best_per_cloud, &go);
}
// starts the staging thread (stager_main) for pieces [b0, b1) of src, copied to dst + b0 on copy_stream; copy_ev holds an event
// per piece, copy_stream already follows the work queued before on the stream
static int start_stager(haf_ctx* ctx, unsigned char* dst, const unsigned char* src, const std::vector<std::pair<size_t, size_t> >& piece_bytes) {
    size_t slot = 0;
    for (size_t i = 0; i < piece_bytes.size(); i++) slot = std::max(slot, piece_bytes[i].second - piece_bytes[i].first);
    slot = round_up(slot, 4096);
    ENSURE(ctx, ctx->h_ring, slot * haf_ctx::kRingSlots);
    ctx->stager.issued = 0; ctx->stager.failed = false;
    try {
        ctx->stager.th = std::thread(stager_main, ctx, dst, src, piece_bytes, slot);
        ctx->stager.active = true;
    } catch (...) {
        return ctx->fail(HAF_ERR_NOMEM, "could not start the staging thread for a pageable host batch (set HAF_STAGE_THREADS=0 to use the driver's copy path)");
    }
    return HAF_OK;
}
// The clouds of a packed batch on the device (cs): device memory is used in place, host memory is staged piece by piece.
// A pageable batch starts the staging thread; the caller joins it (StagerJoin) once run_jobs has returned.
static int prepare_batch(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, CloudSet& cs) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    ctx->last_valid = false;
    cs.stride = 12;
    cs.off.resize(n_clouds + 1);
    for (int c = 0; c <= n_clouds; c++) cs.off[c] = (long long)point_offsets[c];
    for (int c = 0; c < n_clouds; c++) if (cs.off[c + 1] < cs.off[c]) return ctx->fail(HAF_ERR_ARG, "point_offsets must be non-decreasing");
    const size_t total = (size_t)cs.off[n_clouds];
    if (total > 0 && !xyz_all) return ctx->fail(HAF_ERR_ARG, "xyz_all is null");
    bool dev = total > 0 && is_device_ptr(xyz_all);
    ctx->copy_pieces = 0;
    if (total > 0 && !dev) {
        // stage in pieces on a second stream; run_jobs makes each chunk wait only for the pieces it needs, so the
        // host->device copy of later clouds overlaps the kernels of earlier ones (pinned host memory copies truly async)
        ENSURE(ctx, ctx->d_xyz, total * 12 + 16);
        if (!ctx->copy_stream) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        cudaEvent_t start_ev;
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&start_ev, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventRecord(start_ev, ctx->stream));            // copies start no earlier than prior work on the stream
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, start_ev, 0));
        cudaEventDestroy(start_ev);
        ctx->copy_cloud_end.clear();
        const bool own_staging = ctx->stage_threads > 0 && total * 12 >= ((size_t)4 << 20) && !is_pinned_host_ptr(xyz_all);
        std::vector<std::pair<size_t, size_t> > piece_bytes;   // [b0, b1) of every piece (own staging)
        int c = 0, k = 0;
        while (c < n_clouds) {
            int ce = c;
            // the first piece is what the first chunk of run_jobs needs (16 clouds): compute starts ~0.25 ms earlier
            const int piece_clouds = (k == 0) ? 16 : 32;
            while (ce < n_clouds && (ce - c) < piece_clouds && (size_t)(cs.off[ce] - cs.off[c]) * 12 < ((size_t)32 << 20)) ce++;
            if (ce == c) ce = c + 1;
            const size_t b0 = (size_t)cs.off[c] * 12, b1 = (size_t)cs.off[ce] * 12;
            if ((int)ctx->copy_ev.size() <= k) {
                cudaEvent_t e;
                CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx->copy_ev.push_back(e);
            }
            if (own_staging) piece_bytes.push_back(std::make_pair(b0, b1));
            else {
                if (b1 > b0) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_xyz.p + b0, reinterpret_cast<const unsigned char*>(xyz_all) + b0, b1 - b0, cudaMemcpyHostToDevice, ctx->copy_stream));
                CUDA_TRY(ctx, cudaEventRecord(ctx->copy_ev[k], ctx->copy_stream));
            }
            ctx->copy_cloud_end.push_back(ce);
            c = ce;
            k++;
        }
        ctx->copy_pieces = k;
        if (own_staging) {
            const int rc = start_stager(ctx, ctx->d_xyz.p, reinterpret_cast<const unsigned char*>(xyz_all), piece_bytes);
            if (rc) { ctx->copy_pieces = 0; return rc; }
        }
    }
    cs.d_xyz = total == 0 ? nullptr : (dev ? reinterpret_cast<const unsigned char*>(xyz_all) : ctx->d_xyz.p);
    return HAF_OK;
}
struct StagerJoin {
    haf_ctx* c;
    ~StagerJoin() { if (c->stager.active) { c->stager.th.join(); c->stager.active = false; } }
};

static int batch_packed_single(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* req,
                               haf_best* best_per_cloud, const GraspOut* go) {
    if (!point_offsets || n_clouds < 1 || !req || !best_per_cloud) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_packed: bad arguments");
    CloudSet cs;
    { const int rc = prepare_batch(ctx, xyz_all, point_offsets, n_clouds, cs); if (rc) return rc; }
    StagerJoin stager_join{ctx};
    std::vector<Job> jobs(n_clouds);
    for (int c = 0; c < n_clouds; c++) { jobs[c].cloud = c; jobs[c].rq = *req; }
    int rc;
    {
        GraspScope gs(ctx, go);
        rc = run_jobs(ctx, cs, jobs, nullptr, nullptr, nullptr, ctx->debug_keep_batch);
    }
    ctx->copy_pieces = 0;
    if (rc) return rc;
    if (go) {
        if (go->per_job) memcpy(go->per_job, ctx->h_job_grasp.p, (size_t)n_clouds * sizeof(haf_grasp));
        if (go->per_roll) copy_roll_grasps(ctx, jobs, go->per_roll);
    }
    {   // one request for all clouds: the winning roll's transform is built once per roll, not once per cloud
        std::vector<haf_best> per_roll(ctx->R);
        std::vector<char> have(ctx->R, 0);
        for (int c = 0; c < n_clouds; c++) {
            const JobResult& r = ctx->h_results.p[c];
            if (r.roll < 0 || r.roll >= ctx->R) { fill_best(ctx, jobs[c], r, 0, 0, &best_per_cloud[c]); continue; }
            if (!have[r.roll]) { fill_best(ctx, jobs[c], r, 0, 0, &per_roll[r.roll]); have[r.roll] = 1; }
            haf_best& b = best_per_cloud[c];
            b = per_roll[r.roll];   // roll, roll_rad, M, tilt, approach_idx are functions of (request, roll) alone
            b.row = r.row; b.col = r.col; b.topval = r.topval; b.eval = r.topval - 20;
            b.rolls_done = r.rolls_done; b.n_windows_scored = r.n_windows; b.n_guard = 0;
        }
    }
    return HAF_OK;
}

static int batch_requests_entry(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll, const RankOut* rank);
extern "C" int haf_search_batch_requests(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                         const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                         haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll) {
    if (!ctx) return HAF_ERR_ARG;
    if (!point_offsets || n_clouds < 1 || !reqs || !best_per_cloud) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_requests: bad arguments");
    if (!grasp_per_cloud && (grasp_per_request || grasp_per_roll))
        return ctx->fail(HAF_ERR_ARG, "haf_search_batch_requests: grasp_per_request / grasp_per_roll need grasp_per_cloud");
    return batch_requests_entry(ctx, xyz_all, point_offsets, n_clouds, reqs, request_offsets, best_per_cloud, best_per_request, per_roll_top,
                                grasp_per_cloud, grasp_per_request, grasp_per_roll, nullptr);
}
extern "C" int haf_search_batch_candidates(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                           const int* request_offsets, const haf_rank_params* rp, haf_best* best_per_cloud,
                                           haf_grasp* grasp_per_cloud, haf_candidate* candidates, int* n_candidates) {
    if (!ctx) return HAF_ERR_ARG;
    if (!point_offsets || n_clouds < 1 || !reqs || !rp || !best_per_cloud || !grasp_per_cloud || !candidates || !n_candidates)
        return ctx->fail(HAF_ERR_ARG, "haf_search_batch_candidates: bad arguments");
    if (rp->k < 1 || rp->k > 256) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_candidates: k = %d outside 1..256", rp->k);
    const int per_unit = rp->per_unit == 0 ? std::max(rp->k, 64) : rp->per_unit;
    if (per_unit < rp->k || per_unit > 1024)
        return ctx->fail(HAF_ERR_ARG, "haf_search_batch_candidates: per_unit = %d outside k..1024 (0 = max(k, 64))", rp->per_unit);
    if (std::isnan(rp->min_distance)) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_candidates: min_distance is NaN");
    for (int i = 0; i < 4; i++)
        if (rp->reserved[i]) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_candidates: reserved[%d] must be 0", i);
    RankOut ro;
    ro.k = rp->k; ro.per_unit = per_unit;
    ro.md2 = rp->min_distance > 0 ? rp->min_distance * rp->min_distance : -1.0;
    ro.candidates = candidates; ro.n_candidates = n_candidates;
    return batch_requests_entry(ctx, xyz_all, point_offsets, n_clouds, reqs, request_offsets, best_per_cloud, nullptr, nullptr,
                                grasp_per_cloud, nullptr, nullptr, &ro);
}
// arguments checked above, request_offsets aside
static int batch_requests_entry(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll, const RankOut* rank) {
    std::vector<int> one_each;
    if (!request_offsets) {
        one_each.resize(n_clouds + 1);
        for (int c = 0; c <= n_clouds; c++) one_each[c] = c;
        request_offsets = one_each.data();
    }
    if (request_offsets[0] != 0) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_requests: request_offsets[0] must be 0");
    for (int c = 0; c < n_clouds; c++)
        if (request_offsets[c + 1] <= request_offsets[c])
            return ctx->fail(HAF_ERR_ARG, "haf_search_batch_requests: cloud %d has no request (request_offsets must increase)", c);
    if ((long long)request_offsets[n_clouds] * ctx->R > 0x7fffffffLL) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_requests: too many requests");
    if (rank && (long long)request_offsets[n_clouds] * ctx->R * rank->per_unit > 0x7fffffffLL)
        return ctx->fail(HAF_ERR_ARG, "haf_search_batch_candidates: requests x rolls x per_unit above 2^31");
    if (ctx->group.size() > 1)
        return group_batch_requests(ctx, xyz_all, point_offsets, n_clouds, reqs, request_offsets, best_per_cloud, best_per_request, per_roll_top,
                                    grasp_per_cloud, grasp_per_request, grasp_per_roll, rank);
    return batch_requests_single(ctx, xyz_all, point_offsets, n_clouds, reqs, request_offsets, best_per_cloud, best_per_request, per_roll_top,
                                 grasp_per_cloud, grasp_per_request, grasp_per_roll, rank);
}
// request_offsets: checked, request_offsets[0] = 0
static int batch_requests_single(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                 const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                 haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll, const RankOut* rank) {
    CloudSet cs;
    { const int rc = prepare_batch(ctx, xyz_all, point_offsets, n_clouds, cs); if (rc) return rc; }
    StagerJoin stager_join{ctx};
    const int* ro = request_offsets;
    const int n_reqs = ro[n_clouds], R = ctx->R;
    std::vector<Job> jobs(n_reqs);
    for (int c = 0; c < n_clouds; c++)
        for (int r = ro[c]; r < ro[c + 1]; r++) { jobs[r].cloud = c; jobs[r].rq = reqs[r]; }
    int rc;
    {
        GraspOut go;
        go.per_roll = grasp_per_roll;
        GraspScope gs(ctx, grasp_per_cloud ? &go : nullptr);
        DeviceUnitsScope ds(ctx);
        RankScope rs(ctx, rank);
        rc = run_jobs(ctx, cs, jobs, nullptr, nullptr, nullptr, ctx->debug_keep_batch);
    }
    ctx->copy_pieces = 0;
    if (rc) return rc;
    // per cloud what haf_search_grasps returns for its request list (n_guard aside, 0 as in the other batch calls)
    const JobResult* res = ctx->h_results.p;
    for (int c = 0; c < n_clouds; c++) {
        int win = -1, wtop = -1000, rd = 0;
        long long nw = 0;
        for (int r = ro[c]; r < ro[c + 1]; r++) {
            if (best_per_request) fill_best(ctx, jobs[r], res[r], r - ro[c], 0, &best_per_request[r], ctx->h_best_M.p + (size_t)r * 16);
            if (res[r].topval > wtop) { wtop = res[r].topval; win = r; }   // strict >: the earliest request wins ties
            nw += res[r].n_windows; rd += res[r].rolls_done;
        }
        if (win < 0) {
            JobResult none; memset(&none, 0, sizeof none);
            none.row = none.col = none.roll = -1; none.topval = -1000;
            fill_best(ctx, jobs[ro[c]], none, -1, 0, &best_per_cloud[c]);
        } else {
            fill_best(ctx, jobs[win], res[win], win - ro[c], 0, &best_per_cloud[c], ctx->h_best_M.p + (size_t)win * 16);
            best_per_cloud[c].n_windows_scored = (int)nw; best_per_cloud[c].rolls_done = rd;
        }
        if (grasp_per_cloud) memcpy(&grasp_per_cloud[c], ctx->h_job_grasp.p + (win < 0 ? ro[c] : win), sizeof(haf_grasp));
    }
    if (per_roll_top) memcpy(per_roll_top, ctx->h_per_roll_top.p, (size_t)n_reqs * R * 3 * sizeof(int));
    if (grasp_per_request) memcpy(grasp_per_request, ctx->h_job_grasp.p, (size_t)n_reqs * sizeof(haf_grasp));
    if (grasp_per_roll) copy_roll_grasps(ctx, jobs, grasp_per_roll);
    if (rank)   // the slots after a cloud's n_candidates are zeroed
        for (int c = 0; c < n_clouds; c++) {
            const int nc = ctx->h_ncand.p[c];
            rank->n_candidates[c] = nc;
            haf_candidate* dst = rank->candidates + (size_t)c * rank->k;
            memcpy(dst, ctx->h_cand.p + (size_t)c * rank->k, (size_t)nc * sizeof(haf_candidate));
            memset(dst + nc, 0, (size_t)(rank->k - nc) * sizeof(haf_candidate));
        }
    return HAF_OK;
}

extern "C" int haf_search_batch(haf_ctx* ctx, const float* const* clouds, const size_t* n_points, int n_clouds, const haf_request* req,
                                haf_best* best_per_cloud) {
    if (!ctx) return HAF_ERR_ARG;
    if (!clouds || !n_points || n_clouds < 1 || !req || !best_per_cloud) return ctx->fail(HAF_ERR_ARG, "haf_search_batch: bad arguments");
    if (ctx->group.size() > 1) {   // several GPUs: contiguous blocks of clouds, one host thread per GPU, no cross-GPU data
        const int n = (int)ctx->group.size();
        std::vector<int> rcs(n, HAF_OK);
        std::vector<std::thread> th;
        for (int k = 0; k < n; k++) {
            const int c0 = (int)((long long)n_clouds * k / n), c1 = (int)((long long)n_clouds * (k + 1) / n);
            if (c1 <= c0) continue;
            th.emplace_back([=, &rcs]() { rcs[k] = batch_single(ctx->group[k], clouds + c0, n_points + c0, c1 - c0, req, best_per_cloud + c0); });
        }
        for (size_t i = 0; i < th.size(); i++) th[i].join();
        for (int k = 0; k < n; k++)
            if (rcs[k] != HAF_OK) { const std::string msg = ctx->group[k]->err; return ctx->fail(rcs[k], "GPU %d: %s", ctx->group[k]->device, msg.c_str()); }
        group_timing(ctx);
        return HAF_OK;
    }
    return batch_single(ctx, clouds, n_points, n_clouds, req, best_per_cloud);
}
static int batch_single(haf_ctx* ctx, const float* const* clouds, const size_t* n_points, int n_clouds, const haf_request* req,
                        haf_best* best_per_cloud) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<size_t> off(n_clouds + 1, 0);
    for (int c = 0; c < n_clouds; c++) off[c + 1] = off[c] + n_points[c];
    ENSURE(ctx, ctx->d_xyz, off[n_clouds] * 12 + 16);
    for (int c = 0; c < n_clouds; c++) {
        if (n_points[c] == 0) continue;
        if (!clouds[c]) return ctx->fail(HAF_ERR_ARG, "haf_search_batch: clouds[%d] is null", c);
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_xyz.p + off[c] * 12, clouds[c], n_points[c] * 12, cudaMemcpyDefault, ctx->stream));
    }
    return batch_packed_single(ctx, reinterpret_cast<const float*>(ctx->d_xyz.p), off.data(), n_clouds, req, best_per_cloud);
}

// ------------------------------------------------------------------------------------------------------------
// PCD / PointCloud2 ingest on the device (SURVEY 8f-2; kernels and the PCL semantics they restate: pcd_ingest.cuh)
// ------------------------------------------------------------------------------------------------------------
// Host bytes -> dst (device).  Pinned memory, and pageable buffers under 4 MB, take one cudaMemcpyAsync on the stream; larger
// pageable buffers go through the staging thread (stager_main) in pieces that end on `cuts` (ascending offsets into src, the
// last one = bytes), and the call returns once the last piece has arrived (the pinned ring is free for the next call).
static int upload_host_bytes(haf_ctx* ctx, unsigned char* dst, const unsigned char* src, size_t bytes, const std::vector<size_t>& cuts) {
    if (bytes == 0) return HAF_OK;
    if (ctx->stage_threads <= 0 || bytes < ((size_t)4 << 20) || is_pinned_host_ptr(src)) {
        CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
        return HAF_OK;
    }
    std::vector<std::pair<size_t, size_t> > pieces;   // pieces of at least 16 MB (the last one aside)
    size_t b0 = 0;
    for (size_t i = 0; i < cuts.size(); i++)
        if (cuts[i] > b0 && (cuts[i] - b0 >= ((size_t)16 << 20) || cuts[i] == bytes)) { pieces.push_back(std::make_pair(b0, cuts[i])); b0 = cuts[i]; }
    if (!ctx->copy_stream) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    cudaEvent_t start_ev;
    CUDA_TRY(ctx, cudaEventCreateWithFlags(&start_ev, cudaEventDisableTiming));
    CUDA_TRY(ctx, cudaEventRecord(start_ev, ctx->stream));            // dst may still be read by work queued before
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, start_ev, 0));
    cudaEventDestroy(start_ev);
    while (ctx->copy_ev.size() < pieces.size()) {
        cudaEvent_t e;
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->copy_ev.push_back(e);
    }
    { const int rc = start_stager(ctx, dst, src, pieces); if (rc) return rc; }
    ctx->stager.th.join();
    ctx->stager.active = false;
    if (ctx->stager.failed) return ctx->fail(HAF_ERR_CUDA, "staging a pageable host buffer failed");
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->copy_ev[pieces.size() - 1]));
    return HAF_OK;
}

// The tables of one ingest call in one pinned block, sent with one H2D copy: add() places an array (16-byte aligned), open()
// sizes both copies once the previous call's copy has read the pinned one, send() queues the copy.
struct IngestParams {
    haf_ctx* c;
    size_t bytes = 0;
    explicit IngestParams(haf_ctx* ctx) : c(ctx) {}
    size_t add(size_t n) { const size_t o = bytes; bytes = round_up(bytes + n, 16); return o; }
    int open() {
        if (c->pcd_params_ev) CUDA_TRY(c, cudaEventSynchronize(c->pcd_params_ev));
        else CUDA_TRY(c, cudaEventCreateWithFlags(&c->pcd_params_ev, cudaEventDisableTiming));
        ENSURE(c, c->h_pcd_params, bytes + 16);
        ENSURE(c, c->d_pcd_params, bytes + 16);
        return HAF_OK;
    }
    template <typename T> T* h(size_t o) { return reinterpret_cast<T*>(c->h_pcd_params.p + o); }
    template <typename T> T* d(size_t o) { return reinterpret_cast<T*>(c->d_pcd_params.p + o); }
    int send() {
        CUDA_TRY(c, cudaMemcpyAsync(c->d_pcd_params.p, c->h_pcd_params.p, bytes, cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(c, cudaEventRecord(c->pcd_params_ev, c->stream));
        return HAF_OK;
    }
};

// one gather over the segments of a call (hafpcdk::gather_segments_kernel), tables already in the parameter block
static int launch_gather(haf_ctx* ctx, IngestParams& P, size_t o_segs, size_t o_begin, int n_segs, unsigned long long n_points) {
    if (n_segs == 0) return HAF_OK;
    hafpcdk::gather_segments_kernel<<<(unsigned)std::min<unsigned long long>((n_points + 255) / 256, 148 * 16), 256, 0, ctx->stream>>>(
        P.d<hafpcdk::GatherSeg>(o_segs), P.d<unsigned long long>(o_begin), n_segs, ctx->d_pcd_xyz.p);
    LAUNCHED(ctx);
    return HAF_OK;
}

// PCD files [file_offsets[f], file_offsets[f + 1]) of `files` (host memory) -> packed xyz of every cloud in ctx->d_pcd_xyz.
// Every header is parsed and checked on the host first (the lowest failing file is named before any device work); then each
// data kind present runs its fixed launch sequence over all its files, and one stream sync ends the call.  batch: messages
// name the file ("PCD file <i>: ..."); haf_pcd_decode (the batch of one) keeps the bare single-file texts.
static int pcd_decode_files(haf_ctx* ctx, const unsigned char* files, const size_t* file_offsets, int n_files, bool batch,
                            const float** d_xyz, size_t* point_offsets) {
    char buf[512];
    auto fail_file = [&](int f, int code, const char* fmt, ...) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        return batch ? ctx->fail(code, "PCD file %d: %s", f, buf) : ctx->fail(code, "%s", buf);
    };
    for (int f = 0; f < n_files; f++)
        if (file_offsets[f + 1] < file_offsets[f]) return ctx->fail(HAF_ERR_ARG, "haf_pcd_decode_batch: file_offsets must be non-decreasing");
    const size_t base = file_offsets[0], bytes = file_offsets[n_files] - base;
    if (bytes > 0 && !files) return ctx->fail(HAF_ERR_ARG, "haf_pcd_decode_batch: files is null");
    // ---- host: headers, checks and the tables (source addresses as offsets: raw copy or blob, fixed up below)
    std::vector<size_t> pts(n_files + 1, 0);
    std::vector<hafpcdk::AsciiFile> asc;
    std::vector<int> asc_file, tile_file, lzf_file;
    std::vector<hafpcdk::GatherSeg> segs;
    std::vector<unsigned long long> seg_begin(1, 0);
    std::vector<char> seg_in_blob;
    std::vector<hafpcdk::LzfStream> lzf;
    std::vector<size_t> cuts;
    size_t blob_bytes = 0;
    unsigned long long ascii_records_max = 0;
    const size_t tile_bytes = (size_t)HAF_PCD_TILE_THREADS * HAF_PCD_BYTES_PER_THREAD;
    for (int f = 0; f < n_files; f++) {
        const size_t fb = file_offsets[f] - base, nb = file_offsets[f + 1] - file_offsets[f];
        cuts.push_back(fb + nb);
        const unsigned char* raw = files + file_offsets[f];
        hafpcd::PcdHeader hd;
        std::string herr;
        if (!hafpcd::parse_pcd_header(raw, nb, hd, &herr)) return fail_file(f, HAF_ERR_IO, "%s", herr.c_str());
        for (int a = 0; a < 3; a++)
            if (hd.types[hd.idx[a]] != "F" || hd.sizes[hd.idx[a]] != 4) return fail_file(f, HAF_ERR_UNSUPPORTED, "PCD: x / y / z must be float32 fields");
        const size_t npts = (size_t)hd.npts;
        pts[f + 1] = pts[f] + npts;
        if (npts == 0) continue;
        const size_t data = fb + hd.data_begin, dn = nb - hd.data_begin;
        hafpcdk::GatherSeg sg;
        memset(&sg, 0, sizeof sg);
        sg.out_begin = pts[f];
        if (hd.data_kind == "ascii") {
            if (dn == 0) return fail_file(f, HAF_ERR_IO, "fewer records than POINTS in the PCD data");
            std::vector<int> tokoff(hd.fields.size() + 1, 0);
            for (size_t k = 0; k < hd.fields.size(); k++) tokoff[k + 1] = tokoff[k] + hd.counts[k];
            hafpcdk::AsciiFile af;
            memset(&af, 0, sizeof af);
            af.begin = data; af.len = dn; af.n_points = npts; af.out_begin = pts[f];
            const size_t n_tiles = (dn + tile_bytes - 1) / tile_bytes;
            if (tile_file.size() + n_tiles > 0x7fffffffu) return fail_file(f, HAF_ERR_UNSUPPORTED, "ASCII PCD too large");
            af.tile_begin = (int)tile_file.size(); af.tile_end = (int)(tile_file.size() + n_tiles);
            for (int a = 0; a < 3; a++) af.tok[a] = tokoff[hd.idx[a]];
            ascii_records_max += (dn + 1) / 2;     // a record is a token and a line end at least
            if (ascii_records_max > 0xFFFFFFFFull) return fail_file(f, HAF_ERR_UNSUPPORTED, "ASCII PCD too large");
            tile_file.insert(tile_file.end(), n_tiles, (int)asc.size());
            asc.push_back(af);
            asc_file.push_back(f);
        } else if (hd.data_kind == "binary") {
            size_t rec_bytes = 0;
            std::vector<size_t> foff(hd.fields.size());
            for (size_t k = 0; k < hd.fields.size(); k++) { foff[k] = rec_bytes; rec_bytes += (size_t)hd.sizes[k] * hd.counts[k]; }
            if (rec_bytes * npts > dn) return fail_file(f, HAF_ERR_IO, "binary PCD truncated");
            sg.src = reinterpret_cast<const unsigned char*>(data);
            for (int a = 0; a < 3; a++) { sg.off[a] = foff[hd.idx[a]]; sg.stride[a] = rec_bytes; }
            segs.push_back(sg); seg_in_blob.push_back(0); seg_begin.push_back(seg_begin.back() + npts);
        } else if (hd.data_kind == "binary_compressed") {
            if (dn < 8) return fail_file(f, HAF_ERR_IO, "compressed PCD truncated");
            uint32_t comp, uncomp;
            memcpy(&comp, raw + hd.data_begin, 4);
            memcpy(&uncomp, raw + hd.data_begin + 4, 4);
            if ((size_t)comp + 8 > dn) return fail_file(f, HAF_ERR_IO, "compressed PCD truncated");
            std::vector<size_t> foff(hd.fields.size());
            size_t off = 0;
            for (size_t k = 0; k < hd.fields.size(); k++) { foff[k] = off; off += npts * (size_t)hd.sizes[k] * hd.counts[k]; }
            for (int a = 0; a < 3; a++)
                if (foff[hd.idx[a]] + (npts - 1) * 4 * (size_t)hd.counts[hd.idx[a]] + 4 > uncomp)
                    return fail_file(f, HAF_ERR_IO, "compressed PCD: the stream is shorter than the header's fields");
            hafpcdk::LzfStream ls;
            ls.in = reinterpret_cast<const unsigned char*>(data + 8); ls.in_len = comp;
            ls.out = reinterpret_cast<unsigned char*>(blob_bytes); ls.out_len = uncomp;
            lzf.push_back(ls);
            lzf_file.push_back(f);
            sg.src = reinterpret_cast<const unsigned char*>(blob_bytes);
            for (int a = 0; a < 3; a++) { sg.off[a] = foff[hd.idx[a]]; sg.stride[a] = 4 * (size_t)hd.counts[hd.idx[a]]; }
            segs.push_back(sg); seg_in_blob.push_back(1); seg_begin.push_back(seg_begin.back() + npts);
            blob_bytes = round_up(blob_bytes + uncomp, 16);
        } else {
            return fail_file(f, HAF_ERR_UNSUPPORTED, "unsupported PCD DATA kind '%s'", hd.data_kind.c_str());
        }
    }
    const size_t total = pts[n_files];
    if (total > 0) {
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        cudaStream_t st = ctx->stream;
        const int n_asc = (int)asc.size(), n_lzf = (int)lzf.size();
        const unsigned n_tiles = (unsigned)tile_file.size();
        ENSURE(ctx, ctx->d_pcd_xyz, total * 3);
        ENSURE(ctx, ctx->d_pcd_raw, bytes + 16);
        ENSURE(ctx, ctx->d_pcd_blob, blob_bytes + 16);
        ENSURE(ctx, ctx->d_pcd_tiles, (size_t)n_tiles + 1);
        // status: [0] ASCII record total, then u32 count [n_asc], int flags [2 n_asc], int LZF status [n_lzf]
        const size_t status_words = 1 + ((size_t)n_asc * 12 + (size_t)n_lzf * 4 + 7) / 8;
        ENSURE(ctx, ctx->d_pcd_status, status_words);
        ENSURE(ctx, ctx->h_pcd_status, status_words);
        unsigned* d_count = reinterpret_cast<unsigned*>(ctx->d_pcd_status.p + 1);
        int* d_flags = reinterpret_cast<int*>(d_count + n_asc);
        int* d_lzf_status = d_flags + 2 * n_asc;
        for (size_t s = 0; s < segs.size(); s++)
            segs[s].src = (seg_in_blob[s] ? ctx->d_pcd_blob.p : ctx->d_pcd_raw.p) + reinterpret_cast<size_t>(segs[s].src);
        for (int l = 0; l < n_lzf; l++) {
            lzf[l].in = ctx->d_pcd_raw.p + reinterpret_cast<size_t>(lzf[l].in);
            lzf[l].out = ctx->d_pcd_blob.p + reinterpret_cast<size_t>(lzf[l].out);
        }
        IngestParams P(ctx);
        const size_t o_asc = P.add(asc.size() * sizeof(hafpcdk::AsciiFile)), o_tiles = P.add(tile_file.size() * sizeof(int));
        const size_t o_segs = P.add(segs.size() * sizeof(hafpcdk::GatherSeg)), o_begin = P.add(seg_begin.size() * 8);
        const size_t o_lzf = P.add(lzf.size() * sizeof(hafpcdk::LzfStream));
        { const int rc = P.open(); if (rc) return rc; }
        if (n_asc) memcpy(P.h<hafpcdk::AsciiFile>(o_asc), asc.data(), asc.size() * sizeof(hafpcdk::AsciiFile));
        if (n_tiles) memcpy(P.h<int>(o_tiles), tile_file.data(), tile_file.size() * sizeof(int));
        if (!segs.empty()) memcpy(P.h<hafpcdk::GatherSeg>(o_segs), segs.data(), segs.size() * sizeof(hafpcdk::GatherSeg));
        memcpy(P.h<unsigned long long>(o_begin), seg_begin.data(), seg_begin.size() * 8);
        if (n_lzf) memcpy(P.h<hafpcdk::LzfStream>(o_lzf), lzf.data(), lzf.size() * sizeof(hafpcdk::LzfStream));
        { const int rc = upload_host_bytes(ctx, ctx->d_pcd_raw.p, files + base, bytes, cuts); if (rc) return rc; }
        { const int rc = P.send(); if (rc) return rc; }
        CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_pcd_status.p, 0, status_words * 8, st));
        if (n_asc) {
            hafpcdk::ascii_count_kernel<<<n_tiles, HAF_PCD_TILE_THREADS, 0, st>>>(ctx->d_pcd_raw.p, P.d<hafpcdk::AsciiFile>(o_asc), P.d<int>(o_tiles),
                                                                                  ctx->d_pcd_tiles.p);
            LAUNCHED(ctx);
            hafpcdk::ascii_scan_kernel<<<1, 1024, 0, st>>>(ctx->d_pcd_tiles.p, n_tiles, ctx->d_pcd_status.p);
            LAUNCHED(ctx);
            hafpcdk::ascii_parse_kernel<<<n_tiles, HAF_PCD_TILE_THREADS, 0, st>>>(ctx->d_pcd_raw.p, P.d<hafpcdk::AsciiFile>(o_asc), P.d<int>(o_tiles),
                                                                                  ctx->d_pcd_tiles.p, n_tiles, ctx->d_pcd_status.p, ctx->d_pcd_xyz.p,
                                                                                  d_count, d_flags);
            LAUNCHED(ctx);
        }
        if (n_lzf) {
            hafpcdk::lzf_decompress_kernel<<<n_lzf, 32, 0, st>>>(P.d<hafpcdk::LzfStream>(o_lzf), d_lzf_status);
            LAUNCHED(ctx);
        }
        { const int rc = launch_gather(ctx, P, o_segs, o_begin, (int)segs.size(), seg_begin.back()); if (rc) return rc; }
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pcd_status.p, ctx->d_pcd_status.p, status_words * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        // the lowest failing file, with the single-file checks in their order
        const unsigned* h_count = reinterpret_cast<const unsigned*>(ctx->h_pcd_status.p + 1);
        const int* h_flags = reinterpret_cast<const int*>(h_count + n_asc);
        const int* h_lzf_status = h_flags + 2 * n_asc;
        int la = 0, ll = 0;
        while (la < n_asc || ll < n_lzf) {
            const bool take_asc = ll >= n_lzf || (la < n_asc && asc_file[la] < lzf_file[ll]);
            if (take_asc) {
                const int f = asc_file[la], a = la++;
                if (h_count[a] < asc[a].n_points)
                    return fail_file(f, HAF_ERR_IO, "fewer records than POINTS in the PCD data (%llu of %zu)", (unsigned long long)h_count[a], (size_t)asc[a].n_points);
                if (h_flags[2 * a]) return fail_file(f, HAF_ERR_IO, "short ASCII record in the PCD data");
                if (h_flags[2 * a + 1])
                    return fail_file(f, HAF_ERR_UNSUPPORTED, "an ASCII token has more than 19 significant digits and lies next to a float rounding boundary");
            } else {
                const int f = lzf_file[ll], l = ll++;
                if (h_lzf_status[l]) return fail_file(f, HAF_ERR_IO, "corrupt LZF stream in the PCD data");
            }
        }
    }
    for (int f = 0; f <= n_files; f++) point_offsets[f] = pts[f];
    *d_xyz = total ? ctx->d_pcd_xyz.p : nullptr;
    return HAF_OK;
}

// PointCloud2 data: cloud c = bytes [byte_offsets[c], byte_offsets[c + 1]) of data (host or device), records of layouts[4c]
// bytes with x / y / z float32 at layouts[4c + 1 .. 4c + 3] -> packed xyz in ctx->d_pcd_xyz (one gather, no sync).  Clouds of
// no bytes are empty and not checked.  batch: messages name the cloud (haf_pointcloud2_to_xyz is the batch of one).
static int pointcloud2_clouds(haf_ctx* ctx, const void* data, const size_t* byte_offsets, int n_clouds, const int* layouts, bool batch,
                              const float** d_xyz, size_t* point_offsets) {
    const char* who = batch ? "haf_pointcloud2_batch_to_xyz" : "haf_pointcloud2_to_xyz";
    std::vector<size_t> pts(n_clouds + 1, 0);
    for (int c = 0; c < n_clouds; c++) {
        if (byte_offsets[c + 1] < byte_offsets[c]) return ctx->fail(HAF_ERR_ARG, "%s: byte_offsets must be non-decreasing", who);
        const size_t span = byte_offsets[c + 1] - byte_offsets[c];
        pts[c + 1] = pts[c];
        if (span == 0) continue;
        const int* L = layouts + 4 * c;
        if (L[0] < 4 || L[1] < 0 || L[2] < 0 || L[3] < 0 || std::max(L[1], std::max(L[2], L[3])) + 4 > L[0]) {
            if (batch) return ctx->fail(HAF_ERR_ARG, "%s: cloud %d: x / y / z offsets must lie inside point_step", who, c);
            return ctx->fail(HAF_ERR_ARG, "%s: x / y / z offsets must lie inside point_step", who);
        }
        if (span % (size_t)L[0]) return ctx->fail(HAF_ERR_ARG, "%s: cloud %d: %zu bytes are not a whole number of %d-byte records", who, c, span, L[0]);
        pts[c + 1] += span / (size_t)L[0];
    }
    const size_t base = byte_offsets[0], bytes = byte_offsets[n_clouds] - base, total = pts[n_clouds];
    if (bytes > 0 && !data) return ctx->fail(HAF_ERR_ARG, "%s: data is null", who);
    if (total > 0) {
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        const unsigned char* src = reinterpret_cast<const unsigned char*>(data) + base;
        if (!is_device_ptr(data)) {
            ENSURE(ctx, ctx->d_pcd_raw, bytes + 16);
            std::vector<size_t> cuts;
            for (int c = 1; c <= n_clouds; c++) cuts.push_back(byte_offsets[c] - base);
            const int rc = upload_host_bytes(ctx, ctx->d_pcd_raw.p, src, bytes, cuts);
            if (rc) return rc;
            src = ctx->d_pcd_raw.p;
        }
        ENSURE(ctx, ctx->d_pcd_xyz, total * 3);
        std::vector<hafpcdk::GatherSeg> segs;
        std::vector<unsigned long long> seg_begin(1, 0);
        for (int c = 0; c < n_clouds; c++) {
            if (pts[c + 1] == pts[c]) continue;
            hafpcdk::GatherSeg sg;
            sg.src = src + (byte_offsets[c] - base);
            sg.out_begin = pts[c];
            for (int a = 0; a < 3; a++) { sg.off[a] = (unsigned long long)layouts[4 * c + 1 + a]; sg.stride[a] = (unsigned long long)layouts[4 * c]; }
            segs.push_back(sg);
            seg_begin.push_back(pts[c + 1]);
        }
        IngestParams P(ctx);
        const size_t o_segs = P.add(segs.size() * sizeof(hafpcdk::GatherSeg)), o_begin = P.add(seg_begin.size() * 8);
        { const int rc = P.open(); if (rc) return rc; }
        memcpy(P.h<hafpcdk::GatherSeg>(o_segs), segs.data(), segs.size() * sizeof(hafpcdk::GatherSeg));
        memcpy(P.h<unsigned long long>(o_begin), seg_begin.data(), seg_begin.size() * 8);
        { const int rc = P.send(); if (rc) return rc; }
        { const int rc = launch_gather(ctx, P, o_segs, o_begin, (int)segs.size(), seg_begin.back()); if (rc) return rc; }
    }
    if (point_offsets) for (int c = 0; c <= n_clouds; c++) point_offsets[c] = pts[c];
    *d_xyz = total ? ctx->d_pcd_xyz.p : nullptr;
    return HAF_OK;
}

extern "C" int haf_pointcloud2_to_xyz(haf_ctx* ctx, const void* data, size_t n_points, size_t point_step, int off_x, int off_y, int off_z,
                                      const float** d_xyz) {
    if (!ctx || !d_xyz) return HAF_ERR_ARG;
    *d_xyz = nullptr;
    if (n_points == 0) return HAF_OK;
    if (!data || point_step < 4 || point_step > 0x7fffffff)
        return ctx->fail(HAF_ERR_ARG, "haf_pointcloud2_to_xyz: x / y / z offsets must lie inside point_step");
    const size_t byte_offsets[2] = {0, n_points * point_step};
    const int layout[4] = {(int)point_step, off_x, off_y, off_z};
    return pointcloud2_clouds(ctx, data, byte_offsets, 1, layout, false, d_xyz, nullptr);
}

extern "C" int haf_pointcloud2_batch_to_xyz(haf_ctx* ctx, const void* data, const size_t* byte_offsets, int n_clouds, const int* layouts,
                                            const float** d_xyz, size_t* point_offsets) {
    if (!ctx || !d_xyz) return HAF_ERR_ARG;
    *d_xyz = nullptr;
    if (!byte_offsets || n_clouds < 1 || !layouts || !point_offsets) return ctx->fail(HAF_ERR_ARG, "haf_pointcloud2_batch_to_xyz: bad arguments");
    return pointcloud2_clouds(ctx, data, byte_offsets, n_clouds, layouts, true, d_xyz, point_offsets);
}

extern "C" int haf_pcd_decode(haf_ctx* ctx, const void* file_bytes, size_t n_bytes, const float** d_xyz, size_t* n_points) {
    if (!ctx || !d_xyz || !n_points) return HAF_ERR_ARG;
    *d_xyz = nullptr; *n_points = 0;
    if (!file_bytes || n_bytes == 0) return ctx->fail(HAF_ERR_ARG, "haf_pcd_decode: empty buffer");
    const size_t file_offsets[2] = {0, n_bytes};
    size_t point_offsets[2];
    const int rc = pcd_decode_files(ctx, reinterpret_cast<const unsigned char*>(file_bytes), file_offsets, 1, false, d_xyz, point_offsets);
    if (rc == HAF_OK) *n_points = point_offsets[1];
    return rc;
}

extern "C" int haf_pcd_decode_batch(haf_ctx* ctx, const void* files, const size_t* file_offsets, int n_files, const float** d_xyz,
                                    size_t* point_offsets) {
    if (!ctx || !d_xyz) return HAF_ERR_ARG;
    *d_xyz = nullptr;
    if (!file_offsets || n_files < 1 || !point_offsets) return ctx->fail(HAF_ERR_ARG, "haf_pcd_decode_batch: bad arguments");
    return pcd_decode_files(ctx, reinterpret_cast<const unsigned char*>(files), file_offsets, n_files, true, d_xyz, point_offsets);
}

extern "C" int haf_debug_pcd_xyz(haf_ctx* ctx, float* xyz_host, size_t n_points) {
    if (!ctx || !xyz_host) return HAF_ERR_ARG;
    if (n_points * 3 > ctx->d_pcd_xyz.cap) return ctx->fail(HAF_ERR_ARG, "haf_debug_pcd_xyz: more points than the last ingest produced");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpyAsync(xyz_host, ctx->d_pcd_xyz.p, n_points * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return HAF_OK;
}

extern "C" int haf_search_pcd(haf_ctx* ctx, const void* file_bytes, size_t n_bytes, const haf_request* reqs, int n_requests, haf_best* best,
                              haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top) {
    const float* d_xyz = nullptr;
    size_t n = 0;
    const int rc = haf_pcd_decode(ctx, file_bytes, n_bytes, &d_xyz, &n);
    if (rc != HAF_OK) return rc;
    return haf_search(ctx, d_xyz, n, 12, reqs, n_requests, best, best_per_request, graspseval, mask, heights, per_roll_top);
}

extern "C" int haf_search_batch_pcd(haf_ctx* ctx, const void* files, const size_t* file_offsets, int n_files, const haf_request* reqs,
                                    const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                    haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll) {
    if (!ctx) return HAF_ERR_ARG;
    if (!file_offsets || n_files < 1) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_pcd: bad arguments");
    std::vector<size_t> point_offsets(n_files + 1);
    const float* d_xyz = nullptr;
    const int rc = haf_pcd_decode_batch(ctx, files, file_offsets, n_files, &d_xyz, point_offsets.data());
    if (rc != HAF_OK) return rc;
    return haf_search_batch_requests(ctx, d_xyz, point_offsets.data(), n_files, reqs, request_offsets, best_per_cloud, best_per_request,
                                     per_roll_top, grasp_per_cloud, grasp_per_request, grasp_per_roll);
}

// Depth images -> packed xyz in ctx->d_pcd_xyz (hafpcdk::depth_project_kernel; the contract is in hafgpu.h).  Every image is
// checked on the host first; then one upload (host input), one parameter block and one launch over every non-empty image, no sync.
extern "C" int haf_depth_to_xyz_batch(haf_ctx* ctx, const void* data, const size_t* byte_offsets, int n_images, const haf_depth_image* images,
                                      const float** d_xyz, size_t* point_offsets) {
    if (!ctx) return HAF_ERR_ARG;
    if (!d_xyz || !byte_offsets || n_images < 1 || !images || !point_offsets) return ctx->fail(HAF_ERR_ARG, "haf_depth_to_xyz_batch: bad arguments");
    std::vector<size_t> pts(n_images + 1, 0);
    std::vector<hafpcdk::DepthImage> imgs;
    std::vector<unsigned> tile_begin(1, 0);
    std::vector<size_t> cuts;
    const size_t base = byte_offsets[0];
    for (int i = 0; i < n_images; i++) {
        const haf_depth_image& I = images[i];
        auto bad = [&](const char* what) { return ctx->fail(HAF_ERR_ARG, "depth image %d: %s", i, what); };
        if (I.width < 0 || I.width >= (1 << 24) || I.height < 0 || I.height >= (1 << 24)) return bad("width and height must lie in [0, 2^24)");
        if (I.encoding != HAF_DEPTH_U16 && I.encoding != HAF_DEPTH_F32) return bad("unknown encoding");
        const long long esz = I.encoding == HAF_DEPTH_U16 ? 2 : 4;
        if (I.step < (long long)I.width * esz || I.step % esz) return bad("step must be a multiple of the element size and at least width x element size");
        const unsigned long long span = byte_offsets[i + 1] - byte_offsets[i];
        if (byte_offsets[i + 1] < byte_offsets[i] || (I.height && (unsigned long long)I.step > span / (unsigned long long)I.height) ||
            (unsigned long long)I.height * (unsigned long long)I.step != span)
            return bad("the byte span must be height x step");
        if (!std::isfinite(I.fx) || !std::isfinite(I.fy) || !std::isfinite(I.cx) || !std::isfinite(I.cy) || I.fx == 0.0 || I.fy == 0.0)
            return bad("fx, fy, cx, cy must be finite and fx, fy nonzero");
        if (!(I.depth_scale >= 0.0f && I.depth_scale <= 1.0f)) return bad("depth_scale must lie in [0, 1]");
        if (I.has_pose != 0 && I.has_pose != 1) return bad("has_pose must be 0 or 1");
        if (I.has_pose)
            for (int k = 0; k < 16; k++)
                if (!std::isfinite(I.camera_to_base[k])) return bad("camera_to_base has a non-finite entry");
        if (I.reserved[0] || I.reserved[1] || I.reserved[2]) return bad("reserved fields must be 0");
        const unsigned long long npix = (unsigned long long)I.width * (unsigned long long)I.height;
        pts[i + 1] = pts[i] + npix;
        cuts.push_back(byte_offsets[i + 1] - base);
        if (npix == 0) continue;
        const unsigned long long tiles = (npix + HAF_DEPTH_TILE - 1) / HAF_DEPTH_TILE;
        if (tile_begin.back() + tiles > 0x7fffffffull) return bad("the batch has more than 2^31 tiles of pixels");
        hafpcdk::DepthImage d;
        memset(&d, 0, sizeof d);
        d.src = reinterpret_cast<const unsigned char*>(byte_offsets[i] - base);   // offset until the source is known
        d.step = (unsigned long long)I.step;
        d.n_pixels = npix;
        d.out_begin = pts[i];
        d.width = I.width;
        d.encoding = I.encoding;
        d.has_pose = I.has_pose;
        const float s = I.depth_scale != 0.0f ? I.depth_scale : (I.encoding == HAF_DEPTH_U16 ? 0.001f : 1.0f);
        d.s = s;
        d.kx = (float)((double)s / I.fx);
        d.ky = (float)((double)s / I.fy);
        d.cxf = (float)I.cx;
        d.cyf = (float)I.cy;
        for (int k = 0; k < 12; k++) d.m[k] = I.camera_to_base[k];
        imgs.push_back(d);
        tile_begin.push_back((unsigned)(tile_begin.back() + tiles));
    }
    const size_t bytes = byte_offsets[n_images] - base, total = pts[n_images];
    if (total > 0) {
        if (!data) return ctx->fail(HAF_ERR_ARG, "haf_depth_to_xyz_batch: data is null");
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        const unsigned char* src = reinterpret_cast<const unsigned char*>(data) + base;
        if (!is_device_ptr(data)) {
            ENSURE(ctx, ctx->d_pcd_raw, bytes + 16);
            const int rc = upload_host_bytes(ctx, ctx->d_pcd_raw.p, src, bytes, cuts);
            if (rc) return rc;
            src = ctx->d_pcd_raw.p;
        }
        ENSURE(ctx, ctx->d_pcd_xyz, total * 3);
        for (size_t k = 0; k < imgs.size(); k++) imgs[k].src = src + reinterpret_cast<size_t>(imgs[k].src);
        IngestParams P(ctx);
        const size_t o_imgs = P.add(imgs.size() * sizeof(hafpcdk::DepthImage)), o_tiles = P.add(tile_begin.size() * sizeof(unsigned));
        { const int rc = P.open(); if (rc) return rc; }
        memcpy(P.h<hafpcdk::DepthImage>(o_imgs), imgs.data(), imgs.size() * sizeof(hafpcdk::DepthImage));
        memcpy(P.h<unsigned>(o_tiles), tile_begin.data(), tile_begin.size() * sizeof(unsigned));
        { const int rc = P.send(); if (rc) return rc; }
        hafpcdk::depth_project_kernel<<<tile_begin.back(), HAF_DEPTH_THREADS, 0, ctx->stream>>>(P.d<hafpcdk::DepthImage>(o_imgs), P.d<unsigned>(o_tiles),
                                                                                              (int)imgs.size(), ctx->d_pcd_xyz.p);
        LAUNCHED(ctx);
    }
    for (int i = 0; i <= n_images; i++) point_offsets[i] = pts[i];
    *d_xyz = total ? ctx->d_pcd_xyz.p : nullptr;
    return HAF_OK;
}

extern "C" int haf_search_batch_depth(haf_ctx* ctx, const void* data, const size_t* byte_offsets, int n_images, const haf_depth_image* images,
                                      const haf_request* reqs, const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request,
                                      int* per_roll_top, haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll) {
    if (!ctx) return HAF_ERR_ARG;
    if (n_images < 1) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_depth: bad arguments");
    std::vector<size_t> point_offsets(n_images + 1);
    const float* d_xyz = nullptr;
    const int rc = haf_depth_to_xyz_batch(ctx, data, byte_offsets, n_images, images, &d_xyz, point_offsets.data());
    if (rc != HAF_OK) return rc;
    return haf_search_batch_requests(ctx, d_xyz, point_offsets.data(), n_images, reqs, request_offsets, best_per_cloud, best_per_request,
                                     per_roll_top, grasp_per_cloud, grasp_per_request, grasp_per_roll);
}

// ------------------------------------------------------------------------------------------------------------
// several GPUs behind one context (haf_config.n_devices > 1, SURVEY 8b / 8e)
// ------------------------------------------------------------------------------------------------------------
// A cloud given as a DEVICE pointer lives on one GPU: members on other GPUs get their own copy (UVA copy, peer or staged).
static int member_input(haf_ctx* m, const void* src, size_t bytes, const void** use) {
    *use = src;
    if (!bytes || !is_device_ptr(src)) return HAF_OK;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, src) != cudaSuccess) { cudaGetLastError(); return HAF_OK; }
    if (a.device == m->device) return HAF_OK;
    CUDA_TRY(m, cudaSetDevice(m->device));
    {   // NVLink / NVSwitch peer copy instead of a bounce through host memory (already enabled: fine)
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, m->device, a.device) == cudaSuccess && can) cudaDeviceEnablePeerAccess(a.device, 0);
        cudaGetLastError();
    }
    ENSURE(m, m->d_xdense, (bytes + 7) / 8);   // spare buffer of this context, otherwise used by the libsvm front end only
    CUDA_TRY(m, cudaMemcpy(m->d_xdense.p, src, bytes, cudaMemcpyDefault));
    *use = m->d_xdense.p;
    return HAF_OK;
}
static void group_timing(haf_ctx* ctx) {
    haf_timing t;
    memset(&t, 0, sizeof t);
    for (size_t k = 0; k < ctx->group.size(); k++) {
        const haf_timing& c = ctx->group[k]->timing;
        t.ms_total = std::max(t.ms_total, c.ms_total);   // the GPUs run concurrently
        t.ms_bin = std::max(t.ms_bin, c.ms_bin); t.ms_integral = std::max(t.ms_integral, c.ms_integral); t.ms_mask = std::max(t.ms_mask, c.ms_mask);
        t.ms_features = std::max(t.ms_features, c.ms_features); t.ms_svm = std::max(t.ms_svm, c.ms_svm); t.ms_guard = std::max(t.ms_guard, c.ms_guard);
        t.ms_score = std::max(t.ms_score, c.ms_score);
        t.n_points += c.n_points; t.n_units += c.n_units; t.n_windows += c.n_windows; t.n_guard += c.n_guard; t.launches += c.launches;
        t.n_chunks += c.n_chunks; t.n_exact += c.n_exact; t.n_audit += c.n_audit; t.n_clamped += c.n_clamped;
        t.audit_max_rel = std::max(t.audit_max_rel, c.audit_max_rel); t.tc_passes = std::max(t.tc_passes, c.tc_passes); t.escalations += c.escalations;
    }
    ctx->timing = t;
}

// One goal: the units (request, roll) -- independent until the per-roll tops exist (SURVEY 8e) -- go to the GPUs in contiguous
// blocks; every member evaluates its rolls of every request in one haf_search call (roll_begin / roll_limit) and writes the
// per-roll outputs straight into the caller's buffers; the tops are merged HERE with the loop rules of server.cpp:362-365 /
// :953-960 (strict >, earliest roll, early exit when return_only_best), so best / rolls_done / n_windows_scored equal the
// one-GPU result.  The only data that crosses GPUs is R x 3 ints per request.
static int group_search(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* reqs, int n_requests,
                        haf_best* best, haf_best* best_per_request, float* graspseval, unsigned char* mask, float* heights, int* per_roll_top,
                        const GraspOut* go) {
    if (!reqs || n_requests < 1 || !best) return ctx->fail(HAF_ERR_ARG, "haf_search: reqs, n_requests >= 1 and best are required");
    const int n = (int)ctx->group.size(), R = ctx->R;
    if (stride_bytes == 0) stride_bytes = 12;
    // rolls the one-GPU loop would evaluate per request
    std::vector<int> rb(n_requests), re(n_requests);
    std::vector<long long> ubeg(n_requests + 1, 0);
    for (int a = 0; a < n_requests; a++) {
        re[a] = reqs[a].roll_limit > 0 ? std::min(R, reqs[a].roll_limit) : R;
        rb[a] = std::max(0, std::min(reqs[a].roll_begin, re[a]));
        ubeg[a + 1] = ubeg[a] + (re[a] - rb[a]);
    }
    const long long U = ubeg[n_requests];
    // grasp poses with no roll to evaluate anywhere: no member would run, so the head builds the roll -1 poses on its own GPU
    if (go && U == 0)
        return search_single(ctx, xyz, n_points, stride_bytes, reqs, n_requests, best, best_per_request, graspseval, mask, heights, per_roll_top, go);
    std::vector<int> tops((size_t)n_requests * R * 3);
    std::vector<unsigned> uwin((size_t)n_requests * R, 0u);
    for (size_t u = 0; u < (size_t)n_requests * R; u++) { tops[3 * u] = -1; tops[3 * u + 1] = -1; tops[3 * u + 2] = -1000; }
    // grasp poses: every member returns the records of its own units (and, for a request with no roll on it, the roll -1 pose)
    std::vector<GraspRec> ugrasp(go ? (size_t)n_requests * R : 0), nograsp(go ? n_requests : 0);
    std::vector<int> rcs(n, HAF_OK);
    std::vector<long long> guards(n, 0);
    std::vector<std::thread> th;
    int first_member = -1;
    for (int k = 0; k < n; k++) {
        const long long u0 = U * k / n, u1 = U * (k + 1) / n;   // this GPU's block of the active units
        if (u1 <= u0) { memset(&ctx->group[k]->timing, 0, sizeof(haf_timing)); continue; }
        const bool report_nograsp = first_member < 0;   // one member reports the roll -1 poses
        if (first_member < 0) first_member = k;
        th.emplace_back([=, &rcs, &tops, &uwin, &guards, &rb, &re, &ubeg, &ugrasp, &nograsp]() {
            haf_ctx* m = ctx->group[k];
            std::vector<haf_request> rq(reqs, reqs + n_requests);
            for (int a = 0; a < n_requests; a++) {
                const long long b = std::max(u0, ubeg[a]), e = std::min(u1, ubeg[a + 1]);
                rq[a].return_only_best = 0;   // the early exit is replayed on the merged tops
                if (b < e) { rq[a].roll_begin = rb[a] + (int)(b - ubeg[a]); rq[a].roll_limit = rb[a] + (int)(e - ubeg[a]); }
                else { rq[a].roll_begin = R; rq[a].roll_limit = 0; }   // no roll of this request on this GPU
            }
            const void* use = xyz;
            int rc = member_input(m, xyz, n_points * stride_bytes, &use);
            std::vector<int> local((size_t)n_requests * R * 3);
            haf_best b0;
            std::vector<haf_best> bpr(n_requests);
            GraspOut mgo;
            mgo.units = true;
            if (rc == HAF_OK)
                rc = search_single(m, (const float*)use, n_points, stride_bytes, rq.data(), n_requests, &b0, bpr.data(), graspseval, mask, heights, local.data(),
                                   go ? &mgo : nullptr);
            rcs[k] = rc;
            if (rc != HAF_OK) return;
            guards[k] = m->timing.n_guard;
            for (int a = 0; a < n_requests; a++) {
                for (int roll = rq[a].roll_begin; roll < (rq[a].roll_limit > 0 ? rq[a].roll_limit : 0); roll++) {
                    const size_t u = (size_t)a * R + roll;
                    tops[3 * u] = local[3 * u]; tops[3 * u + 1] = local[3 * u + 1]; tops[3 * u + 2] = local[3 * u + 2];
                    uwin[u] = m->h_unit_windows.p[u];
                    if (go) ugrasp[u] = m->h_unit_grasp.p[u];
                }
                if (go && report_nograsp && re[a] <= rb[a]) nograsp[a] = m->h_job_grasp.p[a];   // this request has no roll anywhere
            }
        });
    }
    for (size_t i = 0; i < th.size(); i++) th[i].join();
    for (int k = 0; k < n; k++)
        if (rcs[k] != HAF_OK) { const std::string msg = ctx->group[k]->err; return ctx->fail(rcs[k], "GPU %d: %s", ctx->group[k]->device, msg.c_str()); }
    group_timing(ctx);
    long long n_guard = 0;
    for (int k = 0; k < n; k++) n_guard += guards[k];
    // merge: the reference's loop over rolls per request, then strict > over requests (earliest wins)
    int win = -1, wtop = -1000;
    std::vector<JobResult> res(n_requests);
    std::vector<Job> jobs(n_requests);
    for (int a = 0; a < n_requests; a++) {
        jobs[a].cloud = 0; jobs[a].rq = reqs[a];
        JobResult r; memset(&r, 0, sizeof r);
        r.row = r.col = r.roll = -1; r.topval = -1000;
        for (int roll = rb[a]; roll < re[a]; roll++) {
            if (reqs[a].return_only_best && r.topval >= reqs[a].graspval_top) break;   // :362-365
            const size_t u = (size_t)a * R + roll;
            if (tops[3 * u + 2] > r.topval) { r.topval = tops[3 * u + 2]; r.row = tops[3 * u]; r.col = tops[3 * u + 1]; r.roll = roll; }   // :953
            r.n_windows += (int)uwin[u];
            r.rolls_done++;
        }
        res[a] = r;
        if (best_per_request) fill_best(ctx, jobs[a], r, a, n_guard, &best_per_request[a]);
        if (r.topval > wtop) { wtop = r.topval; win = a; }
    }
    if (go) {   // the winning unit's record from whichever member owns it; eval as the one-GPU gather sets it (:390)
        std::vector<GraspRec> rec(n_requests);
        for (int a = 0; a < n_requests; a++) {
            rec[a] = res[a].roll >= 0 ? ugrasp[(size_t)a * R + res[a].roll] : nograsp[a];
            rec[a].eval = res[a].topval - 20;
        }
        if (go->best) memcpy(go->best, &rec[win < 0 ? 0 : win], sizeof(haf_grasp));
        if (go->per_job) memcpy(go->per_job, rec.data(), (size_t)n_requests * sizeof(haf_grasp));
        if (go->per_roll)
            for (int a = 0; a < n_requests; a++)
                for (int roll = rb[a]; roll < re[a]; roll++) memcpy(go->per_roll + (size_t)a * R + roll, &ugrasp[(size_t)a * R + roll], sizeof(haf_grasp));
    }
    if (per_roll_top) memcpy(per_roll_top, tops.data(), tops.size() * sizeof(int));
    if (win < 0) {
        JobResult none; memset(&none, 0, sizeof none);
        none.row = none.col = none.roll = -1; none.topval = -1000;
        fill_best(ctx, jobs[0], none, -1, n_guard, best);
    } else {
        fill_best(ctx, jobs[win], res[win], win, n_guard, best);
        long long nw = 0; int rd = 0;
        for (int a = 0; a < n_requests; a++) { nw += res[a].n_windows; rd += res[a].rolls_done; }
        best->n_windows_scored = (int)nw; best->rolls_done = rd;
    }
    return HAF_OK;
}

// Throughput mode: contiguous blocks of clouds per GPU, one host thread each, no cross-GPU data at all.
static int group_batch_packed(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* req,
                              haf_best* best_per_cloud, const GraspOut* go) {
    if (!point_offsets || n_clouds < 1 || !req || !best_per_cloud) return ctx->fail(HAF_ERR_ARG, "haf_search_batch_packed: bad arguments");
    const int n = (int)ctx->group.size();
    std::vector<int> rcs(n, HAF_OK);
    std::vector<std::thread> th;
    for (int k = 0; k < n; k++) {
        const int c0 = (int)((long long)n_clouds * k / n), c1 = (int)((long long)n_clouds * (k + 1) / n);
        if (c1 <= c0) { memset(&ctx->group[k]->timing, 0, sizeof(haf_timing)); continue; }
        th.emplace_back([=, &rcs]() {
            haf_ctx* m = ctx->group[k];
            std::vector<size_t> off(c1 - c0 + 1);
            for (int c = c0; c <= c1; c++) off[c - c0] = point_offsets[c] - point_offsets[c0];
            const float* src = xyz_all + point_offsets[c0] * 3;
            const void* use = src;
            GraspOut mgo;   // this member's clouds' records go straight to their place in the caller's arrays
            if (go) { mgo.per_job = go->per_job + c0; mgo.per_roll = go->per_roll ? go->per_roll + (size_t)c0 * ctx->R : nullptr; }
            int rc = member_input(m, src, off[c1 - c0] * 12, &use);
            if (rc == HAF_OK) rc = batch_packed_single(m, (const float*)use, off.data(), c1 - c0, req, best_per_cloud + c0, go ? &mgo : nullptr);
            rcs[k] = rc;
        });
    }
    for (size_t i = 0; i < th.size(); i++) th[i].join();
    for (int k = 0; k < n; k++)
        if (rcs[k] != HAF_OK) { const std::string msg = ctx->group[k]->err; return ctx->fail(rcs[k], "GPU %d: %s", ctx->group[k]->device, msg.c_str()); }
    group_timing(ctx);
    return HAF_OK;
}

// haf_search_batch_requests on several GPUs: contiguous blocks of clouds with all their requests, balanced by unit count
// (requests x R); each member writes its records straight into the caller's arrays.
static int group_batch_requests(haf_ctx* ctx, const float* xyz_all, const size_t* point_offsets, int n_clouds, const haf_request* reqs,
                                const int* request_offsets, haf_best* best_per_cloud, haf_best* best_per_request, int* per_roll_top,
                                haf_grasp* grasp_per_cloud, haf_grasp* grasp_per_request, haf_grasp* grasp_per_roll, const RankOut* rank) {
    const int n = (int)ctx->group.size(), R = ctx->R;
    const int* ro = request_offsets;
    std::vector<int> cb(n + 1, n_clouds);   // member k: clouds [cb[k], cb[k + 1])
    cb[0] = 0;
    for (int k = 1; k < n; k++)
        cb[k] = (int)(std::lower_bound(ro, ro + n_clouds, (int)((long long)ro[n_clouds] * k / n)) - ro);
    std::vector<int> rcs(n, HAF_OK);
    std::vector<std::thread> th;
    for (int k = 0; k < n; k++) {
        const int c0 = cb[k], c1 = cb[k + 1];
        if (c1 <= c0) { memset(&ctx->group[k]->timing, 0, sizeof(haf_timing)); continue; }
        th.emplace_back([=, &rcs]() {
            haf_ctx* m = ctx->group[k];
            std::vector<size_t> off(c1 - c0 + 1);
            std::vector<int> rof(c1 - c0 + 1);
            for (int c = c0; c <= c1; c++) { off[c - c0] = point_offsets[c] - point_offsets[c0]; rof[c - c0] = ro[c] - ro[c0]; }
            const size_t r0 = (size_t)ro[c0];
            const float* src = xyz_all + point_offsets[c0] * 3;
            const void* use = src;
            int rc = member_input(m, src, off[c1 - c0] * 12, &use);
            RankOut mro;   // this member's clouds' candidates go straight to their place in the caller's arrays
            if (rank) { mro = *rank; mro.candidates = rank->candidates + (size_t)c0 * rank->k; mro.n_candidates = rank->n_candidates + c0; }
            if (rc == HAF_OK)
                rc = batch_requests_single(m, (const float*)use, off.data(), c1 - c0, reqs + r0, rof.data(), best_per_cloud + c0,
                                           best_per_request ? best_per_request + r0 : nullptr, per_roll_top ? per_roll_top + r0 * R * 3 : nullptr,
                                           grasp_per_cloud ? grasp_per_cloud + c0 : nullptr, grasp_per_request ? grasp_per_request + r0 : nullptr,
                                           grasp_per_roll ? grasp_per_roll + r0 * R : nullptr, rank ? &mro : nullptr);
            rcs[k] = rc;
        });
    }
    for (size_t i = 0; i < th.size(); i++) th[i].join();
    for (int k = 0; k < n; k++)
        if (rcs[k] != HAF_OK) { const std::string msg = ctx->group[k]->err; return ctx->fail(rcs[k], "GPU %d: %s", ctx->group[k]->device, msg.c_str()); }
    group_timing(ctx);
    return HAF_OK;
}

// ------------------------------------------------------------------------------------------------------------
// parity / inspection entry points
// ------------------------------------------------------------------------------------------------------------
extern "C" int haf_debug_unit_params(haf_ctx* ctx, float* M, float* mask, float* Minv, int cap_units) {
    if (!ctx || cap_units < 0) return HAF_ERR_ARG;
    if (ctx->last_up_n <= 0) return ctx->fail(HAF_ERR_ARG, "haf_debug_unit_params: the context has no search to report");
    if (Minv && !ctx->last_up_pose) return ctx->fail(HAF_ERR_ARG, "haf_debug_unit_params: the last call built no grasp poses");
    const int U = std::min(cap_units, ctx->last_up_n), R = ctx->R;
    if (U == 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<UnitParams> up(U);
    CUDA_TRY(ctx, cudaMemcpy(up.data(), ctx->last_up_units, (size_t)U * sizeof(UnitParams), cudaMemcpyDeviceToHost));
    std::vector<int> jpose;
    std::vector<UnitPose> pose;
    if (Minv) {
        jpose.resize(ctx->last_up_jobs);
        CUDA_TRY(ctx, cudaMemcpy(jpose.data(), ctx->last_up_jpose, jpose.size() * sizeof(int), cudaMemcpyDeviceToHost));
        const int n_sets = *std::max_element(jpose.begin(), jpose.end()) + 1;
        pose.resize((size_t)n_sets * R);
        CUDA_TRY(ctx, cudaMemcpy(pose.data(), ctx->last_up_pose, pose.size() * sizeof(UnitPose), cudaMemcpyDeviceToHost));
    }
    static_assert(offsetof(UnitParams, cy4) - offsetof(UnitParams, sa) == 9 * sizeof(float), "mask constants are contiguous");
    for (int u = 0; u < U; u++) {
        if (M) memcpy(M + (size_t)u * 16, up[u].M, 16 * sizeof(float));
        if (mask) memcpy(mask + (size_t)u * 10, &up[u].sa, 10 * sizeof(float));
        if (Minv) memcpy(Minv + (size_t)u * 16, pose[(size_t)jpose[up[u].job] * R + up[u].roll].Minv, 16 * sizeof(float));
    }
    return U;
}

extern "C" int haf_debug_chunk_copy_waits(const haf_ctx* ctx, int* out, int cap_chunks) {
    if (!ctx || !out || cap_chunks < 0) return HAF_ERR_ARG;
    const int n = std::min(cap_chunks, (int)(ctx->last_chunk_waits.size() / HAF_CHUNK_RECORD));
    memcpy(out, ctx->last_chunk_waits.data(), (size_t)n * HAF_CHUNK_RECORD * sizeof(int));
    return n;
}

// the heights are decoded in place in d_keys by the integral kernels, so they stay there until the next search
extern "C" int haf_debug_heights(haf_ctx* ctx, float* heights, size_t cap_floats) {
    if (!ctx || !ctx->last_valid || !heights) return HAF_ERR_ARG;
    const size_t n = (size_t)ctx->last_units * ctx->G * ctx->G;
    if (cap_floats < n) return ctx->fail(HAF_ERR_ARG, "haf_debug_heights: buffer too small");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpy(heights, ctx->d_keys.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return ctx->last_units;
}

extern "C" int haf_debug_window_count(const haf_ctx* ctx) { return (ctx && ctx->last_valid) ? (int)ctx->last_W : -1; }

extern "C" int haf_debug_windows(haf_ctx* ctx, int* win_unit_cell, int cap) {
    if (!ctx || !ctx->last_valid) return HAF_ERR_ARG;
    const int W = std::min<int>(cap, (int)ctx->last_W);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpy(win_unit_cell, ctx->d_win.p, (size_t)W * sizeof(int2), cudaMemcpyDeviceToHost));
    return W;
}

extern "C" int haf_debug_features(haf_ctx* ctx, float* raw, double* scaled, int cap) {
    if (!ctx || !ctx->last_valid) return HAF_ERR_ARG;
    const int W = std::min<int>(cap, (int)ctx->last_W);
    if (W <= 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    float* d_raw = nullptr;
    double* d_scaled = nullptr;
    if (raw) CUDA_TRY(ctx, cudaMalloc(&d_raw, (size_t)ctx->last_W * ctx->F * sizeof(float)));
    if (scaled) CUDA_TRY(ctx, cudaMalloc(&d_scaled, (size_t)ctx->last_W * ctx->D * sizeof(double)));
    features_kernel<true><<<(ctx->last_W + 31) / 32, 256, 0, ctx->stream>>>(ctx->d_integral.p, ctx->d_win.p, ctx->d_counters.p + 0, ctx->G, ctx->last_unit_base,
                                                                           ctx->d_feats.p, ctx->d_dims.p, ctx->D, ctx->Kpad, ctx->lower, ctx->upper,
                                                                           ctx->cfg.emulate_text_roundtrip, nullptr, ctx->last_ldx, ctx->F, d_raw, d_scaled,
                                                                           (int*)(ctx->d_counters.p + 3));
    LAUNCHED(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (raw) { CUDA_TRY(ctx, cudaMemcpy(raw, d_raw, (size_t)W * ctx->F * sizeof(float), cudaMemcpyDeviceToHost)); cudaFree(d_raw); }
    if (scaled) { CUDA_TRY(ctx, cudaMemcpy(scaled, d_scaled, (size_t)W * ctx->D * sizeof(double), cudaMemcpyDeviceToHost)); cudaFree(d_scaled); }
    return W;
}

// tensor-core mode only: the SVM inputs as the contraction sees them, x_hi + x_lo as float, [W][n_dims]
extern "C" int haf_debug_tensor_inputs(haf_ctx* ctx, float* x, int cap) {
    if (!ctx || !ctx->last_valid || !x) return HAF_ERR_ARG;
    if (ctx->cfg.svm_mode != HAF_SVM_TENSOR_GUARD) return ctx->fail(HAF_ERR_ARG, "haf_debug_tensor_inputs: context is not in tensor mode");
    const int W = std::min<int>(cap, (int)ctx->last_W);
    if (W <= 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t nel = round_up((size_t)W, 128) * ctx->KB * haftc::BK;   // k-block tiled layout (kt_off)
    std::vector<uint16_t> hh(nel), ll(nel, 0);   // lo = 0 where the contraction reads hi only
    CUDA_TRY(ctx, cudaMemcpy(hh.data(), ctx->d_Xh.p, nel * 2, cudaMemcpyDeviceToHost));
    if (ctx->tc_passes >= 3) CUDA_TRY(ctx, cudaMemcpy(ll.data(), ctx->d_Xl.p, nel * 2, cudaMemcpyDeviceToHost));
    for (int w = 0; w < W; w++)
        for (int d = 0; d < ctx->D; d++) x[(size_t)w * ctx->D + d] = h16f(hh[kt_off((size_t)w, d, ctx->KB)]) + h16f(ll[kt_off((size_t)w, d, ctx->KB)]);
    return W;
}

extern "C" int haf_debug_decisions(haf_ctx* ctx, double* dec, int* labels, unsigned char* guard, int cap) {
    if (!ctx || !ctx->last_valid) return HAF_ERR_ARG;
    const int W = std::min<int>(cap, (int)ctx->last_W);
    if (W <= 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<double> hd(W);
    CUDA_TRY(ctx, cudaMemcpy(hd.data(), ctx->d_dec.p, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost));
    if (dec) memcpy(dec, hd.data(), (size_t)W * sizeof(double));
    if (labels) for (int w = 0; w < W; w++) labels[w] = hd[w] > 0 ? ctx->label[0] : ctx->label[1];
    if (guard) CUDA_TRY(ctx, cudaMemcpy(guard, ctx->d_guardflag.p, (size_t)W, cudaMemcpyDeviceToHost));
    return W;
}

extern "C" int haf_debug_integral(haf_ctx* ctx, float* integral, size_t cap_floats) {
    if (!ctx || !ctx->last_valid) return HAF_ERR_ARG;
    const size_t n = (size_t)ctx->last_units * (ctx->G + 1) * (ctx->G + 1);
    if (cap_floats < n) return ctx->fail(HAF_ERR_ARG, "haf_debug_integral: buffer too small");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpy(integral, ctx->d_integral.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return ctx->last_units;
}

extern "C" int haf_debug_cell_indices(haf_ctx* ctx, const float* xyz, size_t n_points, size_t stride_bytes, const haf_request* req, int roll,
                                      int* cell_idx_host) {
    if (!ctx || !req || !cell_idx_host || (!xyz && n_points)) return HAF_ERR_ARG;
    if (stride_bytes == 0) stride_bytes = 12;
    if (n_points == 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    ctx->last_valid = false;
    const int G = ctx->G;
    bool dev = false;
    int rc = stage_points(ctx, xyz, n_points * stride_bytes, &dev);
    if (rc) return rc;
    const unsigned char* dx = dev ? reinterpret_cast<const unsigned char*>(xyz) : ctx->d_xyz.p;
    UnitParams up;
    memset(&up, 0, sizeof up);
    float M[16];
    hafhost::build_transform(*req, roll, ctx->cfg.roll_step_deg, M);
    memcpy(up.M, M, 12 * sizeof(float));
    up.cloud = 0;
    long long off[2] = {0, (long long)n_points};
    int ub[2] = {0, 1};
    ENSURE(ctx, ctx->d_units, 1); ENSURE(ctx, ctx->d_ptoff, 2); ENSURE(ctx, ctx->d_cloud_ubegin, 2); ENSURE(ctx, ctx->d_keys, (size_t)G * G);
    int* d_cells = nullptr;
    CUDA_TRY(ctx, cudaMalloc(&d_cells, n_points * sizeof(int)));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_units.p, &up, sizeof up, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_ptoff.p, off, sizeof off, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_cloud_ubegin.p, ub, sizeof ub, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));  // the staged host arrays live on this stack frame
    fill_u32_kernel<<<64, 256, 0, ctx->stream>>>(ctx->d_keys.p, (size_t)G * G, HAF_KEY_MINUS_ONE);
    LAUNCHED(ctx);
    const float r = (float)((0.5 * (float)G) / 100.0);
    bin_maxz_kernel<4><<<dim3((unsigned)((n_points + 1023) / 1024), 1), 256, 0, ctx->stream>>>(dx, stride_bytes, ctx->d_ptoff.p, ctx->d_cloud_ubegin.p, ctx->d_units.p,
                                                                                            ctx->d_keys.p, G, r, d_cells,
                                                                                            reinterpret_cast<unsigned long long*>(ctx->d_counters.p + 4), 0, 1);
    LAUNCHED(ctx);
    CUDA_TRY(ctx, cudaMemcpyAsync(cell_idx_host, d_cells, n_points * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(d_cells);
    return (int)std::min<size_t>(n_points, 0x7fffffff);
}

// cycle counters of the last svm_rbf_tc3_kernel launch run with HAF_TC_DEBUG bit 5 (svm_tc.cuh, g_tc_probe): [n_ctas][16]
extern "C" int haf_debug_tc_probe(haf_ctx* ctx, unsigned long long* out, int n_ctas) {
    if (!ctx || !out || n_ctas < 1 || n_ctas > 160) return HAF_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaDeviceSynchronize());
    CUDA_TRY(ctx, cudaMemcpyFromSymbol(out, haftc::g_tc_probe, (size_t)n_ctas * 16 * sizeof(unsigned long long)));
    return HAF_OK;
}

extern "C" int haf_debug_text_roundtrip(haf_ctx* ctx, const float* in4, int n4, double* out4, const double* in6, int n6, double* out6) {
    if (!ctx) return HAF_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    float* d4 = nullptr; double *o4 = nullptr, *d6 = nullptr, *o6 = nullptr;
    if (n4 > 0) { CUDA_TRY(ctx, cudaMalloc(&d4, n4 * sizeof(float))); CUDA_TRY(ctx, cudaMalloc(&o4, n4 * sizeof(double))); CUDA_TRY(ctx, cudaMemcpy(d4, in4, n4 * sizeof(float), cudaMemcpyHostToDevice)); }
    if (n6 > 0) { CUDA_TRY(ctx, cudaMalloc(&d6, n6 * sizeof(double))); CUDA_TRY(ctx, cudaMalloc(&o6, n6 * sizeof(double))); CUDA_TRY(ctx, cudaMemcpy(d6, in6, n6 * sizeof(double), cudaMemcpyHostToDevice)); }
    const int n = std::max(n4, n6);
    if (n > 0) {
        text_roundtrip_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d4, n4, o4, d6, n6, o6);
        LAUNCHED(ctx);
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (n4 > 0) { CUDA_TRY(ctx, cudaMemcpy(out4, o4, n4 * sizeof(double), cudaMemcpyDeviceToHost)); cudaFree(d4); cudaFree(o4); }
    if (n6 > 0) { CUDA_TRY(ctx, cudaMemcpy(out6, o6, n6 * sizeof(double), cudaMemcpyDeviceToHost)); cudaFree(d6); cudaFree(o6); }
    return HAF_OK;
}
