// kernels.cuh -- hand-written sm_100a kernels of the grasp-search path.  Compiled with -fmad=false: every
// FP32/FP64 operation whose bit pattern is part of the reference's result is written with the _rn
// intrinsics (no FMA contraction, fixed association); FMA is used explicitly only in the SVM contraction.
//
// Data layout in HBM (G = grid side, U = units = (job, roll) pairs of the chunk in flight):
//   grid_keys / heights  [U][G][G]      u32 ordered keys during binning, decoded in place to f32 heights
//   integral             [U][G+1][G+1]  f32
//   mask                 [U][G][G]      u8        labelgrid [U][G][G] i8 (graspsgrid: -1 = not evaluated)
//   evals                [U][G][G]      f32 (graspseval)
//   win                  [Wcap]         int2 (unit, cell)      compact list of valid windows, any order
//   X                    [Kpad][ldx]    f32 feature-major SVM inputs (dimension d of window w at X[d*ldx+w])
//   svT                  [Kpad][Spad]   f32 feature-major support vectors;  sv64T [D][Spad] f64 for the exact path
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "decimal_round.cuh"
#include "haf_host.hpp"

namespace hafk {

struct UnitParams {      // one (job, roll): 128 bytes
    float M[16];         // mat_transform (row-major); the kernels read rows 0..2, row 3 is kept for haf_best.M
    float sa, ca;        // sinf/cosf(alpha) of pnt_in_box, from the host libm
    float cx1, cy1, cx2, cy2, cx3, cy3, cx4, cy4;
    int cloud;           // cloud index of this unit, -1 = inactive (roll >= roll_limit)
    int job;
    int roll;
    int pad[3];
};
static_assert(sizeof(UnitParams) == 128, "UnitParams layout");

struct __align__(16) FeatDev {  // one feature of data/Features.txt, 64 bytes
    int off[12];         // 3 effective regions x 4 corner offsets into the integral image (row stride G+1):
                         //   [4r+0] (x2+1,y2+1)  [4r+1] (x1,y2+1)  [4r+2] (x2+1,y1)  [4r+3] (x1,y1)
    float w[3];
    int flags;           // bit r: region r active; bit 8: SHAF feature (index >= nr_features_without_shaf)
};
struct __align__(16) DimDev {   // one SVM input dimension (libsvm index d+1), 48 bytes; the fast tier reads the first 32
    double fmin;         // svm-scale feature_min
    double slope;        // (upper - lower) / den, used by the fast (non bit-exact) tier only
    int feat;            // feature index feeding this dimension; -1 = constant cval
    int drop;            // 1: svm-scale skips it (single-valued attribute) -> 0
    double cval;         // value when the dimension is constant (feat < 0)
    double fmax, den;    // den = fmax - fmin
};
static_assert(sizeof(DimDev) == 48, "DimDev layout");

// ---------------------------------------------------------------------------------------------------
// ordered-key float max: key(a) > key(b)  <=>  a > b   (for non-NaN floats)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned fkey(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
#define HAF_KEY_MINUS_ONE 0x407FFFFFu  // fkey(-1.0f): the reference's initial cell value (server.cpp:499-501)

__global__ void fill_u32_kernel(unsigned* __restrict__ p, size_t n, unsigned v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}

// ---------------------------------------------------------------------------------------------------
// a2 + a3: transform + binning with per-cell atomic max-z, all rolls / approach vectors of a cloud fused:
// each point is read ONCE and scattered into every unit grid of its cloud.   (server.cpp:487-520)
// grid = (ceil(max_points / (blockDim*PPT)), n_clouds).  Only the units in [u_lo, u_hi) are binned: a chunk of a batch with
// several requests per cloud may hold part of a cloud's units.
// ---------------------------------------------------------------------------------------------------
// Measured on B200 (profiles/README.md): keeping the points in registers with the unit loop outermost, and a
// read-before-atomic filter, were both SLOWER than this point-outer / fire-and-forget RED form (3.3 / 3.7 vs 2.5 ms).
#define HAF_BIN_MAXU 64
template <int PPT>
__global__ void __launch_bounds__(256) bin_maxz_kernel(const unsigned char* __restrict__ xyz, size_t stride_bytes,
                                                       const long long* __restrict__ pt_off,
                                                       const int* __restrict__ cloud_unit_begin,
                                                       const UnitParams* __restrict__ units,
                                                       unsigned* __restrict__ grid_keys, int G, float r,
                                                       int* __restrict__ cell_idx_out /*debug: [n] or NULL*/,
                                                       unsigned long long* __restrict__ clamp_count, int u_lo, int u_hi) {
    const int c = blockIdx.y;
    const long long p0 = pt_off[c], p1 = pt_off[c + 1];
    const long long first = p0 + (long long)blockIdx.x * (blockDim.x * PPT);
    if (first >= p1) return;
    const int ub = max(cloud_unit_begin[c], u_lo), ue = min(cloud_unit_begin[c + 1], u_hi);   // [u_lo, u_hi): the chunk's units
    __shared__ float sM[HAF_BIN_MAXU][12];
    __shared__ int sActive[HAF_BIN_MAXU];
    const float nr = -r;
    const size_t GG = (size_t)G * G;
    for (int u0 = ub; u0 < ue; u0 += HAF_BIN_MAXU) {
        const int nu = min(HAF_BIN_MAXU, ue - u0);
        __syncthreads();
        for (int t = threadIdx.x; t < nu * 12; t += blockDim.x) sM[t / 12][t % 12] = units[u0 + t / 12].M[t % 12];
        for (int t = threadIdx.x; t < nu; t += blockDim.x) sActive[t] = units[u0 + t].cloud >= 0;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PPT; k++) {
            const long long p = first + (long long)k * blockDim.x + threadIdx.x;
            if (p >= p1) break;
            const float* q = reinterpret_cast<const float*>(xyz + (size_t)p * stride_bytes);
            const float x = __ldg(q), y = __ldg(q + 1), z = __ldg(q + 2);
            for (int u = 0; u < nu; u++) {
                if (!sActive[u]) continue;
                const float* m = sM[u];
                // pcl::transformPointCloud, left-to-right float arithmetic, no FMA (server.cpp:488)
                const float tx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fmul_rn(m[2], z)), m[3]);
                const float ty = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[4], x), __fmul_rn(m[5], y)), __fmul_rn(m[6], z)), m[7]);
                int cell = -1;
                if (tx > nr && tx < r && ty > nr && ty < r) {  // strict (server.cpp:510-511); false for NaN
                    int ix = (int)floorf(__fmul_rn(100.0f, __fadd_rn(tx, r)));  // :513   x - (-r) == x + r
                    int iy = (int)floorf(__fmul_rn(100.0f, __fadd_rn(ty, r)));  // :514
                    if (ix < 0 || ix > G - 1 || iy < 0 || iy > G - 1) {  // impossible at G = 56; defined as clamp otherwise
                        atomicAdd(clamp_count, 1ull);
                        ix = max(0, min(G - 1, ix));
                        iy = max(0, min(G - 1, iy));
                    }
                    cell = ix * G + iy;  // x is the ROW index (:515)
                    const float tz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[8], x), __fmul_rn(m[9], y)), __fmul_rn(m[10], z)), m[11]);
                    if (tz > -1.0f)  // `grid < z` with grid >= -1: NaN and z <= -1 never register (:515-518)
                        atomicMax(grid_keys + (size_t)(u0 + u) * GG + cell, fkey(tz));
                }
                if (cell_idx_out) cell_idx_out[(size_t)(p - p0)] = cell;  // debug: single-unit launches only
            }
        }
    }
}

// Small-grid variant: one CTA walks a whole cloud and keeps, per unit grid, a shared-memory array of LOWER BOUNDS of the
// cell maxima.  The binning is bound by the issue rate of scattered REDG (~0.75 lanes/clk/SM, profiles/); a point whose
// key does not beat the bound cannot change the global cell and skips its RED.  The bound is maintained with plain
// (racy) shared loads/stores: whatever value survives a race was also sent to global memory by its writer, so it never
// exceeds the true maximum and skipping stays safe; with ~30 points per cell only the few running maxima reach L2.
// grid = (n_clouds, unit groups, slices of the cloud), block = 1024, dynamic smem = units_per_group * G * G * 4 bytes.
//
// Round 2 (the kernel was instruction-bound: ~75 instructions per (point, unit), ncu issue slots 86 %):
//   * z row hoisted: rows 0-1 of mat_transform change with the roll, row 2 does not (S * Rroll leaves row 2 = (0, 0, 1, 0)
//     of the approach-vector transform untouched), so the transformed z of a point is computed once per run of units whose
//     row 2 is BITWISE the same as the previous unit's (checked here on the staged matrices, not assumed);
//   * VEC = 4 points per thread, fetched as three 128-bit loads where the slice is 16-byte aligned (packed xyz, stride 12):
//     the unit loop is outermost per group of four points, so each unit's matrix rows are read from shared memory once per
//     four points instead of once per point.
// Round 2, second pass (ncu source view: 66 warp instructions per (point, unit), 15 % of them BSSY / BSYNC / BRA around the
// three nested `if`s, 6 % the ordered key recomputed per unit): the per-point z work -- transformed z, its ordered key and the
// `grid < z` test -- happens once per run of units sharing row 2, and the per-(point, unit) body is straight-line code with
// ONE predicated tail (shared-memory bound update + RED); the index clamp is a rarely taken, almost always uniform branch.
template <int VEC>
__device__ __forceinline__ void bin_points_into_units(const float (&x)[VEC], const float (&y)[VEC], const float (&z)[VEC], int npts, int nu, int GG, int G,
                                                      float r, const float (*sM)[12], const int* sFlags, unsigned* s_bound,
                                                      unsigned* __restrict__ gk /*keys of unit ub*/, unsigned long long* __restrict__ clamp_count) {
    unsigned keyz[VEC];   // ordered key of the transformed z; 0 = the point cannot register (`grid < z` with grid >= -1: z <= -1 or NaN, :515-518)
#pragma unroll
    for (int k = 0; k < VEC; k++) keyz[k] = 0u;
    const int Gm1 = G - 1;
    const uint32_t sb0 = (uint32_t)__cvta_generic_to_shared(s_bound);
    for (int u = 0; u < nu; u++) {
        const int fl = sFlags[u];
        if (fl & 2) {   // row 2 differs from the previous unit's (always true for the first unit)
            const float4 m2 = *reinterpret_cast<const float4*>(sM[u] + 8);
#pragma unroll
            for (int k = 0; k < VEC; k++) {
                const float tz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m2.x, x[k]), __fmul_rn(m2.y, y[k])), __fmul_rn(m2.z, z[k])), m2.w);
                keyz[k] = (k < npts && tz > -1.0f) ? fkey(tz) : 0u;
            }
        }
        if (!(fl & 1)) continue;   // inactive unit (roll outside [roll_begin, roll_limit))
        const float4 m0 = *reinterpret_cast<const float4*>(sM[u]), m1 = *reinterpret_cast<const float4*>(sM[u] + 4);
        const uint32_t sbu = sb0 + (uint32_t)(u * GG) * 4u;
        unsigned* gku = gk + (size_t)u * GG;
#pragma unroll
        for (int k = 0; k < VEC; k++) {
            // pcl::transformPointCloud, left-to-right float arithmetic, no FMA (server.cpp:488)
            const float tx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m0.x, x[k]), __fmul_rn(m0.y, y[k])), __fmul_rn(m0.z, z[k])), m0.w);
            const float ty = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m1.x, x[k]), __fmul_rn(m1.y, y[k])), __fmul_rn(m1.z, z[k])), m1.w);
            // -r < t < r  <=>  |t| < r, exactly (both false for NaN): strict (server.cpp:510-511)
            const bool inbox = fabsf(tx) < r && fabsf(ty) < r;
            const bool in = inbox && keyz[k] != 0u;
            int ix = __float2int_rd(__fmul_rn(100.0f, __fadd_rn(tx, r)));  // :513  (int)floorf(.)
            int iy = __float2int_rd(__fmul_rn(100.0f, __fadd_rn(ty, r)));  // :514
            // t > -r makes t + r >= 0, so an index of a point inside cannot be negative; rounding can push one to G (t just below r).
            // Counted whatever its z, as the reference and bin_maxz_kernel count it: the clamp precedes the height test (:513-518)
            if (inbox && max(ix, iy) > Gm1) atomicAdd(clamp_count, 1ull);
            ix = min(max(ix, 0), Gm1);
            iy = min(max(iy, 0), Gm1);
            const int cell = ix * G + iy;
            unsigned lb;
            asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(lb) : "r"(sbu + (uint32_t)cell * 4u));
            if (in && keyz[k] > lb) {
                asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(sbu + (uint32_t)cell * 4u), "r"(keyz[k]) : "memory");
                atomicMax(gku + cell, keyz[k]);
            }
        }
    }
}
template <int VEC>
__global__ void __launch_bounds__(1024, 1) bin_maxz_cloud_kernel(const unsigned char* __restrict__ xyz, size_t stride_bytes,
                                                                 const long long* __restrict__ pt_off,
                                                                 const int* __restrict__ cloud_unit_begin,
                                                                 const UnitParams* __restrict__ units,
                                                                 unsigned* __restrict__ grid_keys, int G, float r, int units_per_group,
                                                                 unsigned long long* __restrict__ clamp_count, int u_lo, int u_hi) {
    extern __shared__ unsigned s_bound[];  // [units_per_group][G*G]
    __shared__ __align__(16) float sM[16][12];
    __shared__ int sFlags[16];             // bit 0: unit active; bit 1: row 2 of M differs bitwise from the previous unit's
    const int c = blockIdx.x;
    long long p0 = pt_off[c], p1 = pt_off[c + 1];
    {   // blockIdx.z: contiguous slice of the cloud (several CTAs per cloud when there are few clouds)
        const long long per = (p1 - p0 + gridDim.z - 1) / gridDim.z;
        p0 = p0 + per * blockIdx.z;
        p1 = min(p1, p0 + per);
    }
    const int ub = max(cloud_unit_begin[c], u_lo) + blockIdx.y * units_per_group;   // [u_lo, u_hi): as bin_maxz_kernel
    const int ue = min(min(cloud_unit_begin[c + 1], u_hi), ub + units_per_group);
    if (ub >= ue || p0 >= p1) return;
    const int nu = ue - ub, GG = G * G;
    for (int t = threadIdx.x; t < nu * GG; t += blockDim.x) s_bound[t] = HAF_KEY_MINUS_ONE;
    for (int t = threadIdx.x; t < nu * 12; t += blockDim.x) sM[t / 12][t % 12] = units[ub + t / 12].M[t % 12];
    __syncthreads();
    for (int t = threadIdx.x; t < nu; t += blockDim.x) {
        bool diff = t == 0;
        if (t > 0)
            for (int k = 8; k < 12; k++) diff = diff || (__float_as_uint(sM[t][k]) != __float_as_uint(sM[t - 1][k]));
        sFlags[t] = (units[ub + t].cloud >= 0 ? 1 : 0) | (diff ? 2 : 0);
    }
    __syncthreads();
    unsigned* gk = grid_keys + (size_t)ub * GG;
    if (VEC == 4 && stride_bytes == 12) {
        // head: points up to the first 16-byte aligned one; body: groups of four points = three 128-bit loads; tail: the rest
        const unsigned char* base = xyz + (size_t)p0 * 12;
        long long head = 0;
        while (head < p1 - p0 && ((reinterpret_cast<uintptr_t>(base) + (size_t)head * 12) & 15)) head++;   // <= 3
        const long long ngroups = (p1 - p0 - head) / 4;
        const float4* q4 = reinterpret_cast<const float4*>(base + (size_t)head * 12);
        for (long long g = threadIdx.x; g < ngroups; g += blockDim.x) {
            const float4 a = __ldg(q4 + 3 * g), b = __ldg(q4 + 3 * g + 1), d = __ldg(q4 + 3 * g + 2);
            const float x[4] = {a.x, a.w, b.z, d.y}, y[4] = {a.y, b.x, b.w, d.z}, z[4] = {a.z, b.y, d.x, d.w};
            bin_points_into_units<4>(x, y, z, 4, nu, GG, G, r, sM, sFlags, s_bound, gk, clamp_count);
        }
        const long long ntail = (p1 - p0) - ngroups * 4;   // head + tail points, one per thread
        if (threadIdx.x < ntail) {
            const long long p = threadIdx.x < head ? p0 + threadIdx.x : p0 + head + ngroups * 4 + (threadIdx.x - head);
            const float* q = reinterpret_cast<const float*>(xyz + (size_t)p * 12);
            const float x[1] = {__ldg(q)}, y[1] = {__ldg(q + 1)}, z[1] = {__ldg(q + 2)};
            bin_points_into_units<1>(x, y, z, 1, nu, GG, G, r, sM, sFlags, s_bound, gk, clamp_count);
        }
    } else {
        for (long long p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
            const float* q = reinterpret_cast<const float*>(xyz + (size_t)p * stride_bytes);
            const float x[1] = {__ldg(q)}, y[1] = {__ldg(q + 1)}, z[1] = {__ldg(q + 2)};
            bin_points_into_units<1>(x, y, z, 1, nu, GG, G, r, sM, sFlags, s_bound, gk, clamp_count);
        }
    }
}

// decode a key to the final height: cells never hit stay -1 -> "< -0.99 -> 0" (server.cpp:522-528, compare in double)
__device__ __forceinline__ float key_to_height(unsigned k) {
    float h = fkey_inv(k);
    return ((double)h < -0.99) ? 0.0f : h;
}

// ---------------------------------------------------------------------------------------------------
// a4: integral image, cv::integral(CV_64F) order exactly: per row a sequential double running sum s,
// I[y+1][x+1] = I[y][x+1] + s, accumulated top to bottom; cast to float at the end (server.cpp:586-601).
// Small-G variant: one CTA per unit, the whole G x G double tile in shared memory.
//   phase 1: thread t < G walks row t left to right;  phase 2: thread t < G walks column t top to bottom.
// Also decodes the bin keys in place into float heights.
// ---------------------------------------------------------------------------------------------------
__global__ void integral_small_kernel(unsigned* __restrict__ keys_heights, float* __restrict__ integral, int G,
                                      const UnitParams* __restrict__ units) {
    extern __shared__ double sP[];  // [G][G+1]
    const int u = blockIdx.x;
    if (units[u].cloud < 0) return;
    const int ld = G + 1;
    unsigned* kh = keys_heights + (size_t)u * G * G;
    float* I = integral + (size_t)u * ld * ld;
    for (int t = threadIdx.x; t < G * G; t += blockDim.x) {
        float h = key_to_height(kh[t]);
        kh[t] = __float_as_uint(h);
        sP[(t / G) * ld + (t % G)] = (double)h;
    }
    for (int t = threadIdx.x; t < ld; t += blockDim.x) { I[t] = 0.0f; I[(size_t)t * ld] = 0.0f; }
    __syncthreads();
    for (int row = threadIdx.x; row < G; row += blockDim.x) {
        double s = 0.0;
        double* p = sP + row * ld;
        for (int x = 0; x < G; x++) { s = __dadd_rn(s, p[x]); p[x] = s; }
    }
    __syncthreads();
    for (int col = threadIdx.x; col < G; col += blockDim.x) {
        double acc = 0.0;
        for (int y = 0; y < G; y++) {
            acc = __dadd_rn(acc, sP[y * ld + col]);
            I[(size_t)(y + 1) * ld + (col + 1)] = (float)acc;
        }
    }
}

// Large-G variant, pass 1: row prefix sums.  One warp per band of 32 rows (lane = row); 32x32 tiles are
// staged through shared memory so global loads/stores stay coalesced.  P: [U][G][G] double scratch.
__global__ void __launch_bounds__(32) integral_rows_kernel(unsigned* __restrict__ keys_heights, double* __restrict__ P,
                                                           int G, const UnitParams* __restrict__ units) {
    const int u = blockIdx.y;
    if (units[u].cloud < 0) return;
    const int row0 = blockIdx.x * 32;
    const int lane = threadIdx.x;
    __shared__ double tile[32][33];
    unsigned* kh = keys_heights + (size_t)u * G * G;
    double* Pu = P + (size_t)u * G * G;
    double s = 0.0;  // running sum of row (row0 + lane)
    for (int c0 = 0; c0 < G; c0 += 32) {
        for (int rr = 0; rr < 32; rr++) {  // coalesced: lane = column
            int row = row0 + rr, col = c0 + lane;
            double v = 0.0;
            if (row < G && col < G) {
                float h = key_to_height(kh[(size_t)row * G + col]);
                kh[(size_t)row * G + col] = __float_as_uint(h);
                v = (double)h;
            }
            tile[rr][lane] = v;
        }
        __syncwarp();
        for (int cc = 0; cc < 32; cc++) {  // lane = row: sequential left-to-right accumulation
            if (c0 + cc < G) { s = __dadd_rn(s, tile[lane][cc]); tile[lane][cc] = s; }
        }
        __syncwarp();
        for (int rr = 0; rr < 32; rr++) {
            int row = row0 + rr, col = c0 + lane;
            if (row < G && col < G) Pu[(size_t)row * G + col] = tile[rr][lane];
        }
        __syncwarp();
    }
}
// pass 2: thread = column, sequential top-to-bottom accumulation (loads independent of the chain -> unrolled)
__global__ void integral_cols_kernel(const double* __restrict__ P, float* __restrict__ integral, int G,
                                     const UnitParams* __restrict__ units) {
    const int u = blockIdx.y;
    if (units[u].cloud < 0) return;
    const int col = blockIdx.x * blockDim.x + threadIdx.x;  // 0..G  (column index of the integral image)
    const int ld = G + 1;
    if (col > G) return;
    float* I = integral + (size_t)u * ld * ld;
    I[col] = 0.0f;
    if (col == 0) {
        for (int y = 1; y <= G; y++) I[(size_t)y * ld] = 0.0f;
        return;
    }
    const double* Pu = P + (size_t)u * G * G + (col - 1);
    double acc = 0.0;
    int y = 0;
    for (; y + 8 <= G; y += 8) {
        double v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = Pu[(size_t)(y + k) * G];
#pragma unroll
        for (int k = 0; k < 8; k++) { acc = __dadd_rn(acc, v[k]); I[(size_t)(y + k + 1) * ld + col] = (float)acc; }
    }
    for (; y < G; y++) { acc = __dadd_rn(acc, Pu[(size_t)y * G]); I[(size_t)(y + 1) * ld + col] = (float)acc; }
}

// ---------------------------------------------------------------------------------------------------
// a5: valid-window mask (pnt_in_box, server.cpp:666-749) + compaction of the valid windows into `win`.
// Each CTA covers 256*16 consecutive cells of one unit; windows are appended in row-major order within
// the CTA's span with ONE global atomic per CTA.  Also initialises labelgrid to -1 (server.cpp:828-829).
// grid = (ceil(G*G / 4096), U)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_windows_kernel(const float* __restrict__ integral,
                                                           const UnitParams* __restrict__ units, int G,
                                                           unsigned char* __restrict__ mask,
                                                           signed char* __restrict__ labelgrid,
                                                           int2* __restrict__ win, unsigned* __restrict__ win_count,
                                                           unsigned win_cap, int* __restrict__ overflow_flag,
                                                           int unit_base, unsigned* __restrict__ unit_windows) {
    const int u = blockIdx.y;
    const UnitParams up = units[u];
    const int GG = G * G, ld = G + 1;
    const int cell0 = blockIdx.x * 4096;
    const float* I = integral + (size_t)u * ld * ld;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ unsigned s_cnt[16][8];
    __shared__ unsigned s_off[16][8];
    __shared__ unsigned s_base;
    unsigned ballots[16];
    const float nsa = -up.sa;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int cell = cell0 + k * 256 + threadIdx.x;
        bool in = false;
        if (cell < GG && up.cloud >= 0) {
            const int i = cell / G, j = cell - i * G;
            if (i > 6 && i < G - 7 && j > 6 && j < G - 7) {  // :713
                // :714-717  float, left to right:  ((I[i+4][j+4] - I[i-5][j+4]) - I[i+4][j-5]) + I[i-5][j-5]
                const float d = __fadd_rn(__fsub_rn(__fsub_rn(I[(i + 4) * ld + (j + 4)], I[(i - 5) * ld + (j + 4)]), I[(i + 4) * ld + (j - 5)]), I[(i - 5) * ld + (j - 5)]);
                if (d > 0.03f) {
                    const float fj = (float)j, fi = (float)i;
                    const float t1 = __fadd_rn(__fmul_rn(nsa, __fadd_rn(-up.cx1, fj)), __fmul_rn(up.ca, __fadd_rn(-up.cy1, fi)));    // :718
                    const float t2 = __fadd_rn(__fmul_rn(nsa, __fadd_rn(-up.cx2, fj)), __fmul_rn(up.ca, __fadd_rn(-up.cy2, fi)));    // :719
                    const float t3 = __fadd_rn(__fmul_rn(up.ca, __fadd_rn(-up.cx3, fj)), __fmul_rn(up.sa, __fadd_rn(-up.cy3, fi)));  // :720
                    const float t4 = __fadd_rn(__fmul_rn(up.ca, __fadd_rn(-up.cx4, fj)), __fmul_rn(up.sa, __fadd_rn(-up.cy4, fi)));  // :721
                    in = ((double)t1 < 0.00001) && ((double)t2 > -0.00001) && ((double)t3 > -0.00001) && ((double)t4 < 0.00001);
                }
            }
            mask[(size_t)u * GG + cell] = in ? 1 : 0;
            labelgrid[(size_t)u * GG + cell] = -1;
        }
        ballots[k] = __ballot_sync(0xffffffffu, in);
        if (lane == 0) s_cnt[k][warp] = __popc(ballots[k]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // 128-entry exclusive scan in (k, warp) order == ascending cell order
        unsigned run = 0;
        for (int k = 0; k < 16; k++)
            for (int w = 0; w < 8; w++) { s_off[k][w] = run; run += s_cnt[k][w]; }
        unsigned base = run ? atomicAdd(win_count, run) : 0u;
        // overflow (an internal bound bug: window_bound() is an upper bound): the CTA takes its addition back, so that
        // *win_count never ends above win_cap -- every consumer indexes its buffers with it -- and the call fails on the flag.
        // (While an overflowing addition is in place the counter is > win_cap, so later CTAs fail as well: the successful
        // spans stay a contiguous prefix.)
        if (base + run > win_cap) { *overflow_flag = 1; atomicSub(win_count, run); base = 0xFFFFFFFFu; }
        else if (run) atomicAdd(unit_windows + u, run);   // windows of this unit (n_windows_scored); one atomic per CTA
        s_base = base;
    }
    __syncthreads();
    const unsigned base = s_base;
    if (base == 0xFFFFFFFFu) return;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        if (ballots[k] & (1u << lane)) {
            const unsigned pos = base + s_off[k][warp] + __popc(ballots[k] & ((1u << lane) - 1u));
            win[pos] = make_int2(unit_base + u, cell0 + k * 256 + threadIdx.x);
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// a7 + a8 + a9: one SVM input dimension of one window: Haar / SHAF feature value in the reference's float
// order (calc_featurevalue, II2FV.cpp:141-199), "%.4g" round trip, svm-scale output() in double
// (svm-scale.c:333-353), "%g" round trip.  P points at I[row-7][col-7] of the window's integral image.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float rect_sum(const float* __restrict__ P, const int* off) {
    // ((P[x2+1][y2+1] - P[x1][y2+1]) - P[x2+1][y1]) + P[x1][y1]     (II2FV.cpp:161-162)
    return __fadd_rn(__fsub_rn(__fsub_rn(P[off[0]], P[off[1]]), P[off[2]]), P[off[3]]);
}
__device__ __forceinline__ float feature_value(const float* __restrict__ P, const FeatDev& f) {
    if (!(f.flags & 0x100)) {  // HAF: returnval += wgt * rect, regions in order, skipped regions omitted
        float v = 0.0f;
#pragma unroll
        for (int r = 0; r < 3; r++)
            if (f.flags & (1 << r)) v = __fadd_rn(v, __fmul_rn(f.w[r], rect_sum(P, f.off + 4 * r)));
        return v;
    }
    float rr[3];
#pragma unroll
    for (int r = 0; r < 3; r++) rr[r] = (f.flags & (1 << r)) ? __fmul_rn(f.w[r], rect_sum(P, f.off + 4 * r)) : 0.0f;
    if (rr[1] > rr[0] && rr[1] > rr[2]) {  // :187-188
        const float a = __fsub_rn(rr[1], rr[0]), b = __fsub_rn(rr[1], rr[2]);
        return (b < a) ? b : a;
    }
    return -1.0f;
}
template <bool DEBUG>
__global__ void __launch_bounds__(256) features_kernel(const float* __restrict__ integral, const int2* __restrict__ win,
                                                       const unsigned* __restrict__ win_count, int G, int unit_base,
                                                       const FeatDev* __restrict__ feats, const DimDev* __restrict__ dims,
                                                       int D, int Kpad, double lower, double upper, int emulate_text,
                                                       float* __restrict__ X, size_t ldx, int F,
                                                       float* __restrict__ dbg_raw, double* __restrict__ dbg_scaled,
                                                       int* __restrict__ unsupported_flag) {
    const unsigned W = *win_count;
    const unsigned w = blockIdx.x * 32 + (threadIdx.x & 31);
    const int warp = threadIdx.x >> 5;
    if (blockIdx.x * 32 >= W) return;
    const bool valid = w < W;
    const int ld = G + 1;
    const float* P = integral;
    if (valid) {
        const int2 uc = win[w];
        const int row = uc.y / G, col = uc.y - row * G;
        P = integral + (size_t)(uc.x - unit_base) * ld * ld + (size_t)(row - 7) * ld + (col - 7);
    }
    int uns = 0;
    for (int d = warp; d < Kpad; d += 8) {
        double x = 0.0;
        if (d < D && valid) {
            const DimDev dd = dims[d];
            if (dd.feat < 0) {
                x = dd.cval;
            } else {
                const FeatDev f = feats[dd.feat];
                const float raw = feature_value(P, f);
                double v;
                if (emulate_text) {
                    bool u4 = false;
                    v = hafdec::text4(raw, &u4);
                    if (u4) uns = 1;
                } else {
                    v = (double)raw;
                }
                if (dd.drop) x = 0.0;
                else {
                    double val;
                    if (v == dd.fmin) val = lower;
                    else if (v == dd.fmax) val = upper;
                    else val = __dadd_rn(lower, __ddiv_rn(__dmul_rn(__dsub_rn(upper, lower), __dsub_rn(v, dd.fmin)), dd.den));
                    if (val == 0.0) x = 0.0;
                    else if (!emulate_text) x = val;
                    else {
                        bool u6 = false;
                        x = hafdec::text6(val, &u6);
                        if (u6) uns = 1;
                    }
                }
            }
            if (DEBUG && dbg_scaled) dbg_scaled[(size_t)w * D + d] = x;
        }
        if (!DEBUG && valid) X[(size_t)d * ldx + w] = (float)x;
    }
    if (DEBUG && dbg_raw && valid) {
        for (int k = warp; k < F; k += 8) dbg_raw[(size_t)w * F + k] = feature_value(P, feats[k]);
    }
    if (uns) *unsupported_flag = 1;
}

// 10^k for |k| <= 40 (k >= 23 and negative k are rounded doubles: good to 1e-16, enough for the fast tier)
__device__ __forceinline__ double pow10_table(int k) {
    double p = 1.0;
    const int n = k < 0 ? -k : k;
    double b = 10.0;
    int m = n;
    while (m) { if (m & 1) p *= b; b *= b; m >>= 1; }
    return k < 0 ? 1.0 / p : p;
}

#define HAF_FT_ROWS 36  // integral-image rows a features_tc CTA can stage in shared memory (two blocks when its windows straddle two units)

// Joined per-dimension record of the tensor-path feature kernel (built once per context): the feature's corner
// offsets / weights / flags AND the dimension's scaling constants in one 96-byte record, so one dependent-load-free
// group of six 128-bit loads feeds a value (the dims -> feats indirection was the top stall of the first version).
struct __align__(16) DimFeat {
    int off[12];     // BYTE offsets of the corners; skipped regions: four identical corners (and weight +0.0)
    float w[3];
    int flags;       // bit 2: third region present; bit 8: SHAF; bit 9: constant dimension (value = cval); bit 10: dropped (value 0)
    float fmin, slope, cval, padf;   // float copies: the fast tier needs ~1e-7 only
    double pad[2];
};
static_assert(sizeof(DimFeat) == 96, "DimFeat layout");

// one value of the fast tier; I = integral image rows (shared or global), idx0 = index of the window's patch origin.
// Branch-free over regions: the host encodes a skipped region as four identical corners and weight +0.0, for which
// ((P - P) - P) + P == +0.0 exactly, so the reference's "skip" (II2FV.cpp:155-159) and this uniform code give the same
// float (a + (+0.0) == a, and the running sum is never -0.0).  All 12 loads can therefore be issued back to back.
struct FastTab {       // decoded 96-byte DimFeat record
    int off[12];
    float w[3];
    int flags;
    float fmin, slope, cval;
};
__device__ __forceinline__ FastTab load_fast_tab(const DimFeat* __restrict__ table, int d) {
    const uint4* tp = reinterpret_cast<const uint4*>(table + d);
    const uint4 t0 = __ldg(tp), t1 = __ldg(tp + 1), t2 = __ldg(tp + 2), t3 = __ldg(tp + 3), t4 = __ldg(tp + 4);
    FastTab f;
    f.off[0] = (int)t0.x; f.off[1] = (int)t0.y; f.off[2] = (int)t0.z; f.off[3] = (int)t0.w;
    f.off[4] = (int)t1.x; f.off[5] = (int)t1.y; f.off[6] = (int)t1.z; f.off[7] = (int)t1.w;
    f.off[8] = (int)t2.x; f.off[9] = (int)t2.y; f.off[10] = (int)t2.z; f.off[11] = (int)t2.w;
    f.w[0] = __uint_as_float(t3.x); f.w[1] = __uint_as_float(t3.y); f.w[2] = __uint_as_float(t3.z);
    f.flags = (int)t3.w;
    f.fmin = __uint_as_float(t4.x); f.slope = __uint_as_float(t4.y); f.cval = __uint_as_float(t4.z);
    return f;
}
// same record from the copy the CTA staged in shared memory: five broadcast LDS.128 = five wavefronts, where the same
// loads from global memory returned 16 B to each of 32 lanes = twenty (the kernel is bound by the LSU data pipe)
__device__ __forceinline__ FastTab load_fast_tab_smem(uint32_t rec_addr) {
    uint4 t[5];
#pragma unroll
    for (int k = 0; k < 5; k++)
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(t[k].x), "=r"(t[k].y), "=r"(t[k].z), "=r"(t[k].w) : "r"(rec_addr + 16u * k));
    FastTab f;
    f.off[0] = (int)t[0].x; f.off[1] = (int)t[0].y; f.off[2] = (int)t[0].z; f.off[3] = (int)t[0].w;
    f.off[4] = (int)t[1].x; f.off[5] = (int)t[1].y; f.off[6] = (int)t[1].z; f.off[7] = (int)t[1].w;
    f.off[8] = (int)t[2].x; f.off[9] = (int)t[2].y; f.off[10] = (int)t[2].z; f.off[11] = (int)t[2].w;
    f.w[0] = __uint_as_float(t[3].x); f.w[1] = __uint_as_float(t[3].y); f.w[2] = __uint_as_float(t[3].z);
    f.flags = (int)t[3].w;
    f.fmin = __uint_as_float(t[4].x); f.slope = __uint_as_float(t[4].y); f.cval = __uint_as_float(t[4].z);
    return f;
}
struct SmemRows { uint32_t base; };  // 32-bit shared-window byte address of the staged integral rows
__device__ __forceinline__ float load_corner(const float* I, int idx0, int off_bytes) {
    return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(I + idx0) + off_bytes);
}
__device__ __forceinline__ float load_corner(SmemRows I, int idx0_bytes, int off_bytes) {  // one IADD + LDS per corner
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(I.base + (uint32_t)(idx0_bytes + off_bytes)));
    return v;
}
// "%.4g" of the fast tier: powers of ten 10^(i-48) as double and float (built on the host, staged in shared memory by the
// kernel -- as global loads they cost more LSU wavefronts than the instructions they saved).
struct Round4Tab {
    double pwd[96];
    float pwf[96];
};
static_assert(sizeof(Round4Tab) == 96 * 8 + 96 * 4, "Round4Tab layout");
struct Round4Smem { uint32_t pwd, pwf; };   // 32-bit shared-window addresses of the staged tables
// idx0: element index of the window's patch origin for global rows, BYTE offset for staged rows; f.off[] are byte offsets
template <typename PtrT>
__device__ __forceinline__ float fast_tier_value(PtrT I, int idx0, const FastTab& f, float lower, int emulate_text,
                                                 const Round4Smem rt) {
    float c[12];
#pragma unroll
    for (int k = 0; k < 8; k++) c[k] = load_corner(I, idx0, f.off[k]);
    float rr[3];
#pragma unroll
    for (int r = 0; r < 2; r++)  // ((P[x2+1][y2+1] - P[x1][y2+1]) - P[x2+1][y1]) + P[x1][y1]   (II2FV.cpp:161-162)
        rr[r] = __fmul_rn(f.w[r], __fadd_rn(__fsub_rn(__fsub_rn(c[4 * r], c[4 * r + 1]), c[4 * r + 2]), c[4 * r + 3]));
    // 295 of the 323 features of data/Features.txt have no third region: a warp-uniform branch (the dimension is the
    // same for all lanes) saves a third of the corner loads.  rr[2] = +0.0 is what the uniform code computed for them.
    rr[2] = 0.0f;
    if (f.flags & 0x4) {
#pragma unroll
        for (int k = 8; k < 12; k++) c[k] = load_corner(I, idx0, f.off[k]);
        rr[2] = __fmul_rn(f.w[2], __fadd_rn(__fsub_rn(__fsub_rn(c[8], c[9]), c[10]), c[11]));
    }
    float raw;
    if (f.flags & 0x100) {   // SHAF (21 of 323 features): warp-uniform branch
        const float sa = __fsub_rn(rr[1], rr[0]), sb = __fsub_rn(rr[1], rr[2]);
        raw = (rr[1] > rr[0] && rr[1] > rr[2]) ? ((sb < sa) ? sb : sa) : -1.0f;  // II2FV.cpp:187-191
    } else {
        raw = __fadd_rn(__fadd_rn(__fadd_rn(0.0f, rr[0]), rr[1]), rr[2]);
    }
    float v = raw;
    if (emulate_text) {
        // "%.4g": a * 10^(3-E) is formed and rounded in DOUBLE (exact ties stay exact; a mis-decided near-tie needs
        // |frac - 0.5| < 1e-12); everything after the rounding decision only needs float accuracy here.  Branch-free:
        // raw = +-0 runs through the subnormal record and comes out as +-0.
        // E0 = floor(log10 2^k) = (k * 1233) >> 12 exactly for every float binade k in [-126, 127]; subnormals count as
        // binade -126.  (a >= 10^(E0+1) as a float rounded to nearest: a value sitting exactly on a rounded-down power of
        // ten is then scaled by one decade more and still rounds to the same four digits.)
        const float a = fabsf(raw);
        int E = ((max((int)(__float_as_uint(a) >> 23), 1) - 127) * 1233) >> 12;
        float thr;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(thr) : "r"(rt.pwf + (uint32_t)((48 + E + 1) << 2)));
        E += (a >= thr) ? 1 : 0;
        double mul; float inv;
        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(mul) : "r"(rt.pwd + (uint32_t)((48 + 3 - E) << 3)));
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(inv) : "r"(rt.pwf + (uint32_t)((48 + E - 3) << 2)));
        const float r = (float)rint((double)a * mul);
        v = copysignf(r * inv, raw);
    }
    const float x = fmaf(v - f.fmin, f.slope, lower);  // svm-scale.c:344-346
    return (f.flags & 0x400) ? 0.0f : ((f.flags & 0x200) ? f.cval : x);
}

// Tensor-core variant: per-dimension values split into two fp16 terms and written K-major in the k-block tiled layout
// (kt_off: what the UMMA K-major operand / TMA box wants).  Lane = window (WT = 2 windows per lane), warp = one dimension at a time; a
// 64-window x 96-dimension tile of (hi | lo << 16) words is staged in shared memory so that the global writes are whole
// 32-byte sectors of the operand rows; the squared norm of the (hi + lo) representation is accumulated on the way.
// The kernel is bound by the LSU data pipe and the issue rate together (DESIGN.md, "The feature kernel"): hence the
// bank-conflict-free staging of the image rows, the per-pass copy of the table records and the power-of-ten tables in
// shared memory, and the warp-uniform branches around the third region and the SHAF rule.
//
// FAST TIER.  The values written here are rounded to 22 significant bits (fp16 hi + lo) anyway and every window whose
// decision value lands inside the guard band is re-evaluated from the bit-exact emulation (guard_inputs_kernel /
// svm_exact_terms_kernel), so this tier reproduces the text round trips only to ~1e-7 (see fast_tier_value); the
// 6-digit "%g" rounding (<= 5e-6 relative: the largest input error of this tier, tools/dec_error_probe.py) is skipped.
// Raw feature values are the same bit-exact floats as everywhere else.
// (Tables in __constant__ memory were tried and were 1.8x SLOWER: 36 KB of tables thrash the constant cache.)
// OPERAND LAYOUT in global memory ("k-block tiled"): element (row, d) of X / SV lives at
//     ((row / 128) * KB + d / 64) * 8192 + (row % 128) * 64 + d % 64        (fp16 elements; KB = k-blocks of 64)
// i.e. every 128-row x 64-column tile the tensor kernels fetch with ONE TMA box is a contiguous, 128-byte aligned 16 KB
// block.  Round 1 stored plain rows of Krow = 336 elements: a box was then 128 separate 128-byte pieces at a 672-byte pitch,
// every one straddling two cache lines, and the TMA unit -- not L2, not the MMAs, not the epilogue -- bounded the tensor
// kernel at ~5 clocks per box row (profiles/r2_tc_pipeline_probe.txt: the bare TMA + barrier skeleton of the kernel took 70 %
// of its time).
__host__ __device__ __forceinline__ size_t kt_off(size_t row, int d, int KB) {
    return (((row >> 7) * (size_t)KB + (size_t)(d >> 6)) << 13) + ((row & 127) << 6) + (size_t)(d & 63);
}
// the six extra operand columns of a window row (svm_tc.cuh, OPERAND FORMAT): -|x|^2 / 2 as three fp16 terms, then 1 1 1.
// The splits are exact in FP32 (each remainder has fewer significant bits than its predecessor).
__device__ __forceinline__ void write_aug_columns(__half* __restrict__ X, size_t row, int aug0, int KB, float sq, bool ok) {
    const float a = -0.5f * sq;
    const __half h = __float2half_rn(a);
    const float r1 = a - __half2float(h);
    const __half m = __float2half_rn(r1);
    const __half l = __float2half_rn(r1 - __half2float(m));
    const __half one = __float2half_rn(ok ? 1.0f : 0.0f);   // a window outside the fp16 range takes the exact path: keep its row finite
    X[kt_off(row, aug0 + 0, KB)] = h; X[kt_off(row, aug0 + 1, KB)] = m; X[kt_off(row, aug0 + 2, KB)] = l;
    X[kt_off(row, aug0 + 3, KB)] = one; X[kt_off(row, aug0 + 4, KB)] = one; X[kt_off(row, aug0 + 5, KB)] = one;
}

#define HAF_FT_WT 2
#define HAF_FT_KPASS 128  // dimensions per pass of the shared-memory tile: 256 B = two whole k-blocks of a row of Xh / Xl
// dynamic shared memory of features_tc_kernel: fp16 tile(s) [tiles][64 windows][KPASS] + staged image rows + the pass's table records
__host__ __device__ constexpr size_t ft_smem_layout(int G, int tiles) {
    return sizeof(Round4Tab) + (size_t)tiles * 32 * HAF_FT_WT * HAF_FT_KPASS * 2 + (size_t)HAF_FT_ROWS * (G + 1 + 31) * 4 + 16 + (size_t)HAF_FT_KPASS * 96;
}
__global__ void __launch_bounds__(256, 4) features_tc_kernel(const float* __restrict__ integral, const int2* __restrict__ win,
                                                             const unsigned* __restrict__ win_count, int G, int unit_base,
                                                             const DimFeat* __restrict__ table, int D, int Krow, float lower,
                                                             int emulate_text, const Round4Tab* __restrict__ rtab,
                                                             __half* __restrict__ Xh, __half* __restrict__ Xl /*NULL: hi only*/, float* __restrict__ xn,
                                                             int aug0 /*first of the six extra operand columns (svm_tc.cuh)*/, int KB /*k-blocks of the tiled layout*/,
                                                             double* __restrict__ dec_acc, float* __restrict__ asum_acc /*the contraction's accumulators: zeroed here*/) {
    constexpr int WT = HAF_FT_WT, NW = 32 * WT;
    // TILE.  fp16 values [window][KPASS dims] = 256-byte rows of sixteen 16-byte chunks, swizzled so that BOTH sides are free of
    // bank conflicts: element (w, d) sits in chunk (d >> 3) ^ (w & 7), word ((d & 7) >> 1) ^ ((w >> 3) & 3) of its row.  A compute
    // warp stores one dimension of 32 windows per instruction (32 different (chunk & 7, word) pairs = 32 banks); the write-out
    // reads whole chunks with LDS.128 (16 lanes = the 16 chunks of a row, XOR-permuted = all banks) and writes them with
    // STG.128: 8 dimensions per instruction.  Round 1 kept (hi | lo << 16) words and wrote 2 dimensions per STG after two LDS
    // and a PRMT, with 64-bit kt_off arithmetic per word: a quarter of the kernel's instructions (ncu r2, source view).
    // dynamic shared memory: the "%.4g" power-of-ten tables first (their addresses are then tile_base - constant: as a static
    // __shared__ object the compiler re-derived the address -- S2R CgaCtaId, MOV, VIADD, LEA -- for every value, ncu r2), then the
    // tile(s) [1 or 2][NW][KPASS] fp16, then float s_int[ROWS][ld .. ld + 31], then the pass's table records
    extern __shared__ __align__(16) uint32_t s_dyn[];
    static_assert(sizeof(Round4Tab) % 16 == 0, "the tile behind the tables must stay 16-byte aligned");
    uint32_t* const s_words = s_dyn + sizeof(Round4Tab) / 4;
    const int tiles = Xl ? 2 : 1;
    constexpr int TILE_WORDS = NW * HAF_FT_KPASS / 2;
    const unsigned W = *win_count;
    const unsigned w0 = blockIdx.x * NW;
    if (w0 >= W) return;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // provably warp-uniform for the compiler
    const int ld = G + 1;
    float* s_int = reinterpret_cast<float*>(s_words + tiles * TILE_WORDS);  // [HAF_FT_ROWS][ld .. ld + 31]
    uint4* s_tab = reinterpret_cast<uint4*>(s_words + ((tiles * TILE_WORDS + HAF_FT_ROWS * (ld + 31) + 3) & ~3));  // [KPASS] DimFeat records of the pass
    __shared__ int s_box[9];       // unit A, its first row, rows (0 = no staging), row stride of the staged image; unit B, first row, rows
    int unit[WT], row[WT], col[WT];
    bool valid[WT];
#pragma unroll
    for (int t = 0; t < WT; t++) {
        const unsigned w = w0 + t * 32 + lane;
        valid[t] = w < W;
        unit[t] = 0; row[t] = 7; col[t] = 7;
        if (valid[t]) {
            const int2 uc = win[w];
            unit[t] = uc.x;
            row[t] = uc.y / G;
            col[t] = uc.y - row[t] * G;
        }
    }
    if (threadIdx.x < 32) {
        // The CTA's 64 consecutive windows belong to one unit or -- one CTA in ~9 on the bench workload -- to the end of
        // one unit and the start of the next (each unit's windows are contiguous in the list).  Both units' image rows are
        // staged, one block after the other; only a CTA touching three units (masks with < 64 windows) reads global memory.
        const int uA = __shfl_sync(0xffffffffu, unit[0], 0);  // window w0 is always valid
        int uB = uA;
#pragma unroll
        for (int t = 0; t < WT; t++) {   // unit of the last valid window
            const unsigned vm = __ballot_sync(0xffffffffu, valid[t]);
            if (vm) uB = __shfl_sync(0xffffffffu, unit[t], 31 - __clz(vm));
        }
        bool two = true;
        int rminA = 0x7fffffff, rmaxA = -1, rminB = 0x7fffffff, rmaxB = -1, cmin = 0x7fffffff, cmax = -1;
#pragma unroll
        for (int t = 0; t < WT; t++) {
            two = two && (!valid[t] || unit[t] == uA || unit[t] == uB);
            if (valid[t]) { cmin = min(cmin, col[t]); cmax = max(cmax, col[t]); }
            if (valid[t] && unit[t] == uA) { rminA = min(rminA, row[t]); rmaxA = max(rmaxA, row[t]); }
            else if (valid[t]) { rminB = min(rminB, row[t]); rmaxB = max(rmaxB, row[t]); }
        }
        two = __all_sync(0xffffffffu, two);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            rminA = min(rminA, __shfl_xor_sync(0xffffffffu, rminA, o));
            rmaxA = max(rmaxA, __shfl_xor_sync(0xffffffffu, rmaxA, o));
            rminB = min(rminB, __shfl_xor_sync(0xffffffffu, rminB, o));
            rmaxB = max(rmaxB, __shfl_xor_sync(0xffffffffu, rmaxB, o));
            cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
            cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        }
        // BANK-CONFLICT-FREE STAGING.  Lanes are consecutive windows of the compact list: a warp-load touches columns
        // a..b of one image row and a'..b' of the next.  With the natural row stride G + 1 the two runs overlap in banks
        // and EVERY corner load took two wavefronts (ncu: 13 conflict wavefronts per 12 loads; the kernel is LSU-bound).
        // The rows are therefore staged with the stride s = (b + 1 - a') mod 32 that makes the second run continue in the
        // bank after the first; the per-dimension corner offsets for each of the 32 stride classes are precomputed
        // (table[cls][d]).  The first row break of the CTA's windows picks s (axis-aligned masks break identically in
        // every row; rotated ones differ by +-1 between rows, which leaves some two-wavefront loads).
        int o = ld;
        bool have = false;
#pragma unroll
        for (int t = 0; t < WT; t++) {
            const int pc = __shfl_up_sync(0xffffffffu, col[t], 1), pr = __shfl_up_sync(0xffffffffu, row[t], 1);
            const int pu = __shfl_up_sync(0xffffffffu, unit[t], 1);
            const bool brk = lane > 0 && valid[t] && pu == unit[t] && row[t] == pr + 1;
            const unsigned m = __ballot_sync(0xffffffffu, brk);
            if (m && !have) { o = __shfl_sync(0xffffffffu, pc + 1 - col[t], __ffs(m) - 1); have = true; }
        }
        if (lane == 0) {
            const int nA = rmaxA - rminA + 15, nB = (uB != uA) ? rmaxB - rminB + 15 : 0;
            const bool ok = two && nA + nB <= HAF_FT_ROWS;
            s_box[0] = uA; s_box[1] = rminA - 7; s_box[2] = ok ? nA : 0;
            s_box[3] = ld + (((o - ld) % 32) + 32) % 32;
            s_box[4] = uB; s_box[5] = rminB - 7; s_box[6] = ok ? nB : 0;
            s_box[7] = cmin - 7; s_box[8] = cmax - cmin + 15;   // columns the patches touch: only these are copied
        }
    }
    for (int t = threadIdx.x; t < (int)(sizeof(Round4Tab) / 8); t += blockDim.x)
        reinterpret_cast<uint2*>(s_dyn)[t] = __ldg(reinterpret_cast<const uint2*>(rtab) + t);
    __syncthreads();
    Round4Smem rt;
    rt.pwd = (uint32_t)__cvta_generic_to_shared(s_dyn);                                                  // Round4Tab::pwd at offset 0
    asm volatile("" : "+r"(rt.pwd));   // opaque: keep the base in a register instead of re-deriving it (S2R CgaCtaId, MOV, VIADD, LEA) per value
    rt.pwf = rt.pwd + (uint32_t)(96 * sizeof(double));                                                   // Round4Tab::pwf behind it
    const int nrows = s_box[2];
    const int sst = nrows > 0 ? s_box[3] : ld;           // row stride the corner offsets must be built for
    table += (size_t)(sst - ld) * D;                      // stride class
    int idx0[WT];
    const float* gI[WT];
#pragma unroll
    for (int t = 0; t < WT; t++) {
        idx0[t] = (row[t] - 7) * ld + (col[t] - 7);
        gI[t] = integral + (size_t)(unit[t] - unit_base) * ld * ld;
    }
    if (nrows > 0) {
        const int nB = s_box[6];
        const float* srcA = integral + (size_t)(s_box[0] - unit_base) * ld * ld + (size_t)s_box[1] * ld;
        const float* srcB = integral + (size_t)(s_box[4] - unit_base) * ld * ld + (size_t)s_box[5] * ld - (size_t)nrows * ld;
        // only the columns the CTA's patches touch (all of them at G = 56, a sixth of the row at G = 512); the staged image
        // keeps the full-width addressing the offset tables are built for
        const int c0 = s_box[7], wd = s_box[8];
        for (int t = threadIdx.x; t < (nrows + nB) * wd; t += blockDim.x) {
            const int r = t / wd, c = c0 + (t - r * wd);
            s_int[r * sst + c] = (r < nrows ? srcA : srcB)[r * ld + c];
        }
#pragma unroll
        for (int t = 0; t < WT; t++) {   // padding lanes read row 0 harmlessly
            const int r0 = (unit[t] == s_box[0]) ? row[t] - 7 - s_box[1] : nrows + row[t] - 7 - s_box[5];
            idx0[t] = valid[t] ? r0 * sst + (col[t] - 7) : 0;
        }
    }
    const uint32_t tab_base = (uint32_t)__cvta_generic_to_shared(s_tab);
    SmemRows srows;
    srows.base = (uint32_t)__cvta_generic_to_shared(s_int);
    float nrm[WT];  // squared-norm partials of this lane's windows over the dimensions this warp evaluates
#pragma unroll
    for (int t = 0; t < WT; t++) nrm[t] = 0.0f;
    const uint32_t tile_base = rt.pwd + (uint32_t)sizeof(Round4Tab);
    const uint32_t row0 = tile_base + (uint32_t)lane * (HAF_FT_KPASS * 2), row1 = row0 + 32u * (HAF_FT_KPASS * 2);   // windows lane, 32 + lane
    const uint32_t sw = (uint32_t)(((lane & 7) << 2) | ((lane >> 3) & 3));   // swizzle of this lane's two rows (same low five bits)
    for (int d0 = 0; d0 < Krow; d0 += HAF_FT_KPASS) {
        const int KP = min(HAF_FT_KPASS, Krow - d0);   // a multiple of 16
        {   // this pass's records of the stride class, coalesced
            const int nrec = min(KP, D - d0);
            const uint4* src = reinterpret_cast<const uint4*>(table + d0);
            for (int t = threadIdx.x; t < nrec * 6; t += blockDim.x) s_tab[t] = __ldg(src + t);
        }
        __syncthreads();
        for (int dl = warp; dl < KP; dl += 8) {
            const int d = d0 + dl;
            float xf[WT];
#pragma unroll
            for (int t = 0; t < WT; t++) xf[t] = 0.0f;
            if (d < D) {
                const FastTab f = load_fast_tab_smem(tab_base + 96u * dl);
                if (nrows > 0) {
#pragma unroll
                    for (int t = 0; t < WT; t++) xf[t] = fast_tier_value(srows, idx0[t] * 4, f, lower, emulate_text, rt);
                } else {
#pragma unroll
                    for (int t = 0; t < WT; t++) xf[t] = valid[t] ? fast_tier_value(gI[t], idx0[t], f, lower, emulate_text, rt) : 0.0f;
                }
            }
            // fp16 hi + fp16 lo = 22 significant bits (absolute floor 2^-25 once lo is subnormal), two windows per conversion.
            // A value beyond the fp16 range becomes hi = +-inf, lo = -+inf: the NaN / inf it produces stays inside this
            // window's own accumulator row, and the window is sent to the FP64 exact path (xn = +inf below).
            static_assert(WT == 2, "the packing below converts the two windows of a lane together");
            const __half2 hi2 = __floats2half2_rn(xf[0], xf[1]);
            const float2 hif = __half22float2(hi2);
            const __half2 lo2 = __floats2half2_rn(xf[0] - hif.x, xf[1] - hif.y);
            {   // squared norm of what the contraction will see (hi + lo), accumulated per lane over this warp's dimensions
                const float2 lof = __half22float2(lo2);
                const float v0 = hif.x + lof.x, v1 = hif.y + lof.y;
                nrm[0] = fmaf(v0, v0, nrm[0]);
                nrm[1] = fmaf(v1, v1, nrm[1]);
            }
            const uint32_t hu = *reinterpret_cast<const uint32_t*>(&hi2), lu = *reinterpret_cast<const uint32_t*>(&lo2);
            // swizzled byte offset of dimension dl inside a tile row (see TILE above)
            const uint32_t toff = ((((uint32_t)dl >> 1) ^ sw) << 2) | (((uint32_t)dl & 1u) << 1);
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(row0 + toff), "h"((unsigned short)(hu & 0xffffu)) : "memory");
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(row1 + toff), "h"((unsigned short)(hu >> 16)) : "memory");
            if (Xl) {   // three products only
                asm volatile("st.shared.b16 [%0], %1;" ::"r"(row0 + TILE_WORDS * 4 + toff), "h"((unsigned short)(lu & 0xffffu)) : "memory");
                asm volatile("st.shared.b16 [%0], %1;" ::"r"(row1 + TILE_WORDS * 4 + toff), "h"((unsigned short)(lu >> 16)) : "memory");
            }
        }
        __syncthreads();
        {   // write-out: lane = (window of a pair, chunk): 16 lanes x 16 bytes = two whole 128-byte k-block rows of one window
            const int c = lane & 15, nch = KP >> 3;
            // k-block tiled layout (kt_off): chunk c of this pass = dimensions d0 + 8c .. + 7 = 16 contiguous bytes of the window's row
            const size_t coff = ((size_t)((d0 >> 6) + (c >> 3)) << 13) + (size_t)((c & 7) << 3);
#pragma unroll
            for (int k = 0; k < NW / 16; k++) {
                const int wi = 16 * k + 2 * warp + (lane >> 4);
                const unsigned ww = w0 + wi;
                if (ww < W && c < nch) {
                    const uint32_t a = tile_base + (uint32_t)wi * (HAF_FT_KPASS * 2) + (uint32_t)((c ^ (wi & 7)) << 4);
                    const size_t off = ((size_t)(ww >> 7) * (size_t)KB << 13) + ((size_t)(ww & 127) << 6) + coff;
                    const int kx = (wi >> 3) & 3;   // the row's word permutation: stored word q ^ kx holds dimensions 2q, 2q + 1
#pragma unroll
                    for (int tl = 0; tl < 2; tl++) {
                        if (tl == 1 && !Xl) break;
                        uint4 v;
                        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a + tl * TILE_WORDS * 4));
                        if (kx & 1) { uint32_t t0 = v.x; v.x = v.y; v.y = t0; t0 = v.z; v.z = v.w; v.w = t0; }
                        if (kx & 2) { uint32_t t0 = v.x; v.x = v.z; v.z = t0; t0 = v.y; v.y = v.w; v.w = t0; }
                        *reinterpret_cast<uint4*>((tl ? Xl : Xh) + off) = v;
                    }
                }
            }
        }
    }
    // squared norms: the 8 warps' partials of each window are summed through the (now free) tile; a value that left the fp16
    // range made its window's partial inf - inf = NaN (or inf): such windows get xn = +inf = "always take the exact path"
    __syncthreads();
    float* s_nrm = reinterpret_cast<float*>(s_words);   // [8][NW]
#pragma unroll
    for (int t = 0; t < WT; t++) s_nrm[warp * NW + t * 32 + lane] = nrm[t];
    __syncthreads();
    if (threadIdx.x < NW && w0 + threadIdx.x < W) {
        float sq = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; k++) sq += s_nrm[k * NW + threadIdx.x];
        // -|x|^2 / 2 has to fit the fp16 extra columns as well (|x|^2 / 2 <= 65504)
        const bool ok = sq < 1.3e5f;
        xn[w0 + threadIdx.x] = ok ? sq : __int_as_float(0x7f800000);
        dec_acc[w0 + threadIdx.x] = 0.0;
        asum_acc[w0 + threadIdx.x] = 0.0f;
        write_aug_columns(Xh, w0 + threadIdx.x, aug0, KB, ok ? sq : 0.0f, ok);
    }
}

// squared norm of every window's SVM input (FP32)
__global__ void xnorm_kernel(const float* __restrict__ X, size_t ldx, int Kpad, const unsigned* __restrict__ win_count,
                             float* __restrict__ xn) {
    const unsigned W = *win_count;
    const unsigned w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    float s = 0.0f;
    for (int d = 0; d < Kpad; d++) { const float v = X[(size_t)d * ldx + w]; s = fmaf(v, v, s); }
    xn[w] = s;
}

// ---------------------------------------------------------------------------------------------------
// a11 (FP32 SIMT): dec[w] = sum_i coef_i * exp(-gamma * ||x_w - sv_i||^2) - rho with
// ||x - sv||^2 = ||x||^2 + ||sv||^2 - 2 x.sv; the x.sv contraction is a register-tiled SGEMM
// (CTA tile 128 windows x 128 SVs, BK = 16, 8x8 micro-tiles, 3-stage cp.async pipeline) with the
// exp / coef / row-sum epilogue fused, decision sums accumulated in FP64.
// A window whose |dec| <= guard_rel * sum_i |coef_i| K_i is appended to the guard list and re-evaluated by
// svm_exact_kernel in FP64 in libsvm's own order, so LABELS equal the reference's.
// ---------------------------------------------------------------------------------------------------
#define SVM_BM 128
#define SVM_BN 128
#define SVM_BK 16
#define SVM_STAGES 3
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__global__ void __launch_bounds__(256, 2) svm_rbf_simt_kernel(const float* __restrict__ X, size_t ldx,
                                                               const float* __restrict__ svT, int Spad, int Kpad,
                                                               const float* __restrict__ xn, const float* __restrict__ svn,
                                                               const float* __restrict__ coef, float neg_gamma_log2e,
                                                               double rho, float guard_rel, float e_floor /*see svm_finalize_kernel*/,
                                                               const unsigned* __restrict__ win_count,
                                                               double* __restrict__ dec, unsigned char* __restrict__ guard_flag,
                                                               int* __restrict__ guard_list, unsigned* __restrict__ guard_count) {
    const unsigned W = *win_count;
    const unsigned m0 = blockIdx.x * SVM_BM;
    if (m0 >= W) return;
    extern __shared__ __align__(16) float smem[];
    float* As = smem;                                       // [STAGES][BK][BM]
    float* Bs = smem + SVM_STAGES * SVM_BK * SVM_BM;        // [STAGES][BK][BN]
    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;                 // 16 x 16 threads, each 8 (m) x 8 (n) as 2x(4) + 2x(4)
    const int nk = Kpad / SVM_BK;
    const int ntiles = Spad / SVM_BN;

    double dsum[8];
    float asum[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { dsum[i] = 0.0; asum[i] = 0.0f; }
    float xnr[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const unsigned m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        xnr[i] = (m < W) ? xn[m] : 0.0f;
    }

    // one stage = 16 rows x 128 floats for A and for B = 2 x 512 16-byte chunks; 256 threads -> 2 + 2 chunks each
    auto load_stage = [&](int stage, int kb, int n0) {
        const int k0 = kb * SVM_BK;
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const int chunk = tid + c * 256;        // 0..511
            const int kr = chunk >> 5, mc = (chunk & 31) * 4;
            cp_async16(As + (stage * SVM_BK + kr) * SVM_BM + mc, X + (size_t)(k0 + kr) * ldx + m0 + mc);
            cp_async16(Bs + (stage * SVM_BK + kr) * SVM_BN + mc, svT + (size_t)(k0 + kr) * Spad + n0 + mc);
        }
    };

    const int total = ntiles * nk;  // flattened (n-tile, k-block) iteration space
    int issued = 0;
    for (; issued < SVM_STAGES - 1 && issued < total; issued++) {
        load_stage(issued % SVM_STAGES, issued % nk, (issued / nk) * SVM_BN);
        cp_async_commit();
    }
    for (int s = issued; s < SVM_STAGES - 1; s++) cp_async_commit();

    float acc[8][8];
    for (int it = 0; it < total; it++) {
        const int kb = it % nk, nt = it / nk;
        if (kb == 0) {
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 8; j++) acc[i][j] = 0.0f;
        }
        cp_async_wait<SVM_STAGES - 2>();
        __syncthreads();
        if (issued < total) load_stage(issued % SVM_STAGES, issued % nk, (issued / nk) * SVM_BN);
        cp_async_commit();
        issued++;
        const float* a = As + (it % SVM_STAGES) * SVM_BK * SVM_BM;
        const float* b = Bs + (it % SVM_STAGES) * SVM_BK * SVM_BN;
#pragma unroll
        for (int k = 0; k < SVM_BK; k++) {
            const float4 a0 = *reinterpret_cast<const float4*>(a + k * SVM_BM + ty * 4);
            const float4 a1 = *reinterpret_cast<const float4*>(a + k * SVM_BM + 64 + ty * 4);
            const float4 b0 = *reinterpret_cast<const float4*>(b + k * SVM_BN + tx * 4);
            const float4 b1 = *reinterpret_cast<const float4*>(b + k * SVM_BN + 64 + tx * 4);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 8; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (kb == nk - 1) {  // epilogue of this SV tile
            const int n0 = nt * SVM_BN;
            float cf[8], sn[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                cf[j] = __ldg(coef + n);
                sn[j] = __ldg(svn + n);
            }
#pragma unroll
            for (int i = 0; i < 8; i++) {
                float ps = 0.0f, pa = 0.0f;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const float base = xnr[i] + sn[j];
                    const float d2 = fmaxf(fmaf(-2.0f, acc[i][j], base), 0.0f);
                    const float kv = exp2f(neg_gamma_log2e * d2);
                    ps = fmaf(cf[j], kv, ps);
                    // guard scale: |coef| K (1 + |c| (xn + svn)) -- the exponent's absolute FP32 error grows with the
                    // magnitude of the numbers it is assembled from (see svm_tc.cuh, GUARD SCALE)
                    pa = fmaf(fabsf(cf[j]) * kv, fmaf(-neg_gamma_log2e, base, 1.0f), pa);
                }
                dsum[i] += (double)ps;
                asum[i] += pa;
            }
        }
    }
    cp_async_wait<0>();
    // reduce over the 16 tx lanes that share the same window rows (lanes 0-15 / 16-31 of a warp)
#pragma unroll
    for (int i = 0; i < 8; i++) {
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) {
            dsum[i] += __shfl_xor_sync(0xffffffffu, dsum[i], o);
            asum[i] += __shfl_xor_sync(0xffffffffu, asum[i], o);
        }
    }
    if (tx == 0) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const unsigned m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
            if (m < W) {
                const double dv = dsum[i] - rho;
                dec[m] = dv;
                const bool g = !(fabs(dv) > (double)guard_rel * ((double)asum[i] + fabs(rho))) || !(asum[i] >= e_floor);   // NaN-safe
                guard_flag[m] = g ? 1 : 0;
                if (g) guard_list[atomicAdd(guard_count, 1u)] = (int)m;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// a11 (FP64, libsvm order): one CTA per listed window.  x is re-derived in double from the integral image
// (same device functions as features_kernel), K_i = exp(-gamma * sum_d (x_d - sv_i,d)^2) with the d loop
// sequential and un-fused (Kernel::k_function, svm.cpp:326-365: absent entries are zeros, adding 0.0 is
// exact), then ONE thread sums coef_i * K_i in file order and subtracts rho (svm.cpp:2500-2514).
// list == NULL: all windows (HAF_SVM_FP64_EXACT).  grid-stride over the list; kscratch: [gridDim.x][Spad].
// ---------------------------------------------------------------------------------------------------
#define HAF_EXACT_WB 8     // windows evaluated together by one CTA: every support-vector element is loaded once per 8 windows
#define HAF_EXACT_SVT 2    // support vectors per thread (register tile WB x SVT)
#define HAF_EXACT_SLICE (256 * HAF_EXACT_SVT)   // support vectors per CTA
struct ExactArgs {
    const int* list; const unsigned* list_count; const unsigned* win_count; const float* integral; const int2* win;
    int G, unit_base; const FeatDev* feats; const DimDev* dims; int D; double lower, upper; int emulate_text;
    const double* sv64T; int Spad, S, Dsv; const double* coef64; double gamma, rho; double* terms; double* dec;
    int* unsupported_flag;
    int* overflow_flag;   // set when the list holds more entries than this launch covers (guard mode: one launch only)
    int entry_begin;      // this launch covers list entries [entry_begin, entry_begin + max_entries)
    int max_entries;      // capacity of `terms` in windows
    const double* xdense; // haf_svm_predict: the SVM inputs are GIVEN ([window][Dsv] doubles) instead of derived from a cloud
    int x_global;         // 1: the inputs of HAF_EXACT_WB windows do not fit in shared memory (svm_exact_terms_xglobal_kernel)
};
// SVM input d of window w, re-derived in double from the integral image with the bit-exact emulation of both text round
// trips (a7-a9: calc_featurevalue, "%.4g", svm-scale.c:339-352 with "%g"): exactly what svm-predict parses.
__device__ __forceinline__ double exact_scaled_input(const ExactArgs& A, int w, int d) {
    if (A.xdense) return A.xdense[(size_t)w * A.Dsv + d];
    const int ld = A.G + 1;
    const int2 uc = A.win[w];
    const int row = uc.y / A.G, col = uc.y - row * A.G;
    const float* P = A.integral + (size_t)(uc.x - A.unit_base) * ld * ld + (size_t)(row - 7) * ld + (col - 7);
    const DimDev dd = A.dims[d];
    if (dd.feat < 0) return dd.cval;
    double x = 0.0;
    const float raw = feature_value(P, A.feats[dd.feat]);
    bool u4 = false, u6 = false;
    const double v = A.emulate_text ? hafdec::text4(raw, &u4) : (double)raw;
    if (!dd.drop) {
        double val;
        if (v == dd.fmin) val = A.lower;
        else if (v == dd.fmax) val = A.upper;
        else val = __dadd_rn(A.lower, __ddiv_rn(__dmul_rn(__dsub_rn(A.upper, A.lower), __dsub_rn(v, dd.fmin)), dd.den));
        if (val != 0.0) x = A.emulate_text ? hafdec::text6(val, &u6) : val;
    }
    if (u4 || u6) *A.unsupported_flag = 1;
    return x;
}

// Phase 1: terms[e][i] = coef_i * K_i for list entry e (window list[e], or window e when list == NULL).
// grid = (window blocks, SV slices).  x is re-derived in double from the integral image with the bit-exact emulation of
// both text round trips; K_i = exp(-gamma * sum_d (x_d - sv_i,d)^2) with the d loop sequential and un-fused
// (Kernel::k_function, svm.cpp:326-365: absent entries are zeros, adding 0.0 is exact).  WB = 8 windows share every SV
// element (throughput); WB = 1 spreads a short list over many CTAs (latency of a single goal).  XG (models too wide for
// the shared-memory copy, WB = 1 only): every thread reads x_d in place -- one broadcast load per d.
template <int WB, bool XG = false>
__device__ __forceinline__ void svm_exact_terms_body(const ExactArgs& A, double* xs, unsigned n) {
    const int Dsv = A.Dsv, Spad = A.Spad;
    const int i0 = blockIdx.y * HAF_EXACT_SLICE;
    if (i0 >= A.S) return;
    for (unsigned e0 = A.entry_begin + blockIdx.x * WB; e0 < n; e0 += gridDim.x * WB) {
        const int nb = min((unsigned)WB, n - e0);
        const int w0 = XG ? (A.list ? A.list[e0] : (int)e0) : 0;   // XG: the one window of this step
        if (!XG) {
            __syncthreads();
            for (int t = threadIdx.x; t < WB * Dsv; t += blockDim.x) {
                const int b = t / Dsv, d = t - b * Dsv;
                double x = 0.0;
                if (b < nb && d < A.D) x = exact_scaled_input(A, A.list ? A.list[e0 + b] : (int)(e0 + b), d);
                xs[t] = x;
            }
            __syncthreads();
        }
        double sum[WB][HAF_EXACT_SVT];
#pragma unroll
        for (int b = 0; b < WB; b++)
#pragma unroll
            for (int k = 0; k < HAF_EXACT_SVT; k++) sum[b][k] = 0.0;
        const int ia = i0 + threadIdx.x;  // this thread's SVs: ia, ia + 256 (padding SVs are all-zero columns, coef 0)
        for (int d = 0; d < Dsv; d++) {
            double sv[HAF_EXACT_SVT];
#pragma unroll
            for (int k = 0; k < HAF_EXACT_SVT; k++) sv[k] = A.sv64T[(size_t)d * Spad + ia + 256 * k];
#pragma unroll
            for (int b = 0; b < WB; b++) {
                const double xb = XG ? (d < A.D ? exact_scaled_input(A, w0, d) : 0.0) : xs[b * Dsv + d];
#pragma unroll
                for (int k = 0; k < HAF_EXACT_SVT; k++) {
                    const double diff = __dsub_rn(xb, sv[k]);
                    sum[b][k] = __dadd_rn(sum[b][k], __dmul_rn(diff, diff));
                }
            }
        }
#pragma unroll
        for (int k = 0; k < HAF_EXACT_SVT; k++) {
            const int i = ia + 256 * k;
            if (i < A.S) {
                const double cf = A.coef64[i];
#pragma unroll
                for (int b = 0; b < WB; b++)
                    if (b < nb) A.terms[(size_t)(e0 - A.entry_begin + b) * Spad + i] = __dmul_rn(cf, exp(__dmul_rn(-A.gamma, sum[b][k])));
            }
        }
    }
}
__global__ void __launch_bounds__(256) svm_exact_terms_kernel(const ExactArgs A) {
    extern __shared__ double xs[];  // [HAF_EXACT_WB][Dsv]
    unsigned n = A.list ? *A.list_count : *A.win_count;
    n = min(n, (unsigned)(A.entry_begin + A.max_entries));
    if (n <= (unsigned)A.entry_begin) return;
    if (n - A.entry_begin >= (unsigned)gridDim.x * 2u) svm_exact_terms_body<HAF_EXACT_WB>(A, xs, n);
    else svm_exact_terms_body<1>(A, xs, n);
}
// the same for models whose inputs of HAF_EXACT_WB windows do not fit in shared memory (ExactArgs.x_global): one window per
// CTA step, x read in place (a kernel of its own, so that the register allocation of the one above stays as it is)
__global__ void __launch_bounds__(256) svm_exact_terms_xglobal_kernel(const ExactArgs A) {
    unsigned n = A.list ? *A.list_count : *A.win_count;
    n = min(n, (unsigned)(A.entry_begin + A.max_entries));
    if (n <= (unsigned)A.entry_begin) return;
    svm_exact_terms_body<1, true>(A, nullptr, n);
}
// Phase 2: dec = (sum of the terms in FILE ORDER, one sequential chain) - rho   (svm.cpp:2500-2514).  One warp per
// entry: 32 terms are fetched with one coalesced load and broadcast lane by lane, every lane runs the same chain.
__global__ void __launch_bounds__(128) svm_exact_sum_kernel(const ExactArgs A) {
    const unsigned total = A.list ? *A.list_count : *A.win_count;
    if (A.overflow_flag && total > (unsigned)(A.entry_begin + A.max_entries) && blockIdx.x == 0 && threadIdx.x == 0) *A.overflow_flag = 1;
    const unsigned n = min(total, (unsigned)(A.entry_begin + A.max_entries));
    const int lane = threadIdx.x & 31;
    for (unsigned e = A.entry_begin + blockIdx.x * 4 + (threadIdx.x >> 5); e < n; e += gridDim.x * 4) {
        const double* t = A.terms + (size_t)(e - A.entry_begin) * A.Spad;
        double sum = 0.0;
        for (int i0 = 0; i0 < A.S; i0 += 32) {
            const double mine = (i0 + lane < A.S) ? t[i0 + lane] : 0.0;
            const int cnt = min(32, A.S - i0);
            for (int k = 0; k < cnt; k++) sum = __dadd_rn(sum, __shfl_sync(0xffffffffu, mine, k));
        }
        if (lane == 0) A.dec[A.list ? A.list[e] : (int)e] = __dsub_rn(sum, A.rho);
    }
}

// ---------------------------------------------------------------------------------------------------
// Guard band, tier 2: FP64 FMA contraction.  Every window the FP32 / tensor contraction left inside the guard band is
// re-evaluated from the bit-exact inputs with  d^2 = |x|^2 + |sv|^2 - 2 x.sv  in FP64 (one DFMA per element instead of
// the reference order's sub / mul / add) and an unordered FP64 sum.  Its error is <= ~1e-12 of
// E = sum |coef_i| K_i (1 + gamma log2(e) (|x|^2 + |sv_i|^2)) -- the same order as the distance between libsvm's own
// sequential evaluation and the real number -- so a window whose |dec| > tol2 * (E + |rho|) (tol2 = 1e-10) has the sign
// libsvm computes; the rest (practically none) go on to tier 3, the exact-order kernels above.
//   guard_inputs_kernel : Xg[e][d] = exact_scaled_input(list[e], d)           (entries e < cap)
//   guard_fma_kernel    : grid (window blocks, SV slices); 16 windows x SVT support vectors per thread in registers;
//                         partial sums per slice -> atomicAdd; the last slice to arrive finalises the 16 windows
//                         (and re-zeroes the accumulators, so they need zeroing only once at allocation).
// Entries beyond cap (a guard band mis-configured to be huge) are handed to tier 3 unchanged.
// ---------------------------------------------------------------------------------------------------
#define HAF_G2_WB 16
struct Guard2Args {
    const int* list; const unsigned* list_count; int cap;   // tier-1 guard list, capacity of Xg in entries
    double* Xg;                  // [cap][ldx]: the exact inputs of the listed windows, columns Dsv .. ldx-1 zero
    int ldx;                     // row stride of Xg in doubles: Dsv rounded up to 16 (the DMMA kernel's k-chunks)
    double* xn64;                // [cap] |x|^2 of the rows (guard_norms_kernel; DMMA kernel only)
    const double* svn64;         // [Spad]  sum_d sv_d^2 in double
    double* accum;               // [cap][2]  (decision sum, E), zero on entry, left zero
    unsigned* tickets;           // [cap / WB + 1], zero on entry, left zero
    double tol2;
    int* list2; unsigned* list2_count;   // tier-3 list
    const double* dec_tc;        // audit: the contraction's decision value of every listed window (NaN = not comparable) or NULL
    unsigned* audit_max;         // audit: max over listed windows of |dec_tc - dec_fp64| / (E + |rho|), as float bits
    const unsigned char* guard_flag;   // [W] 1 = inside the guard band; listed windows with 0 are the audit sample: measured, not rewritten
};
// a single goal's handful of guard windows: one THREAD per element (a warp per row would leave most of the GPU idle while
// each lane walks 11 text-emulated values), |x|^2 in a second small kernel
__global__ void __launch_bounds__(256) guard_inputs_flat_kernel(const ExactArgs A, const Guard2Args Q) {
    const unsigned n = min(*Q.list_count, (unsigned)Q.cap);
    const size_t total = (size_t)n * Q.ldx;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const unsigned e = (unsigned)(t / Q.ldx);
        const int d = (int)(t - (size_t)e * Q.ldx);
        Q.Xg[t] = d < A.D ? exact_scaled_input(A, Q.list[e], d) : 0.0;
    }
}
__global__ void __launch_bounds__(256) guard_norms_kernel(const Guard2Args Q) {
    const unsigned n = min(*Q.list_count, (unsigned)Q.cap);
    const int lane = threadIdx.x & 31;
    for (unsigned e = blockIdx.x * 8 + (threadIdx.x >> 5); e < n; e += gridDim.x * 8) {
        double sq = 0.0;
        for (int d = lane; d < Q.ldx; d += 32) { const double v = Q.Xg[(size_t)e * Q.ldx + d]; sq = fma(v, v, sq); }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) Q.xn64[e] = sq;
    }
}
// batches: one warp per listed row: its exact inputs (columns >= D zero up to ldx) and |x|^2 (for the DMMA kernel)
__global__ void __launch_bounds__(256) guard_inputs_kernel(const ExactArgs A, const Guard2Args Q) {
    const unsigned n = min(*Q.list_count, (unsigned)Q.cap);
    const int lane = threadIdx.x & 31;
    for (unsigned e = blockIdx.x * 8 + (threadIdx.x >> 5); e < n; e += gridDim.x * 8) {
        const int w = Q.list[e];
        double sq = 0.0;
        for (int d = lane; d < Q.ldx; d += 32) {
            const double v = d < A.D ? exact_scaled_input(A, w, d) : 0.0;
            Q.Xg[(size_t)e * Q.ldx + d] = v;
            sq = fma(v, v, sq);
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) Q.xn64[e] = sq;
    }
}
// one finished window of tier 2 (its decision sum and guard scale are complete in accum): audit, decision value, tier-3 list
__device__ __forceinline__ void guard_finalize_entry(const ExactArgs& A, const Guard2Args& Q, unsigned e) {
    const double sum = atomicAdd(Q.accum + (size_t)e * 2, 0.0), E = atomicAdd(Q.accum + (size_t)e * 2 + 1, 0.0);
    Q.accum[(size_t)e * 2] = 0.0; Q.accum[(size_t)e * 2 + 1] = 0.0;
    const int w = Q.list[e];
    const double dv = sum - A.rho;
    if (Q.dec_tc) {   // audit of the FP32 / tensor contraction against this FP64 value, in the guard band's own unit
        const double tcv = Q.dec_tc[w];
        const float rel = (float)(fabs(tcv - dv) / (E + fabs(A.rho)));
        if (rel == rel) atomicMax(Q.audit_max, __float_as_uint(rel));
    }
    // a sample window keeps the contraction's value: what a row gets must not depend on whether its index was sampled
    if (!Q.guard_flag || Q.guard_flag[w]) {
        A.dec[w] = dv;
        if (!(fabs(dv) > Q.tol2 * (E + fabs(A.rho)))) Q.list2[atomicAdd(Q.list2_count, 1u)] = w;
    }
}
// Work item = (group of 16 windows, slice of 256 * SVT support vectors), items walked grid-stride by one CTA per SM: a
// launch of ~5 k guard windows is 344 groups x 4 slices = 1376 items = 9.3 rounds over 148 SMs (the round-1 grid of
// (SMs, slices) CTAs walked groups per slice: 2.3 rounds, the last one a third full).  The SV matrix (L2-resident, 5 MB)
// is read DB = 8 dimensions ahead into registers: one 176-register CTA per SM has only two warps per scheduler, and two
// dimensions of look-ahead (128 DFMA issue clocks) did not cover an L2 round trip (ncu r2: long-scoreboard 2.6 of 4.5 stall
// cycles per issue, FP64 pipe 32 %).
template <int SVT>
__global__ void __launch_bounds__(256, 1) guard_fma_kernel(const ExactArgs A, const Guard2Args Q, int nslices) {
    constexpr int WB = HAF_G2_WB, DB = 8;
    extern __shared__ double g2s[];       // xs [Dsv][WB], then xn [WB], red [8][WB][2]
    const int Dsv = A.Dsv, Spad = A.Spad;
    double* xs = g2s;
    double* xn = g2s + (size_t)Dsv * WB;
    double* red = xn + WB;
    __shared__ unsigned s_ticket;
    const unsigned total = *Q.list_count;
    const unsigned n = min(total, (unsigned)Q.cap);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x == 0)   // overflow of the tier-2 buffers: straight to tier 3
        for (unsigned e = (unsigned)Q.cap + threadIdx.x; e < total; e += blockDim.x)
            if (!Q.guard_flag || Q.guard_flag[Q.list[e]]) Q.list2[atomicAdd(Q.list2_count, 1u)] = Q.list[e];
    const double g2 = A.gamma * 1.4426950408889634;
    const unsigned ngroups = (n + WB - 1) / WB;
    const unsigned nitems = ngroups * (unsigned)nslices;
    for (unsigned item = blockIdx.x; item < nitems; item += gridDim.x) {
        const unsigned e0 = (item / (unsigned)nslices) * WB;
        const int i0 = (int)(item % (unsigned)nslices) * (256 * SVT);
        const int nb = min((unsigned)WB, n - e0);
        __syncthreads();
        for (int t = threadIdx.x; t < WB * Dsv; t += blockDim.x) {
            const int b = t / Dsv, d = t - b * Dsv;    // coalesced read of Xg rows
            xs[d * WB + b] = b < nb ? Q.Xg[(size_t)(e0 + b) * Q.ldx + d] : 0.0;
        }
        __syncthreads();
        for (int b = warp; b < WB; b += 8) {
            double sq = 0.0;
            for (int d = lane; d < Dsv; d += 32) { const double v = xs[d * WB + b]; sq = fma(v, v, sq); }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
            if (lane == 0) xn[b] = sq;
        }
        __syncthreads();
        double acc[WB][SVT];
#pragma unroll
        for (int b = 0; b < WB; b++)
#pragma unroll
            for (int k = 0; k < SVT; k++) acc[b][k] = 0.0;
        const int ia = i0 + threadIdx.x;
        bool in[SVT];
#pragma unroll
        for (int k = 0; k < SVT; k++) in[k] = ia + 256 * k < Spad;
        double cur[DB][SVT], nxt[DB][SVT];
#pragma unroll
        for (int q = 0; q < DB; q++)
#pragma unroll
            for (int k = 0; k < SVT; k++) cur[q][k] = (q < Dsv && in[k]) ? A.sv64T[(size_t)q * Spad + ia + 256 * k] : 0.0;
        for (int d0 = 0; d0 < Dsv; d0 += DB) {
#pragma unroll
            for (int q = 0; q < DB; q++)
#pragma unroll
                for (int k = 0; k < SVT; k++) nxt[q][k] = (d0 + DB + q < Dsv && in[k]) ? A.sv64T[(size_t)(d0 + DB + q) * Spad + ia + 256 * k] : 0.0;
#pragma unroll
            for (int q = 0; q < DB; q++) {
                if (d0 + q < Dsv) {   // uniform
                    const double2* xr = reinterpret_cast<const double2*>(xs + (d0 + q) * WB);
#pragma unroll
                    for (int b2 = 0; b2 < WB / 2; b2++) {
                        const double2 xv = xr[b2];   // broadcast 128-bit shared load: two windows
#pragma unroll
                        for (int k = 0; k < SVT; k++) {
                            acc[2 * b2][k] = fma(xv.x, cur[q][k], acc[2 * b2][k]);
                            acc[2 * b2 + 1][k] = fma(xv.y, cur[q][k], acc[2 * b2 + 1][k]);
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < DB; q++)
#pragma unroll
                for (int k = 0; k < SVT; k++) cur[q][k] = nxt[q][k];
        }
        double ds[WB], es[WB];
#pragma unroll
        for (int b = 0; b < WB; b++) { ds[b] = 0.0; es[b] = 0.0; }
#pragma unroll
        for (int k = 0; k < SVT; k++) {
            const int i = ia + 256 * k;
            if (i < A.S) {
                const double cf = A.coef64[i], sn = Q.svn64[i];
#pragma unroll
                for (int b = 0; b < WB; b++) {
                    const double base = xn[b] + sn;
                    const double d2 = fmax(fma(-2.0, acc[b][k], base), 0.0);
                    const double tk = cf * exp(-A.gamma * d2);
                    ds[b] += tk;
                    es[b] = fma(fabs(tk), fma(g2, base, 1.0), es[b]);
                }
            }
        }
#pragma unroll
        for (int b = 0; b < WB; b++) {
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) {
                ds[b] += __shfl_xor_sync(0xffffffffu, ds[b], o);
                es[b] += __shfl_xor_sync(0xffffffffu, es[b], o);
            }
            if (lane == 0) { red[(warp * WB + b) * 2] = ds[b]; red[(warp * WB + b) * 2 + 1] = es[b]; }
        }
        __syncthreads();
        if (threadIdx.x < 2 * WB) {
            const int b = threadIdx.x >> 1, c = threadIdx.x & 1;
            double v = 0.0;
            for (int w8 = 0; w8 < 8; w8++) v += red[(w8 * WB + b) * 2 + c];
            if (b < nb) atomicAdd(Q.accum + (size_t)(e0 + b) * 2 + c, v);
        }
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = atomicAdd(Q.tickets + e0 / WB, 1u);
        __syncthreads();
        if (s_ticket == (unsigned)nslices - 1) {   // every slice of these windows has been added: finalise
            __threadfence();
            if (threadIdx.x < nb) guard_finalize_entry(A, Q, e0 + threadIdx.x);
            if (threadIdx.x == 0) Q.tickets[e0 / WB] = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Guard band tier 2 on the FP64 TENSOR CORES (mma.sync.m8n8k4.f64, DMMA).  The DFMA kernel above reached 29-32 % of the FP64
// pipe (ncu r2: two warps per scheduler at 176-232 registers cannot cover the latencies of a 32-accumulator register tile)
// and spends one issue slot per 32 FMAs; a DMMA does 256 FMAs per slot with 4 registers of operands, which frees both the
// schedulers and the register file (2 CTAs per SM).  B200 keeps full-rate FP64 tensor cores (the B300 of the guides does not).
// Same contraction: C[w][i] = x_w . sv_i over the zero-padded K = ldx dimensions, then d^2 = |x|^2 + |sv|^2 - 2C, the
// exp / coef / row-sum epilogue and the ticket that lets the last SV block of a window block finalise it.  A DMMA is a chain
// of FP64 FMAs in an unspecified order: the error is a few 1e-16 of the operands' products, the band's tolerance is 1e-10 E.
//   CTA tile 64 windows x 128 SVs, 8 warps (2 x 4) of 32 x 32 = 4 x 4 m8n8 tiles; k-chunks of 16 dimensions through a 3-stage
//   cp.async ring: X chunk [64][16 (+4)] from Xg, SV chunk [16][128 (+4)] from sv64T (row paddings make every fragment load
//   conflict-free: 8-byte lanes of a half-warp fall into 16 distinct bank pairs).
// grid-stride over items = (window blocks) x nsb SV blocks; sv64T must hold ldx rows (rows >= Dsv zero).
// ---------------------------------------------------------------------------------------------------
#define HAF_GD_WB 64
#define HAF_GD_SB 128
#define HAF_GD_KC 16
#define HAF_GD_APAD 20
#define HAF_GD_BPAD 132
#define HAF_GD_STAGES 3
#define HAF_GD_STAGE_DOUBLES (HAF_GD_WB * HAF_GD_APAD + HAF_GD_KC * HAF_GD_BPAD)
#define HAF_GD_SMEM_BYTES (HAF_GD_STAGES * HAF_GD_STAGE_DOUBLES * 8)
__device__ __forceinline__ void cp_async16_zfill(void* smem, const void* gmem, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    const int n = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(n));
}
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__global__ void __launch_bounds__(256, 2) guard_dmma_kernel(const ExactArgs A, const Guard2Args Q, int nsb) {
    extern __shared__ __align__(16) double gds[];   // [STAGES][ X chunk | SV chunk ]
    __shared__ unsigned s_ticket;
    const unsigned total = *Q.list_count;
    const unsigned n = min(total, (unsigned)Q.cap);
    if (blockIdx.x == 0)   // overflow of the tier-2 buffers: straight to tier 3
        for (unsigned e = (unsigned)Q.cap + threadIdx.x; e < total; e += blockDim.x)
            if (!Q.guard_flag || Q.guard_flag[Q.list[e]]) Q.list2[atomicAdd(Q.list2_count, 1u)] = Q.list[e];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp & 1, wn = warp >> 1;           // warp tile: windows wm * 32 .., SVs wn * 32 ..
    const int g4 = lane >> 2, t4 = lane & 3;
    const int Spad = A.Spad, ldx = Q.ldx, nk = ldx / HAF_GD_KC;
    const double g2 = A.gamma * 1.4426950408889634;
    const unsigned ngroups = (n + HAF_GD_WB - 1) / HAF_GD_WB;
    const unsigned nitems = ngroups * (unsigned)nsb;
    for (unsigned item = blockIdx.x; item < nitems; item += gridDim.x) {
        const unsigned e0 = (item / (unsigned)nsb) * HAF_GD_WB;
        const int i0 = (int)(item % (unsigned)nsb) * HAF_GD_SB;
        const int nrows = (int)min((unsigned)HAF_GD_WB, n - e0);
        auto load_stage = [&](int stage, int kc) {
            double* As = gds + (size_t)stage * HAF_GD_STAGE_DOUBLES;
            double* Bs = As + HAF_GD_WB * HAF_GD_APAD;
            const int d0 = kc * HAF_GD_KC;
#pragma unroll
            for (int q = 0; q < 2; q++) {   // X chunk: 64 rows x 8 sixteen-byte pieces
                const int idx = tid + 256 * q, row = idx >> 3, c = idx & 7;
                const bool ok = row < nrows;
                cp_async16_zfill(As + row * HAF_GD_APAD + 2 * c, Q.Xg + (size_t)(e0 + (ok ? row : 0)) * ldx + d0 + 2 * c, ok);
            }
#pragma unroll
            for (int q = 0; q < 4; q++) {   // SV chunk: 16 rows x 64 sixteen-byte pieces
                const int idx = tid + 256 * q, row = idx >> 6, c = idx & 63;
                cp_async16_zfill(Bs + row * HAF_GD_BPAD + 2 * c, A.sv64T + (size_t)(d0 + row) * Spad + i0 + 2 * c, true);
            }
        };
        double acc[4][4][2];
#pragma unroll
        for (int mb = 0; mb < 4; mb++)
#pragma unroll
            for (int nb = 0; nb < 4; nb++) { acc[mb][nb][0] = 0.0; acc[mb][nb][1] = 0.0; }
        __syncthreads();   // the previous item's readers are done with the ring
        for (int s = 0; s < HAF_GD_STAGES - 1; s++) { if (s < nk) load_stage(s, s); cp_async_commit(); }
        for (int kc = 0; kc < nk; kc++) {
            cp_async_wait<HAF_GD_STAGES - 2>();
            __syncthreads();
            if (kc + HAF_GD_STAGES - 1 < nk) load_stage((kc + HAF_GD_STAGES - 1) % HAF_GD_STAGES, kc + HAF_GD_STAGES - 1);
            cp_async_commit();
            const double* As = gds + (size_t)(kc % HAF_GD_STAGES) * HAF_GD_STAGE_DOUBLES;
            const double* Bs = As + HAF_GD_WB * HAF_GD_APAD;
#pragma unroll
            for (int ks = 0; ks < HAF_GD_KC / 4; ks++) {
                double a[4], b[4];
#pragma unroll
                for (int mb = 0; mb < 4; mb++) a[mb] = As[(wm * 32 + mb * 8 + g4) * HAF_GD_APAD + ks * 4 + t4];
#pragma unroll
                for (int nb = 0; nb < 4; nb++) b[nb] = Bs[(ks * 4 + t4) * HAF_GD_BPAD + wn * 32 + nb * 8 + g4];
#pragma unroll
                for (int mb = 0; mb < 4; mb++)
#pragma unroll
                    for (int nb = 0; nb < 4; nb++) dmma_m8n8k4(acc[mb][nb][0], acc[mb][nb][1], a[mb], b[nb]);
            }
        }
        cp_async_wait<0>();
        // epilogue: this thread's rows e0 + wm*32 + mb*8 + g4, columns i0 + wn*32 + nb*8 + 2*t4 + {0, 1}
        double cf[4][2], sn[4][2];
#pragma unroll
        for (int nb = 0; nb < 4; nb++)
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int i = i0 + wn * 32 + nb * 8 + 2 * t4 + j;
                cf[nb][j] = A.coef64[i];     // padding support vectors: coef 0
                sn[nb][j] = Q.svn64[i];
            }
#pragma unroll
        for (int mb = 0; mb < 4; mb++) {
            const int r = wm * 32 + mb * 8 + g4;
            const bool live = r < nrows;
            const double xn = live ? Q.xn64[e0 + r] : 0.0;
            double ds = 0.0, es = 0.0;
#pragma unroll
            for (int nb = 0; nb < 4; nb++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const double base = xn + sn[nb][j];
                    const double d2 = fmax(fma(-2.0, acc[mb][nb][j], base), 0.0);
                    const double tk = cf[nb][j] * exp(-A.gamma * d2);
                    ds += tk;
                    es = fma(fabs(tk), fma(g2, base, 1.0), es);
                }
            ds += __shfl_xor_sync(0xffffffffu, ds, 1); es += __shfl_xor_sync(0xffffffffu, es, 1);
            ds += __shfl_xor_sync(0xffffffffu, ds, 2); es += __shfl_xor_sync(0xffffffffu, es, 2);
            if (t4 == 0 && live) {
                atomicAdd(Q.accum + (size_t)(e0 + r) * 2, ds);
                atomicAdd(Q.accum + (size_t)(e0 + r) * 2 + 1, es);
            }
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) s_ticket = atomicAdd(Q.tickets + e0 / HAF_GD_WB, 1u);
        __syncthreads();
        if (s_ticket == (unsigned)nsb - 1) {   // every SV block of these windows has been added: finalise
            __threadfence();
            if (tid < nrows) guard_finalize_entry(A, Q, e0 + tid);
            if (tid == 0) Q.tickets[e0 / HAF_GD_WB] = 0;
        }
    }
}

// label -> graspsgrid value (server.cpp:843) scattered into the unit grids
__global__ void label_scatter_kernel(const double* __restrict__ dec, const int2* __restrict__ win,
                                     const unsigned* __restrict__ win_count, int G, int unit_base, int gv_pos, int gv_neg,
                                     signed char* __restrict__ labelgrid) {
    const unsigned W = *win_count;
    const unsigned w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    const int2 uc = win[w];
    labelgrid[(size_t)(uc.x - unit_base) * G * G + uc.y] = (signed char)((dec[w] > 0.0) ? gv_pos : gv_neg);  // svm.cpp:2516
}

// ---------------------------------------------------------------------------------------------------
// a13: 29-tap weighted neighbourhood score + first strict maximum per unit (server.cpp:865-897).
// grid = (ceil(G*G/256), U).  unit_top key: (val + 2^20) << 32 | (0xFFFFFFFF - cell): max == first strict max.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) score_kernel(const signed char* __restrict__ labelgrid, int G,
                                                    const UnitParams* __restrict__ units, float* __restrict__ evals,
                                                    unsigned long long* __restrict__ unit_top) {
    const int u = blockIdx.y;
    if (units[u].cloud < 0) return;
    const int GG = G * G;
    const int cell = blockIdx.x * 256 + threadIdx.x;
    const signed char* L = labelgrid + (size_t)u * GG;
    int e = 0;
    bool have = cell < GG;
    if (have) {
        const int row = cell / G, col = cell - row * G;
        if (L[cell] >= 0) {  // graspsgrid >= 0 only where the mask is true, i.e. 7 <= row,col <= G-8: taps stay inside
#define LG(dr, dc) ((int)L[(row + (dr)) * G + (col + (dc))])
            e = 1 * LG(-2, -2) + 2 * LG(-2, -1) + 3 * LG(-2, 0) + 2 * LG(-2, 1) + 1 * LG(-2, 2) +
                2 * LG(-1, -2) + 3 * LG(-1, -1) + 4 * LG(-1, 0) + 3 * LG(-1, 1) + 2 * LG(-1, 2) +
                2 * LG(0, -4) + 2 * LG(0, -3) + 3 * LG(0, -2) + 4 * LG(0, -1) + 55 * LG(0, 0) + 4 * LG(0, 1) + 3 * LG(0, 2) + 2 * LG(0, 3) + 2 * LG(0, 4) +
                2 * LG(1, -2) + 3 * LG(1, -1) + 4 * LG(1, 0) + 3 * LG(1, 1) + 2 * LG(1, 2) +
                1 * LG(2, -2) + 2 * LG(2, -1) + 3 * LG(2, 0) + 2 * LG(2, 1) + 1 * LG(2, 2);
#undef LG
        }
        evals[(size_t)u * GG + cell] = (float)e;
    }
    unsigned long long key = have ? (((unsigned long long)(unsigned)(e + (1 << 20))) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)cell) : 0ull;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    __shared__ unsigned long long sk[8];
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) key = sk[w] > key ? sk[w] : key;
        atomicMax(unit_top + u, key);
    }
}

// a14: among cells == topval, the first (row-major) strictly longest horizontal run; cell = (row, col_end - len/2)
// (server.cpp:905-932).  One warp per (unit, row).  unit_run key: len << 32 | (0xFFFF - row) << 16 | col_mid.
__global__ void __launch_bounds__(256) tie_rule_kernel(const float* __restrict__ evals, int G,
                                                       const UnitParams* __restrict__ units,
                                                       const unsigned long long* __restrict__ unit_top,
                                                       unsigned long long* __restrict__ unit_run) {
    const int u = blockIdx.y;
    if (units[u].cloud < 0) return;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= G) return;
    const int lane = threadIdx.x & 31;
    const float topval = (float)((int)(unsigned)(unit_top[u] >> 32) - (1 << 20));
    const float* E = evals + (size_t)u * G * G + (size_t)row * G;
    // sequential semantics reproduced with a warp-wide segmented scan over chunks of 32 columns
    int carry = 0;       // length of the run ending at the previous column
    int best_len = 0, best_col = 0;
    for (int c0 = 0; c0 < G; c0 += 32) {
        const int col = c0 + lane;
        const bool hit = (col < G) && (E[col] == topval);
        const unsigned b = __ballot_sync(0xffffffffu, hit);
        // run length ending at this lane = number of consecutive set bits ending at `lane` (+ carry if they reach bit 0)
        const unsigned upto = b << (31 - lane);          // bit 31 = this lane, lower lanes below
        const int ones = __clz(~upto);                   // consecutive ones from the top
        int len = hit ? ones : 0;
        if (hit && ones == lane + 1) len += carry;
        // the reference updates "longest" incrementally while a run grows, so the winner is the FIRST run whose final
        // length is the maximum, at position col_end - len/2; a later run replaces it only if strictly longer.
        const bool next_hit = (col + 1 < G) && (E[col + 1] == topval);
        const bool run_end = hit && !next_hit;
        // candidate key: longer run wins, equal length -> smaller column (the earlier run)
        unsigned cand = run_end ? (((unsigned)len << 16) | (0xFFFFu - (unsigned)(col - len / 2))) : 0u;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const unsigned other = __shfl_xor_sync(0xffffffffu, cand, o);
            cand = other > cand ? other : cand;
        }
        const int cand_len = (int)(cand >> 16);
        if (cand_len > best_len) { best_len = cand_len; best_col = 0xFFFF - (int)(cand & 0xFFFFu); }
        carry = __shfl_sync(0xffffffffu, len, 31);
    }
    if (lane == 0 && best_len > 0) {
        const unsigned long long key = ((unsigned long long)(unsigned)best_len << 32) |
                                       ((unsigned long long)(0xFFFFu - (unsigned)row) << 16) | (unsigned long long)(unsigned)best_col;
        atomicMax(unit_run + u, key);
    }
}

struct JobResult {  // per job (cloud x request)
    int row, col, roll, topval;
    int rolls_done, n_windows, pad0, pad1;
};
struct JobParams {
    int return_only_best, graspval_top, n_rolls_active, roll_begin;  // rolls [roll_begin, n_rolls_active) are evaluated
};

// top cell of a unit after the tie rule (id_row_top_all, id_col_top_all, topval_gp_all of show_predicted_gps, :881-932)
__device__ __forceinline__ int unit_top_cell(const unsigned long long* __restrict__ unit_top, const unsigned long long* __restrict__ unit_run,
                                             int u, int G, int* row, int* col) {
    const int val = (int)(unsigned)(unit_top[u] >> 32) - (1 << 20);
    const unsigned long long rk = unit_run[u];
    if (rk) {
        *row = 0xFFFF - (int)((rk >> 16) & 0xFFFFu);
        *col = (int)(rk & 0xFFFFu);
    } else {   // no cell EQUALS topval (probability mode: topval is a truncated float): the first-maximum cell stays (:881-892)
        const unsigned cell = 0xFFFFFFFFu - (unsigned)(unit_top[u] & 0xFFFFFFFFull);
        *row = (int)(cell / (unsigned)G);
        *col = (int)(cell % (unsigned)G);
    }
    return val;
}

// per-unit tops (after the tie rule) + a15 cross-roll reduction with the loop_control rules
// (server.cpp:362-365 early exit, :953-960 strict >).  One thread per job.  best_M (optional, pinned host memory [n_jobs][16]):
// mat_transform of each job's winning roll, taken from units (jobs whose unit parameters were built on the device).
__global__ void reduce_rolls_kernel(const unsigned long long* __restrict__ unit_top, const unsigned long long* __restrict__ unit_run,
                                    const unsigned* __restrict__ unit_windows, const JobParams* __restrict__ jobs, int n_jobs,
                                    int R, int G, int* __restrict__ per_roll_top /*[n_jobs][R][3]*/,
                                    JobResult* __restrict__ results, const UnitParams* __restrict__ units, float* __restrict__ best_M) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_jobs) return;
    const JobParams jp = jobs[j];
    int best = -1000, brow = -1, bcol = -1, broll = -1, done = 0, nwin = 0;
    for (int roll = 0; roll < R; roll++) {
        const int u = j * R + roll;
        int row = -1, col = -1, val = -1000;
        if (roll >= jp.roll_begin && roll < jp.n_rolls_active) val = unit_top_cell(unit_top, unit_run, u, G, &row, &col);
        per_roll_top[(j * R + roll) * 3 + 0] = row;
        per_roll_top[(j * R + roll) * 3 + 1] = col;
        per_roll_top[(j * R + roll) * 3 + 2] = val;
    }
    for (int roll = jp.roll_begin; roll < jp.n_rolls_active; roll++) {
        if (jp.return_only_best && best >= jp.graspval_top) break;  // :362-365
        const int u = j * R + roll;
        const int val = per_roll_top[u * 3 + 2];
        if (val > best) { best = val; brow = per_roll_top[u * 3]; bcol = per_roll_top[u * 3 + 1]; broll = roll; }  // :953
        nwin += (int)unit_windows[u];
        done++;
    }
    JobResult r;
    r.row = brow; r.col = bcol; r.roll = broll; r.topval = best; r.rolls_done = done; r.n_windows = nwin; r.pad0 = r.pad1 = 0;
    results[j] = r;
    if (best_M && broll >= 0) {   // four 16-byte stores (UnitParams and the pinned rows are 64-byte aligned)
        const float4* src = reinterpret_cast<const float4*>(units[j * R + broll].M);
        float4* dst = reinterpret_cast<float4*>(best_M + (size_t)j * 16);
        for (int k = 0; k < 4; k++) dst[k] = src[k];
    }
}

// ---------------------------------------------------------------------------------------------------
// a16: grasp pose in world coordinates (transform_gp_in_wcs_and_publish, server.cpp:1274-1401).  Launched only by the
// grasp entry points: grasp_unit_kernel once per chunk while the chunk's heights are resident, grasp_gather_kernel once per
// call after reduce_rolls_kernel.
// ---------------------------------------------------------------------------------------------------
struct GraspRec {      // = haf_grasp (include/hafgpu.h)
    int eval;
    float roll;
    double gp1[3], gp2[3], avg[3], approach[3];
    int row, col, roll_index, reserved;
};
static_assert(sizeof(GraspRec) == 120, "GraspRec layout");
struct UnitPose {      // one (request, roll): inverse of the transform rebuilt from the double approach vector (:1276-1334), row-major
    float Minv[16];
};

// Minv: the roll's UnitPose; Mrow2: third row of generate_grid's matrix of the roll (:1370-1374); heights: the roll's G x G grid,
// not read when roll < 0 (no roll evaluated: h_locmax stays -10).  Float / double operations in the reference's order, no FMA.
__device__ void grasp_pose(const float* __restrict__ Minv, const float* __restrict__ Mrow2, const float* __restrict__ heights, int G,
                           int row, int col, int roll, int roll_step_deg, int eval, GraspRec* __restrict__ out) {
    const float x_gp = __fdiv_rn(-(float)(G / 2 - row), 100.0f);   // :1339
    const float y_gp = __fdiv_rn(-(float)(G / 2 - col), 100.0f);   // :1340
    float h = -10.0f;
    if (roll >= 0)
        for (int rz = -4; rz < 5; rz++)           // :1343
            for (int cz = -4; cz < 4; cz++) {     // :1344 (asymmetric column range)
                const int r = row + rz, c = col + cz;
                if (r >= 0 && c >= 0 && r < G && c < G) {
                    const float v = heights[r * G + c];
                    if (h < v) h = v;
                }
            }
    const float z_gp = __double2float_rn(__dsub_rn((double)h, 0.01));   // :1354 (float -= double)
    const float gp1[4] = {__fsub_rn(x_gp, 0.03f), y_gp, z_gp, 1.0f};   // :1360-1367
    const float gp2[4] = {__fadd_rn(x_gp, 0.03f), y_gp, z_gp, 1.0f};
    out->eval = eval;
    out->roll = __double2float_rn(__ddiv_rn(__dmul_rn((double)(roll * roll_step_deg), 3.141592653), 180.0));   // :1401
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const float* m = Minv + 4 * i;
        const float g1 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], gp1[0]), __fmul_rn(m[1], gp1[1])), __fmul_rn(m[2], gp1[2])), __fmul_rn(m[3], gp1[3]));
        const float g2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], gp2[0]), __fmul_rn(m[1], gp2[1])), __fmul_rn(m[2], gp2[2])), __fmul_rn(m[3], gp2[3]));
        out->gp1[i] = (double)g1;                                   // :1389-1394
        out->gp2[i] = (double)g2;
        out->avg[i] = __ddiv_rn((double)__fadd_rn(g1, g2), 2.0);   // :1395-1397 (float sum, double division)
        out->approach[i] = (double)Mrow2[i];
    }
    out->row = row; out->col = col; out->roll_index = roll; out->reserved = 0;
}

// one thread per unit of the chunk, right after tie_rule_kernel: the unit's top cell (as reduce_rolls_kernel decodes it) and its
// pose, eval = max(top - 20, 10) (:962-972), into unit_grasp -- an array of the whole call, so it outlives the chunk's buffers.
// units / unit_top / unit_run / keys_heights / unit_grasp: the chunk's slices; poses [n_requests][R], job_pose [job] -> request.
__global__ void grasp_unit_kernel(const unsigned* __restrict__ keys_heights, int G, const UnitParams* __restrict__ units, int n_units,
                                  const unsigned long long* __restrict__ unit_top, const unsigned long long* __restrict__ unit_run,
                                  const UnitPose* __restrict__ poses, const int* __restrict__ job_pose, int R, int roll_step_deg,
                                  GraspRec* __restrict__ unit_grasp) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_units) return;
    const UnitParams* up = units + u;
    if (up->cloud < 0) return;   // roll not evaluated: its record is left as it is
    int row, col;
    const int val = unit_top_cell(unit_top, unit_run, u, G, &row, &col);
    grasp_pose(poses[job_pose[up->job] * R + up->roll].Minv, up->M + 8, reinterpret_cast<const float*>(keys_heights) + (size_t)u * G * G, G,
               row, col, up->roll, roll_step_deg, max(val - 20, 10), unit_grasp + u);
}

// one thread per job, after reduce_rolls_kernel: the winning unit's record with eval = topval - 20 (:390); a job that evaluated
// no roll gets the reference's pose for roll -1 (roll 0's transforms, no height).  job_grasp: pinned host memory (UVA)
__global__ void grasp_gather_kernel(const JobResult* __restrict__ results, int n_jobs, const UnitParams* __restrict__ units,
                                    const UnitPose* __restrict__ poses, const int* __restrict__ job_pose, int R, int G, int roll_step_deg,
                                    const GraspRec* __restrict__ unit_grasp, GraspRec* __restrict__ job_grasp) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_jobs) return;
    const JobResult r = results[j];
    if (r.roll >= 0) {
        GraspRec g = unit_grasp[j * R + r.roll];
        g.eval = r.topval - 20;
        job_grasp[j] = g;
    } else {
        grasp_pose(poses[job_pose[j] * R].Minv, units[j * R].M + 8, nullptr, G, r.row, r.col, -1, roll_step_deg, r.topval - 20, job_grasp + j);
    }
}

// ---------------------------------------------------------------------------------------------------
// Unit parameters built on the device (haf_search_batch_requests): the host evaluates the libm calls once per distinct
// approach vector (hafhost::ApproachTrig) and once per roll (hafhost::RollTrig); one thread per unit composes the rest with
// the host's own source (haf_host.hpp: compose_transform, compose_mask, invert4), so the result is bit-equal to the host
// build of haf_search.
// ---------------------------------------------------------------------------------------------------
struct JobSpec {         // one (cloud, request): 64 bytes
    double center[3];
    int cloud, approach;     // approach: index into the ApproachTrig table
    int gripper_opening_width, area_x, area_y;   // area truncated to int like server.cpp:266-267
    int roll_begin, n_rolls_active, return_only_best, graspval_top, pad;
};
static_assert(sizeof(JobSpec) == 64, "JobSpec layout");
// one thread per unit u = job * R + roll: UnitParams (the full matrix), JobParams (roll 0's thread) and, with poses != NULL, the
// inverse of the WCS transform (one UnitPose per unit)
__global__ void expand_units_kernel(const JobSpec* __restrict__ specs, const hafhost::ApproachTrig* __restrict__ approaches,
                                    const hafhost::RollTrig* __restrict__ rolls, int n_jobs, int R, int G, UnitParams* __restrict__ units,
                                    JobParams* __restrict__ jobs, UnitPose* __restrict__ poses) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_jobs * R) return;
    const int j = u / R, roll = u - j * R;
    const JobSpec js = specs[j];
    const hafhost::ApproachTrig at = approaches[js.approach];
    const hafhost::RollTrig rt = rolls[roll];
    UnitParams up;
    hafhost::compose_transform(at.grid, rt, js.gripper_opening_width, js.center, up.M);
    const hafhost::MaskConsts mc = hafhost::compose_mask(G, rt, js.area_x, js.area_y);
    up.sa = mc.sa; up.ca = mc.ca; up.cx1 = mc.cx1; up.cy1 = mc.cy1; up.cx2 = mc.cx2; up.cy2 = mc.cy2;
    up.cx3 = mc.cx3; up.cy3 = mc.cy3; up.cx4 = mc.cx4; up.cy4 = mc.cy4;
    up.cloud = (roll >= js.roll_begin && roll < js.n_rolls_active) ? js.cloud : -1;
    up.job = j; up.roll = roll;
    up.pad[0] = up.pad[1] = up.pad[2] = 0;
    units[u] = up;
    if (roll == 0) {
        JobParams jp;
        jp.return_only_best = js.return_only_best; jp.graspval_top = js.graspval_top;
        jp.n_rolls_active = js.n_rolls_active; jp.roll_begin = js.roll_begin;
        jobs[j] = jp;
    }
    if (poses) {
        float Mw[16];
        hafhost::compose_transform(at.wcs, rt, js.gripper_opening_width, js.center, Mw);
        hafhost::invert4(Mw, poses[u].Minv);
    }
}

// parameter block upload: src is pinned HOST memory read over PCIe through its UVA address (see run_jobs)
__global__ void copy_params_kernel(const uint4* __restrict__ src_host, uint4* __restrict__ dst, size_t n16) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n16; i += stride) dst[i] = src_host[i];
}

// counters: [0] windows of this chunk, [1] guard list entries, [13] of which audit-only, [6] exact-order windows of this chunk
// -> running totals in [8], [9] (guard band), [14] (audit only), [11]; [12] = audit maximum (float bits, whole call)
__global__ void accumulate_counts_kernel(unsigned* cnt) {
    cnt[8] += cnt[0];
    cnt[9] += cnt[1] - cnt[13];   // [1] counts the audit sample too; [13] = listed windows outside the guard band (audit only)
    cnt[14] += cnt[13];
    cnt[13] = 0;
    cnt[11] += cnt[6];   // windows that went on to the exact-order kernels (tier 3)
    cnt[6] = 0;
}

// host-staged batches run their chunks alternately on several streams, each with its own counter block of 16 words: fold the
// others' totals into the first
__global__ void merge_counts_kernel(unsigned* cnt, int n_more) {
    for (int k = 1; k <= n_more; k++) {
        const unsigned* o = cnt + 16 * k;
        cnt[8] += o[8]; cnt[9] += o[9]; cnt[14] += o[14]; cnt[11] += o[11];
        cnt[2] |= o[2]; cnt[3] |= o[3]; cnt[10] |= o[10];
        cnt[12] = max(cnt[12], o[12]);   // audit maximum: bits of a non-negative float order like the float
        *reinterpret_cast<unsigned long long*>(cnt + 4) += *reinterpret_cast<const unsigned long long*>(o + 4);
    }
}

// ---------------------------------------------------------------------------------------------------
// libsvm front ends (SURVEY 8f-3): svm-predict / svm-scale on rows given in libsvm's sparse text layout (CSR here).
// ---------------------------------------------------------------------------------------------------
// dense[r][index-1] = value for the entries of rows [0, n_rows); dense must be zeroed (absent = 0, svm.cpp:328-364).
__global__ void csr_to_dense_kernel(const long long* __restrict__ row_ptr, const int* __restrict__ index, const double* __restrict__ value,
                                    int n_rows, int width, double* __restrict__ dense) {
    const int r = blockIdx.x;
    if (r >= n_rows) return;
    const long long base = row_ptr[0];
    for (long long e = row_ptr[r] - base + threadIdx.x; e < row_ptr[r + 1] - base; e += blockDim.x) {
        const int i = index[e];
        if (i >= 1 && i <= width) dense[(size_t)r * width + (i - 1)] = value[e];
    }
}
// SVM operands of given inputs: tensor mode (Xh != NULL): fp16 hi/lo in the k-block tiled layout (kt_off) + ||x||^2 of the float values;
// SIMT mode (Xf != NULL): feature-major floats [Kpad][ldx] + ||x||^2.  One warp per row.
__global__ void __launch_bounds__(256) pack_svm_inputs_kernel(const double* __restrict__ dense, int n_rows, int width, int Krow, int KB,
                                                              __half* __restrict__ Xh, __half* __restrict__ Xl /*NULL: hi only*/, float* __restrict__ Xf,
                                                              size_t ldx, int Kpad, float* __restrict__ xn, double* __restrict__ dec_acc, float* __restrict__ asum_acc) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    float sq = 0.0f;
    const int K = Xh ? Krow : Kpad;
    for (int d = lane; d < K; d += 32) {
        const float xf = d < width ? (float)dense[(size_t)r * width + d] : 0.0f;
        if (Xh) {
            const float xc = fminf(fmaxf(xf, -65504.0f), 65504.0f);
            const __half hi = __float2half_rn(xc);
            const __half lo = __float2half_rn(xc - __half2float(hi));
            Xh[kt_off((size_t)r, d, KB)] = hi;
            if (Xl) Xl[kt_off((size_t)r, d, KB)] = lo;
            const float v = __half2float(hi) + __half2float(lo);
            sq = fmaf(v, v, sq);
            if (!(fabsf(xf) < 65504.0f)) sq = __int_as_float(0x7f800000);   // clamped or NaN: force the exact path
        } else {
            Xf[(size_t)d * ldx + r] = xf;
            sq = fmaf(xf, xf, sq);
        }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    __syncwarp();   // the zeros the lanes wrote into the extra columns above come first
    if (lane == 0) {
        const bool ok = !Xh || sq < 1.3e5f;
        xn[r] = ok ? sq : __int_as_float(0x7f800000);
        if (dec_acc) { dec_acc[r] = 0.0; asum_acc[r] = 0.0f; }   // the tensor contraction accumulates into them
        if (Xh) write_aug_columns(Xh, (size_t)r, width, KB, ok ? sq : 0.0f, ok);   // extra operand columns (svm_tc.cuh)
    }
}
// predicted label per row: dec > 0 ? label[0] : label[1]   (svm.cpp:2516-2531)
__global__ void labels_from_dec_kernel(const double* __restrict__ dec, int n, double l0, double l1, double* __restrict__ labels) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) labels[i] = dec[i] > 0.0 ? l0 : l1;
}
// svm-scale pass 2 (svm-scale.c:165-198): per-feature min / max over all rows, absent entries counting as 0.
// dense [n_rows][width]; ordered 64-bit keys so that atomicMax / atomicMin on integers order doubles.
__device__ __forceinline__ unsigned long long dkey(double v) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(unsigned long long k) {
    const unsigned long long u = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)u);
}
__global__ void scale_minmax_kernel(const double* __restrict__ dense, int n_rows, int width, int rows_per_block,
                                    unsigned long long* __restrict__ kmin, unsigned long long* __restrict__ kmax, int* __restrict__ nan_flag) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= width) return;
    const int r0 = blockIdx.y * rows_per_block, r1 = min(n_rows, r0 + rows_per_block);
    if (r0 >= r1) return;
    double mn = dense[(size_t)r0 * width + d], mx = mn;
    bool bad = mn != mn;
    for (int r = r0 + 1; r < r1; r++) {
        const double v = dense[(size_t)r * width + d];
        bad = bad || (v != v);
        mn = v < mn ? v : mn;
        mx = v > mx ? v : mx;
    }
    if (bad) *nan_flag = 1;
    atomicMin(kmin + d, dkey(mn));
    atomicMax(kmax + d, dkey(mx));
}
__global__ void scale_minmax_decode_kernel(const unsigned long long* __restrict__ kmin, const unsigned long long* __restrict__ kmax, int width,
                                           double* __restrict__ fmin, double* __restrict__ fmax) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < width) { fmin[d] = dkey_inv(kmin[d]); fmax[d] = dkey_inv(kmax[d]); }
}
// svm-scale pass 3, output() (svm-scale.c:333-353), in place on the dense matrix: single-valued features become 0
// (they are skipped, i.e. absent, in the output), the rest  v == min -> lower, v == max -> upper, else
// lower + (upper - lower) * (v - min) / (max - min)  evaluated left to right in double.
__global__ void scale_apply_kernel(double* __restrict__ dense, size_t n_elems, int width, const double* __restrict__ fmin,
                                   const double* __restrict__ fmax, double lower, double upper) {
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_elems; t += (size_t)gridDim.x * blockDim.x) {
        const int d = (int)(t % (size_t)width);
        const double mn = fmin[d], mx = fmax[d];
        double v = dense[t];
        if (mx == mn) v = 0.0;
        else if (v == mn) v = lower;
        else if (v == mx) v = upper;
        else v = __dadd_rn(lower, __ddiv_rn(__dmul_rn(__dsub_rn(upper, lower), __dsub_rn(v, mn)), __dsub_rn(mx, mn)));
        dense[t] = v;
    }
}

// ---------------------------------------------------------------------------------------------------
// Probability estimates (SURVEY 8f-4): svm-predict -b 1 and the server's svm_with_probability branch.
// ---------------------------------------------------------------------------------------------------
// svm_predict_probability for nr_class = 2 (svm.cpp:2550-2590): sigmoid_predict (:1818-1826), the clamp to
// [1e-7, 1 - 1e-7] with libsvm's own min / max templates, then multiclass_probability (:1829-1890, "method 2" of Wu, Lin
// and Weng) -- an ITERATION stopped at eps = 0.005 / k, so its result is not the sigmoid value and has to be replayed
// operation by operation (double, no FMA, the reference's association).  Only exp() differs from the host (glibc vs CUDA,
// <= 1 ulp): the estimates agree to ~1e-16 relative, i.e. the "%g" text is the same unless a value sits within that of a
// 6-digit rounding boundary.  Returns the index of the predicted label (strict >, first wins: :2577-2580).
__device__ __forceinline__ int svm_probability_2class(double dec, double A, double B, double p[2]) {
    const double fApB = __dadd_rn(__dmul_rn(dec, A), B);
    double s;
    if (fApB >= 0) { const double e = exp(-fApB); s = __ddiv_rn(e, __dadd_rn(1.0, e)); }   // 1-p used later; avoid catastrophic cancellation
    else s = __ddiv_rn(1.0, __dadd_rn(1.0, exp(fApB)));
    const double min_prob = 1e-7, hi = __dsub_rn(1.0, min_prob);
    double r01 = (s > min_prob) ? s : min_prob;     // max(x, y) = (x > y) ? x : y
    r01 = (r01 < hi) ? r01 : hi;                    // min(x, y) = (x < y) ? x : y
    const double r10 = __dsub_rn(1.0, r01);
    // Q[t][t] += r[j][t] * r[j][t];  Q[t][j] = -r[j][t] * r[t][j]
    const double Q00 = __dadd_rn(0.0, __dmul_rn(r10, r10)), Q01 = __dmul_rn(-r10, r01), Q11 = __dadd_rn(0.0, __dmul_rn(r01, r01)), Q10 = Q01;
    const double eps = 0.005 / 2;
    double p0 = 1.0 / 2, p1 = 1.0 / 2;
    for (int iter = 0; iter < 100; iter++) {
        double Qp0 = __dadd_rn(__dadd_rn(0.0, __dmul_rn(Q00, p0)), __dmul_rn(Q01, p1));
        double pQp = __dadd_rn(0.0, __dmul_rn(p0, Qp0));
        double Qp1 = __dadd_rn(__dadd_rn(0.0, __dmul_rn(Q10, p0)), __dmul_rn(Q11, p1));
        pQp = __dadd_rn(pQp, __dmul_rn(p1, Qp1));
        double max_error = 0;
        const double e0 = fabs(__dsub_rn(Qp0, pQp)), e1 = fabs(__dsub_rn(Qp1, pQp));
        if (e0 > max_error) max_error = e0;
        if (e1 > max_error) max_error = e1;
        if (max_error < eps) break;
        {   // t = 0
            const double diff = __ddiv_rn(__dadd_rn(-Qp0, pQp), Q00), od = __dadd_rn(1.0, diff);
            p0 = __dadd_rn(p0, diff);
            pQp = __ddiv_rn(__ddiv_rn(__dadd_rn(pQp, __dmul_rn(diff, __dadd_rn(__dmul_rn(diff, Q00), __dmul_rn(2.0, Qp0)))), od), od);
            Qp0 = __ddiv_rn(__dadd_rn(Qp0, __dmul_rn(diff, Q00)), od); p0 = __ddiv_rn(p0, od);
            Qp1 = __ddiv_rn(__dadd_rn(Qp1, __dmul_rn(diff, Q01)), od); p1 = __ddiv_rn(p1, od);
        }
        {   // t = 1
            const double diff = __ddiv_rn(__dadd_rn(-Qp1, pQp), Q11), od = __dadd_rn(1.0, diff);
            p1 = __dadd_rn(p1, diff);
            pQp = __ddiv_rn(__ddiv_rn(__dadd_rn(pQp, __dmul_rn(diff, __dadd_rn(__dmul_rn(diff, Q11), __dmul_rn(2.0, Qp1)))), od), od);
            Qp0 = __ddiv_rn(__dadd_rn(Qp0, __dmul_rn(diff, Q10)), od); p0 = __ddiv_rn(p0, od);
            Qp1 = __ddiv_rn(__dadd_rn(Qp1, __dmul_rn(diff, Q11)), od); p1 = __ddiv_rn(p1, od);
        }
    }
    p[0] = p0; p[1] = p1;
    return p1 > p0 ? 1 : 0;
}
// haf_svm_predict_probability: labels [n], prob_estimates [n][2] (the order of the model's labels, svm-predict.c:111-118)
__global__ void prob_from_dec_kernel(const double* __restrict__ dec, int n, double A, double B, double l0, double l1,
                                     double* __restrict__ labels, double* __restrict__ probs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double p[2];
    const int idx = svm_probability_2class(dec[i], A, B, p);
    labels[i] = idx ? l1 : l0;
    probs[2 * (size_t)i] = p[0];
    probs[2 * (size_t)i + 1] = p[1];
}
// The server's probability branch (server.cpp:831-841) reads "<label> <p0> <p1>" lines: res = atof(first two characters),
// prob = atof of the SECOND estimate when res > 0, else of the first (whatever the model's label order is), the grid value is
// res * prob in float.  res0 / res1: atof of the first two characters of "%g" of the two labels (host); the estimate goes
// through the "%g" text (text6) and a double -> float conversion.  Values land in pv[unit][cell]; the reference's one-line
// shift (below) is applied afterwards.
__global__ void prob_value_kernel(const double* __restrict__ dec, const int2* __restrict__ win, const unsigned* __restrict__ win_count,
                                  int G, int unit_base, double A, double B, int res0, int res1, float* __restrict__ pv,
                                  int* __restrict__ unsupported_flag) {
    const unsigned W = *win_count;
    const unsigned w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    double p[2];
    const int idx = svm_probability_2class(dec[w], A, B, p);
    const int res = idx ? res1 : res0;
    bool uns = false;
    const float prob = (float)hafdec::text6(res > 0 ? p[1] : p[0], &uns);
    if (uns) *unsupported_flag = 1;
    const int2 uc = win[w];
    pv[(size_t)(uc.x - unit_base) * G * G + uc.y] = __fmul_rn((float)res, prob);
}
// THE ONE-LINE SHIFT.  show_predicted_gps reads the first line of the output file BEFORE its loop (server.cpp:817-818) and
// the next one after every valid window (:846).  With -b 1 the file starts with the header "labels <l0> <l1>"
// (svm-predict.c:57-66), so the k-th valid window (row-major) of a roll gets the prediction of window k - 1, the first one
// gets the header parsed as a prediction (res = atof("la") = 0, prob = atof(" <l0>"): header_val = 0 * (float)l0, i.e. -0.0f
// for a negative first label) and the last prediction is never read.  grid[cell] = -1 outside the mask (:828-829).
// One CTA per unit walks the cells in order carrying the last valid cell seen.
__global__ void __launch_bounds__(1024) prob_shift_grid_kernel(const unsigned char* __restrict__ mask, const float* __restrict__ pv, int G,
                                                               const UnitParams* __restrict__ units, float header_val, float* __restrict__ grid) {
    const int u = blockIdx.x;
    if (units[u].cloud < 0) return;
    const int GG = G * G;
    const unsigned char* m = mask + (size_t)u * GG;
    const float* v = pv + (size_t)u * GG;
    float* g = grid + (size_t)u * GG;
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    if (threadIdx.x == 0) s_carry = -1;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int c0 = 0; c0 < GG; c0 += 1024) {
        const int cell = c0 + threadIdx.x;
        const bool valid = cell < GG && m[cell];
        // last valid cell strictly before this one: exclusive max-scan of (valid ? cell : -1)
        int mine = valid ? cell : -1, incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl = max(incl, up);
        }
        int excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = -1;
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int before = s_carry;
        for (int k = 0; k < warp; k++) before = max(before, s_warp[k]);
        const int prev = max(before, excl);
        if (cell < GG) g[cell] = valid ? (prev >= 0 ? v[prev] : header_val) : -1.0f;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = max(prev, mine);
        __syncthreads();
    }
}
// a13 on the float grid (server.cpp:865-897): the 29 products int * float and their sum in the reference's order, in float;
// topval_gp = (int)graspseval (truncation) whenever graspseval > topval_gp, and the overall top follows only when that
// integer strictly grows (:881-892) -> the per-roll top is the FIRST cell reaching the maximum of trunc(graspseval):
// the same ordered key as score_kernel with trunc(v) in the value field.  The tie rule (graspseval == topval_gp) runs
// unchanged on evals.
__global__ void __launch_bounds__(256) score_prob_kernel(const float* __restrict__ grid, int G, const UnitParams* __restrict__ units,
                                                         float* __restrict__ evals, unsigned long long* __restrict__ unit_top) {
    const int u = blockIdx.y;
    if (units[u].cloud < 0) return;
    const int GG = G * G;
    const int cell = blockIdx.x * 256 + threadIdx.x;
    const float* L = grid + (size_t)u * GG;
    float e = 0.0f;
    const bool have = cell < GG;
    if (have) {
        const int row = cell / G, col = cell - row * G;
        if (!(L[cell] < 0.0f) && row >= 2 && row < G - 2 && col >= 4 && col < G - 4) {   // mask-true cells are >= 7 from the border
            float s = 0.0f;
            bool first = true;
#define PG(w, dr, dc) { const float t = __fmul_rn((float)(w), L[(row + (dr)) * G + (col + (dc))]); s = first ? t : __fadd_rn(s, t); first = false; }
            PG(1, -2, -2) PG(2, -2, -1) PG(3, -2, 0) PG(2, -2, 1) PG(1, -2, 2)
            PG(2, -1, -2) PG(3, -1, -1) PG(4, -1, 0) PG(3, -1, 1) PG(2, -1, 2)
            PG(2, 0, -4) PG(2, 0, -3) PG(3, 0, -2) PG(4, 0, -1) PG(55, 0, 0) PG(4, 0, 1) PG(3, 0, 2) PG(2, 0, 3) PG(2, 0, 4)
            PG(2, 1, -2) PG(3, 1, -1) PG(4, 1, 0) PG(3, 1, 1) PG(2, 1, 2)
            PG(1, 2, -2) PG(2, 2, -1) PG(3, 2, 0) PG(2, 2, 1) PG(1, 2, 2)
#undef PG
            e = s;
        }
        evals[(size_t)u * GG + cell] = e;
    }
    const int ti = (int)e;   // float -> int truncates toward zero, like the reference's assignment
    unsigned long long key = have ? (((unsigned long long)(unsigned)(ti + (1 << 20))) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)cell) : 0ull;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    __shared__ unsigned long long sk[8];
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) key = sk[w] > key ? sk[w] : key;
        atomicMax(unit_top + u, key);
    }
}

// debug: device text round trips
__global__ void text_roundtrip_kernel(const float* in4, int n4, double* out4, const double* in6, int n6, double* out6) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n4) out4[i] = hafdec::text4(in4[i]);
    if (i < n6) out6[i] = hafdec::text6(in6[i]);
}

}  // namespace hafk
