// pcd_ingest.cuh -- PCD ingest on the device (SURVEY 8f-2): the DATA section of a PCD v0.7 file, or a PointCloud2 buffer,
// becomes packed xyz floats in HBM without a host decode pass.
//
// Reference: the client loads the file with pcl::io::loadPCDFile<pcl::PointXYZ> (src/calc_grasppoints_action_client.cpp:137-157)
// and ships a PointCloud2; the server turns it back into points with pcl::fromROSMsg (src/calc_grasppoints_action_server.cpp
// :313-316).  PCL is a dependency of the reference, not vendored in it (ROS hydro / indigo: PCL 1.7); what is restated here is
// its published reader (io/src/pcd_io.cpp, PCDReader::read):
//   * ascii             -- one record per non-empty line, fields split on blank / tab / CR, FLOAT32 fields through
//                          `istringstream >> float` (= strtof: correctly rounded, hafdec::parse_float_token); exactly POINTS
//                          records are taken, further lines are ignored (pcd4 / pcd5 carry 208 lines for POINTS 200);
//   * binary            -- POINTS records of the header's layout;
//   * binary_compressed -- u32 compressed size, u32 uncompressed size, one LZF stream (liblzf, as embedded in PCL), fields
//                          stored struct-of-arrays;
//   * fromROSMsg        -- x / y / z FLOAT32 at their declared byte offsets inside records of point_step bytes.
// A call takes a batch of files / buffers (haf_pcd_decode and haf_pointcloud2_to_xyz are batches of one): every cloud keeps
// the semantics above, and each data kind present runs one fixed sequence of launches over all its clouds.
// The text header stays on the host (csrc/host/pcd_io.hpp, parse_pcd_header).  Parity: byte-equal xyz with the host reader
// (csrc/host/pcd_io.hpp, haf_grasping_b200/pcd.py) on every bundled PCD and on generated files (tests/test_pcd_device.py).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "decimal_round.cuh"

namespace hafpcdk {

__device__ __forceinline__ float load_f32_any(const unsigned char* p) {   // records need not be 4-byte aligned
    if ((reinterpret_cast<uintptr_t>(p) & 3) == 0) return *reinterpret_cast<const float*>(p);
    const uint32_t u = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    return __uint_as_float(u);
}

// ---------------------------------------------------------------------------------------------------------------------
// A call decodes a BATCH of files or PointCloud2 buffers (a single one is the batch of one): each data kind present runs one
// fixed sequence of launches over all its clouds, described by tables the host sends in one parameter block.
// ---------------------------------------------------------------------------------------------------------------------
// Gather: point i of segment s has x / y / z at src + off[a] + i * stride[a]; it becomes point out_begin + i of the packed
// output.  Binary PCD records (stride = record bytes for all three), the struct-of-arrays blob of binary_compressed files
// after the LZF stage (stride = 4 * COUNT), PointCloud2 records (stride = point_step).
struct GatherSeg {
    const unsigned char* src;
    unsigned long long out_begin;
    unsigned long long off[3], stride[3];
};
// seg_begin [n_segs + 1]: exclusive prefix of the segments' point counts (no empty segment); a point finds its segment by
// binary search
__global__ void gather_segments_kernel(const GatherSeg* __restrict__ segs, const unsigned long long* __restrict__ seg_begin, int n_segs,
                                       float* __restrict__ xyz) {
    const unsigned long long n = seg_begin[n_segs];
    for (unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (unsigned long long)gridDim.x * blockDim.x) {
        int lo = 0, hi = n_segs - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (seg_begin[mid] <= p) lo = mid; else hi = mid - 1;
        }
        const GatherSeg& S = segs[lo];
        const unsigned long long i = p - seg_begin[lo], o = 3 * (S.out_begin + i);
        xyz[o] = load_f32_any(S.src + S.off[0] + i * S.stride[0]);
        xyz[o + 1] = load_f32_any(S.src + S.off[1] + i * S.stride[1]);
        xyz[o + 2] = load_f32_any(S.src + S.off[2] + i * S.stride[2]);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// LZF (liblzf lzf_d.c): ctrl < 32: literal run of ctrl + 1 bytes; else back reference: len = ctrl >> 5 (7: + next byte) + 2,
// distance = ((ctrl & 31) << 8 | next byte) + 1 <= 8192.  The token chain is sequential, the bytes of a token are not: one
// WARP per stream -- all lanes read the control bytes from a shared-memory ring of the input, the lanes copy a token's bytes
// together (an overlapping reference repeats its `distance` bytes: source index (k mod distance)), back references read a
// 16 KB shared-memory ring of the output, so no global load sits on the token chain.  status: 0 ok, 1 corrupt stream.
// grid = streams (a batch of files decodes one stream per CTA, each into its own range of one blob buffer), block = 32.
// ---------------------------------------------------------------------------------------------------------------------
#define HAF_LZF_IN_RING 8192
#define HAF_LZF_OUT_RING 16384
struct LzfStream { const unsigned char* in; unsigned long long in_len; unsigned char* out; unsigned long long out_len; };
__global__ void __launch_bounds__(32) lzf_decompress_kernel(const LzfStream* __restrict__ streams, int* __restrict__ status) {
    __shared__ unsigned char s_in[HAF_LZF_IN_RING];
    __shared__ unsigned char s_out[HAF_LZF_OUT_RING];
    const LzfStream S = streams[blockIdx.x];
    const int lane = threadIdx.x;
    unsigned long long ip = 0, op = 0, loaded = 0;   // loaded: input bytes [.., loaded) are in the ring
    bool bad = false;
    while (ip < S.in_len) {
        // keep at least 512 bytes of look-ahead in the ring (a token is at most 3 + 32 bytes); refill in 4 KB blocks, which
        // only overwrites input more than 4 KB behind ip
        while (loaded < S.in_len && loaded < ip + 512) {
            const unsigned long long n = min((unsigned long long)4096, S.in_len - loaded);
            for (unsigned long long k = lane; k < n; k += 32) s_in[(loaded + k) & (HAF_LZF_IN_RING - 1)] = S.in[loaded + k];
            loaded += n;
            __syncwarp();
        }
        const unsigned ctrl = s_in[ip & (HAF_LZF_IN_RING - 1)];
        if (ctrl < 32) {
            const unsigned n = ctrl + 1;
            if (op + n > S.out_len || ip + 1 + n > S.in_len) { bad = true; break; }
            if (lane < n) {
                const unsigned char v = s_in[(ip + 1 + lane) & (HAF_LZF_IN_RING - 1)];
                s_out[(op + lane) & (HAF_LZF_OUT_RING - 1)] = v;
                S.out[op + lane] = v;
            }
            ip += 1 + n;
            op += n;
        } else {
            unsigned len = ctrl >> 5;
            unsigned long long q = ip + 1;
            if (len == 7) { if (q >= S.in_len) { bad = true; break; } len += s_in[q & (HAF_LZF_IN_RING - 1)]; q++; }
            if (q >= S.in_len) { bad = true; break; }
            const unsigned dist = ((ctrl & 0x1f) << 8) + s_in[q & (HAF_LZF_IN_RING - 1)] + 1;
            q++;
            len += 2;
            if (dist > op || op + len > S.out_len) { bad = true; break; }
            // bytes [op - dist, op) are final; byte k of the token copies byte (k mod dist) of them
            for (unsigned k0 = 0; k0 < len; k0 += 32) {
                const unsigned k = k0 + lane;
                if (k < len) {
                    const unsigned char v = s_out[(op - dist + (k % dist)) & (HAF_LZF_OUT_RING - 1)];
                    S.out[op + k] = v;
                    // the ring slot of byte op + k may be a source of this same token only if dist > 16384 - len: never (dist <= 8192)
                    s_out[(op + k) & (HAF_LZF_OUT_RING - 1)] = v;
                }
            }
            ip = q;
            op += len;
        }
        __syncwarp();
    }
    if (lane == 0 && (bad || op != S.out_len)) status[blockIdx.x] = 1;
}

// ---------------------------------------------------------------------------------------------------------------------
// ASCII.  A byte is a RECORD START when it begins a line that holds at least one token.  Three passes over the data sections
// of all ASCII files of a batch, in tiles of 256 threads x 16 bytes; each section starts a new tile (tile_file: tile -> file):
// count record starts per tile; exclusive scan of the tile counts over the whole batch (one CTA); rank the starts -- the
// rank within a file is the batch rank minus the scan value at the file's first tile -- and the thread that owns start number
// r < POINTS of its file parses the record into point out_begin + r.
// ---------------------------------------------------------------------------------------------------------------------
#define HAF_PCD_TILE_THREADS 256
#define HAF_PCD_BYTES_PER_THREAD 16
struct AsciiFile {
    unsigned long long begin, len;           // data section in the device copy of the batch
    unsigned long long n_points, out_begin;  // POINTS, first output point
    int tile_begin, tile_end;                // tiles [tile_begin, tile_end)
    int tok[3];                              // token numbers of x, y, z inside a record (COUNT-aware)
    int pad;
};
__device__ __forceinline__ bool is_blank(unsigned char c) { return c == ' ' || c == '\t' || c == '\r'; }
// t: one file's data section of n bytes (its first byte is a line start, the scan stops at its end)
__device__ __forceinline__ bool record_starts_at(const unsigned char* __restrict__ t, size_t n, size_t i) {
    if (i > 0 && t[i - 1] != '\n') return false;
    for (size_t k = i; k < n; k++) {     // a line of blanks only is no record
        const unsigned char c = t[k];
        if (c == '\n') return false;
        if (!is_blank(c)) return true;
    }
    return false;
}
__device__ __forceinline__ unsigned block_exclusive_scan(unsigned v, unsigned* s_warp /*[8]*/, unsigned* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned before = 0, all = 0;
    for (int k = 0; k < HAF_PCD_TILE_THREADS / 32; k++) { if (k < warp) before += s_warp[k]; all += s_warp[k]; }
    *total = all;
    return before + incl - v;
}
// record-start bit mask of this thread's 16 bytes of tile blockIdx.x
__device__ __forceinline__ unsigned tile_starts(const unsigned char* __restrict__ raw, const AsciiFile& F, size_t* b0_out) {
    const unsigned char* text = raw + F.begin;
    const size_t b0 = ((size_t)(blockIdx.x - F.tile_begin) * HAF_PCD_TILE_THREADS + threadIdx.x) * HAF_PCD_BYTES_PER_THREAD;
    unsigned mask = 0;
    for (int k = 0; k < HAF_PCD_BYTES_PER_THREAD; k++)
        if (b0 + k < F.len && record_starts_at(text, F.len, b0 + k)) mask |= 1u << k;
    *b0_out = b0;
    return mask;
}
__global__ void __launch_bounds__(HAF_PCD_TILE_THREADS) ascii_count_kernel(const unsigned char* __restrict__ raw, const AsciiFile* __restrict__ files,
                                                                           const int* __restrict__ tile_file, unsigned* __restrict__ tile_count) {
    __shared__ unsigned s_warp[HAF_PCD_TILE_THREADS / 32];
    const AsciiFile F = files[tile_file[blockIdx.x]];
    size_t b0;
    const unsigned c = __popc(tile_starts(raw, F, &b0));
    unsigned total;
    block_exclusive_scan(c, s_warp, &total);
    if (threadIdx.x == 0) tile_count[blockIdx.x] = total;
}
// in place: tile_count -> exclusive offsets (the host keeps the records of a batch below 2^32); total[0] = number of records
__global__ void __launch_bounds__(1024) ascii_scan_kernel(unsigned* __restrict__ tile_count, unsigned n_tiles, unsigned long long* __restrict__ total) {
    __shared__ unsigned s_warp[32];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (unsigned t0 = 0; t0 < n_tiles; t0 += 1024) {
        const unsigned t = t0 + threadIdx.x;
        const unsigned v = t < n_tiles ? tile_count[t] : 0u;
        unsigned incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned before = 0, all = 0;
        for (int k = 0; k < 32; k++) { if (k < warp) before += s_warp[k]; all += s_warp[k]; }
        const unsigned long long carry = s_carry;
        if (t < n_tiles) tile_count[t] = (unsigned)min(carry + before + incl - v, (unsigned long long)0xFFFFFFFFu);
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + all;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}
// Per ASCII file a: count[a] = its records (the first tile's CTA writes it: scan value at the next file's first tile, or the
// batch total, minus the scan value at its own); flags[2a]: a record had fewer tokens than the three fields need;
// flags[2a + 1]: a token outside what the conversion reproduces exactly (> 19 digits next to a rounding boundary)
__global__ void __launch_bounds__(HAF_PCD_TILE_THREADS) ascii_parse_kernel(const unsigned char* __restrict__ raw, const AsciiFile* __restrict__ files,
                                                                           const int* __restrict__ tile_file, const unsigned* __restrict__ tile_offset,
                                                                           unsigned n_tiles, const unsigned long long* __restrict__ total,
                                                                           float* __restrict__ xyz, unsigned* __restrict__ count, int* __restrict__ flags) {
    __shared__ unsigned s_warp[HAF_PCD_TILE_THREADS / 32];
    const int a = tile_file[blockIdx.x];
    const AsciiFile F = files[a];
    const unsigned base = tile_offset[F.tile_begin];
    if (blockIdx.x == (unsigned)F.tile_begin && threadIdx.x == 0)
        count[a] = ((unsigned)F.tile_end < n_tiles ? tile_offset[F.tile_end] : (unsigned)*total) - base;
    const unsigned char* text = raw + F.begin;
    const size_t n = F.len;
    size_t b0;
    unsigned mask = tile_starts(raw, F, &b0);
    unsigned tile_total;
    unsigned long long rank = (unsigned long long)(tile_offset[blockIdx.x] - base) + block_exclusive_scan(__popc(mask), s_warp, &tile_total);
    const int tok_x = F.tok[0], tok_y = F.tok[1], tok_z = F.tok[2];
    const int tmax = max(tok_x, max(tok_y, tok_z));
    while (mask) {
        const int k = __ffs(mask) - 1;
        mask &= mask - 1;
        const unsigned long long r = rank++;
        if (r >= F.n_points) break;      // exactly POINTS records; further lines are ignored
        size_t p = b0 + k;
        float v[3] = {0.0f, 0.0f, 0.0f};
        int tok = 0;
        bool uns = false;
        while (p < n && text[p] != '\n' && tok <= tmax) {
            while (p < n && is_blank(text[p])) p++;
            if (p >= n || text[p] == '\n') break;
            size_t e = p;
            while (e < n && text[e] != '\n' && !is_blank(text[e])) e++;
            if (tok == tok_x || tok == tok_y || tok == tok_z) {
                const float f = hafdec::parse_float_token(text + p, text + e, &uns);
                if (tok == tok_x) v[0] = f;
                if (tok == tok_y) v[1] = f;
                if (tok == tok_z) v[2] = f;
            }
            tok++;
            p = e;
        }
        if (tok <= tmax) flags[2 * a] = 1;
        if (uns) flags[2 * a + 1] = 1;
        const unsigned long long o = 3 * (F.out_begin + r);
        xyz[o] = v[0]; xyz[o + 1] = v[1]; xyz[o + 2] = v[2];
    }
}

}  // namespace hafpcdk
