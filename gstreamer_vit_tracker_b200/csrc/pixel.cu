// pixel.cu — byte/integer kernels of the per-frame path (HBM-bound; no tensor cores on purpose).
//
//   K1  nv12_to_rgb_*        ≙ nv12_full_to_rgb_parallel        /root/reference/src/nv12_convert.rs:46-169
//   K2  crop_resize_norm     ≙ K1 fused with VitTrack's crop/resize/blob (OpenCV TrackerVit semantics, SURVEY.md App. A)
//   K9  overlay / box_overlay ≙ draw_*_nv12 (src/nv12_convert.rs:172-343), draw_cursor/draw_selection (src/drawing.rs:5-50),
//                               draw_*_rgb (src/drawing_rgb.rs:30-128)
#include <stdlib.h>

#include "vt_internal.h"

namespace vt {

// ------------------------------------------------------------------------------------------------
// BT.601 limited-range integer conversion, bit-exact with src/nv12_convert.rs:24-30,124-126,41-43
// (arithmetic >> on negative int, clamp to 0..255).
// ------------------------------------------------------------------------------------------------
struct Chroma { int rv, guv, bu; };
__device__ __forceinline__ Chroma chroma_terms(int u, int v) {
    Chroma c;
    c.rv = 409 * (v - 128) + 128;
    c.guv = -100 * (u - 128) - 208 * (v - 128) + 128;
    c.bu = 516 * (u - 128) + 128;
    return c;
}
__device__ __forceinline__ int clamp255(int v) { return min(max(v, 0), 255); }
__device__ __forceinline__ void yuv_px(int y, const Chroma& c, int& r, int& g, int& b) {
    const int yv = 298 * (y - 16);
    r = clamp255((yv + c.rv) >> 8);
    g = clamp255((yv + c.guv) >> 8);
    b = clamp255((yv + c.bu) >> 8);
}

// Vectorised form used by the full-frame kernels: the -16 of the luma term and the +128 rounding are folded into three per-chroma
// constants, so a pixel costs 3 IMAD + 3 SHR + 3 clamp (VIMNMX.relu) — (298*(y-16) + k + 128) >> 8 == (298*y + (k + 128 - 4768)) >> 8
// exactly.  Eight pixels (24 bytes) are packed into six words with byte-weight IMADs.
struct ChromaF { int r, g, b; };
__device__ __forceinline__ ChromaF chroma_folded(int u, int v) {
    ChromaF c;
    c.r = 409 * (v - 128) + (128 - 298 * 16);
    c.g = -100 * (u - 128) - 208 * (v - 128) + (128 - 298 * 16);
    c.b = 516 * (u - 128) + (128 - 298 * 16);
    return c;
}
__device__ __forceinline__ void yuv_px_fast(int y, const ChromaF& c, int& r, int& g, int& b) {
    r = __vimin_s32_relu((298 * y + c.r) >> 8, 255);
    g = __vimin_s32_relu((298 * y + c.g) >> 8, 255);
    b = __vimin_s32_relu((298 * y + c.b) >> 8, 255);
}
// r/g/b[0..7] (each 0..255) -> 24 interleaved bytes as three uint2
__device__ __forceinline__ void pack_rgb8(const int (&r)[8], const int (&g)[8], const int (&b)[8], uint2* dst) {
    uint32_t w[6];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int o = 4 * h;
        w[3 * h + 0] = (uint32_t)(r[o] + (g[o] << 8) + (b[o] << 16) + (r[o + 1] << 24));
        w[3 * h + 1] = (uint32_t)(g[o + 1] + (b[o + 1] << 8) + (r[o + 2] << 16) + (g[o + 2] << 24));
        w[3 * h + 2] = (uint32_t)(b[o + 2] + (r[o + 3] << 8) + (g[o + 3] << 16) + (b[o + 3] << 24));
    }
    dst[0] = make_uint2(w[0], w[1]), dst[1] = make_uint2(w[2], w[3]), dst[2] = make_uint2(w[4], w[5]);
}

// ------------------------------------------------------------------------------------------------
// K1 fast path: W % 16 == 0, H even.  One warp converts a 256-px segment of one row pair:
// each lane loads 8 Y bytes from two rows + 4 UV pairs (8-byte loads, 256 B contiguous per warp),
// converts 16 pixels, stages 2 x 768 B in shared memory and the warp writes them back as
// 16-byte coalesced stores.  Algorithmic traffic: 1.5*W*H read + 3*W*H written.
// ------------------------------------------------------------------------------------------------
constexpr int kCvtWarps = 8;

__global__ void __launch_bounds__(kCvtWarps * 32) nv12_to_rgb_vec_kernel(const uint8_t* __restrict__ in, size_t stride_in,
                                                                       uint8_t* __restrict__ out, size_t stride_out, int W, int H,
                                                                       int n_frames) {
    __shared__ __align__(16) uint8_t stage[kCvtWarps][2][768];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // grid = (segment groups, row pairs, frames): no index division in the kernel
    const int segs = (W + 255) >> 8;
    (void)n_frames;
    {
        const int seg = blockIdx.x * (blockDim.x >> 5) + warp, pair = blockIdx.y, frame = blockIdx.z;
        if (seg >= segs) return;
        const uint8_t* yp = in + (size_t)frame * stride_in;
        const uint8_t* uvp = yp + (size_t)W * H;
        uint8_t* op = out + (size_t)frame * stride_out;
        const int x = seg * 256 + lane * 8;
        const int seg_px = min(256, W - seg * 256);
        if (x < W) {
            const uint2 ya = __ldg(reinterpret_cast<const uint2*>(yp + (size_t)(2 * pair) * W + x));
            const uint2 yb = __ldg(reinterpret_cast<const uint2*>(yp + (size_t)(2 * pair + 1) * W + x));
            const uint2 uv = __ldg(reinterpret_cast<const uint2*>(uvp + (size_t)pair * W + x));
            const uint32_t yw[2][2] = {{ya.x, ya.y}, {yb.x, yb.y}};
            const uint32_t uvw[2] = {uv.x, uv.y};
            int r[2][8], g[2][8], b[2][8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {  // 4 chroma pairs
                const uint32_t w = uvw[q >> 1] >> ((q & 1) * 16);
                const ChromaF c = chroma_folded((int)(w & 0xff), (int)((w >> 8) & 0xff));
#pragma unroll
                for (int row = 0; row < 2; ++row)
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        const int i = q * 2 + k;
                        yuv_px_fast((int)((yw[row][i >> 2] >> ((i & 3) * 8)) & 0xff), c, r[row][i], g[row][i], b[row][i]);
                    }
            }
#pragma unroll
            for (int row = 0; row < 2; ++row) pack_rgb8(r[row], g[row], b[row], reinterpret_cast<uint2*>(&stage[warp][row][lane * 24]));
        }
        __syncwarp();
        const int row_bytes = seg_px * 3;  // multiple of 48
#pragma unroll
        for (int row = 0; row < 2; ++row) {
            uint8_t* g = op + ((size_t)(2 * pair + row) * W + (size_t)seg * 256) * 3;
            for (int off = lane * 16; off < row_bytes; off += 32 * 16)
                *reinterpret_cast<uint4*>(g + off) = *reinterpret_cast<const uint4*>(&stage[warp][row][off]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K1 wide path: W % 16 == 0, H % 4 == 0.  One warp converts a 512-px segment of FOUR rows (two chroma rows): every lane has six
// 16-byte loads in flight (4 x 16 luma bytes + 2 x 8 chroma pairs = 96 B per thread, 3 KB per warp) before it converts anything —
// the kernel is a pure stream (4.5 B of traffic per pixel, no reuse), so what counts is bytes in flight per SM; the 8-byte / two-row
// form above left ~25 % of the HBM rate on the table.  Rows are staged one at a time in 1.5 KB of shared memory per warp and leave as
// 16-byte coalesced stores (a warp instruction writes 512 contiguous bytes).
// ------------------------------------------------------------------------------------------------
constexpr int kCvt4Warps = 4;

__global__ void __launch_bounds__(kCvt4Warps * 32) nv12_to_rgb_vec4_kernel(const uint8_t* __restrict__ in, size_t stride_in,
                                                                         uint8_t* __restrict__ out, size_t stride_out, int W, int H) {
    __shared__ __align__(16) uint8_t stage[kCvt4Warps][1536];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int segs = (W + 511) >> 9;
    const int seg = blockIdx.x * (blockDim.x >> 5) + warp, quad = blockIdx.y, frame = blockIdx.z;
    if (seg >= segs) return;
    const uint8_t* yp = in + (size_t)frame * stride_in;
    const uint8_t* uvp = yp + (size_t)W * H;
    uint8_t* op = out + (size_t)frame * stride_out;
    const int x = seg * 512 + lane * 16;
    const int seg_px = min(512, W - seg * 512);
    uint4 yq[4], uvq[2];
    if (x < W) {
#pragma unroll
        for (int k = 0; k < 4; ++k) yq[k] = __ldg(reinterpret_cast<const uint4*>(yp + (size_t)(4 * quad + k) * W + x));
#pragma unroll
        for (int k = 0; k < 2; ++k) uvq[k] = __ldg(reinterpret_cast<const uint4*>(uvp + (size_t)(2 * quad + k) * W + x));
    }
    const int row_bytes = seg_px * 3;  // multiple of 48
#pragma unroll
    for (int row = 0; row < 4; ++row) {
        if (x < W) {
            const uint32_t yw[4] = {yq[row].x, yq[row].y, yq[row].z, yq[row].w};
            const uint32_t uvw[4] = {uvq[row >> 1].x, uvq[row >> 1].y, uvq[row >> 1].z, uvq[row >> 1].w};
#pragma unroll
            for (int half = 0; half < 2; ++half) {  // 8 pixels = 4 chroma pairs per half
                int r[8], g[8], b[8];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t w = uvw[2 * half + (q >> 1)] >> ((q & 1) * 16);
                    const ChromaF c = chroma_folded((int)(w & 0xff), (int)((w >> 8) & 0xff));
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        const int i = q * 2 + k;
                        yuv_px_fast((int)((yw[2 * half + (i >> 2)] >> ((i & 3) * 8)) & 0xff), c, r[i], g[i], b[i]);
                    }
                }
                pack_rgb8(r, g, b, reinterpret_cast<uint2*>(&stage[warp][lane * 48 + half * 24]));
            }
        }
        __syncwarp();
        uint8_t* gp = op + ((size_t)(4 * quad + row) * W + (size_t)seg * 512) * 3;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int off = lane * 16 + j * 512;
            if (off < row_bytes) *reinterpret_cast<uint4*>(gp + off) = *reinterpret_cast<const uint4*>(&stage[warp][off]);
        }
        __syncwarp();
    }
}

// K1 generic path (odd sizes, W % 16 != 0): one thread per 2x2 quad, byte accesses.
__global__ void nv12_to_rgb_generic_kernel(const uint8_t* __restrict__ in, size_t stride_in, uint8_t* __restrict__ out,
                                           size_t stride_out, int W, int H, int n_frames) {
    const int qw = (W + 1) >> 1, qh = (H + 1) >> 1;
    const long long total = (long long)n_frames * qw * qh;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int qx = (int)(i % qw);
        const long long t = i / qw;
        const int qy = (int)(t % qh);
        const int frame = (int)(t / qh);
        const uint8_t* yp = in + (size_t)frame * stride_in;
        const uint8_t* uvp = yp + (size_t)W * H;
        uint8_t* op = out + (size_t)frame * stride_out;
        const int x = qx * 2, y = qy * 2;
        const size_t uvi = (size_t)qy * W + x;  // src/nv12_convert.rs:109 / :152 (odd-width tail uses the pair at even col)
        const Chroma c = chroma_terms(uvp[uvi], uvp[uvi + 1]);
        for (int dy = 0; dy < 2 && y + dy < H; ++dy)
            for (int dx = 0; dx < 2 && x + dx < W; ++dx) {
                int r, g, b;
                yuv_px(yp[(size_t)(y + dy) * W + x + dx], c, r, g, b);
                uint8_t* o = op + ((size_t)(y + dy) * W + x + dx) * 3;
                o[0] = (uint8_t)r, o[1] = (uint8_t)g, o[2] = (uint8_t)b;
            }
    }
}

cudaError_t launch_nv12_to_rgb(const uint8_t* d_nv12, size_t stride_in, uint8_t* d_rgb, size_t stride_out, int width, int height,
                               int n_frames, cudaStream_t s) {
    if (width <= 0 || height <= 0 || n_frames <= 0) return cudaSuccess;
    const bool aligned = (width % 16 == 0) && (height % 2 == 0) && (height / 2 <= 65535) && (n_frames <= 65535) && (stride_in % 16 == 0) &&
                         (stride_out % 16 == 0) &&
                         ((reinterpret_cast<uintptr_t>(d_nv12) | reinterpret_cast<uintptr_t>(d_rgb)) % 16 == 0);
    if (aligned && height % 4 == 0) {
        const int segs = (width + 511) / 512;
        const int wpb = segs < kCvt4Warps ? segs : kCvt4Warps;
        const dim3 grid((segs + wpb - 1) / wpb, height / 4, n_frames);  // one warp per 512-px x 4-row item
        nv12_to_rgb_vec4_kernel<<<grid, wpb * 32, 0, s>>>(d_nv12, stride_in, d_rgb, stride_out, width, height);
    } else if (aligned) {
        const int segs = (width + 255) / 256;
        const int wpb = segs < kCvtWarps ? segs : kCvtWarps;  // narrow frames: no idle warps
        const dim3 grid((segs + wpb - 1) / wpb, height / 2, n_frames);  // one warp per 256-px x 2-row item
        nv12_to_rgb_vec_kernel<<<grid, wpb * 32, 0, s>>>(d_nv12, stride_in, d_rgb, stride_out, width, height, n_frames);
    } else {
        const long long items = (long long)n_frames * ((width + 1) / 2) * ((height + 1) / 2);
        long long blocks = (items + 255) / 256;
        if (blocks > 148LL * 32) blocks = 148LL * 32;
        nv12_to_rgb_generic_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_nv12, stride_in, d_rgb, stride_out, width, height, n_frames);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// YUY2 (packed 4:2:2: Y0 U Y1 V) -> RGB, SURVEY.md §8(f) row 1 (≙ the videoconvert step of src/pipeline_ir.rs:27-56), same
// integer arithmetic as K1.  Fast path (W % 8 == 0): one warp converts a 256-px row segment — each lane loads 16 B (8 px),
// stages 24 B in shared memory, the warp writes 768 B as 16-byte coalesced stores.  2*W*H read + 3*W*H written.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kCvtWarps * 32) yuy2_to_rgb_vec_kernel(const uint8_t* __restrict__ in, size_t stride_in,
                                                                       uint8_t* __restrict__ out, size_t stride_out, int W, int H,
                                                                       int n_frames) {
    __shared__ __align__(16) uint8_t stage[kCvtWarps][768];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int segs = (W + 255) >> 8;
    const size_t row_in = (size_t)W * 2;
    (void)n_frames, (void)H;
    {
        const int seg = blockIdx.x * (blockDim.x >> 5) + warp, row = blockIdx.y, frame = blockIdx.z;
        if (seg >= segs) return;
        const uint8_t* ip = in + (size_t)frame * stride_in + (size_t)row * row_in;
        uint8_t* op = out + (size_t)frame * stride_out + ((size_t)row * W + (size_t)seg * 256) * 3;
        const int x = seg * 256 + lane * 8;
        const int seg_px = min(256, W - seg * 256);
        if (x < W) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(ip + (size_t)x * 2));
            const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
            int r[8], g[8], b[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {  // one Y0 U Y1 V word = two pixels
                const ChromaF c = chroma_folded((int)((w4[k] >> 8) & 0xff), (int)(w4[k] >> 24));
                yuv_px_fast((int)(w4[k] & 0xff), c, r[2 * k], g[2 * k], b[2 * k]);
                yuv_px_fast((int)((w4[k] >> 16) & 0xff), c, r[2 * k + 1], g[2 * k + 1], b[2 * k + 1]);
            }
            pack_rgb8(r, g, b, reinterpret_cast<uint2*>(&stage[warp][lane * 24]));
        }
        __syncwarp();
        const int row_bytes = seg_px * 3;  // multiple of 24; the tail (< 16 B) is written bytewise
        for (int off = lane * 16; off + 16 <= row_bytes; off += 32 * 16)
            *reinterpret_cast<uint4*>(op + off) = *reinterpret_cast<const uint4*>(&stage[warp][off]);
        if ((row_bytes & 15) && lane < (row_bytes & 15)) op[(row_bytes & ~15) + lane] = stage[warp][(row_bytes & ~15) + lane];
    }
}

// YUY2 word [Y0 U Y1 V] -> the six colour values of its two pixels with two-way dot products (dp2a: 16-bit coefficients x unsigned bytes):
// the luma term and the chroma term that sits next to it in the word are one instruction, the other chroma term and the folded
// constant ride in the accumulator operand (G) or come from one byte permute (R0, B1).  Identical integer sums as yuv_px_fast, then
// >> 8 and a saturating pack (cvt.pack.sat.u8.s32: clamp to 0..255 and place two bytes per instruction): ~10 instead of ~17
// instructions per pixel — the kernel was instruction-issue bound (ncu: SM 85 %, DRAM 48 %).
__device__ __forceinline__ int dp2a_lo_su(int coef16x2, uint32_t bytes, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(coef16x2), "r"(bytes), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_su(int coef16x2, uint32_t bytes, int c) {
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(coef16x2), "r"(bytes), "r"(c));
    return d;
}
// (sat_u8(hi) << 8 | sat_u8(lo)) | (upper << 16)
__device__ __forceinline__ uint32_t pack_sat2(int hi, int lo, uint32_t upper) {
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(hi), "r"(lo), "r"(upper));
    return d;
}
constexpr int kC16(int lo, int hi) { return (int)((uint32_t)(lo & 0xffff) | ((uint32_t)(hi & 0xffff) << 16)); }
// v[0..5] = R0 G0 B0 R1 G1 B1, each (sum >> 8) before saturation
__device__ __forceinline__ void yuy2_word6(uint32_t w, int (&v)[6]) {
    constexpr int cR = 128 - 298 * 16 - 409 * 128, cG = 128 - 298 * 16 + 100 * 128 + 208 * 128, cB = 128 - 298 * 16 - 516 * 128;
    const uint32_t w2 = __byte_perm(w, 0, 0x1230);                 // [Y0 V Y1 U]
    const int gv = (int)(w >> 24) * -208 + cG, gu = (int)((w >> 8) & 0xff) * -100 + cG;
    v[0] = dp2a_lo_su(kC16(298, 409), w2, cR) >> 8;                // 298 Y0 + 409 V
    v[1] = dp2a_lo_su(kC16(298, -100), w, gv) >> 8;                // 298 Y0 - 100 U (- 208 V)
    v[2] = dp2a_lo_su(kC16(298, 516), w, cB) >> 8;                 // 298 Y0 + 516 U
    v[3] = dp2a_hi_su(kC16(298, 409), w, cR) >> 8;                 // 298 Y1 + 409 V
    v[4] = dp2a_hi_su(kC16(298, -208), w, gu) >> 8;                // 298 Y1 - 208 V (- 100 U)
    v[5] = dp2a_hi_su(kC16(298, 516), w2, cB) >> 8;                // 298 Y1 + 516 U
}

// wide path (W % 16 == 0): rows are tightly packed on both sides (2 W bytes in, 3 W bytes out), so a frame is a flat array of 16-pixel
// items (32 bytes in, 48 bytes out).  One warp converts 64 consecutive items: every lane has four 16-byte loads in flight before it
// converts anything, the 3072 output bytes are staged in shared memory and leave as 16-byte stores, 512 contiguous bytes per warp
// instruction.  (The row-segment form left 37 % of the lanes idle on 640-pixel rows: 512 + 128.)
__global__ void __launch_bounds__(kCvt4Warps * 32) yuy2_to_rgb_vec2_kernel(const uint8_t* __restrict__ in, size_t stride_in,
                                                                         uint8_t* __restrict__ out, size_t stride_out, int W, int H) {
    __shared__ __align__(16) uint8_t stage[kCvt4Warps][3072];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long items = (long long)W * H / 16;
    const long long base = ((long long)blockIdx.x * kCvt4Warps + warp) * 64;
    if (base >= items) return;
    const int frame = blockIdx.z;
    const uint8_t* ip = in + (size_t)frame * stride_in;
    uint8_t* op = out + (size_t)frame * stride_out;
    uint4 q[2][2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const long long it = base + 32 * r + lane;
        if (it < items) {
#pragma unroll
            for (int k = 0; k < 2; ++k) q[r][k] = __ldg(reinterpret_cast<const uint4*>(ip + (size_t)it * 32 + 16 * k));
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        if (base + 32 * r + lane < items) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const uint32_t w4[4] = {q[r][half].x, q[r][half].y, q[r][half].z, q[r][half].w};
                int v[24];  // 8 pixels x RGB, interleaved
#pragma unroll
                for (int k = 0; k < 4; ++k) {  // one Y0 U Y1 V word = two pixels
                    int v6[6];
                    yuy2_word6(w4[k], v6);
#pragma unroll
                    for (int j = 0; j < 6; ++j) v[6 * k + j] = v6[j];
                }
                uint32_t o[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) o[j] = pack_sat2(v[4 * j + 1], v[4 * j], pack_sat2(v[4 * j + 3], v[4 * j + 2], 0));
                uint2* dst = reinterpret_cast<uint2*>(&stage[warp][r * 1536 + lane * 48 + half * 24]);
                dst[0] = make_uint2(o[0], o[1]), dst[1] = make_uint2(o[2], o[3]), dst[2] = make_uint2(o[4], o[5]);
            }
        }
    }
    __syncwarp();
    const long long n_here = items - base < 64 ? items - base : 64;
    const int bytes = (int)n_here * 48;
    uint8_t* gp = op + (size_t)base * 48;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const int off = lane * 16 + j * 512;
        if (off < bytes) *reinterpret_cast<uint4*>(gp + off) = *reinterpret_cast<const uint4*>(&stage[warp][off]);
    }
}

// generic path: one thread per pixel pair, byte accesses, GStreamer row stride (width*2 rounded up to 4)
__global__ void yuy2_to_rgb_generic_kernel(const uint8_t* __restrict__ in, size_t stride_in, uint8_t* __restrict__ out, size_t stride_out,
                                           int W, int H, int n_frames) {
    const int pw = (W + 1) >> 1;
    const size_t row_in = ((size_t)W * 2 + 3) & ~(size_t)3;
    const long long total = (long long)n_frames * H * pw;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int p = (int)(i % pw);
        const long long t = i / pw;
        const int row = (int)(t % H), frame = (int)(t / H);
        const uint8_t* q = in + (size_t)frame * stride_in + (size_t)row * row_in + (size_t)p * 4;
        const Chroma c = chroma_terms(q[1], q[3]);
        for (int k = 0; k < 2 && 2 * p + k < W; ++k) {
            int r, g, b;
            yuv_px(q[2 * k], c, r, g, b);
            uint8_t* o = out + (size_t)frame * stride_out + ((size_t)row * W + 2 * p + k) * 3;
            o[0] = (uint8_t)r, o[1] = (uint8_t)g, o[2] = (uint8_t)b;
        }
    }
}

cudaError_t launch_yuy2_to_rgb(const uint8_t* d_yuy2, size_t stride_in, uint8_t* d_rgb, size_t stride_out, int width, int height,
                               int n_frames, cudaStream_t s) {
    if (width <= 0 || height <= 0 || n_frames <= 0) return cudaSuccess;
    const bool aligned = (width % 8 == 0) && (height <= 65535) && (n_frames <= 65535) && (stride_in % 16 == 0) && (stride_out % 16 == 0) &&
                         ((size_t)width * 3 % 16 == 0) &&
                         ((reinterpret_cast<uintptr_t>(d_yuy2) | reinterpret_cast<uintptr_t>(d_rgb)) % 16 == 0);
    if (aligned && width % 16 == 0) {
        const long long items = (long long)width * height / 16;  // flat 16-pixel items, 64 per warp
        const dim3 grid((unsigned)((items + 64 * kCvt4Warps - 1) / (64 * kCvt4Warps)), 1, n_frames);
        yuy2_to_rgb_vec2_kernel<<<grid, kCvt4Warps * 32, 0, s>>>(d_yuy2, stride_in, d_rgb, stride_out, width, height);
    } else if (aligned) {
        const int segs = (width + 255) / 256;
        const int wpb = segs < kCvtWarps ? segs : kCvtWarps;
        const dim3 grid((segs + wpb - 1) / wpb, height, n_frames);  // one warp per 256-px row segment
        yuy2_to_rgb_vec_kernel<<<grid, wpb * 32, 0, s>>>(d_yuy2, stride_in, d_rgb, stride_out, width, height, n_frames);
    } else {
        const long long items = (long long)n_frames * height * ((width + 1) / 2);
        long long blocks = (items + 255) / 256;
        if (blocks > 148LL * 32) blocks = 148LL * 32;
        yuy2_to_rgb_generic_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_yuy2, stride_in, d_rgb, stride_out, width, height, n_frames);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K2: fused crop (zero border) + NV12->RGB + OpenCV INTER_LINEAR (fixed point) + normalise.
// One thread per output pixel; output goes straight into the patch-major A operand of the
// patch-embed GEMM: patches[target][token][c*256 + py*16 + px].
// ------------------------------------------------------------------------------------------------
struct Tap { int ofs; int a0, a1; };

// OpenCV resize coefficient for destination index i (SURVEY.md App. A.3). clamp_frac: horizontal taps clamp
// the fraction at the borders, vertical taps keep it and clamp the row index instead.
__device__ __forceinline__ Tap lin_tap(int i, int s, int d, bool clamp_frac) {
    const double scale = __ddiv_rn(1.0, __ddiv_rn((double)d, (double)s));
    float f = (float)__dadd_rn(__dmul_rn((double)i + 0.5, scale), -0.5);
    int ix = (int)floorf(f);
    f = __fsub_rn(f, (float)ix);
    if (clamp_frac) {
        if (ix < 0) ix = 0, f = 0.f;
        if (ix >= s - 1) ix = s - 1, f = 0.f;
    }
    Tap t;
    t.ofs = ix;
    t.a0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
    t.a1 = __float2int_rn(__fmul_rn(f, 2048.f));
    return t;
}

// Where the pixels of this frame live: the device frame inside the valid window (the part that was uploaded this frame), the
// caller's pinned host frame (zero-copy loads over PCIe) outside of it.  With whole-frame uploads the window is the frame.  The device
// frame may be a pitched surface; the host frame has the device frame's pitches and plane offset (see FrameRef).
struct PixelSrc {
    const uint8_t *dev, *dev_uv;  // device planes: Y / RGB / gray, NV12 chroma / I420 U
    size_t pitch, uv_pitch;       // their row pitches
    const uint8_t* host;          // null: everything is on the device
    int x0, y0, x1, y1;           // valid window of the device frame (even-aligned, so a pixel and its chroma pair sit on the same side;
                                  // x1 >= x0, y1 >= y0)
    bool dev_words, host_words;   // YUY2 / RGBA / BGRA: the plane's words (pixel pairs, pixels) are 4-byte aligned (base and pitch), one
                                  // 32-bit load each
    int format;                   // vt_format of this target's frame
    int xlim, ylim;               // pixels [0, xlim) x [0, ylim) are read, the rest is border (0 x 0 for a short frame)
};

// the 4 bytes at q (a YUY2 Y0 U Y1 V word, an RGBA / BGRA pixel): one 32-bit load when aligned, else four byte loads (surfaces may have
// any pitch)
__device__ __forceinline__ uint32_t plane_word(const uint8_t* q, bool aligned) {
    if (aligned) return *reinterpret_cast<const uint32_t*>(q);
    return (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
}

// RGB of the frame pixel (fx, fy); zero outside the frame (constant border of the crop).  pad: the kernel's pad_plus1.
__device__ __forceinline__ void frame_rgb(const PixelSrc& ps, int pad, int fx, int fy, int& r, int& g, int& b) {
    r = g = b = 0;
    if (fx < 0 || fy < 0 || fx >= ps.xlim || fy >= ps.ylim) return;
    const bool host = ps.host && ((unsigned)(fx - ps.x0) >= (unsigned)(ps.x1 - ps.x0) || (unsigned)(fy - ps.y0) >= (unsigned)(ps.y1 - ps.y0));
    const uint8_t* data = host ? ps.host : ps.dev;  // (same pitches: see PixelSrc)
    if (ps.format == VT_FMT_RGB24) {
        const uint8_t* p = data + (size_t)fy * ps.pitch + (size_t)fx * 3;
        r = p[0], g = p[1], b = p[2];
    } else if (ps.format == VT_FMT_GRAY8) {
        r = g = b = data[(size_t)fy * ps.pitch + fx];
    } else if (ps.format == VT_FMT_YUY2) {
        const uint32_t w = plane_word(data + (size_t)fy * ps.pitch + 4 * (fx >> 1), host ? ps.host_words : ps.dev_words);
        const Chroma c = chroma_terms((int)((w >> 8) & 0xff), (int)(w >> 24));
        yuv_px((int)((w >> ((fx & 1) * 16)) & 0xff), c, r, g, b);
    } else if (format_is_rgb32(ps.format)) {  // byte 3 is loaded with the word but never used
        const uint32_t w = plane_word(data + (size_t)fy * ps.pitch + 4 * (size_t)fx, host ? ps.host_words : ps.dev_words);
        const RgbOffsets o = fmt_rgb_offsets(ps.format);
        r = (int)((w >> (8 * o.r)) & 0xff), g = (int)((w >> (8 * o.g)) & 0xff), b = (int)((w >> (8 * o.b)) & 0xff);
    } else {
        const int yv = data[(size_t)fy * ps.pitch + fx];
        const uint8_t* uv = host ? ps.host + (ps.dev_uv - ps.dev) : ps.dev_uv;
        int u, v;
        if (ps.format == VT_FMT_I420) {
            // U of the pixel's 2x2 block in plane 1; V at the same place one chroma plane further, uv_pitch * ceil(H / 2): only packed
            // frames are I420 (no surfaces), and a pixel is read only when the frame is valid, where H = ylim + pad.  (H is not kept in
            // PixelSrc: one more live register would make ptxas spill at 32.)
            const uint8_t* q = uv + (size_t)(fy >> 1) * ps.uv_pitch + (fx >> 1);
            u = q[0], v = q[ps.uv_pitch * (size_t)((ps.ylim + pad + 1) >> 1)];
        } else {
            const size_t uvi = (size_t)(fy >> 1) * ps.uv_pitch + (fx & ~1);
            u = uv[uvi], v = uv[uvi + 1];
        }
        const Chroma c = chroma_terms(u, v);
        yuv_px(yv, c, r, g, b);
    }
}

// (minimum of 8 CTAs per SM stated: without it ptxas takes 40 registers, 6 CTAs of 256 per SM)
__global__ void __launch_bounds__(256, 8) crop_resize_norm_kernel(FrameDesc f, TargetState* __restrict__ state,
                                                               const int32_t* __restrict__ slots, int factor, int S,
                                                               const float* __restrict__ lut, float* __restrict__ patches,
                                                               size_t patches_stride, __nv_bfloat16* __restrict__ p_hi,
                                                               __nv_bfloat16* __restrict__ p_lo, unsigned long long* stamp) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the template gather behind this kernel does not depend on it
    if (stamp && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) *stamp = device_time_ns();
    const int bi = blockIdx.y;
    // this target's frame (one target per blockIdx.y: the format branch varies between CTAs, never within one), and with a control block
    // which part of the device frame holds this frame's pixels
    const FrameRef& fr = f.ctl ? target_frame(*f.ctl, bi) : f.frame;
    const int4 g = *reinterpret_cast<const int4*>(fr.geom);
    const int format = g.x, width = g.y, height = g.z, valid = g.w;
    PixelSrc ps{fr.plane[0], fr.plane[1], fr.pitch[0], fr.pitch[1], nullptr, 0, 0, width, height, false, false, format, 0, 0};
    if (f.ctl && f.ctl->n_win >= 0) {
        const int nw = f.ctl->n_win;
        ps.host = fr.host;
        if (bi < nw) ps.x0 = f.ctl->win[bi][0], ps.y0 = f.ctl->win[bi][1], ps.x1 = f.ctl->win[bi][2], ps.y1 = f.ctl->win[bi][3];
        else ps.x1 = ps.y1 = 0;  // nothing of this target was uploaded
    }
    ps.dev_words = ((reinterpret_cast<uintptr_t>(ps.dev) | ps.pitch) & 3) == 0;
    ps.host_words = (reinterpret_cast<uintptr_t>(ps.host) & 3) == 0;  // (packed YUY2 / RGBA / BGRA rows are whole words)
    // pad_plus1 (App. A.7, older OpenCV): a crop that reaches the right / bottom edge pads one pixel more, i.e. the last column / row of
    // the frame reads as border; a crop that stays inside never addresses it, so the bound can move unconditionally
    ps.xlim = valid ? width - f.pad_plus1 : 0, ps.ylim = valid ? height - f.pad_plus1 : 0;
    const int slot = slots[bi];
    TargetState* st = state + slot;
    const int bx = st->rect[0], by = st->rect[1], bw = st->rect[2], bh = st->rect[3];
    // A.1: c = ceil(sqrt(w*h) * factor); origin by C truncating division
    const long long area = (long long)bw * bh;
    int c = 0;
    if (bw > 0 && bh > 0) c = (int)ceil(__dmul_rn(sqrt((double)(int)area), (double)factor));
    const int x1 = bx + (bw - c) / 2, y1 = by + (bh - c) / 2;
    const int pl = max(0, -x1), pt = max(0, -y1);
    const int pr = max(x1 + c - width + f.pad_plus1, 0), pb = max(y1 + c - height + f.pad_plus1, 0);
    const bool outside = (c <= 0) || (c - pl - pr <= 0) || (c - pt - pb <= 0);
    if (threadIdx.x == 0 && blockIdx.x == 0 && factor == 4) st->crop_err = outside ? 1 : 0;
    if (outside) return;

    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= S * S) return;
    const int dx = idx % S, dy = idx / S;
    const Tap tx = lin_tap(dx, c, S, true);
    const Tap ty = lin_tap(dy, c, S, false);
    const int cx0 = tx.ofs, cx1 = min(tx.ofs + 1, c - 1);
    const int cy0 = min(max(ty.ofs, 0), c - 1), cy1 = min(max(ty.ofs + 1, 0), c - 1);
    // each pair of horizontal taps is blended as soon as it is read (three sums stay live instead of six samples: with the I420 read in
    // frame_rgb this keeps the kernel at 32 registers without spills; the arithmetic is unchanged)
    int qa[3], qb[3], t0[3], t1[3];
    frame_rgb(ps, f.pad_plus1, x1 + cx0, y1 + cy0, qa[0], qa[1], qa[2]);
    frame_rgb(ps, f.pad_plus1, x1 + cx1, y1 + cy0, qb[0], qb[1], qb[2]);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) t0[ch] = qa[ch] * tx.a0 + qb[ch] * tx.a1;
    frame_rgb(ps, f.pad_plus1, x1 + cx0, y1 + cy1, qa[0], qa[1], qa[2]);
    frame_rgb(ps, f.pad_plus1, x1 + cx1, y1 + cy1, qb[0], qb[1], qb[2]);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) t1[ch] = qa[ch] * tx.a0 + qb[ch] * tx.a1;
    const int nt = S >> 4;
    const int token = (dy >> 4) * nt + (dx >> 4);
    const size_t off = (size_t)bi * patches_stride + (size_t)token * kPatchK + (dy & 15) * 16 + (dx & 15);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const int v = (((ty.a0 * (t0[ch] >> 4)) >> 16) + ((ty.a1 * (t1[ch] >> 4)) >> 16) + 2) >> 2;
        const float val = lut[ch * 256 + (v & 255)];
        patches[off + ch * 256] = val;
        if (p_hi && !p_lo) {  // single-pass fp16 operands
            reinterpret_cast<unsigned short*>(p_hi)[off + ch * 256] = operand_bits(val, true);
        } else if (p_hi) {
            const __nv_bfloat16 h = __float2bfloat16_rn(val);
            p_hi[off + ch * 256] = h;
            p_lo[off + ch * 256] = __float2bfloat16_rn(val - __bfloat162float(h));
        }
    }
}

cudaError_t launch_crop_resize_norm(FrameDesc f, TargetState* d_state, const int32_t* d_slots, int n, int factor, int out_size,
                                    const float* d_norm_lut, float* d_patches, size_t patches_stride, __nv_bfloat16* p_hi,
                                    __nv_bfloat16* p_lo, cudaStream_t s, unsigned long long* stamp) {
    if (n <= 0) return cudaSuccess;
    dim3 grid((out_size * out_size + 255) / 256, n);
    crop_resize_norm_kernel<<<grid, 256, 0, s>>>(f, d_state, d_slots, factor, out_size, d_norm_lut, d_patches, patches_stride, p_hi, p_lo, stamp);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// RGB24 resize, OpenCV INTER_LINEAR fixed-point semantics (SURVEY.md App. A.3; bit-exact with cv2.resize) — SURVEY.md §8(f)
// row 1: the display upscale after the probe (≙ rgaconvert 640x512 -> 1280x1024, src/pipeline_ir.rs:62-73).  One thread per
// destination pixel; a warp reads two source rows segments and writes 96 contiguous bytes.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) resize_rgb_linear_kernel(const uint8_t* __restrict__ src, int sw, int sh, uint8_t* __restrict__ dst,
                                                                int dw, int dh) {
    const long long total = (long long)dw * dh;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int dx = (int)(i % dw), dy = (int)(i / dw);
        const Tap tx = lin_tap(dx, sw, dw, true);
        const Tap ty = lin_tap(dy, sh, dh, false);
        const int x0 = tx.ofs, x1 = min(tx.ofs + 1, sw - 1);
        const int y0 = min(max(ty.ofs, 0), sh - 1), y1 = min(max(ty.ofs + 1, 0), sh - 1);
        const uint8_t *r0 = src + (size_t)y0 * sw * 3, *r1 = src + (size_t)y1 * sw * 3;
        uint8_t* o = dst + (size_t)i * 3;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const int t0 = r0[x0 * 3 + ch] * tx.a0 + r0[x1 * 3 + ch] * tx.a1;
            const int t1 = r1[x0 * 3 + ch] * tx.a0 + r1[x1 * 3 + ch] * tx.a1;
            o[ch] = (uint8_t)((((ty.a0 * (t0 >> 4)) >> 16) + ((ty.a1 * (t1 >> 4)) >> 16) + 2) >> 2);
        }
    }
}

// Batched form with the taps of every destination column / row precomputed on the host (ResizeTaps: the same float arithmetic, done
// once per geometry instead of two double divisions per pixel): one warp produces 128 destination pixels of a row — 4 per lane, 12
// bytes staged in shared memory — and writes them as 24 coalesced 16-byte stores.  0.98 MB read + 3.9 MB written per 640x512 ->
// 1280x1024 frame: write bound.
constexpr int kRszWarps = 8;
__global__ void __launch_bounds__(kRszWarps * 32) resize_rgb_tab_kernel(const uint8_t* __restrict__ src, size_t stride_in, int sw, int sh,
                                                                      uint8_t* __restrict__ dst, size_t stride_out, int dw, int dh,
                                                                      const int4* __restrict__ xt, const int4* __restrict__ yt) {
    __shared__ __align__(16) uint8_t stage[kRszWarps][384];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int seg = blockIdx.x * kRszWarps + warp, dy = blockIdx.y, frame = blockIdx.z;
    if (seg * 128 >= dw) return;
    const uint8_t* sp = src + (size_t)frame * stride_in;
    const int4 ty = __ldg(yt + dy);  // y0, y1 (clamped rows), b0, b1
    const uint8_t *r0 = sp + (size_t)ty.x * sw * 3, *r1 = sp + (size_t)ty.y * sw * 3;
    const int seg_px = min(128, dw - seg * 128);
    uint32_t w3[3] = {0, 0, 0};
    uint8_t px[12];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int dx = seg * 128 + lane * 4 + k;
        if (dx < dw) {
            const int4 tx = __ldg(xt + dx);  // x0, x1 (clamped), a0, a1
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const int t0 = r0[tx.x * 3 + ch] * tx.z + r0[tx.y * 3 + ch] * tx.w;
                const int t1 = r1[tx.x * 3 + ch] * tx.z + r1[tx.y * 3 + ch] * tx.w;
                px[3 * k + ch] = (uint8_t)((((ty.z * (t0 >> 4)) >> 16) + ((ty.w * (t1 >> 4)) >> 16) + 2) >> 2);
            }
        } else {
            px[3 * k] = px[3 * k + 1] = px[3 * k + 2] = 0;
        }
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) w3[j] = px[4 * j] | (px[4 * j + 1] << 8) | (px[4 * j + 2] << 16) | ((uint32_t)px[4 * j + 3] << 24);
    uint32_t* st = reinterpret_cast<uint32_t*>(&stage[warp][lane * 12]);
    st[0] = w3[0], st[1] = w3[1], st[2] = w3[2];
    __syncwarp();
    uint8_t* gp = dst + (size_t)frame * stride_out + ((size_t)dy * dw + (size_t)seg * 128) * 3;
    const int row_bytes = seg_px * 3;
    const int off = lane * 16;
    if (off + 16 <= row_bytes) *reinterpret_cast<uint4*>(gp + off) = *reinterpret_cast<const uint4*>(&stage[warp][off]);
    else if (off < row_bytes)
        for (int b = off; b < row_bytes; ++b) gp[b] = stage[warp][b];
}

// Tiled separable form (up-scales: a tile of 16 destination rows needs at most kRszSrcRows source rows).  One CTA produces 16 rows x 256
// pixels: phase 1 blends every needed source row horizontally ONCE — T[row][dx][ch] = (p0 a0 + p1 a1) >> 4 as u16 in shared memory (the
// per-row kernel above recomputes it for every destination row: 12 scattered byte loads per pixel) — phase 2 blends two T rows vertically,
// 16 output bytes per thread from four 16-byte shared-memory loads, written as one 16-byte store.  Same integer formulas, bit-exact.
constexpr int kRszTileRows = 16, kRszTilePx = 256, kRszSrcRows = 12, kRszThreads = 256;
__global__ void __launch_bounds__(kRszThreads) resize_rgb_tile_kernel(const uint8_t* __restrict__ src, size_t stride_in, int sw, int sh,
                                                                     uint8_t* __restrict__ dst, size_t stride_out, int dw, int dh,
                                                                     const int4* __restrict__ xt, const int4* __restrict__ yt) {
    __shared__ __align__(16) uint16_t T[kRszSrcRows][kRszTilePx * 3];
    const int x0 = blockIdx.x * kRszTilePx, dy0 = blockIdx.y * kRszTileRows, frame = blockIdx.z;
    const int npx = min(kRszTilePx, dw - x0), nrow_out = min(kRszTileRows, dh - dy0);
    const uint8_t* sp = src + (size_t)frame * stride_in;
    const int ylo = __ldg(yt + dy0).x, yhi = __ldg(yt + dy0 + nrow_out - 1).y;  // (row taps are monotonic)
    const int nsrc = min(yhi - ylo + 1, kRszSrcRows);
    // ---- phase 1: thread t owns the flat (dx, ch) elements t, t + 256, t + 512 of a row, for every source row of the tile
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int e = threadIdx.x + k * kRszThreads;
        if (e < npx * 3) {
            const int dx = e / 3, ch = e - 3 * dx;
            const int4 tx = __ldg(xt + x0 + dx);  // x0, x1 (clamped), a0, a1
            const int rs = sw * 3;
            const uint8_t *p0 = sp + (size_t)ylo * rs + tx.x * 3 + ch, *p1 = sp + (size_t)ylo * rs + tx.y * 3 + ch;
            int v0[kRszSrcRows], v1[kRszSrcRows];  // every load of the column issued before the first use (one L2 round trip, not nsrc)
#pragma unroll
            for (int r = 0; r < kRszSrcRows; ++r)
                if (r < nsrc) v0[r] = p0[r * rs], v1[r] = p1[r * rs];
#pragma unroll
            for (int r = 0; r < kRszSrcRows; ++r)
                if (r < nsrc) T[r][e] = (uint16_t)((v0[r] * tx.z + v1[r] * tx.w) >> 4);
        }
    }
    __syncthreads();
    // ---- phase 2: 16 bytes (flat elements 16 q ..) of destination row dy0 + row per thread and step
    const int q_per_row = npx * 3 / 16;
    constexpr int kQ = kRszTilePx * 3 / 16;  // 48 16-byte slots per full tile row (constant divisor; slots past a narrow tile's row are skipped)
    for (int u = threadIdx.x; u < nrow_out * kQ; u += kRszThreads) {
        const int row = u / kQ, q = u - row * kQ;
        if (q >= q_per_row) continue;
        const int4 ty = __ldg(yt + dy0 + row);  // y0, y1 (clamped rows), b0, b1
        const uint4* t0 = reinterpret_cast<const uint4*>(&T[ty.x - ylo][16 * q]);
        const uint4* t1 = reinterpret_cast<const uint4*>(&T[ty.y - ylo][16 * q]);
        uint32_t a[8], b[8], o[4];
        *reinterpret_cast<uint4*>(a) = t0[0], *reinterpret_cast<uint4*>(a + 4) = t0[1];
        *reinterpret_cast<uint4*>(b) = t1[0], *reinterpret_cast<uint4*>(b + 4) = t1[1];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            uint32_t x[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t wa = a[2 * w + (j >> 1)], wb = b[2 * w + (j >> 1)];
                const int ta = (j & 1) ? (int)(wa >> 16) : (int)(wa & 0xffff), tb = (j & 1) ? (int)(wb >> 16) : (int)(wb & 0xffff);
                x[j] = (uint32_t)((((ty.z * ta) >> 16) + ((ty.w * tb) >> 16) + 2) >> 2);
            }
            o[w] = __byte_perm(__byte_perm(x[0], x[1], 0x0040), __byte_perm(x[2], x[3], 0x0040), 0x5410);
        }
        uint8_t* gp = dst + (size_t)frame * stride_out + ((size_t)(dy0 + row) * dw + x0) * 3 + 16 * q;
        *reinterpret_cast<uint4*>(gp) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

cudaError_t launch_resize_rgb_tab(const uint8_t* d_src, size_t stride_in, int sw, int sh, uint8_t* d_dst, size_t stride_out, int dw, int dh,
                                  int n_frames, const int4* d_xt, const int4* d_yt, cudaStream_t s, int max_src_rows) {
    if (sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || n_frames <= 0) return cudaSuccess;
    if (max_src_rows > 0 && max_src_rows <= kRszSrcRows) {
        const dim3 grid((dw + kRszTilePx - 1) / kRszTilePx, (dh + kRszTileRows - 1) / kRszTileRows, n_frames);
        resize_rgb_tile_kernel<<<grid, kRszThreads, 0, s>>>(d_src, stride_in, sw, sh, d_dst, stride_out, dw, dh, d_xt, d_yt);
        return cudaGetLastError();
    }
    const dim3 grid((dw + 128 * kRszWarps - 1) / (128 * kRszWarps), dh, n_frames);
    resize_rgb_tab_kernel<<<grid, kRszWarps * 32, 0, s>>>(d_src, stride_in, sw, sh, d_dst, stride_out, dw, dh, d_xt, d_yt);
    return cudaGetLastError();
}

cudaError_t launch_resize_rgb_linear(const uint8_t* d_src, int sw, int sh, uint8_t* d_dst, int dw, int dh, cudaStream_t s) {
    if (sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0) return cudaSuccess;
    long long blocks = ((long long)dw * dh + 255) / 256;
    if (blocks > 148LL * 32) blocks = 148LL * 32;
    resize_rgb_linear_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_src, sw, sh, d_dst, dw, dh);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K9 overlay.  One CTA walks the command list in order (a barrier between commands keeps the
// reference's draw order where commands overlap: background dim -> text -> cursor -> box).
// Each primitive is a flattened parallel loop over exactly the pixels the reference loop nests
// visit; usize/i32 semantics of the Rust code are reproduced with 64-bit integers.
// ------------------------------------------------------------------------------------------------
typedef unsigned long long u64;
__device__ __forceinline__ u64 i32_as_usize(int v) { return (u64)(long long)v; }
__device__ __forceinline__ u64 sat_sub(u64 a, u64 b) { return a > b ? a - b : 0; }
__device__ __forceinline__ u64 umin64(u64 a, u64 b) { return a < b ? a : b; }

struct Surface {
    uint8_t* d;
    size_t len;            // bytes of the drawn plane (RGB writes are bounds-checked against it)
    int W, H, fmt;
    size_t pitch;          // row pitch of the drawn plane in bytes (Y plane / RGB image)
    int step;              // bytes between the pixels of a row: luma formats, between the Y samples (1; YUY2: 2, the chroma bytes in
                           // between are never written); RGB formats, the pixel size (RGB24: 3; RGBA / BGRA: 4, byte 3 is never written)
    RgbOffsets ch;         // RGB formats: the bytes of R, G, B within a pixel
};
__device__ __forceinline__ Surface make_surface(uint8_t* d, size_t len, int W, int H, int fmt, size_t pitch) {
    return Surface{d, len, W, H, overlay_format(fmt), pitch, fmt_px_step(fmt), fmt_rgb_offsets(fmt)};
}
// NV12: luma write (Y plane). RGB: bounds-checked colour write (src/drawing_rgb.rs:18-28); the pixel's last colour byte is byte 2 in
// every RGB format.
__device__ __forceinline__ void put_y(const Surface& s, u64 x, u64 y, uint8_t v) { s.d[y * (u64)s.pitch + x * (u64)s.step] = v; }
__device__ __forceinline__ void put_rgb(const Surface& s, int x, int y, uint8_t r, uint8_t g, uint8_t b) {
    if (x < 0 || y < 0 || x >= s.W || y >= s.H) return;
    const size_t off = (size_t)y * s.pitch + (size_t)x * s.step;
    if (off + 2 < s.len) s.d[off + s.ch.r] = r, s.d[off + s.ch.g] = g, s.d[off + s.ch.b] = b;
}

__device__ void ov_rect_nv12(const Surface& s, int x, int y, int w, int h, int thickness, uint8_t v) {  // src/nv12_convert.rs:172-213
    const u64 W = s.W, H = s.H, th = (u64)max(thickness, 0);
    const u64 x1 = (u64)max(x, 0), y1 = (u64)max(y, 0);
    const u64 x2 = umin64(i32_as_usize((int)((unsigned)x + (unsigned)w)), sat_sub(W, 1));
    const u64 y2 = umin64(i32_as_usize((int)((unsigned)y + (unsigned)h)), sat_sub(H, 1));
    const u64 nx = x2 >= x1 ? x2 - x1 + 1 : 0, ny = y2 >= y1 ? y2 - y1 + 1 : 0;
    const u64 n_h = th * 2 * nx;  // horizontal runs
    // (index decomposition in 32 bits when the counts fit — every real frame: a 64-bit division costs ~100 instructions, and this code
    // is most of the frame's last kernel)
    const bool small = n_h < (1ull << 31) && ny * th * 2 < (1ull << 31);
    for (u64 i = threadIdx.x; i < n_h; i += blockDim.x) {
        const u64 kq = small ? (u64)((uint32_t)i / (uint32_t)nx) : i / nx;
        const u64 px = x1 + (i - kq * nx), k = kq, t = k >> 1;
        if ((k & 1) == 0) {
            if (y1 + t < H) put_y(s, px, y1 + t, v);
        } else if (y2 >= t && y2 - t < H) {
            put_y(s, px, y2 - t, v);
        }
    }
    const u64 n_v = ny * th * 2;  // vertical runs
    for (u64 i = threadIdx.x; i < n_v; i += blockDim.x) {
        const u64 rq = small ? (u64)((uint32_t)i / (uint32_t)(th * 2)) : i / (th * 2);
        const u64 py = y1 + rq, k = i - rq * (th * 2), t = k >> 1;
        if ((k & 1) == 0) {
            if (x1 + t < W) put_y(s, x1 + t, py, v);
        } else if (x2 >= t && x2 - t < W) {
            put_y(s, x2 - t, py, v);
        }
    }
}
__device__ void ov_rect_rgb(const Surface& s, int x, int y, int rw, int rh, int thickness, uint8_t r, uint8_t g, uint8_t b) {  // src/drawing_rgb.rs:55-66
    const long long nw = max(rw, 0), nh = max(rh, 0), th = max(thickness, 0);
    for (long long i = threadIdx.x; i < th * nw * 2; i += blockDim.x) {
        const int t = (int)(i / (nw * 2)), j = (int)(i % (nw * 2)), k = j >> 1;
        if ((j & 1) == 0) put_rgb(s, x + k, y + t, r, g, b);
        else put_rgb(s, x + k, y + rh - 1 - t, r, g, b);
    }
    for (long long i = threadIdx.x; i < th * nh * 2; i += blockDim.x) {
        const int t = (int)(i / (nh * 2)), j = (int)(i % (nh * 2)), k = j >> 1;
        if ((j & 1) == 0) put_rgb(s, x + t, y + k, r, g, b);
        else put_rgb(s, x + rw - 1 - t, y + k, r, g, b);
    }
}
__device__ void ov_crosshair_nv12(const Surface& s, int cx_, int cy_, int size_, uint8_t v) {  // src/nv12_convert.rs:216-242
    const u64 W = s.W, H = s.H, cx = (u64)max(cx_, 0), cy = (u64)max(cy_, 0), size = i32_as_usize(size_);
    if (cy < H) {
        const u64 a = sat_sub(cx, size), b = umin64(cx + size, W - 1);
        for (u64 x = a + threadIdx.x; x <= b && b >= a; x += blockDim.x) put_y(s, x, cy, v);
    }
    if (cx < W) {
        const u64 a = sat_sub(cy, size), b = umin64(cy + size, H - 1);
        for (u64 y = a + threadIdx.x; y <= b && b >= a; y += blockDim.x) put_y(s, cx, y, v);
    }
}
__device__ void ov_crosshair_rgb(const Surface& s, int cx, int cy, int size, uint8_t r, uint8_t g, uint8_t b) {  // src/drawing_rgb.rs:68-73
    for (int i = -size + (int)threadIdx.x; i <= size; i += blockDim.x) {
        put_rgb(s, cx + i, cy, r, g, b);
        put_rgb(s, cx, cy + i, r, g, b);
    }
}
__device__ void ov_text(const Surface& s, const OverlayCmdDev& c) {  // src/nv12_convert.rs:245-321 / src/drawing_rgb.rs:86-104
    const int scale = max(c.a, 0);
    const long long per_char = 35LL * scale * scale;
    const long long total = per_char * c.nchar;
    const bool small = total < (1LL << 31);  // 32-bit index decomposition (see ov_rect_nv12)
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
        const int ch = small ? (int)((uint32_t)i / (uint32_t)per_char) : (int)(i / per_char);
        long long r = i - (long long)ch * per_char;
        const int cell = small ? (int)((uint32_t)r / (uint32_t)(scale * scale)) : (int)(r / (scale * scale));
        const int sub = (int)(r - (long long)cell * (scale * scale));
        const int row = cell / 5, col = cell % 5, dy = sub / scale, dx = sub % scale;
        if (!c.known[ch] || !((c.glyph[ch][row] >> (4 - col)) & 1)) continue;
        if (s.fmt == VT_FMT_NV12) {
            const u64 px = (u64)c.x + (u64)ch * 6 * scale + (u64)col * scale + dx, py = (u64)c.y + (u64)row * scale + dy;
            if (px < (u64)s.W && py < (u64)s.H) put_y(s, px, py, c.r);
        } else {
            put_rgb(s, c.x + ch * 6 * scale + col * scale + dx, c.y + row * scale + dy, c.r, c.r, c.r);
        }
    }
}
__device__ void ov_background(const Surface& s, const OverlayCmdDev& c) {
    if (s.fmt == VT_FMT_NV12) {  // src/nv12_convert.rs:324-343: Y = (Y * (255-darkness)) / 255 in u16
        const u64 x0 = (u64)c.x, y0 = (u64)c.y;
        const u64 x1 = umin64(x0 + (u64)c.w, (u64)s.W), y1 = umin64(y0 + (u64)c.h, (u64)s.H);
        if (x1 <= x0 || y1 <= y0) return;
        const u64 nx = x1 - x0, n = nx * (y1 - y0);
        const unsigned factor = 255u - (unsigned)(uint8_t)c.a;
        for (u64 i = threadIdx.x; i < n; i += blockDim.x) {
            const u64 idx = (y0 + i / nx) * (u64)s.pitch + (x0 + i % nx) * (u64)s.step;
            s.d[idx] = (uint8_t)(((unsigned)s.d[idx] * factor) / 255u);
        }
    } else {  // src/drawing_rgb.rs:30-53: fill with 30
        const u64 xs = (u64)max(c.x, 0), xe = umin64(i32_as_usize((int)((unsigned)c.x + (unsigned)c.w)), (u64)s.W);
        const u64 ys = (u64)max(c.y, 0), ye = umin64(i32_as_usize((int)((unsigned)c.y + (unsigned)c.h)), (u64)s.H);
        if (xe <= xs || ye <= ys) return;
        // (every colour byte of the row span; of a 32-bit pixel, byte 3 is skipped)
        const u64 rb = (xe - xs) * (u64)s.step, n = rb * (ye - ys);
        for (u64 i = threadIdx.x; i < n; i += blockDim.x) {
            const u64 row = ys + i / rb, col = i % rb;
            const u64 off = row * (u64)s.pitch + xs * (u64)s.step;
            if (off + rb <= s.len && (s.step != 4 || (col & 3) != 3)) s.d[off + col] = 30;
        }
    }
}
__device__ void ov_cursor(const Surface& s, int x_, int y_) {
    if (s.fmt == VT_FMT_NV12) {  // src/drawing.rs:5-23
        const u64 W = s.W, H = s.H;
        const u64 x = (u64)min(max(x_, 0), s.W - 1), y = (u64)min(max(y_, 0), s.H - 1);
        const u64 ax = sat_sub(x, 25), bx = umin64(x + 25, W - 1);
        for (u64 px = ax + threadIdx.x; px <= bx; px += blockDim.x)
            if (!(px >= sat_sub(x, 5) && px <= x + 5)) put_y(s, px, y, 255);
        const u64 ay = sat_sub(y, 25), by = umin64(y + 25, H - 1);
        for (u64 py = ay + threadIdx.x; py <= by; py += blockDim.x)
            if (!(py >= sat_sub(y, 5) && py <= y + 5)) put_y(s, x, py, 255);
    } else {  // src/drawing_rgb.rs:75-84
        for (int i = 5 + (int)threadIdx.x; i <= 25; i += blockDim.x) {
            put_rgb(s, x_ + i, y_, 0, 255, 0);
            put_rgb(s, x_ - i, y_, 0, 255, 0);
            put_rgb(s, x_, y_ + i, 0, 255, 0);
            put_rgb(s, x_, y_ - i, 0, 255, 0);
        }
    }
}
__device__ void ov_selection(const Surface& s, int sx, int sy, int cx, int cy) {
    if (s.fmt == VT_FMT_NV12) {  // src/drawing.rs:25-50
        const u64 x1 = (u64)max(min(sx, cx), 0), y1 = (u64)max(min(sy, cy), 0);
        const u64 x2 = umin64(i32_as_usize(max(sx, cx)), (u64)s.W - 1), y2 = umin64(i32_as_usize(max(sy, cy)), (u64)s.H - 1);
        for (u64 x = x1 + threadIdx.x; x <= x2; x += blockDim.x)
            if ((x / 6) % 2 == 0) put_y(s, x, y1, 255), put_y(s, x, y2, 255);
        for (u64 y = y1 + threadIdx.x; y <= y2; y += blockDim.x)
            if ((y / 6) % 2 == 0) put_y(s, x1, y, 255), put_y(s, x2, y, 255);
    } else {  // src/drawing_rgb.rs:106-128
        const int x1 = max(min(sx, cx), 0), y1 = max(min(sy, cy), 0);
        const int x2 = min(max(sx, cx), s.W - 1), y2 = min(max(sy, cy), s.H - 1);
        for (int x = x1 + (int)threadIdx.x; x <= x2; x += blockDim.x)
            if ((x / 6) % 2 == 0) put_rgb(s, x, y1, 255, 255, 0), put_rgb(s, x, y2, 255, 255, 0);
        for (int y = y1 + (int)threadIdx.x; y <= y2; y += blockDim.x)
            if ((y / 6) % 2 == 0) put_rgb(s, x1, y, 255, 255, 0), put_rgb(s, x2, y, 255, 255, 0);
    }
}

__device__ void ov_dispatch(const Surface& s, const OverlayCmdDev& c) {
    switch (c.kind) {
        case VT_OV_RECT:
            if (s.fmt == VT_FMT_NV12) ov_rect_nv12(s, c.x, c.y, c.w, c.h, c.a, c.r);
            else ov_rect_rgb(s, c.x, c.y, c.w, c.h, c.a, c.r, c.g, c.b);
            break;
        case VT_OV_CROSSHAIR:
            if (s.fmt == VT_FMT_NV12) ov_crosshair_nv12(s, c.x, c.y, c.a, c.r);
            else ov_crosshair_rgb(s, c.x, c.y, c.a, c.r, c.g, c.b);
            break;
        case VT_OV_TEXT: ov_text(s, c); break;
        case VT_OV_BACKGROUND: ov_background(s, c); break;
        case VT_OV_CURSOR: ov_cursor(s, c.x, c.y); break;
        case VT_OV_SELECTION: ov_selection(s, c.x, c.y, c.w, c.h); break;
        default: break;
    }
}

__global__ void __launch_bounds__(1024) overlay_kernel(uint8_t* frame, size_t len, int W, int H, int fmt,
                                                       const OverlayCmdDev* __restrict__ cmds, int n) {
    const Surface s = make_surface(frame, len, W, H, fmt, fmt_row_bytes(fmt, W));
    for (int i = 0; i < n; ++i) {
        ov_dispatch(s, cmds[i]);
        __syncthreads();
    }
}

cudaError_t launch_overlay(uint8_t* d_frame, size_t len, int width, int height, int format, const OverlayCmdDev* d_cmds, int n,
                           cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    overlay_kernel<<<1, 1024, 0, s>>>(d_frame, len, width, height, format, d_cmds, n);
    return cudaGetLastError();
}

// Last kernel of a frame.  (a) Box overlay straight from the device-side decode result: one CTA per target, rect (thickness 3) then
// crosshair (size 15) at the box centre ≙ src/pipeline.rs:165-168 / src/pipeline_ir.rs:192-195.  (b) The frame's HUD command list
// (probe: ≙ src/pipeline.rs:125-174 / src/pipeline_ir.rs:165-202), CTA 0: the list holds the commands of BOTH outcomes of the frame
// and the kernel picks by the gate (status ok && success && score > gate, src/tracker_context.rs:93,122), takes the box geometry and
// the score digits from the decode result — the host queued it before the frame's result existed, so the whole probe needs ONE
// synchronisation.  (c) With a pinned caller frame (FrameRef::host) the touched pixels are also written straight into the host frame
// (zero-copy stores over PCIe; the dimmed background is copied out of the device frame), so no device->host row copy and no second
// synchronisation is needed to hand the overlaid frame back.  (d) The result block is published into the pinned host block.
__device__ void hud_score_glyphs(OverlayCmdDev& c, float score) {  // "score: " + "{:.0}%" of score*100 (src/pipeline.rs:146-156)
    const float pct = rintf(__fmul_rn(score, 100.0f));            // round-half-even, as Rust's {:.0} / printf("%.0f")
    int v = pct > 0.f ? (pct < 999.f ? (int)pct : 999) : 0;
    int dig[3], nd = 0;
    do { dig[nd++] = v % 10, v /= 10; } while (v && nd < 3);
    int k = c.nchar;
    for (int i = nd - 1; i >= 0 && k < 36; --i, ++k) {
        for (int r = 0; r < 7; ++r) c.glyph[k][r] = c.glyph[kHudDigitSlot + dig[i]][r];
        c.known[k] = c.known[kHudDigitSlot + dig[i]];
    }
    if (k < 36) {
        for (int r = 0; r < 7; ++r) c.glyph[k][r] = c.glyph[kHudPercentSlot][r];
        c.known[k] = c.known[kHudPercentSlot], ++k;
    }
    c.nchar = (uint8_t)k;
}

// The luma background dim of the probe HUD (src/nv12_convert.rs:324-343: Y = Y * (255 - darkness) / 255 over a rectangle) is the one
// read-modify-write of the overlay.  Its pixels are fetched in 4-byte words, ALL loads of a thread issued before anything else
// (a byte-wise loop whose loads wait for the previous iteration's stores — same array — costs one L2 round trip per pixel: measured
// ~90 us for the 400x80 HUD block on one CTA), from the caller's pinned host frame when there is one: that needs no upload of the region
// and, issued before the dependency wait, overlaps the kernels ahead.  The dimmed words go to the device frame and the host frame.
constexpr int kOvThreads = 512;
constexpr int kBgEdge = 2;    // ragged-edge bytes per thread held in registers (rows x <= 6 columns)
constexpr int kBgWords = 20;  // words per thread held in registers: 512 x 20 x 4 = 40 KB >= the 400 x 80 HUD block
// Pixels are addressed as row * y + step * x (step: the Y sample step of the format, 1 or 2); a word holds 4 / step pixels, and of a
// YUY2 word only bytes 0 and 2 (Y0, Y1) are dimmed.
struct BgRegion {
    long long x0, y0, x1, y1;  // clipped pixel rectangle (usize arithmetic of the reference), empty when x1 <= x0
    long long ax0, ax1;        // word-aligned interior of a row in pixels: [ax0, ax1), ax0 >= x0, ax1 <= x1
    int wpr;                   // words per row
    bool vec;                  // rows are word addressable (pitch % 4 == 0)
};
// pitch: bytes between the rows of the plane the region is read from and written to
__device__ BgRegion bg_region(const OverlayCmdDev& c, int W, int H, size_t pitch, int step) {
    BgRegion g;
    const u64 x0 = (u64)c.x, y0 = (u64)c.y;
    const u64 x1 = umin64(x0 + (u64)c.w, (u64)W), y1 = umin64(y0 + (u64)c.h, (u64)H);
    g.x0 = (long long)x0, g.y0 = (long long)y0, g.x1 = x1 > x0 && y1 > y0 ? (long long)x1 : (long long)x0, g.y1 = (long long)y1;
    g.vec = (pitch % 4) == 0;
    const long long ppw = 4 / step;  // pixels per word
    g.ax0 = (g.x0 + ppw - 1) & ~(ppw - 1), g.ax1 = g.x1 & ~(ppw - 1);
    g.wpr = g.vec && g.ax1 > g.ax0 ? (int)((g.ax1 - g.ax0) / ppw) : 0;
    return g;
}
__device__ __forceinline__ uint32_t dim4(uint32_t v, unsigned factor, int step) {
    const uint32_t d = ((v & 0xff) * factor / 255u) | ((((v >> 8) & 0xff) * factor / 255u) << 8) |
                       ((((v >> 16) & 0xff) * factor / 255u) << 16) | (((v >> 24) * factor / 255u) << 24);
    return step == 2 ? (d & 0x00ff00ffu) | (v & 0xff00ff00u) : d;
}

// The body of both last-kernel forms.  kGroup = false: box_overlay_kernel — CTA x draws the box of active target x (stream group: into
// that target's own frame), CTA 0 also runs the frame's HUD list.  kGroup = true: probe_group_overlay_kernel — CTA pair x draws stream x
// of a probe group (ProbeGroupCtl::s[x]: its frames, geometry, slot or -1, HUD list and background-dim handshake), whether or not the
// stream took part in the forward.  (Two instances of one body rather than one kernel with a runtime switch: the per-stream addressing
// stays out of the single probe's last kernel, whose size and register use are what they were.)
template <bool kGroup>
__device__ __forceinline__ void box_overlay_body(const DeviceResult* __restrict__ res, const int32_t* __restrict__ slots, int n, float gate,
                                                 const FrameCtl* ctl, unsigned long long* stamp_end, const uint32_t* __restrict__ blk,
                                                 int blk_words, int draw_box, OverlayCmdDev* s_cmd) {
    // the control block was written at the start of the frame (complete long before the kernel ahead of this one): every thread fetches
    // what it needs in one batch, and the HUD list comes out of pinned host memory, BEFORE the dependency wait: only the decode result
    // waits for the preceding kernel
    const ProbeStreamCtl* const e = kGroup ? &reinterpret_cast<const ProbeGroupCtl*>(ctl)->s[blockIdx.x] : nullptr;
    // the frame this CTA draws into — block i: target i's (stream group: stream i's own frame); probe group: pair x, stream x's — with its
    // format and size (nothing is written outside its plane 0), and its HUD list and background-dim flags: the frame's (CTA 0), or its
    // stream's (probe group)
    const FrameRef* const fr = kGroup ? &e->frame : &target_frame(*ctl, blockIdx.x);
    const HudCtl* const hud = kGroup ? &e->hud : &ctl->hud;
    const int4 g = *reinterpret_cast<const int4*>(fr->geom);
    const int fmt = g.x, W = g.y, H = g.z;
    // HUD mode runs two CTAs per target (gridDim.y = 2): y = 0 draws on the device frame (and publishes), y = 1 on the pinned host frame —
    // the two passes over the command list (~8 us each on one CTA) run side by side
    const bool split = gridDim.y > 1;
    uint8_t* const frame = const_cast<uint8_t*>(fr->plane[0]);
    uint8_t* const host = fr->host;
    if (split && blockIdx.y == 1 && !host) return;  // nothing to mirror into
    // row pitch of the drawn plane: the caller's surface pitch for the device frame; the pinned host frame is packed, and only ever goes
    // with a packed device frame (fpitch == row, see FrameRef): a surface step has no host frame, so no host-pass CTA and no bg_ready
    // handshake (host == nullptr above and below).  The background dim therefore addresses both frames by fpitch.
    // fmt is the frame's format: drawn with the overlay semantics of ofmt
    const size_t row = fmt_row_bytes(fmt, W);
    const int ofmt = overlay_format(fmt), step = fmt_px_step(fmt);
    const size_t fpitch = fr->pitch[0];
    const size_t plen = (size_t)(H - 1) * fpitch + row;  // bytes from the plane's first row to the end of its last
    const bool do_dev = !split || blockIdx.y == 0, do_host = host != nullptr && (!split || blockIdx.y == 1);
    const int32_t* const bg_on_dev = &hud->bg_on_device;
    const int32_t* const bg_ready = &hud->bg_ready;
    int n_hud = kGroup || blockIdx.x == 0 ? hud->n : 0;
    if (n_hud > kMaxCmds) n_hud = kMaxCmds;
    if (n_hud > 0) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(hud->list);
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_cmd);
        for (int i = threadIdx.x; i < n_hud * (int)(sizeof(OverlayCmdDev) / 4); i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    // the luma background dim, if it leads the list unconditionally (the probe's HUD): prefetch its pixels from the host frame now (or
    // from the device frame: a surface too, which no earlier kernel of the frame writes)
    const bool bg_first = n_hud > 0 && ofmt == VT_FMT_NV12 && s_cmd[0].kind == VT_OV_BACKGROUND && s_cmd[0].cond == VT_HUD_ALWAYS;
    BgRegion bg{0, 0, 0, 0, 0, 0, 0, false};
    uint32_t bgw[kBgWords];
    uint8_t bge[kBgEdge];
    bool bg_pre = false, bg_edge_pre = false;
    if (bg_first) {
        bg = bg_region(s_cmd[0], W, H, fpitch, step);
        const long long rows = bg.y1 - bg.y0;
        if (((reinterpret_cast<uintptr_t>(host) | reinterpret_cast<uintptr_t>(frame)) & 3) != 0) bg.wpr = 0;  // bytewise (as a pitch % 4)
        // source of the region: the device frame when it was uploaded with the windows (a copy-engine transfer ahead of the graph; an L2 hit
        // here), else the pinned host frame (PCIe reads: ~12 us for the 260 x 90 block, on the critical path of a short frame)
        const uint8_t* bsrc = (host && !*bg_on_dev) ? host : frame;
        bg_pre = (host || *bg_on_dev) && bg.wpr > 0 && rows * bg.wpr <= (long long)kBgWords * kOvThreads && (size_t)(bg.y1 - 1) * fpitch + row <= plen;
        if (bg_pre) {
            const int total = (int)rows * bg.wpr;
#pragma unroll
            for (int k = 0; k < kBgWords; ++k) {
                const int i = threadIdx.x + k * kOvThreads;
                if (i < total) bgw[k] = *reinterpret_cast<const volatile uint32_t*>(bsrc + (size_t)(bg.y0 + i / bg.wpr) * fpitch + bg.ax0 * step + 4 * (i % bg.wpr));
            }
            // ... and the columns outside the word interior (<= 3 + 3 per row), so that nothing of the region is read after the dependency
            // wait: with two CTAs per target the other CTA dims the device frame's copy of the region after its own wait
            const long long eh = bg.ax0 - bg.x0, ec = eh + (bg.x1 - bg.ax1);
            bg_edge_pre = rows * ec <= (long long)kBgEdge * kOvThreads;
            if (bg_edge_pre) {
#pragma unroll
                for (int k = 0; k < kBgEdge; ++k) {
                    const long long i = threadIdx.x + (long long)k * kOvThreads;
                    if (i < rows * ec) {
                        const uint32_t rq = (uint32_t)i / (uint32_t)ec;
                        const long long yy = bg.y0 + rq, kk = i - (long long)rq * ec, xx = kk < eh ? bg.x0 + kk : bg.ax1 + (kk - eh);
                        bge[k] = *reinterpret_cast<const volatile uint8_t*>(bsrc + (size_t)yy * fpitch + (size_t)xx * step);
                    }
                }
            }
        }
    }
    // two CTAs, both prefetched the region from the DEVICE frame: the device-pass CTA may only dim it there once the host-pass CTA holds
    // its copy (the loads are consumed below before the flag is raised)
    const bool bg_handshake = split && host != nullptr && bg_pre && *bg_on_dev;
    if (bg_handshake && blockIdx.y == 1) {
        uint32_t acc = 0;
#pragma unroll
        for (int k = 0; k < kBgWords; ++k) acc |= bgw[k];
#pragma unroll
        for (int k = 0; k < kBgEdge; ++k) acc |= bge[k];
        asm volatile("" ::"r"(acc));
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            atomicExch(const_cast<int32_t*>(bg_ready), 1);
        }
    }
    const int slot = kGroup ? e->slot : (int)blockIdx.x < n ? slots[blockIdx.x] : -1;
    if (stamp_end && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) stamp_end[1] = device_time_ns();  // diagnostics: prologue done
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (stamp_end && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) stamp_end[2] = device_time_ns();  // diagnostics: dependency satisfied
    DeviceResult r;
    r.status = VT_ERR_NOT_INIT, r.success = 0, r.score = 0.f, r.bbox[0] = r.bbox[1] = r.bbox[2] = r.bbox[3] = 0, r.best = 0;
    if (slot >= 0) r = res[slot];
    const bool pass = r.status == VT_OK && r.success && r.score > gate;
    if (draw_box && pass) {
        const int x = r.bbox[0], y = r.bbox[1], w = r.bbox[2], h = r.bbox[3];
        for (int p = 0; p < 2; ++p) {
            uint8_t* dst = p == 0 ? frame : host;
            if (!dst) break;
            if ((p == 0 && !do_dev) || (p == 1 && !do_host)) continue;
            const size_t pitch = p == 0 ? fpitch : row;
            const Surface s = make_surface(dst, plen, W, H, fmt, pitch);
            if (ofmt == VT_FMT_NV12) {
                ov_rect_nv12(s, x, y, w, h, 3, 255);
                __syncthreads();
                ov_crosshair_nv12(s, x + w / 2, y + h / 2, 15, 255);
            } else {
                ov_rect_rgb(s, x, y, w, h, 3, 0, 255, 0);
                __syncthreads();
                ov_crosshair_rgb(s, x + w / 2, y + h / 2, 15, 0, 255, 0);
            }
            __syncthreads();
        }
    }
    if (!kGroup && blockIdx.x != 0) return;
    if (n_hud > 0) {
        // resolve the result-dependent commands once (shared copy), drop the ones of the other outcome
        if ((int)threadIdx.x < n_hud) {
            OverlayCmdDev& c = s_cmd[threadIdx.x];
            if ((c.cond == VT_HUD_IF_PASS && !pass) || (c.cond == VT_HUD_IF_FAIL && pass)) c.kind = -1;
            else if (c.from_result == VT_HUD_RESULT_RECT) c.x = r.bbox[0], c.y = r.bbox[1], c.w = r.bbox[2], c.h = r.bbox[3];
            else if (c.from_result == VT_HUD_RESULT_CROSS) c.x = r.bbox[0] + r.bbox[2] / 2, c.y = r.bbox[1] + r.bbox[3] / 2;
            else if (c.from_result == VT_HUD_SCORE_TEXT) hud_score_glyphs(c, r.score);
        }
        __syncthreads();
        int first = 0;
        if (bg_handshake && blockIdx.y == 0) {  // (bounded: a protocol error must not hang the GPU; the flag is normally long set)
            if (threadIdx.x == 0) {
                const volatile int32_t* f = bg_ready;
                for (int i = 0; i < (1 << 18) && *f == 0; ++i) {}
            }
            __syncthreads();
        }
        if (bg_first) {  // ---- the background dim: word interior from registers (or the device frame), ragged edges bytewise
            const unsigned factor = 255u - (unsigned)(uint8_t)s_cmd[0].a;
            const long long rows = bg.y1 - bg.y0;
            if (bg.x1 > bg.x0 && (size_t)(bg.y1 - 1) * fpitch + row <= plen) {
                if (bg.wpr > 0) {
                    const long long total = rows * bg.wpr;
                    for (long long base = 0; base < total; base += (long long)kBgWords * kOvThreads) {
                        if (!bg_pre || base > 0) {  // not prefetched (no pinned frame, or a region larger than the register budget)
                            // (pinned frame: the region may not have been uploaded; a host-pass CTA always reads the host frame — the device
                            // frame's copy is being dimmed by the other CTA)
                            const uint8_t* src = ((host && !*bg_on_dev) || (split && do_host)) ? host : frame;
#pragma unroll
                            for (int k = 0; k < kBgWords; ++k) {
                                const long long i = base + threadIdx.x + (long long)k * kOvThreads;
                                if (i < total) {
                                    const uint32_t rr = (uint32_t)i / (uint32_t)bg.wpr, cc = (uint32_t)i - rr * (uint32_t)bg.wpr;
                                    bgw[k] = *reinterpret_cast<const uint32_t*>(src + (size_t)(bg.y0 + rr) * fpitch + bg.ax0 * step + 4 * cc);
                                }
                            }
                        }
#pragma unroll
                        for (int k = 0; k < kBgWords; ++k) {
                            const long long i = base + threadIdx.x + (long long)k * kOvThreads;
                            if (i < total) {
                                const uint32_t rr = (uint32_t)i / (uint32_t)bg.wpr, cc = (uint32_t)i - rr * (uint32_t)bg.wpr;
                                const size_t o = (size_t)(bg.y0 + rr) * fpitch + bg.ax0 * step + 4 * cc;
                                const uint32_t d = dim4(bgw[k], factor, step);
                                if (do_dev) *reinterpret_cast<uint32_t*>(frame + o) = d;
                                if (do_host) *reinterpret_cast<uint32_t*>(host + o) = d;
                            }
                        }
                    }
                }
                // columns outside the word interior (<= 3 + 3 per row; every column when rows are not word addressable)
                const long long eh = bg.wpr > 0 ? bg.ax0 - bg.x0 : bg.x1 - bg.x0, et = bg.wpr > 0 ? bg.x1 - bg.ax1 : 0, ec = eh + et;
                const bool edge_host = (host && !*bg_on_dev) || (split && do_host);
                for (long long i = threadIdx.x, kk = 0; i < rows * ec; i += blockDim.x, ++kk) {
                    const uint32_t rq = (uint32_t)i / (uint32_t)ec;  // (rows * ec < 2^31)
                    const long long yy = bg.y0 + rq, k = i - (long long)rq * ec, xx = k < eh ? bg.x0 + k : bg.ax1 + (k - eh);
                    const size_t o = (size_t)yy * fpitch + (size_t)xx * step;
                    const unsigned v = (bg_edge_pre && bg.wpr > 0) ? (unsigned)bge[kk < kBgEdge ? kk : 0] : (unsigned)(edge_host ? host[o] : frame[o]);
                    const uint8_t d = (uint8_t)((v * factor) / 255u);
                    if (do_dev) frame[o] = d;
                    if (do_host) host[o] = d;
                }
            }
            __syncthreads();
            first = 1;
        }
        for (int p = 0; p < 2; ++p) {
            uint8_t* dst = p == 0 ? frame : host;
            if (!dst) break;
            if ((p == 0 && !do_dev) || (p == 1 && !do_host)) continue;
            const size_t pitch = p == 0 ? fpitch : row;
            const Surface s = make_surface(dst, plen, W, H, fmt, pitch);
            for (int i = first; i < n_hud; ++i) {
                const OverlayCmdDev& c = s_cmd[i];
                if (c.kind < 0) continue;
                if (p == 1 && c.kind == VT_OV_BACKGROUND && ofmt == VT_FMT_NV12 && !split) {  // (split: this CTA dims the host pixels itself)
                    // a dim that does not lead the list: the host copy takes the final pixels of the region from the device frame (the
                    // later commands of this pass re-draw what lies on top of it; both packed, as every frame that has a host copy)
                    const BgRegion g = bg_region(c, W, H, row, step);
                    for (long long j = threadIdx.x; j < (g.y1 - g.y0) * (g.x1 - g.x0); j += blockDim.x) {
                        const size_t o = (size_t)(g.y0 + j / (g.x1 - g.x0)) * row + (size_t)(g.x0 + j % (g.x1 - g.x0)) * step;
                        if (o < plen) host[o] = frame[o];
                    }
                } else {
                    ov_dispatch(s, c);
                }
                __syncthreads();
            }
        }
    }
    if (split && blockIdx.y == 1) return;  // (the host waits for the whole grid: the mirrored pixels are complete when it reads the result)
    if (kGroup && blockIdx.x != 0) return;  // (pair 0 publishes; the host waits for the whole grid, as above)
    if (stamp_end && threadIdx.x == 0) *stamp_end = device_time_ns();
    if (blk) {  // last kernel of the frame: publish the result block (see publish_kernel) — one kernel boundary less
        uint32_t* dst = ctl->hblk;
        __threadfence();  // the end stamp above is part of the block
        __syncthreads();
        if (dst)
            for (int i = threadIdx.x; i < blk_words; i += blockDim.x) dst[i] = __ldcg(blk + i);
    }
}

__global__ void __launch_bounds__(kOvThreads) box_overlay_kernel(const DeviceResult* __restrict__ res, const int32_t* __restrict__ slots, int n,
                                                                 float gate, const FrameCtl* ctl, unsigned long long* stamp_end,
                                                                 const uint32_t* __restrict__ blk, int blk_words, int draw_box) {
    __shared__ OverlayCmdDev s_cmd[kMaxCmds];
    box_overlay_body<false>(res, slots, n, gate, ctl, stamp_end, blk, blk_words, draw_box, s_cmd);
}

// (minimum of one CTA per SM stated: without it ptxas holds this instance to 64 registers and spills the background-dim prefetch; the grid
// is one CTA pair per stream, at most 32 CTAs)
__global__ void __launch_bounds__(kOvThreads, 1) probe_group_overlay_kernel(const DeviceResult* __restrict__ res, float gate, const ProbeGroupCtl* ctl,
                                                                         unsigned long long* stamp_end, const uint32_t* __restrict__ blk,
                                                                         int blk_words) {
    __shared__ OverlayCmdDev s_cmd[kMaxCmds];
    box_overlay_body<true>(res, nullptr, 0, gate, &ctl->f, stamp_end, blk, blk_words, 0, s_cmd);
}

cudaError_t launch_group_overlay(int n_streams, const DeviceResult* d_res, float gate, const ProbeGroupCtl* d_ctl, unsigned long long* stamp_end,
                                 cudaStream_t s, bool pdl, const void* d_blk, size_t blk_bytes) {
    return launch_ex(probe_group_overlay_kernel, dim3(n_streams, 2), dim3(kOvThreads), 0, s, pdl, 1, d_res, gate, d_ctl, stamp_end,
                     (const uint32_t*)d_blk, (int)(blk_bytes / 4));
}

cudaError_t launch_box_overlay(const DeviceResult* d_res, const int32_t* d_slots, int n, float gate, const FrameCtl* d_ctl,
                               unsigned long long* stamp_end, cudaStream_t s, bool pdl, const void* d_blk, size_t blk_bytes, int draw_box) {
    const bool split = (draw_box >> 16) != 0;  // HUD mode: device pass and host pass in two CTAs
    return launch_ex(box_overlay_kernel, dim3(n > 0 ? n : 1, split ? 2 : 1), dim3(kOvThreads), 0, s, pdl, 1, d_res, d_slots, n, gate, d_ctl,
                     stamp_end, (const uint32_t*)d_blk, (int)(blk_bytes / 4), draw_box & 0xffff);
}

// per-frame, outside the graph: submit stamp + the control block (addresses and parameters that change from frame to frame)
__global__ void stamp_kernel(unsigned long long* stamp, FrameCtl* dst, const FrameCtl val) {
    if (threadIdx.x == 0) *stamp = device_time_ns();
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&val);
    for (int i = threadIdx.x; i < (int)(sizeof(FrameCtl) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(dst)[i] = src[i];
}
struct HudInline {
    OverlayCmdDev c[kHudInline];
};
__global__ void stamp_hud_kernel(unsigned long long* stamp, FrameCtl* dst, const FrameCtl val, const __grid_constant__ HudInline list, int n,
                                 OverlayCmdDev* d_list) {
    if (threadIdx.x == 0) *stamp = device_time_ns();
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&val);
    for (int i = threadIdx.x; i < (int)(sizeof(FrameCtl) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(dst)[i] = src[i];
    const uint32_t* ls = reinterpret_cast<const uint32_t*>(&list);
    for (int i = threadIdx.x; i < n * (int)(sizeof(OverlayCmdDev) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(d_list)[i] = ls[i];
}
cudaError_t launch_stamp(unsigned long long* stamp, FrameCtl* d_ctl, const FrameCtl& ctl, cudaStream_t s, const OverlayCmdDev* h_list, int n,
                         OverlayCmdDev* d_list) {
    static_assert(sizeof(FrameCtl) % 4 == 0 && sizeof(OverlayCmdDev) % 4 == 0, "word copy");
    // stamp_hud_kernel's parameters (the control block by value next to the inline HUD list) stay within the 32764-byte parameter limit
    static_assert(sizeof(FrameCtl) + sizeof(HudInline) + 4 * sizeof(void*) + sizeof(int) <= 32764, "stamp_hud_kernel parameter block");
    if (h_list && d_list && n > 0 && n <= kHudInline) {
        HudInline blk;
        memcpy(blk.c, h_list, sizeof(OverlayCmdDev) * (size_t)n);
        stamp_hud_kernel<<<1, 256, 0, s>>>(stamp, d_ctl, ctl, blk, n, d_list);
    } else {
        stamp_kernel<<<1, 96, 0, s>>>(stamp, d_ctl, ctl);
    }
    return cudaGetLastError();
}
__global__ void stamp_group_kernel(unsigned long long* stamp, ProbeGroupCtl* dst, const ProbeGroupCtl val) {
    if (threadIdx.x == 0) *stamp = device_time_ns();
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&val);
    for (int i = threadIdx.x; i < (int)(sizeof(ProbeGroupCtl) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(dst)[i] = src[i];
}
cudaError_t launch_stamp_group(unsigned long long* stamp, ProbeGroupCtl* d_ctl, const ProbeGroupCtl& ctl, cudaStream_t s) {
    static_assert(sizeof(ProbeGroupCtl) % 4 == 0 && sizeof(ProbeGroupCtl) + 2 * sizeof(void*) <= 32764, "stamp_group_kernel parameter block");
    stamp_group_kernel<<<1, 256, 0, s>>>(stamp, d_ctl, ctl);
    return cudaGetLastError();
}

// Last kernel of a frame: the result block (results, stage stamps, error flag; < 2 KB) is written straight into the pinned host block
// of the frame's queue slot (zero-copy stores).  A kernel -> copy-engine -> kernel hand-over on the stream costs ~14 us per frame
// (measured between the overlay's end stamp and the next frame's submit stamp); a dependent kernel costs ~4 us.
__global__ void __launch_bounds__(128) publish_kernel(const uint32_t* __restrict__ blk, const FrameCtl* ctl, int words) {
    uint32_t* dst = ctl->hblk;  // written by stamp_kernel at the start of the frame
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (!dst) return;
    for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = __ldcg(blk + i);
}
cudaError_t launch_publish(const void* d_blk, const FrameCtl* d_ctl, size_t bytes, cudaStream_t s, bool pdl) {
    return launch_ex(publish_kernel, dim3(1), dim3(128), 0, s, pdl, 1, (const uint32_t*)d_blk, d_ctl, (int)(bytes / 4));
}

}  // namespace vt
