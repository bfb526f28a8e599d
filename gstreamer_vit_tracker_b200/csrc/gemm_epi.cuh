// gemm_epi.cuh — epilogue helpers shared by the tensor-core GEMM kernels (gemm_tc.cu: one tile per CTA; gemm_as.cu: the
// A-stationary throughput form): GELU, the swizzled shared-memory staging tiles and their coalesced copy-out into the dense
// [targets][heads][rows][cols] outputs (TcOut), the Q / K / V^T scatter.  Both kernels run the epilogue with 512 threads: four
// threads per accumulator row (TMEM lane), column group g = 16 (8) consecutive columns.
#pragma once

#include "tc_common.cuh"
#include "vt_internal.h"

namespace vt {

using namespace tc;

constexpr int kTcBM = 128, kTcBK = 64;
constexpr int kTileABytes = kTcBM * kTcBK * 2;  // 16 KB, one precision part

// GELU(x) = 0.5 x (1 + erf(x / sqrt 2)) with erf by Abramowitz & Stegun 7.1.26 (one rcp, five FMAs, one ex2): |abs error| < 7e-7 in fp32
// for erf, < 3e-7 for GELU — an order of magnitude below the bf16x3 operand error.  The FC1 epilogue is instruction-issue bound (16 GELUs
// per thread and chunk: 1.25 us of a 2.2 us epilogue step at 5120 rows), so two values go through the polynomial as one packed fp32 pair
// (FFMA2 / FMUL2: half the issue slots; only the two MUFU ops per value stay scalar).  Every operation is written out (no contraction
// left to the compiler), so every GEMM form computes bit-identical GELUs.
__device__ __forceinline__ void gelu_erf2(float& x0, float& x1) {
    const uint64_t x = f2_pack(x0, x1);
    const uint64_t z = f2_mul(x & 0x7fffffff7fffffffull, f2_bcast(0.70710678118654752440f));
    float d0, d1, t0, t1;
    f2_unpack(f2_fma(f2_bcast(0.3275911f), z, f2_bcast(1.f)), d0, d1);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
    const uint64_t t = f2_pack(t0, t1);
    uint64_t p = f2_fma(f2_bcast(1.061405429f), t, f2_bcast(-1.453152027f));
    p = f2_fma(p, t, f2_bcast(1.421413741f)), p = f2_fma(p, t, f2_bcast(-0.284496736f)), p = f2_fma(p, t, f2_bcast(0.254829592f));
    float a0, a1;
    f2_unpack(f2_mul(f2_mul(z, f2_bcast(-1.4426950408889634f)), z), a0, a1);
    const uint64_t e = f2_pack(ex2_approx(a0), ex2_approx(a1));
    // s = copysign(1 - p t e, x)  (1 - p t e is in [0, 1): its sign bit is clear)
    const uint64_t s = f2_fma(f2_mul(f2_mul(p, t), e), f2_bcast(-1.f), f2_bcast(1.f)) | (x & 0x8000000080000000ull);
    const uint64_t h = f2_mul(x, f2_bcast(0.5f));
    f2_unpack(f2_fma(h, s, h), x0, x1);
}
__device__ __forceinline__ float gelu_erf(float x) {
    float y = x, dummy = 0.f;
    gelu_erf2(y, dummy);
    return y;
}

constexpr int kTcThreads = 512;                         // 16 warps: warp w reads TMEM lane quarter w % 4, column group w / 4
constexpr int kTcColGroups = kTcThreads / kTcBM;        // 4 threads per accumulator row, BN / 4 columns each

// Staging tiles live in shared memory as [128 rows][RB bytes] (RB = 128: 64 bf16 or 32 fp32 columns; RB = 64: 32 bf16 columns) with
// the 16-byte chunks of a row XOR-swizzled so that both the per-row writes of the epilogue threads and the row-major reads of the
// copy-out are bank-conflict free; RB = 128 is the hardware 128B swizzle (the staged hidden tile is a valid UMMA A operand).
template <int RB>
__device__ __forceinline__ int swz(int row, int chunk) {
    return RB == 128 ? (chunk ^ (row & 7)) : (chunk ^ ((row >> 1) & 3));
}

// CPT (16 or 8) fp32 -> bf16 (hi, lo) into the staging tiles: thread (row, g) holds columns CPT g .. of a tile with RB bytes per row
// (RB = 8 CPT: four threads per row; RB = 128 with CPT = 8: eight threads per row, the 64-row tiles of gemm_tc_kernel)
template <int CPT, bool F16, int RB = CPT * 8>
__device__ __forceinline__ void stage_split(const float (&v)[CPT], uint8_t* tile_hi, uint8_t* tile_lo, int row, int g, bool with_lo) {
    uint32_t hi[CPT / 2], lo[CPT / 2];
#pragma unroll
    for (int j = 0; j < CPT; j += 2) split2_h<F16>(v[j], v[j + 1], hi[j >> 1], lo[j >> 1]);
#pragma unroll
    for (int q = 0; q < CPT / 8; ++q) {
        const int off = row * RB + (swz<RB>(row, (CPT / 8) * g + q) << 4);
        *reinterpret_cast<uint4*>(tile_hi + off) = make_uint4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
        if (with_lo) *reinterpret_cast<uint4*>(tile_lo + off) = make_uint4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
    }
}

// Staged tile -> global memory.  Row m of the GEMM is row (m % period + row_off) of target (m / period + batch_off) of a dense
// [targets][heads][rows][cols] output (TcOut); periods are multiples of 64, so each 64-row half of a tile stays inside one target
// and its (row, target) is computed once (TileRows).  Rows outside [0, rows) — the template rows the final LayerNorm drops, the
// padding rows of the last tile — and targets >= batch are skipped.
// The copy is done by all 512 threads with fully coalesced 16-byte stores: RB / 16 lanes cover one tile row, a warp instruction
// writes 4 (8) rows.  (Measured alternatives: thread-per-row stores straight from registers touch 32 lines per instruction and run at
// ~9 B/clk/SM; TMA tile stores cost ~0.16 us per 8 KB box on the issuing SM, 2 us for the 96 KB partial tile of the chained GEMM.)
constexpr int kHalfRows = 64;
struct TileRows {  // (row-in-target, target) of the two 64-row halves of a tile; computed once, before the accumulator wait
    int t[2], b[2];
    __device__ __forceinline__ TileRows(int m0, int period, int batch_off) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int mr = m0 + k * kHalfRows;
            b[k] = mr / period, t[k] = mr - b[k] * period, b[k] += batch_off;
        }
    }
};
// one [ROWS (128 or 64) rows][RB bytes] swizzled tile; col_bytes = byte offset of the tile's first column inside a destination row
template <int RB, int ROWS = kTcBM>
__device__ __forceinline__ void tile_to_global(const uint8_t* tile, const TcOut& o, int64_t col_bytes, const TileRows& r, int row_off, int head,
                                               int plane, int tid) {
    constexpr int CH = RB / 16, kRowsPerPass = kTcThreads / CH;  // 8 chunks, 64 rows per pass / 4 chunks, 128 rows in one pass
    static_assert(ROWS % kRowsPerPass == 0, "whole passes");
#pragma unroll
    for (int i = 0; i < ROWS / kRowsPerPass; ++i) {
        const int row = tid / CH + kRowsPerPass * i, ch = tid % CH, half = row >> 6;
        const int tt = r.t[half] + (row & 63) + row_off, b = r.b[half];
        if (tt >= 0 && tt < o.rows && b < o.batch) {
            const uint4 v = *reinterpret_cast<const uint4*>(tile + row * RB + (swz<RB>(row, ch) << 4));
            uint8_t* dst = o.base + (int64_t)plane * o.plane_bytes + (((int64_t)b * o.heads + head) * o.rows + tt) * o.row_bytes + col_bytes + ch * 16;
            *reinterpret_cast<uint4*>(dst) = v;
        }
    }
}
// V^T: SUBS (two, or one for a 64-row tile) unswizzled [BN d][64 tokens] sub-tiles -> rows d_off.. of [targets][heads][64 d][tokens];
// sub-tile k holds tokens t[k]..t[k]+63
template <int BN, int SUBS = 2>
__device__ __forceinline__ void vt_tile_to_global(const uint8_t* tile, const TcOut& o, const TileRows& r, int head, int d_off, int tid) {
    constexpr int kPasses = SUBS * BN * 8 / kTcThreads;  // SUBS sub-tiles x BN rows x 8 chunks over 512 threads
#pragma unroll
    for (int i = 0; i < kPasses; ++i) {
        const int idx = tid + i * kTcThreads, sub = idx / (BN * 8), d = (idx >> 3) % BN, ch = idx & 7, b = r.b[sub];
        if (b < o.batch && r.t[sub] + kHalfRows <= o.rows) {
            const uint4 v = *reinterpret_cast<const uint4*>(tile + sub * (BN * 128) + d * 128 + ch * 16);
            uint8_t* dst = o.base + (((int64_t)b * o.heads + head) * 64 + d_off + d) * o.row_bytes + (int64_t)r.t[sub] * 2 + ch * 16;
            *reinterpret_cast<uint4*>(dst) = v;
        }
    }
}

}  // namespace vt
