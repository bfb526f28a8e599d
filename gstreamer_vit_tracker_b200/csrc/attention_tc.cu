// attention_tc.cu — joint attention over the 320-token sequence on tcgen05 tensor cores (head_dim 64).
//
// One CTA (16 softmax warps + 1 control warp) per (128-query tile, head, target):
//   TMA        Q tile [128 x 64], K [320 x 64] and V^T [64 x 320] (bf16 hi/lo parts, 128B swizzle) -> shared memory
//   tcgen05    S[128 x 320] = Q K^T  -> TMEM columns 0..319 (two N = 160 UMMAs per K-step and precision term)
//   control    warp 16 issues every TMA load and every UMMA (one elected lane) and owns the TMEM allocation, so that no softmax
//              warp ever serialises MMA issue with its share of the exp work; chunks are handed over through mbarriers
//              (p_full[c]: one arrival per softmax warp) — there is no CTA-wide barrier in the chunk loop
//   softmax    FOUR threads per query row (warp w reads TMEM lane quarter w % 4; column group g = w / 4): the exp work is what
//              bounds this kernel, so it is spread over 16 warps.  Per 64-key chunk thread (row, g) owns 16 keys:
//              tcgen05.ld.x16 -> ex2(s * k - max * k) -> bf16 (hi, lo) split -> tcgen05.st of the packed pairs back into the thread's
//              OWN 16 S columns (8 columns P_hi, 8 columns P_lo): P never leaves tensor memory; row max / row sum partials are
//              combined through shared memory in a fixed order
//   tcgen05    O[128 x 64] += P_chunk V_chunk with the A operand (P) read from TMEM, so each UMMA fetches only V from shared memory
//              (the smem-operand form was fetch bound: 0.39 us per chunk, longer than the chunk's softmax) -> TMEM columns 320..383
//              (+ 384..447 for the hi*lo term), overlapped with the next chunk's softmax
//   epilogue   O / sum -> bf16 (hi, lo) tile staged in shared memory -> coalesced 16-byte stores into the proj GEMM's A operand.
// The output staging tile aliases the Q/K area once S is complete (~192 KB of shared memory per CTA).
//
// Chained form (latency mode, `chain`): the proj GEMM is folded in.  The normalised O tile goes back into tensor memory as packed
// bf16 (hi, lo) — a UMMA A operand, like P — and the CTA multiplies it with a kAttChainW-row slice of W_proj[:, 64 h .. 64 h + 64)
// (fetched before the dependency wait) into TMEM columns 0.. (dead P) and stores the fp32 partial product [128 x kAttChainW] of
// head h to plane h of the partial buffer; reduce_ln_kernel adds the heads in index order with bias, residual and LayerNorm 2.
// Each (query tile, head) is computed by D / kAttChainW CTAs, one per column slice of the product, so that every CTA stores only
// 16 KB: one kernel and one dependency edge less per block.
// 64-row query tiles (QT = 64, chained form only): five tiles instead of 128 + 128 + 64, M = 64 UMMAs.  Row 16 q + i of an M = 64
// accumulator sits in lane 32 q + i (i < 16), so the 16 softmax warps split each row 8 ways (8 keys per thread per chunk) through the
// 16x32bx2 TMEM shapes; the P / O column layout and the MMA issue loops are those of the 128-row tile.
#include "tc_common.cuh"
#include "vt_internal.h"

namespace vt {

using namespace tc;

constexpr int kDh = 64;
constexpr int kKeyChunk = 64;
constexpr int kNChunks = kNTok / kKeyChunk;       // 5
constexpr int kKBytes = kNTok * kDh * 2;          // 40 KB
constexpr int kVBytes = kDh * kNTok * 2;          // 40 KB (5 blocks of [64 x 64])
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColO = 320;
constexpr uint32_t kColA = 128;  // chained form: normalised O as a packed bf16 A operand (dead P columns; the product uses 0..63)
constexpr int kSoftmaxWarps = 16, kSoftmaxThreads = kSoftmaxWarps * 32;
constexpr int kAttThreads = kSoftmaxThreads + 32;     // + one control warp (TMA, MMA issue, TMEM alloc)

// QT: query rows per CTA, 128 (M = 128 UMMAs, tiles 128 + 128 + 64) or 64 (M = 64 UMMAs, five full tiles; chained form only)
template <int NSPLIT, int QT>
struct AttSmem {
    static constexpr int kParts = NSPLIT == 3 ? 2 : 1;  // NSPLIT: 1 = bf16, 2 = fp16 (single pass), 3 = bf16 hi + lo
    static constexpr int kQBytes = QT * kDh * 2;        // 16 / 8 KB
    static constexpr int kPBytes = QT * kKeyChunk * 2;  // 16 / 8 KB
    static constexpr int kQTiles = (kNTok + QT - 1) / QT;
    static constexpr int kColGroups = kSoftmaxThreads / QT;    // threads per query row: 4 / 8
    static constexpr int kKeys = kKeyChunk / kColGroups;       // keys of every chunk per thread: 16 / 8
    static constexpr int kQK = kParts * (kQBytes + kKBytes);
    static constexpr int kP = kParts * kPBytes;  // output staging tile
    static constexpr int kRegion1 = kQK > kP ? kQK : kP;
    static constexpr int kV = kParts * kVBytes;
    static constexpr int kW2 = kParts * kAttChainW * 128;  // chained form: [W_proj slice hi W x 128 B][lo], adjacent = one N = 2 W B operand
    static constexpr int kTotal = kRegion1 + kV + kW2 + 1024;
};

// named barrier over the 16 softmax warps only (the control warp never joins it)
__device__ __forceinline__ void softmax_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kSoftmaxThreads) : "memory"); }

// A thread's columns of its query row: the 32x32b shapes for the 128-row tile (thread l = lane l of the quarter), the 16x32bx2 shapes for
// the 64-row tile (threads 16..31 take the columns after those of threads 0..15)
template <int QT, int N>
__device__ __forceinline__ void ld_row_issue(uint32_t a, uint32_t (&r)[N]) {
    if constexpr (QT == 64) tmem_ld_16x2_x8_issue(a, r); else tmem_ld_32x16_issue(a, r);
}
template <int QT, int N>
__device__ __forceinline__ void ld_row(uint32_t a, float (&v)[N]) {
    if constexpr (QT == 64) tmem_ld_16x2(a, v); else tmem_ld_cols(a, v);
}
template <int QT, int N>
__device__ __forceinline__ void st_row(uint32_t a, const uint32_t (&r)[N]) {
    if constexpr (QT == 64) tmem_st_16x2_x4(a, r); else tmem_st_32x8(a, r);
}

template <int NSPLIT, int QT>
__global__ void __launch_bounds__(kAttThreads, 1)
attention_tc_kernel(const __grid_constant__ TcAttentionPlan mp, __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, int D,
                    int heads, int* err, unsigned long long* trace, int dup) {
    using SM = AttSmem<NSPLIT, QT>;
    constexpr bool kQ64 = QT == 64;
    constexpr int P = SM::kParts, kQBytes = SM::kQBytes, kPBytes = SM::kPBytes, kQTiles = SM::kQTiles;
    constexpr int kColGroups = SM::kColGroups, kKeys = SM::kKeys;
    const CUtensorMap &mQhi = kQ64 ? mp.mQ64hi : mp.mQhi, &mQlo = kQ64 ? mp.mQ64lo : mp.mQlo;
    const CUtensorMap &mKhi = mp.mKhi, &mKlo = mp.mKlo, &mVhi = mp.mVhi, &mVlo = mp.mVlo;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_qk, bar_k1, bar_v, bar_s, p_full[kNChunks], bar_o, bar_w2, bar_a2, bar_o2;
    __shared__ uint32_t tmem_base_s;
    __shared__ float red[kColGroups][QT];  // row-max partials, then row-sum partials
    __shared__ unsigned long long* trace_slot;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sQ = smem;                       // [P][QT x 128B]
    uint8_t* sK = smem + P * kQBytes;         // [P][320 x 128B]
    uint8_t* sV = smem + SM::kRegion1;        // [P][5 blocks][64 x 128B]
    uint8_t* sW2 = sV + SM::kV;               // chained form: W_proj slice

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool ctrl = warp == kSoftmaxWarps;  // warp 16: TMA + MMA issue (one elected lane), TMEM alloc / dealloc
    // query row inside the tile; warp w reads TMEM lane quarter w % 4 and owns the 16 columns 16 g .. of every key chunk
    const int row = kQ64 ? (warp & 3) * 16 + (lane & 15) : (warp & 3) * 32 + lane;
    const int g = (warp >> 2) & 3;
    const int cg = kQ64 ? 2 * g + (lane >> 4) : g;  // column group of the thread: keys kKeys cg .. of every chunk
    // dup ("spread" form, idle SMs available): every (query tile, head, target) is computed by two CTAs, replica 0 stores the hi tile
    // and replica 1 the lo tile (a CTA's store rate is what bounds the end of the kernel)
    const int replica = blockIdx.x / kQTiles;
    const bool st_hi = !dup || replica == 0, st_lo = P == 2 && (!dup || replica == 1);
    const bool chain = kQ64 || mp.chain != 0;  // replica = column slice of the chained proj product
    const int q0 = (blockIdx.x % kQTiles) * QT, h = blockIdx.y, b = blockIdx.z;
    const int bh = b * heads + h;
    const bool q_ok = q0 + row < kNTok;       // uniform per warp (320 = 2 * 128 + 64 = 5 * 64)
    bool ok = true;
    TraceRec tr;
    tr.begin(&trace_slot, trace, 10);

    if (tid == 0) {
        mbar_init(&bar_qk, 1), mbar_init(&bar_k1, 1), mbar_init(&bar_v, 1), mbar_init(&bar_s, 1), mbar_init(&bar_o, 1);
        mbar_init(&bar_w2, 1), mbar_init(&bar_a2, kSoftmaxWarps), mbar_init(&bar_o2, 1);
        for (int c = 0; c < kNChunks; ++c) mbar_init(&p_full[c], kSoftmaxWarps);
        fence_barrier_init();
    }
    if (ctrl) {
        if (elect_one_sync()) {
            tma_prefetch_desc(&mQhi), tma_prefetch_desc(&mKhi), tma_prefetch_desc(&mVhi);
            if (P == 2) tma_prefetch_desc(&mQlo), tma_prefetch_desc(&mKlo), tma_prefetch_desc(&mVlo);
        }
        tmem_alloc(&tmem_base_s, kTmemCols);
        tmem_relinquish();
    }
    tcgen05_fence_before();
    __syncthreads();
    if (chain && ctrl && elect_one_sync()) {  // weights never depend on the preceding kernel: W_proj[W replica .. + W)[64 h .. 64 h + 64)
        tma_prefetch_desc(&mp.mW2hi);
        mbar_arrive_expect_tx(&bar_w2, P * kAttChainW * 128);
        tma_load_2d(sW2, &mp.mW2hi, &bar_w2, h * kDh, replica * kAttChainW);
        if (P == 2) tma_load_2d(sW2 + kAttChainW * 128, &mp.mW2lo, &bar_w2, h * kDh, replica * kAttChainW);
    }
    tcgen05_fence_after();
    const uint32_t tmem = tmem_base_s;

    pdl_wait();               // Q, K, V^T come from the QKV GEMM
    if (tid == 0) tr.mark(2);
    pdl_launch_dependents();

    if (ctrl) {
        // (elect.sync instead of lane == 0: the compiler then knows that the region runs in one thread and emits the uniform-datapath
        // instructions — tcgen05.mma, TMA — without a per-thread election loop around each of them)
        if (elect_one_sync()) {
            // ---- TMA: Q + the first 160 keys on one barrier, the other 160 keys on a second (their UMMAs start while the first half
            // computes), V^T on a third (only needed after the softmax of the first chunk)
            constexpr int kHalfK = kNTok / 2, kHalfKBytes = kHalfK * kDh * 2;
            mbar_arrive_expect_tx(&bar_qk, P * (kQBytes + kHalfKBytes));
            tma_load_3d(sQ, &mQhi, &bar_qk, 0, q0, bh);
            tma_load_3d(sK, &mKhi, &bar_qk, 0, 0, bh);
            if (P == 2) tma_load_3d(sQ + kQBytes, &mQlo, &bar_qk, 0, q0, bh), tma_load_3d(sK + kKBytes, &mKlo, &bar_qk, 0, 0, bh);
            mbar_arrive_expect_tx(&bar_k1, P * kHalfKBytes);
            tma_load_3d(sK + kHalfKBytes, &mKhi, &bar_k1, 0, kHalfK, bh);
            if (P == 2) tma_load_3d(sK + kKBytes + kHalfKBytes, &mKlo, &bar_k1, 0, kHalfK, bh);
            mbar_arrive_expect_tx(&bar_v, P * kVBytes);
            for (int c = 0; c < kNChunks; ++c) {  // per key chunk: [V^T hi 64 x 128 B][V^T lo 64 x 128 B], adjacent = one N = 128 B operand
                tma_load_3d(sV + c * (P * kDh * 128), &mVhi, &bar_v, c * kKeyChunk, 0, bh);
                if (P == 2) tma_load_3d(sV + c * (P * kDh * 128) + kDh * 128, &mVlo, &bar_v, c * kKeyChunk, 0, bh);
            }
            // ---- S = Q K^T
            ok &= mbar_wait(&bar_qk, 0);
            tcgen05_fence_after();
            const uint64_t dQ = umma_desc_sw128(smem_u32(sQ)), dK = umma_desc_sw128(smem_u32(sK));
            constexpr int kHalf = kNTok / 2;  // 160 keys per UMMA: two equal N = 160 instructions instead of N = 256 + a fetch-bound N = 64
            constexpr uint32_t idescS = umma_idesc_h<NSPLIT == 2>(QT, kHalf);
            constexpr uint64_t kLoQ = kQBytes >> 4, kLoK = kKBytes >> 4, kK2 = (kHalf * 128) >> 4;  // descriptor address units (16 B)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                if (half) {
                    ok &= mbar_wait(&bar_k1, 0);
                    tcgen05_fence_after();
                }
#pragma unroll
                for (int k = 0; k < kDh / 16; ++k) {
                    const uint64_t qh = dQ + 2 * k, kh = dK + 2 * k + half * kK2;
                    umma_bf16(tmem + half * kHalf, qh, kh, idescS, k != 0);
                    if (NSPLIT == 3) {
                        umma_bf16(tmem + half * kHalf, qh, kh + kLoK, idescS, 1);
                        umma_bf16(tmem + half * kHalf, qh + kLoQ, kh, idescS, 1);
                    }
                }
            }
            umma_commit(&bar_s);
            // ---- O += P_c V_c as the softmax warps hand the chunks over
            const uint64_t dV = umma_desc_sw128(smem_u32(sV));
            // bf16x3 as P_hi x [V_hi; V_lo] (ONE N = 128 UMMA into O columns [0, 64) = hi*hi and [64, 128) = hi*lo) + P_lo x V_hi; the epilogue
            // adds the two column halves.  K-step k of chunk c = the 16 keys of softmax warp column group k: P_hi in TMEM columns
            // 64 c + 16 k .. + 7, P_lo in the next 8 (two bf16 per column).
            constexpr uint32_t idesc = umma_idesc_h<NSPLIT == 2>(QT, kDh), idesc2n = umma_idesc_h<NSPLIT == 2>(QT, 2 * kDh);
            constexpr uint64_t kBlkV = (uint64_t)(P * kDh * 128) >> 4;
            ok &= mbar_wait(&bar_v, 0);
            for (int c = 0; c < kNChunks; ++c) {
                ok &= mbar_wait(&p_full[c], 0);
                tcgen05_fence_after();
#pragma unroll
                for (int k = 0; k < kKeyChunk / 16; ++k) {
                    const uint32_t ph = tmem + c * kKeyChunk + k * 16;
                    const uint64_t vh = dV + c * kBlkV + 2 * k;
                    if (NSPLIT == 3) {
                        umma_bf16_ta(tmem + kColO, ph, vh, idesc2n, (c | k) != 0);
                        umma_bf16_ta(tmem + kColO, ph + 8, vh, idesc, 1);
                    } else {
                        umma_bf16_ta(tmem + kColO, ph, vh, idesc, (c | k) != 0);
                    }
                }
            }
            umma_commit(&bar_o);
            if (chain) {  // ---- partial proj product of this head: O (staged by the softmax warps) x W_proj slice^T -> TMEM columns 0..127
                ok &= mbar_wait(&bar_w2, 0);
                ok &= mbar_wait(&bar_a2, 0);
                tcgen05_fence_after();
                // A = normalised O, written by the softmax warps as packed bf16 into TMEM columns kColA.. (K-step k = their warp column
                // group k: 8 columns hi, 8 columns lo), so the UMMA fetches only the weight slice from shared memory
                const uint64_t dW = umma_desc_sw128(smem_u32(sW2));
                constexpr uint32_t idescW = umma_idesc_h<NSPLIT == 2>(QT, kAttChainW), idescW2 = umma_idesc_h<NSPLIT == 2>(QT, 2 * kAttChainW);
#pragma unroll
                for (int k = 0; k < kDh / 16; ++k) {
                    const uint32_t ah = tmem + kColA + k * 16;
                    if (NSPLIT == 3) {
                        umma_bf16_ta(tmem, ah, dW + 2 * k, idescW2, k != 0);  // O_hi x [W_hi; W_lo]
                        umma_bf16_ta(tmem, ah + 8, dW + 2 * k, idescW, 1);    // O_lo x W_hi
                    } else {
                        umma_bf16_ta(tmem, ah, dW + 2 * k, idescW, k != 0);
                    }
                }
                umma_commit(&bar_o2);
            }
        }
        __syncwarp();
    } else {
        // ---- softmax: thread (row, cg) owns keys 64 c + kKeys cg .. + kKeys - 1 of every chunk c; a warp owns 16 columns of each chunk
        ok &= mbar_wait(&bar_s, 0);
        tcgen05_fence_after();
        if (tid == 0) tr.mark(4);
        const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const float k2 = 1.4426950408889634f / sqrtf((float)kDh);  // scale * log2(e)
        float mx = -INFINITY;
        const uint32_t col0 = lane_addr + g * 16;
        uint32_t r[2][kKeys];  // software pipeline over the key chunks: the TMEM load of chunk c + 1 is in flight while chunk c is processed
        if (q_ok) {
            ld_row_issue<QT>(col0, r[0]);
#pragma unroll
            for (int c = 0; c < kNChunks; ++c) {
                tmem_ld_wait(r[c & 1]);
                if (c + 1 < kNChunks) ld_row_issue<QT>(col0 + (c + 1) * kKeyChunk, r[(c + 1) & 1]);
#pragma unroll
                for (int j = 0; j < kKeys; ++j) mx = fmaxf(mx, __uint_as_float(r[c & 1][j]));
            }
            ld_row_issue<QT>(col0, r[0]);  // chunk 0 again, for the exp pass: in flight across the row-max exchange
        }
        red[cg][row] = mx;
        softmax_bar_sync();
        mx = fmaxf(fmaxf(red[0][row], red[1][row]), fmaxf(red[2][row], red[3][row]));
        if constexpr (kColGroups == 8) mx = fmaxf(mx, fmaxf(fmaxf(red[4][row], red[5][row]), fmaxf(red[6][row], red[7][row])));
        if (tid == 0) tr.mark(5);
        const float mk = mx * k2;
        float sum = 0.f;
#pragma unroll
        for (int c = 0; c < kNChunks; ++c) {
            uint32_t hi[kKeys / 2], lo[kKeys / 2];
            if (q_ok) {
                tmem_ld_wait(r[c & 1]);
                if (c + 1 < kNChunks) ld_row_issue<QT>(col0 + (c + 1) * kKeyChunk, r[(c + 1) & 1]);
#pragma unroll
                for (int j = 0; j < kKeys; j += 2) {
                    const float e0 = ex2_approx(fmaf(__uint_as_float(r[c & 1][j]), k2, -mk));
                    const float e1 = ex2_approx(fmaf(__uint_as_float(r[c & 1][j + 1]), k2, -mk));
                    sum += e0;
                    sum += e1;
                    split2_h<NSPLIT == 2>(e0, e1, hi[j >> 1], lo[j >> 1]);
                }
            }
            if (q_ok) {  // P replaces the S values the warp has just consumed: columns [0, 8) of its 16 hold P_hi, [8, 16) P_lo
                st_row<QT>(col0 + c * kKeyChunk, hi);
                if (P == 2) st_row<QT>(col0 + c * kKeyChunk + 8, lo);
                tmem_st_wait();
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_full[c]);  // one arrival per softmax warp: no CTA-wide barrier in this loop
            if (tid == 0 && c == 0) tr.mark(6);
        }
        if (tid == 0) tr.mark(7);
        // the row-max partials were consumed before the first hand-over: reuse the array for the row sums
        red[cg][row] = sum;
        softmax_bar_sync();
        sum = (red[0][row] + red[1][row]) + (red[2][row] + red[3][row]);
        if constexpr (kColGroups == 8) sum += (red[4][row] + red[5][row]) + (red[6][row] + red[7][row]);

        // ---- epilogue: O / sum -> bf16 (hi, lo): the chained product's A operand in tensor memory, or a tile staged in (dead) shared
        // memory and copied with coalesced stores into columns h*64.. of the proj GEMM's A operand [B][320][D]; query rows >= 320 are skipped
        ok &= mbar_wait(&bar_o, 0);
        tcgen05_fence_after();
        {
            const float inv = q_ok ? 1.f / sum : 0.f;
            float v[kKeys];  // output columns 16 g .. + 15 of the row, kKeys of them per thread
            ld_row<QT>(lane_addr + kColO + g * 16, v);
            if (NSPLIT == 3) {
                float hl[kKeys];
                ld_row<QT>(lane_addr + kColO + kDh + g * 16, hl);
#pragma unroll
                for (int j = 0; j < kKeys; ++j) v[j] += hl[j];
            }
            uint32_t hi[kKeys / 2], lo[kKeys / 2];
#pragma unroll
            for (int j = 0; j < kKeys; j += 2) split2_h<NSPLIT == 2>(v[j] * inv, v[j + 1] * inv, hi[j >> 1], lo[j >> 1]);
            if (chain) {  // A operand of the chained product, in tensor memory
                st_row<QT>(lane_addr + kColA + g * 16, hi);
                if (P == 2) st_row<QT>(lane_addr + kColA + g * 16 + 8, lo);
                tmem_st_wait();
            } else if constexpr (!kQ64) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int off = row * 128 + (((2 * g + j) ^ (row & 7)) << 4);
                    *reinterpret_cast<uint4*>(smem + off) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
                    if (P == 2) *reinterpret_cast<uint4*>(smem + kPBytes + off) = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
                }
            }
        }
        if (chain) {
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_a2);
            ok &= mbar_wait(&bar_o2, 0);
            tcgen05_fence_after();
            // product columns per thread: kAttChainW / 4 per warp column group g, split over its two half-warps in the 64-row tile
            constexpr int CW = kAttChainW / kColGroups;
            float v[CW];
            ld_row<QT>(lane_addr + g * (kAttChainW / 4), v);
            if (NSPLIT == 3) {
                float hl[CW];
                ld_row<QT>(lane_addr + kAttChainW + g * (kAttChainW / 4), hl);
#pragma unroll
                for (int j = 0; j < CW; ++j) v[j] += hl[j];
            }
            // fp32 tile [QT][W] staged as swizzled boxes of [QT rows][128 B] behind the O tiles (dead K area)
            uint8_t* prow = smem + 2 * kPBytes + ((cg * CW) >> 5) * (QT * 128) + row * 128;
            const int ch0 = ((cg * CW) & 31) >> 2;
#pragma unroll
            for (int q = 0; q < CW / 4; ++q)
                *reinterpret_cast<float4*>(prow + (((ch0 + q) ^ (row & 7)) << 4)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            softmax_bar_sync();
            // -> partial plane h: [B][320][D] fp32, columns W replica ..: W * 4 contiguous bytes per row
            constexpr int CH = kAttChainW / 4, RPP = kSoftmaxThreads / CH;  // 16-byte chunks per row, rows per pass
#pragma unroll
            for (int i = 0; i < QT / RPP; ++i) {
                const int r = tid / CH + RPP * i, c16 = tid % CH, bx = c16 >> 3, ch = c16 & 7;
                if (q0 + r < kNTok) {
                    const float4 val = *reinterpret_cast<const float4*>(smem + 2 * kPBytes + bx * (QT * 128) + r * 128 + ((ch ^ (r & 7)) << 4));
                    float* dst = mp.p2 + (int64_t)h * mp.p2_plane + ((int64_t)b * kNTok + q0 + r) * D + replica * kAttChainW + c16 * 4;
                    *reinterpret_cast<float4*>(dst) = val;
                }
            }
        } else if constexpr (!kQ64) {
        softmax_bar_sync();
        // staged [128][128 B] tiles -> att_hi / att_lo [B][320][D], columns h*64..: coalesced 16-byte stores, 4 rows per warp instruction
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int r = (tid >> 3) + 64 * i, ch = tid & 7;
            if (q0 + r < kNTok) {
                const int off = r * 128 + ((ch ^ (r & 7)) << 4);
                const int64_t dst = (((int64_t)b * kNTok + q0 + r) * D + h * kDh) * 2 + ch * 16;
                if (st_hi) *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(out_hi) + dst) = *reinterpret_cast<const uint4*>(smem + off);
                if (st_lo) *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(out_lo) + dst) = *reinterpret_cast<const uint4*>(smem + kPBytes + off);
            }
        }
        }
    }
    if (!ok && err) atomicExch(err, 2);
    tcgen05_fence_before();
    __syncthreads();
    if (tid == 0) tr.mark(3);
    if (ctrl) tmem_dealloc(tmem, kTmemCols);
}

bool tc_make_map(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box);

bool tc_attention_plan_init(TcAttentionPlan* p, const __nv_bfloat16* Qhi, const __nv_bfloat16* Qlo, const __nv_bfloat16* Khi, const __nv_bfloat16* Klo,
                            const __nv_bfloat16* Vthi, const __nv_bfloat16* Vtlo, int batch_heads, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, int D,
                            int batch) {
    bool ok = true;
    p->out_hi = out_hi, p->out_lo = out_lo, p->D = D;
    p->p2 = nullptr, p->p2_plane = 0, p->chain = 0;
    (void)batch;
    {   // Q, K: [batch*heads][320][64], box {64, rows, 1}
        const uint64_t dims[3] = {kDh, kNTok, (uint64_t)batch_heads}, strides[2] = {kDh * 2, (uint64_t)kDh * 2 * kNTok};
        const uint32_t boxq[3] = {kDh, 128, 1}, boxq64[3] = {kDh, 64, 1}, boxk[3] = {kDh, kNTok / 2, 1};  // K: two boxes of 160 keys
        ok &= tc_make_map(&p->mQhi, Qhi, 3, dims, strides, boxq) && tc_make_map(&p->mQlo, Qlo, 3, dims, strides, boxq);
        ok &= tc_make_map(&p->mQ64hi, Qhi, 3, dims, strides, boxq64) && tc_make_map(&p->mQ64lo, Qlo, 3, dims, strides, boxq64);
        ok &= tc_make_map(&p->mKhi, Khi, 3, dims, strides, boxk) && tc_make_map(&p->mKlo, Klo, 3, dims, strides, boxk);
    }
    {   // V^T: [batch*heads][64][320], box {64 keys, 64 rows, 1}
        const uint64_t dims[3] = {kNTok, kDh, (uint64_t)batch_heads}, strides[2] = {kNTok * 2, (uint64_t)kNTok * 2 * kDh};
        const uint32_t box[3] = {kKeyChunk, kDh, 1};
        ok &= tc_make_map(&p->mVhi, Vthi, 3, dims, strides, box) && tc_make_map(&p->mVlo, Vtlo, 3, dims, strides, box);
    }
    return ok;
}

template <int NSPLIT, int QT>
static cudaError_t att_set_smem() {
    return cudaFuncSetAttribute(attention_tc_kernel<NSPLIT, QT>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttSmem<NSPLIT, QT>::kTotal);
}
cudaError_t tc_attention_setup() {
    const cudaError_t e[6] = {att_set_smem<1, 128>(), att_set_smem<2, 128>(), att_set_smem<3, 128>(),
                              att_set_smem<1, 64>(),  att_set_smem<2, 64>(),  att_set_smem<3, 64>()};
    for (cudaError_t x : e)
        if (x != cudaSuccess) return x;
    return cudaSuccess;
}

template <int QT>
static cudaError_t att_launch(dim3 grid, const TcAttentionPlan& q, int heads, int nsplit, int* err, cudaStream_t s, bool pdl, unsigned long long* trace,
                              int dup) {
    if (nsplit == 3)
        return launch_ex(attention_tc_kernel<3, QT>, grid, dim3(kAttThreads), AttSmem<3, QT>::kTotal, s, pdl, 1, q, q.out_hi, q.out_lo, q.D, heads, err, trace, dup);
    if (nsplit == 2)
        return launch_ex(attention_tc_kernel<2, QT>, grid, dim3(kAttThreads), AttSmem<2, QT>::kTotal, s, pdl, 1, q, q.out_hi, q.out_lo, q.D, heads, err, trace, dup);
    return launch_ex(attention_tc_kernel<1, QT>, grid, dim3(kAttThreads), AttSmem<1, QT>::kTotal, s, pdl, 1, q, q.out_hi, q.out_lo, q.D, heads, err, trace, dup);
}

cudaError_t tc_attention_launch(const TcAttentionPlan& p, int B, int heads, int nsplit, int* err, cudaStream_t s, bool pdl, unsigned long long* trace,
                                int form) {
    if (B <= 0) return cudaSuccess;
    const bool q64 = form == VT_ATT_CHAIN_Q64;
    dim3 grid(q64 ? AttSmem<3, 64>::kQTiles : AttSmem<3, 128>::kQTiles, heads, B);
    const int ctas = (int)(grid.x * grid.y * grid.z);
    int dup = 0;
    TcAttentionPlan q = p;
    q.chain = 0;
    if (form == VT_ATT_CHAIN || q64) {
        if (!p.p2 || ctas * (p.D / kAttChainW) > kSpreadCtas) return cudaErrorInvalidValue;
        q.chain = 1, grid.x *= p.D / kAttChainW;
    } else if (form == VT_ATT_DUP && nsplit == 3 && ctas * 2 <= kSpreadCtas) {
        dup = 1, grid.x *= 2;
    }
    return q64 ? att_launch<64>(grid, q, heads, nsplit, err, s, pdl, trace, dup) : att_launch<128>(grid, q, heads, nsplit, err, s, pdl, trace, dup);
}

// chained form: W_proj [D out][D in] (bf16 hi / lo) and the fp32 partial planes [heads][batch][320][D]
bool tc_attention_plan_chain(TcAttentionPlan* p, const __nv_bfloat16* Whi, const __nv_bfloat16* Wlo, float* P2, int64_t plane_elems) {
    const uint64_t dims[2] = {(uint64_t)p->D, (uint64_t)p->D}, strides[1] = {(uint64_t)p->D * 2};
    const uint32_t box[2] = {64, kAttChainW};
    const bool ok = tc_make_map(&p->mW2hi, Whi, 2, dims, strides, box) && tc_make_map(&p->mW2lo, Wlo ? Wlo : Whi, 2, dims, strides, box);
    p->p2 = P2, p->p2_plane = plane_elems;
    return ok;
}

}  // namespace vt
