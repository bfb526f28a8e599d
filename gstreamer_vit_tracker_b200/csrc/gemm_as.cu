// gemm_as.cu — the A-stationary throughput form of the K <= 192 contractions (QKV, FC1) for many rows (cfg4: 16 targets = 5120 rows;
// cfg5: stream groups), where the one-tile-per-CTA kernel of gemm_tc.cu spends most of a CTA's life in prologue, first-TMA latency and
// epilogue with the tensor pipe idle, and re-reads the activation tile once per column tile.
//
//   C[M, N] = epilogue( A[M, K] * W[N, K]^T + bias ),   K = 64 * num_kb <= 192
//
// One CTA (18 warps) owns one 128-row tile of A and a contiguous range of 64-column chunks of N:
//   * the A tile (all of K, bf16 hi + lo: <= 96 KB) is loaded ONCE and stays in shared memory;
//   * warp 0 streams the weight chunks through a ring of k-block stages ([W_hi; W_lo] of one 64 x 64 block = 16 KB; the first
//     stages are in flight before griddepcontrol.wait — weights never depend on the preceding kernel);
//   * warp 1 issues the UMMAs of chunk i into TMEM accumulator i % 2 (bf16x3: A_hi x [W_hi; W_lo] as one N = 128 UMMA + A_lo x W_hi,
//     as in gemm_tc.cu), so the main loop of chunk i + 1 runs under the epilogue of chunk i;
//   * warps 2..17 are the epilogue: tcgen05.ld -> release the accumulator -> bias / GELU -> bf16 (hi, lo) split -> staging tile in
//     shared memory (double buffered) -> fully coalesced 16-byte stores (same staging and copy-out as gemm_tc.cu; Q / K / V^T scatter).
// L2 -> SM traffic per row tile: the A tile once per CTA + every weight chunk once, instead of (A tile + chunk) per 128 x 64 tile.
// The sums are the same as in gemm_tc.cu, in the same order (k ascending; hi*hi + lo*hi in one accumulator half, hi*lo in the
// other, added in the epilogue): results are bit-identical to the one-tile form.
#include <stdlib.h>
#include <string.h>

#include "gemm_epi.cuh"

namespace vt {

#ifndef VT_AS_STAGES
#define VT_AS_STAGES 4
#endif
constexpr int kAsStages = VT_AS_STAGES;  // weight k-block stages in flight (3 .. 4 fit beside the activation tile and two staging buffers)
constexpr int kAsMaxKb = 3;            // K <= 192
constexpr int kAsThreads = 64 + kTcThreads;  // TMA warp, MMA warp, 16 epilogue warps
constexpr int kAsChunk = 64;           // columns per accumulator / epilogue step
constexpr int kMaxAsChainN = 192;      // widest chained second GEMM (TMEM: 2 x 128 + 64 + N2 <= 512 columns)

template <int NSPLIT>
struct AsSmem {
    static constexpr int kParts = NSPLIT == 3 ? 2 : 1;
    static constexpr int kABytes = kAsMaxKb * kParts * kTileABytes;      // 96 / 48 KB
    static constexpr int kStageBytes = kParts * kAsChunk * kTcBK * 2;    // 16 / 8 KB
    static constexpr int kTileOBytes = kTcBM * kAsChunk * 2;             // 16 KB: one bf16 output tile
    static constexpr int kOffB = kABytes;
    static constexpr int kOffO = kOffB + kAsStages * kStageBytes;        // 2 buffers x (hi, lo)
    static constexpr int kTotal = kOffO + 2 * kParts * kTileOBytes + 1024;
};

template <int NSPLIT>
__global__ void __launch_bounds__(kAsThreads, 1) gemm_as_kernel(const __grid_constant__ TcMaps mp, const TcGemmArgs a, const int chunks_per_cta) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t a_bar[kAsMaxKb], full_bar[kAsStages], empty_bar[kAsStages], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ unsigned long long* trace_slot;
    using SM = AsSmem<NSPLIT>;
    constexpr bool kLo = NSPLIT == 3, kF16 = NSPLIT == 2;
    constexpr int kParts = SM::kParts, CPT = kAsChunk / kTcColGroups;  // 16 accumulator columns per epilogue thread
    constexpr uint32_t kAccCols = kLo ? 2 * kAsChunk : kAsChunk;      // bf16x3 keeps hi*lo in a second column half
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.y * kTcBM;
    const int num_kb = a.K / kTcBK, n_chunks = a.N / kAsChunk;
    // chunk i of this CTA = blockIdx.x + i gridDim.x (strided: with the QKV scatter every CTA then gets its share of the V^T chunks, whose
    // transposing epilogue is the slow one — a contiguous range gave one CTA of a row tile all of them: 9.4 against 8.1 us)
    (void)chunks_per_cta;
    const int c_begin = blockIdx.x, c_step = gridDim.x;
    const int my_chunks = c_begin < n_chunks ? (n_chunks - 1 - c_begin) / c_step + 1 : 0, n_items = my_chunks * num_kb;  // item = (chunk, k-block)
    // ... and the CTA's LAST chunk (QKV: its V^T chunk) goes first, so that the slow epilogue runs under the main loops of the others
    auto chunk_of = [&](int i) { return c_begin + ((i + my_chunks - 1) % my_chunks) * c_step; };
    bool ok = true;
    TraceRec tr;
    tr.begin(&trace_slot, a.trace, a.trace_id);

    // ---- prologue: independent of the preceding kernel
    if (warp == 0 && elect_one_sync()) {
        tma_prefetch_desc(&mp.Ahi), tma_prefetch_desc(&mp.Bhi);
        if (kLo) tma_prefetch_desc(&mp.Alo), tma_prefetch_desc(&mp.Blo);
        for (int i = 0; i < kAsMaxKb; ++i) mbar_init(&a_bar[i], 1);
        for (int s = 0; s < kAsStages; ++s) mbar_init(&full_bar[s], 1), mbar_init(&empty_bar[s], 1);
        for (int b = 0; b < 2; ++b) mbar_init(&acc_full[b], 1), mbar_init(&acc_empty[b], kTcThreads / 32);
        fence_barrier_init();
        const int npre = n_items < kAsStages ? n_items : kAsStages;
        for (int it = 0; it < npre; ++it) {
            const int c = chunk_of(it / num_kb), kb = it % num_kb;
            uint8_t* sb = smem + SM::kOffB + it * SM::kStageBytes;
            mbar_arrive_expect_tx(&full_bar[it], SM::kStageBytes);
            tma_load_2d(sb, &mp.Bhi, &full_bar[it], kb * kTcBK, c * kAsChunk);
            if (kLo) tma_load_2d(sb + kAsChunk * 128, &mp.Blo, &full_bar[it], kb * kTcBK, c * kAsChunk);
        }
    }
    if (warp == 1) {
        tmem_alloc(&tmem_base_s, 2 * kAccCols);
        tmem_relinquish();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = tmem_base_s;

    pdl_wait();
    if (tid == 0) tr.mark(2);
    pdl_launch_dependents();

    if (warp == 0) {
        if (elect_one_sync()) {  // ---- TMA producer: the activation tile once, then the rest of the weight stream
            for (int kb = 0; kb < num_kb; ++kb) {
                uint8_t* sa = smem + kb * kParts * kTileABytes;
                mbar_arrive_expect_tx(&a_bar[kb], kParts * kTileABytes);
                tma_load_2d(sa, &mp.Ahi, &a_bar[kb], kb * kTcBK, m0);
                if (kLo) tma_load_2d(sa + kTileABytes, &mp.Alo, &a_bar[kb], kb * kTcBK, m0);
            }
            for (int it = kAsStages; it < n_items; ++it) {
                const int s = it % kAsStages, c = chunk_of(it / num_kb), kb = it % num_kb;
                ok &= mbar_wait(&empty_bar[s], ((it / kAsStages) - 1) & 1);
                uint8_t* sb = smem + SM::kOffB + s * SM::kStageBytes;
                mbar_arrive_expect_tx(&full_bar[s], SM::kStageBytes);
                tma_load_2d(sb, &mp.Bhi, &full_bar[s], kb * kTcBK, c * kAsChunk);
                if (kLo) tma_load_2d(sb + kAsChunk * 128, &mp.Blo, &full_bar[s], kb * kTcBK, c * kAsChunk);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issuer: one elected lane (elect.sync: no per-thread election loop around tcgen05.mma); descriptors step by one add
        constexpr uint32_t idesc = umma_idesc_h<kF16>(kTcBM, kAsChunk), idesc2n = umma_idesc_h<kF16>(kTcBM, 2 * kAsChunk);
        const uint32_t a_lo0 = umma_desc_lo(smem_u32(smem)), b_lo0 = umma_desc_lo(smem_u32(smem + SM::kOffB));
        if (elect_one_sync()) {
            int it = 0;
            for (int i = 0; i < my_chunks; ++i) {
                const int buf = i & 1;
                if (i >= 2) {  // the epilogue of chunk i - 2 has read this accumulator
                    ok &= mbar_wait(&acc_empty[buf], ((i >> 1) - 1) & 1);
                    tcgen05_fence_after();
                }
                const uint32_t acc = tmem + buf * kAccCols;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % kAsStages;
                    if (i == 0) ok &= mbar_wait(&a_bar[kb], 0);
                    ok &= mbar_wait(&full_bar[s], (it / kAsStages) & 1);
                    tcgen05_fence_after();
                    const uint32_t sa = a_lo0 + kb * (kParts * kTileABytes >> 4), sb = b_lo0 + s * (SM::kStageBytes >> 4);
#pragma unroll
                    for (int k = 0; k < kTcBK / 16; ++k) {
                        const uint64_t dAhi = umma_desc_from_lo(sa + 2 * k), dBhi = umma_desc_from_lo(sb + 2 * k);
                        if (kLo) {
                            umma_bf16(acc, dAhi, dBhi, idesc2n, (kb | k) != 0);
                            umma_bf16(acc, umma_desc_from_lo(sa + (kTileABytes >> 4) + 2 * k), dBhi, idesc, 1);
                        } else {
                            umma_bf16(acc, dAhi, dBhi, idesc, (kb | k) != 0);
                        }
                    }
                    umma_commit(&empty_bar[s]);
                }
                umma_commit(&acc_full[buf]);
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue warps: thread (row, g) owns 16 accumulator columns of its row in every chunk
        const int e = tid - 64, ew = e >> 5;
        const int quarter = warp & 3, row = quarter * 32 + lane, g = ew >> 2;
        const TileRows tr_rows(m0, a.period, a.batch_off);
        const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
        const int Dm = a.N / 3;
        for (int i = 0; i < my_chunks; ++i) {
            const int buf = i & 1, n0 = chunk_of(i) * kAsChunk, nc = n0 + g * CPT;
            float bias_v[CPT];
            if (a.bias) {
#pragma unroll
                for (int j = 0; j < CPT; j += 4) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.bias + nc + j));
                    bias_v[j] = b4.x, bias_v[j + 1] = b4.y, bias_v[j + 2] = b4.z, bias_v[j + 3] = b4.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < CPT; ++j) bias_v[j] = 0.f;
            }
            ok &= mbar_wait(&acc_full[buf], (i >> 1) & 1);
            tcgen05_fence_after();
            if (e == 0 && i == 0) tr.mark(6);
            float v[CPT];
            tmem_ld_cols(lane_base + buf * kAccCols + g * CPT, v);
            if (kLo) {
                float hl[CPT];
                tmem_ld_cols(lane_base + buf * kAccCols + kAsChunk + g * CPT, hl);
#pragma unroll
                for (int j = 0; j < CPT; ++j) v[j] += hl[j];
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);  // accumulator i % 2 may be overwritten by chunk i + 2
            if (e == 0 && i == 0) tr.mark(4);
#pragma unroll
            for (int j = 0; j < CPT; ++j) v[j] += bias_v[j];
            if (a.gelu) {
#pragma unroll
                for (int j = 0; j < CPT; j += 2) gelu_erf2(v[j], v[j + 1]);
            }
            uint8_t* t_hi = smem + SM::kOffO + buf * kParts * SM::kTileOBytes;
            uint8_t* t_lo = t_hi + SM::kTileOBytes;
            int o_which = 0, o_h = 0;
            if (a.o_mode == 2) o_which = n0 / Dm, o_h = (n0 - o_which * Dm) / 64;  // this chunk is one head of Q, K or V
            if (o_which < 2) {
                stage_split<CPT, kF16>(v, t_hi, t_lo, row, g, kLo);
            } else {  // V^T: two unswizzled [64 d][64 tokens] sub-tiles (see gemm_tc.cu)
                const int sub = (row >> 6) * (kAsChunk * kHalfRows) + (g * CPT) * kHalfRows + (row & 63);
                unsigned short* uh = reinterpret_cast<unsigned short*>(t_hi) + sub;
                unsigned short* ul = reinterpret_cast<unsigned short*>(t_lo) + sub;
#pragma unroll
                for (int j = 0; j < CPT; j += 2) {
                    uint32_t h2, l2;
                    split2_h<kF16>(v[j], v[j + 1], h2, l2);
                    uh[j * kHalfRows] = (unsigned short)(h2 & 0xffffu), uh[(j + 1) * kHalfRows] = (unsigned short)(h2 >> 16);
                    if (kLo) ul[j * kHalfRows] = (unsigned short)(l2 & 0xffffu), ul[(j + 1) * kHalfRows] = (unsigned short)(l2 >> 16);
                }
            }
            // all 512 epilogue threads have staged chunk i (and, having passed this barrier for chunk i - 1 after copying chunk i - 2 out,
            // nobody still reads the buffer chunk i + ... writes next: two staging buffers, one barrier per chunk)
            if (e == 0 && i == 0) tr.mark(5);
            asm volatile("bar.sync 1, %0;" ::"n"(kTcThreads) : "memory");
            if (a.o_mode == 1) {
                tile_to_global<128>(t_hi, a.o[0], (int64_t)n0 * 2, tr_rows, a.o_row_off, 0, 0, e);
                if (kLo) tile_to_global<128>(t_lo, a.o[1], (int64_t)n0 * 2, tr_rows, a.o_row_off, 0, 0, e);
            } else if (o_which < 2) {  // Q / K: [B][heads][320][64]
                tile_to_global<128>(t_hi, a.o[2 * o_which], 0, tr_rows, 0, o_h, 0, e);
                if (kLo) tile_to_global<128>(t_lo, a.o[2 * o_which + 1], 0, tr_rows, 0, o_h, 0, e);
            } else {                   // V^T: [B][heads][64][320]
                vt_tile_to_global<kAsChunk>(t_hi, a.o[4], tr_rows, o_h, 0, e);
                if (kLo) vt_tile_to_global<kAsChunk>(t_lo, a.o[5], tr_rows, o_h, 0, e);
            }
            if (e == 0 && i == 0) tr.mark(7);  // chunk 0 copied out
        }
    }
    if (!ok && a.err) atomicExch(a.err, 1);
    tcgen05_fence_before();
    __syncthreads();
    if (tid == 0) tr.mark(3);
    if (warp == 1) tmem_dealloc(tmem, 2 * kAccCols);
}

// ---- chained MLP, A-stationary ---------------------------------------------------------------------------------------------------------
//   P[z][M, N2] = GELU( A[M, K] * W1[hidden range z, K]^T + b1 ) * W2[N2, hidden range z]^T        (bf16x3 only)
// One CTA owns a 128-row tile and a contiguous range of 64-column hidden chunks.  Per chunk: MMA1 (as above) -> the epilogue warps apply
// bias + GELU and write the hidden tile back into TENSOR MEMORY as packed bf16 (hi, lo) — a UMMA A operand — -> MMA2 multiplies it with
// the matching 64-wide K-slice of W2 and accumulates into a third TMEM accumulator [128 x N2] that lives across all chunks of the CTA.
// The hidden activations [M, hidden] never exist in memory (unchained: 15.7 MB written and read back three times at 5120 rows), and a
// row tile leaves (hidden / 64) / chunks-per-CTA fp32 partial planes instead of hidden / 64; reduce_ln_kernel adds them in plane order
// with bias, residual and the next LayerNorm.  W1 k-blocks and W2 row blocks share one ring of 16 KB stages, in MMA issue order:
//   W1(0) | W1(1) W2(0) | W1(2) W2(1) | ... | W2(n-1)       (MMA1 of chunk c + 1 is issued before MMA2 of chunk c: it runs under c's GELU)
// TMEM: accumulators of MMA1 2 x 128 columns, hidden tile 64, MMA2 accumulator N2 <= 192  = 512 columns.
#ifndef VT_MLP_STAGES
#define VT_MLP_STAGES 6
#endif
constexpr int kMlpStages = VT_MLP_STAGES;
constexpr int kMlpStageBytes = 2 * kAsChunk * kTcBK * 2;  // [W_hi; W_lo] of a 64 x 64 block
constexpr int kMlpABytes = kAsMaxKb * 2 * kTileABytes;
constexpr int kMlpSmemTotal = kMlpABytes + kMlpStages * kMlpStageBytes + 1024;
constexpr uint32_t kMlpColH = 256, kMlpColAcc2 = 320;
static_assert(kTcBM * kMaxAsChainN * 4 <= kMlpABytes + kMlpStages * kMlpStageBytes, "the partial tile is staged over the dead operand buffers");

__device__ __forceinline__ void mlp_group(int g, int n, bool& is_w2, int& chunk) {
    if (g == 0) is_w2 = false, chunk = 0;
    else if (g == 2 * n - 1) is_w2 = true, chunk = n - 1;
    else if (g & 1) is_w2 = false, chunk = (g + 1) >> 1;
    else is_w2 = true, chunk = (g >> 1) - 1;
}

__global__ void __launch_bounds__(kAsThreads, 1) gemm_as_mlp_kernel(const __grid_constant__ TcMaps mp, const TcGemmArgs a, const int chunks_per_cta) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t a_bar[kAsMaxKb], full_bar[kMlpStages], empty_bar[kMlpStages], acc_full[2], acc_empty[2], h_full, h_free, acc2_full;
    __shared__ uint32_t tmem_base_s;
    __shared__ unsigned long long* trace_slot;
    constexpr int CPT = kAsChunk / kTcColGroups;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* ring = smem + kMlpABytes;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.y * kTcBM;
    const int num_kb = a.K / kTcBK, n_chunks = a.N / kAsChunk, N2 = a.chain_n, nb2 = N2 / 64;
    const int c_begin = blockIdx.x * chunks_per_cta;
    const int c_end = c_begin + chunks_per_cta < n_chunks ? c_begin + chunks_per_cta : n_chunks;
    const int n = c_end - c_begin, n_groups = 2 * n, n_items = n * (num_kb + nb2);
    bool ok = true;
    TraceRec tr;
    tr.begin(&trace_slot, a.trace, a.trace_id);
    __shared__ unsigned long long ev_buf[kTraceEvents][2];
    __shared__ unsigned ev_cnt;
    TraceEvents ev;
    ev.begin(ev_buf, &ev_cnt, &tr);

    // weight stream walker of the producer warp (all lanes keep the same state; one elected lane issues): (group, index in group, item)
    int p_g = 0, p_j = 0, p_it = 0;
    auto issue_next = [&](bool wait_empty) {
        bool w2;
        int ch;
        mlp_group(p_g, n, w2, ch);
        const int st = p_it % kMlpStages, c = c_begin + ch;
        uint8_t* sb = ring + st * kMlpStageBytes;
        if (elect_one_sync()) {  // (the elected lane alone polls the stage: 31 lanes spinning beside it cost issue slots of the MMA-heavy SM)
            if (wait_empty) ok &= mbar_wait(&empty_bar[st], ((p_it / kMlpStages) - 1) & 1);
            mbar_arrive_expect_tx(&full_bar[st], kMlpStageBytes);
            if (!w2) {  // W1[64 c .., 64 j ..]: k-block j of hidden chunk c
                tma_load_2d(sb, &mp.Bhi, &full_bar[st], p_j * kTcBK, c * kAsChunk);
                tma_load_2d(sb + kAsChunk * 128, &mp.Blo, &full_bar[st], p_j * kTcBK, c * kAsChunk);
            } else {    // W2[64 j .., 64 c ..]: output row block j, K-slice = hidden chunk c
                tma_load_2d(sb, &mp.B2hi, &full_bar[st], c * kAsChunk, p_j * 64);
                tma_load_2d(sb + kAsChunk * 128, &mp.B2lo, &full_bar[st], c * kAsChunk, p_j * 64);
            }
        }
        __syncwarp();
        ++p_it;
        if (++p_j == (w2 ? nb2 : num_kb)) p_j = 0, ++p_g;
    };

    if (warp == 0) {
        if (elect_one_sync()) {
            tma_prefetch_desc(&mp.Ahi), tma_prefetch_desc(&mp.Alo), tma_prefetch_desc(&mp.Bhi), tma_prefetch_desc(&mp.Blo);
            tma_prefetch_desc(&mp.B2hi), tma_prefetch_desc(&mp.B2lo);
            for (int i = 0; i < kAsMaxKb; ++i) mbar_init(&a_bar[i], 1);
            for (int s = 0; s < kMlpStages; ++s) mbar_init(&full_bar[s], 1), mbar_init(&empty_bar[s], 1);
            for (int b = 0; b < 2; ++b) mbar_init(&acc_full[b], 1), mbar_init(&acc_empty[b], kTcThreads / 32);
            mbar_init(&h_full, kTcThreads / 32), mbar_init(&h_free, 1), mbar_init(&acc2_full, 1);
            fence_barrier_init();
        }
        __syncwarp();
        while (p_it < n_items && p_it < kMlpStages) issue_next(false);  // weights never depend on the preceding kernel
    }
    if (warp == 1) {
        tmem_alloc(&tmem_base_s, 512);
        tmem_relinquish();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = tmem_base_s;

    pdl_wait();
    if (tid == 0) tr.mark(2);
    pdl_launch_dependents();

    if (warp == 0) {
        // ---- TMA producer
        if (elect_one_sync()) {
            for (int kb = 0; kb < num_kb; ++kb) {
                uint8_t* sa = smem + kb * 2 * kTileABytes;
                mbar_arrive_expect_tx(&a_bar[kb], 2 * kTileABytes);
                tma_load_2d(sa, &mp.Ahi, &a_bar[kb], kb * kTcBK, m0);
                tma_load_2d(sa + kTileABytes, &mp.Alo, &a_bar[kb], kb * kTcBK, m0);
            }
        }
        __syncwarp();
        while (p_it < n_items) issue_next(true);
    } else if (warp == 1) {
        // ---- MMA issuer: one elected lane
        constexpr uint32_t idesc = umma_idesc_bf16(kTcBM, kAsChunk), idesc2n = umma_idesc_bf16(kTcBM, 2 * kAsChunk);
        const uint32_t a_lo0 = umma_desc_lo(smem_u32(smem)), b_lo0 = umma_desc_lo(smem_u32(ring));
        if (elect_one_sync()) {
            int it = 0;
            for (int g = 0; g < n_groups; ++g) {
                bool w2;
                int ch;
                mlp_group(g, n, w2, ch);
                if (!w2) {  // MMA1 of hidden chunk ch -> accumulator ch % 2
                    const int buf = ch & 1;
                    if (ch >= 2) {
                        ok &= mbar_wait(&acc_empty[buf], ((ch >> 1) - 1) & 1);
                        tcgen05_fence_after();
                    }
                    const uint32_t acc = tmem + buf * 128;
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % kMlpStages;
                        if (ch == 0) ok &= mbar_wait(&a_bar[kb], 0);
                        ok &= mbar_wait(&full_bar[s], (it / kMlpStages) & 1);
                        tcgen05_fence_after();
                        const uint32_t sa = a_lo0 + kb * (2 * kTileABytes >> 4), sb = b_lo0 + s * (kMlpStageBytes >> 4);
#pragma unroll
                        for (int k = 0; k < kTcBK / 16; ++k) {
                            const uint64_t dAhi = umma_desc_from_lo(sa + 2 * k), dBhi = umma_desc_from_lo(sb + 2 * k);
                            umma_bf16(acc, dAhi, dBhi, idesc2n, (kb | k) != 0);
                            umma_bf16(acc, umma_desc_from_lo(sa + (kTileABytes >> 4) + 2 * k), dBhi, idesc, 1);
                        }
                        umma_commit(&empty_bar[s]);
                    }
                    umma_commit(&acc_full[buf]);
                } else {    // MMA2: acc2[:, 64 j ..] += H(ch) x W2[64 j .., chunk ch]^T, H read from tensor memory
                    ok &= mbar_wait(&h_full, ch & 1);
                    tcgen05_fence_after();
                    for (int j = 0; j < nb2; ++j, ++it) {
                        const int s = it % kMlpStages;
                        ok &= mbar_wait(&full_bar[s], (it / kMlpStages) & 1);
                        tcgen05_fence_after();
                        const uint32_t sb = b_lo0 + s * (kMlpStageBytes >> 4);
                        const uint32_t acc2 = tmem + kMlpColAcc2 + 64 * j;
#pragma unroll
                        for (int k = 0; k < kAsChunk / 16; ++k) {
                            const uint32_t ah = tmem + kMlpColH + 16 * k;
                            const uint64_t dBhi = umma_desc_from_lo(sb + 2 * k), dBlo = umma_desc_from_lo(sb + (kAsChunk * 128 >> 4) + 2 * k);
                            umma_bf16_ta(acc2, ah, dBhi, idesc, (ch | k) != 0);
                            umma_bf16_ta(acc2, ah, dBlo, idesc, 1);
                            umma_bf16_ta(acc2, ah + 8, dBhi, idesc, 1);
                        }
                        umma_commit(&empty_bar[s]);
                    }
                    umma_commit(&h_free);  // the hidden-tile columns may be rewritten once these MMAs have read them
                    if (ch == n - 1) umma_commit(&acc2_full);
                }
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue warps
        const int e = tid - 64, ew = e >> 5;
        const int quarter = warp & 3, row = quarter * 32 + lane, g = ew >> 2;
        const TileRows tr_rows(m0, a.period, a.batch_off);
        const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
        for (int i = 0; i < n; ++i) {
            const int buf = i & 1, nc = (c_begin + i) * kAsChunk + g * CPT;
            float bias_v[CPT];
#pragma unroll
            for (int j = 0; j < CPT; j += 4) {
                const float4 b4 = a.bias ? __ldg(reinterpret_cast<const float4*>(a.bias + nc + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
                bias_v[j] = b4.x, bias_v[j + 1] = b4.y, bias_v[j + 2] = b4.z, bias_v[j + 3] = b4.w;
            }
            ok &= mbar_wait(&acc_full[buf], (i >> 1) & 1);
            tcgen05_fence_after();
            if (e == 0 && i == 0) tr.mark(6);
            if (e == 0) ev.event(10 + i);  // epilogue: accumulator of chunk i ready
            float v[CPT], hl[CPT];
            tmem_ld_cols(lane_base + buf * 128 + g * CPT, v);
            tmem_ld_cols(lane_base + buf * 128 + kAsChunk + g * CPT, hl);
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
#pragma unroll
            for (int j = 0; j < CPT; ++j) v[j] += hl[j];
#pragma unroll
            for (int j = 0; j < CPT; ++j) v[j] += bias_v[j];
            if (a.gelu) {
#pragma unroll
                for (int j = 0; j < CPT; j += 2) gelu_erf2(v[j], v[j + 1]);
            }
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int j = 0; j < 16; j += 2) split2_bf16(v[j], v[j + 1], hi[j >> 1], lo[j >> 1]);
            if (e == 0) ev.event(20 + i);  // epilogue: GELU of chunk i done
            if (i >= 1) {  // MMA2 of chunk i - 1 has read the hidden-tile columns
                ok &= mbar_wait(&h_free, (i - 1) & 1);
                tcgen05_fence_after();
            }
            if (e == 0) ev.event(30 + i);  // epilogue: hidden-tile columns free
            const uint32_t ta = lane_base + kMlpColH + g * 16;   // thread (row, g) = K-step g of MMA2: 8 columns hi, 8 columns lo
            tmem_st_32x8(ta, hi);
            tmem_st_32x8(ta + 8, lo);
            tmem_st_wait();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&h_full);
            if (e == 0 && i == 0) tr.mark(4);
        }
        // ---- the CTA's partial product [128, N2] -> plane blockIdx.x (staged over the dead operand buffers: every MMA has completed)
        ok &= mbar_wait(&acc2_full, 0);
        tcgen05_fence_after();
        if (e == 0) tr.mark(5);
        const int cols_per = N2 / kTcColGroups, sw = row & 7;
        for (int c = g * cols_per; c < (g + 1) * cols_per; c += 16) {
            float pv[16];
            tmem_ld_32x16(lane_base + kMlpColAcc2 + c, pv);
            uint8_t* prow = smem + (c >> 5) * (kTcBM * 128) + row * 128;
            const int ch0 = (c & 31) >> 2;
#pragma unroll
            for (int q = 0; q < 4; ++q)
                *reinterpret_cast<float4*>(prow + (((ch0 + q) ^ sw) << 4)) = make_float4(pv[4 * q], pv[4 * q + 1], pv[4 * q + 2], pv[4 * q + 3]);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTcThreads) : "memory");
        for (int cb = 0; cb < N2 / 32; ++cb)
            tile_to_global<128>(smem + cb * (kTcBM * 128), a.p, (int64_t)cb * 128, tr_rows, 0, 0, blockIdx.x, e);
        if (e == 0) tr.mark(7);
    }
    if (!ok && a.err) atomicExch(a.err, 1);
    tcgen05_fence_before();
    __syncthreads();
    if (tid == 0) tr.mark(3), ev.flush(a.trace);
    if (warp == 1) tmem_dealloc(tmem, 512);
}

cudaError_t tc_gemm_as_setup() {
    cudaError_t e = cudaFuncSetAttribute(gemm_as_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, AsSmem<1>::kTotal);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_as_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, AsSmem<2>::kTotal);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_as_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, AsSmem<3>::kTotal);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_as_mlp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMlpSmemTotal);
    return e;
}

// The plan's epilogue must be a bf16 (hi, lo) tile store or the QKV scatter.
bool tc_gemm_as_supported(const TcGemmPlan& p) {
    const TcGemmArgs& a = p.args;
    return a.K % kTcBK == 0 && a.K / kTcBK <= kAsMaxKb && a.N % kAsChunk == 0 && !a.conv_feat && !a.kb_per_split && !a.chain_n &&
           !a.ln_g && !a.c_on && !a.residual && !a.pos && !a.relu && (a.o_mode == 1 || a.o_mode == 2) && (a.o_mode != 2 || (a.N / 3) % 64 == 0);
}

// as many CTAs per row tile as fit in one wave (or `forced` > 0 of them), chunks dealt out evenly (the makespan is the largest share);
// returns CTAs per row tile
int tc_gemm_as_split(int M, int n_chunks, int sm_count, int forced, int* per_cta) {
    const int row_tiles = (M + kTcBM - 1) / kTcBM;
    int smax = forced > 0 ? forced : sm_count / row_tiles;
    if (smax < 1) smax = 1;
    if (smax > n_chunks) smax = n_chunks;
    *per_cta = (n_chunks + smax - 1) / smax;
    return (n_chunks + *per_cta - 1) / *per_cta;
}

// plan = an FC1 plan with tc_plan_chain applied (bf16x3 operands); writes *planes partial planes to the chain output
bool tc_gemm_as_mlp_supported(const TcGemmPlan& p, int nsplit) {
    const TcGemmArgs& a = p.args;
    return nsplit == 3 && a.K % kTcBK == 0 && a.K / kTcBK <= kAsMaxKb && a.N % kAsChunk == 0 && !a.conv_feat && !a.kb_per_split &&
           a.chain_n > 0 && a.chain_n % 64 == 0 && a.chain_n <= kMaxAsChainN && !a.ln_g && !a.c_on && !a.residual && !a.pos && !a.relu && a.o_mode == 3;
}
cudaError_t tc_gemm_as_mlp_launch(const TcGemmPlan& p, int M, cudaStream_t s, bool pdl, int sm_count, int forced_split, int* planes) {
    if (!tc_gemm_as_mlp_supported(p, 3) || M <= 0) return cudaErrorInvalidValue;
    TcGemmArgs a = p.args;
    a.M = M;
    a.chain_slices = 0, a.dup_hl = 0, a.dup_ln = 0;
    int per_cta = 1;
    *planes = tc_gemm_as_split(M, a.N / kAsChunk, sm_count, forced_split, &per_cta);
    const dim3 grid(*planes, (M + kTcBM - 1) / kTcBM, 1);
    return launch_ex(gemm_as_mlp_kernel, grid, dim3(kAsThreads), kMlpSmemTotal, s, pdl, 1, p.maps, a, per_cta);
}

cudaError_t tc_gemm_as_launch(const TcGemmPlan& p, int M, int nsplit, cudaStream_t s, bool pdl, int sm_count, int forced_split) {
    if (M <= 0) return cudaSuccess;
    if (!tc_gemm_as_supported(p)) return cudaErrorInvalidValue;
    TcGemmArgs a = p.args;
    a.M = M;
    a.chain_slices = 0, a.dup_hl = 0, a.dup_ln = 0;
    int per_cta = 1;
    dim3 grid(tc_gemm_as_split(M, a.N / kAsChunk, sm_count, forced_split, &per_cta), (M + kTcBM - 1) / kTcBM, 1);
    if (nsplit == 3) return launch_ex(gemm_as_kernel<3>, grid, dim3(kAsThreads), AsSmem<3>::kTotal, s, pdl, 1, p.maps, a, per_cta);
    if (nsplit == 2) return launch_ex(gemm_as_kernel<2>, grid, dim3(kAsThreads), AsSmem<2>::kTotal, s, pdl, 1, p.maps, a, per_cta);
    return launch_ex(gemm_as_kernel<1>, grid, dim3(kAsThreads), AsSmem<1>::kTotal, s, pdl, 1, p.maps, a, per_cta);
}

}  // namespace vt
