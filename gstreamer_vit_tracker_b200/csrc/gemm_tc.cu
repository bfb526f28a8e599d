// gemm_tc.cu — the dense contractions of the ViT on 5th-generation tensor cores.
//
//   C[M,N] = epilogue( A[M,K] * W[N,K]^T + bias )      A, W: bf16 (optionally split hi+lo), accumulate fp32 in TMEM
//
// One CTA (512 threads) computes one 128 x 64 output tile:
//   warp 0 (one elected lane)  TMA producer: cp.async.bulk.tensor 128B-swizzled boxes of A and W into a 3-stage smem ring,
//                              completion counted on mbarriers (expect_tx); the weight boxes of the first stages are issued
//                              BEFORE griddepcontrol.wait (they never depend on the preceding kernel), the activation boxes and
//                              the fp32 residual tile right after it;
//   warp 1 (one elected lane)  issues tcgen05.mma (UMMA 128x64x16, kind::f16) from smem descriptors into a TMEM accumulator,
//                              tcgen05.commit releases each stage and finally signals the accumulator;
//   all 16 warps               epilogue: four threads per accumulator row (tcgen05.ld.x16: warp w reads lane quarter w % 4, columns
//                              16 (w / 4) ..) -> bias / GELU / ReLU / pos-embed / residual -> the output tile is STAGED IN SHARED
//                              MEMORY (128B-swizzled, conflict free) and copied out by all 16 warps with fully coalesced 16-byte
//                              stores (a warp instruction writes four 128-byte rows).  A thread-per-row epilogue that stores
//                              straight from registers touches 32 lines per warp instruction (measured ~9 B/clk per SM, 2 us per
//                              32 KB tile); TMA tile stores were measured at ~0.16 us per 8 KB box on the issuing SM.
//                              Optionally LayerNorm of the full row through a cluster exchange (see below).
// Output rows are addressed as (target, row-in-target) of dense [targets][heads][rows][cols] tensors (TcOut): each 64-row half of a
// tile stays inside one target, rows outside a target's range are skipped; the same mechanism scatters Q / K / V^T into the
// per-(target, head) layout of the attention kernel and drops the template rows of the final LayerNorm.
//
// Precision: VT_GEMM_TCGEN05_BF16 issues A_hi*W_hi only; VT_GEMM_TCGEN05_BF16X3 adds A_hi*W_lo + A_lo*W_hi into the same
// accumulator (error ~2^-17 relative per product), which is what the 1e-3 score / exact-box parity needs; the extra tensor
// FLOPs are free at these sizes (the step is latency bound).
// Forms selected at launch (tc_gemm_launch): split-K over blockIdx.z (patch embed, head conv: fp32 partial planes); a chained second
// GEMM (FC1 -> FC2 partial products, the hidden tile never leaves the SM); LayerNorm fused through a cluster exchange; and, in latency
// mode (`spread`: at most two live handles on the GPU, most SMs idle), replicas of a tile over blockIdx.z so that each replica stores
// a share of the epilogue output — a CTA stores at ~26 B/clk, which is what bounds the 32..96 KB epilogues: FC1 chain in three
// 64-column slices (the GELU'd hidden tile then is a TMEM A operand), QKV scatter as hi / lo replicas, fused-LN GEMM as fp32 / LN-hi /
// LN-lo replicas.  All forms are re-associations of the same sums (tests/test_gpu_tracker.py::test_kernel_forms_agree).
// With one target the QKV scatter and the chained FC1 run on 64-row tiles (M = 64 UMMAs: five tiles of 320 rows instead of
// 128 + 128 + 64, half the epilogue per CTA), the chained product in two slices of 96 columns (tests/test_gpu_gemm_q64.py).
// 128 x 32 tiles and TMA multicast of the activation tile across column-tile CTAs were measured without gain (DESIGN.md §7).
// The 3x3 head convolution runs through the same kernel: its A operand is gathered by TMA from the [B,16,16,D] token grid with
// shifted (possibly negative) coordinates; out-of-bounds elements are zero-filled by the TMA unit = zero padding of the conv.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "gemm_epi.cuh"

namespace vt {

constexpr int kTcStages = 3;
constexpr int kMaxChainN = 192;                 // widest chained second GEMM (TMEM: 128 + N2 <= 512 columns)
constexpr int kTcBN = 64;                       // column-tile width; the chained GEMM consumes the 64-column hidden tile as its K

// 64-row tiles (BM = 64, M = 64 UMMAs; bf16x3 only): the QKV scatter and the chained FC1 in two slices of kMaxChainN / 2 columns
constexpr int kChainN64 = kMaxChainN / 2;

template <int NSPLIT, int BM = kTcBM>
struct TcSmem {
    static constexpr int kParts = NSPLIT == 3 ? 2 : 1;  // NSPLIT: 1 = bf16, 2 = fp16 (single pass), 3 = bf16 hi + lo
    static constexpr int kTileABytes = BM * kTcBK * 2;  // 16 / 8 KB, one precision part
    static constexpr int kTileBBytes = kTcBN * kTcBK * 2;   // 8 KB
    static constexpr int kTileOBytes = BM * kTcBN * 2;      // 16 / 8 KB: one bf16 output tile, rows of 128 bytes
    static constexpr int kTileCBytes = BM * kTcBN * 4;      // 32 / 16 KB: the fp32 tile as two boxes of [BM rows][128 B]
    static constexpr int kStageBytes = kParts * (kTileABytes + kTileBBytes);
    // the ring is padded (bf16 mode) so that the chained GEMM's result tile fits behind the staged hidden tile
    static constexpr int kRingMin = 2 * kTileOBytes + BM * kMaxChainN * 4;
    static constexpr int kPipeBytes = kTcStages * kStageBytes > kRingMin ? kTcStages * kStageBytes : kRingMin;
    // after the main loop the pipeline ring is dead and holds the staged output tiles
    static constexpr int kOffOhi = 0, kOffOlo = kTileOBytes, kOffLnHi = 2 * kTileOBytes, kOffLnLo = 3 * kTileOBytes;
    static constexpr int kOffC = kPipeBytes;  // fp32 tile: residual in (TMA load during the main loop), C out, in place
    // chained second GEMM (FC2 partial inside the FC1 kernel): its weight slice [N2 <= 192][64] per part lives where the fp32
    // tile would be, its fp32 result tile [BM][N2] is staged in the dead ring behind the two hidden-tile parts
    static constexpr int kOffB2 = kPipeBytes, kB2PartBytes = kMaxChainN * 128, kOffP = 2 * kTileOBytes;
    static constexpr int kTailBytes = kParts * kB2PartBytes > kTileCBytes ? kParts * kB2PartBytes : kTileCBytes;
    static constexpr int kTotal = kPipeBytes + kTailBytes + 1024;  // + alignment slack
    static_assert(4 * kTileOBytes <= kPipeBytes, "staging must fit in the dead pipeline ring");
};


// LayerNorm fused into the epilogue of the GEMMs that produce the residual stream (patch-embed, proj, FC2): the N / 64 CTAs
// that hold the column tiles of one 128-row tile form a thread-block cluster; every thread computes the (sum, M2) of its 16
// columns from registers, pushes the pair into every peer's shared memory with st.async (the store itself signals the peer's
// mbarrier: no cluster barrier on the critical path), and every CTA combines the partials in a fixed order (Chan's parallel variance) — every CTA gets bit-identical statistics — normalises its
// own columns and stages the bf16 (hi, lo) A operand of the next GEMM for a TMA tile store.
constexpr int kMaxLnCluster = 8;


// BM = 64 (tc_gemm_launch: q64): a 64-row tile with M = 64 UMMAs, for the QKV scatter (hi / lo replicas) and the sliced chained FC1
// (hidden tile as a TMEM A operand) only.  Row 16 q + i of an M = 64 accumulator sits in TMEM lane 32 q + i (i < 16), so the 16 warps
// split each row 8 ways (8 columns per thread) through the 16x32bx2 shapes; the fused-LN, split-K, residual, fp32-tile, bf16-tile,
// conv and unsliced chained epilogues exist for BM = 128 only.
template <int NSPLIT, int BM>
__global__ void __launch_bounds__(kTcThreads, 1) gemm_tc_kernel(const __grid_constant__ TcMaps mp, const TcGemmArgs a) {
    static_assert(BM == kTcBM || (BM == 64 && NSPLIT == 3), "64-row tiles: bf16x3 only");
    constexpr bool kQ64 = BM == 64;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kTcStages], empty_bar[kTcStages], accum_bar, resid_bar, b2_bar, accum2_bar, ln_bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ float2 ln_loc[kTcColGroups][kTcBM];   // (sum, M2) of the CPT columns of thread (row, g)
    __shared__ float2 ln_part[kMaxLnCluster][kTcBM];  // (sum, M2) of the 64 columns of every CTA of the cluster, per row
    __shared__ unsigned long long* trace_slot;
    using SM = TcSmem<NSPLIT, BM>;
    constexpr int BN = kTcBN;
    constexpr int CPT = BN * BM / kTcThreads;  // accumulator columns per thread: 16 (4 threads per row) / 8 (8 threads per row)
    constexpr int RB = BN * 2;                 // bytes per row of a bf16 staging tile
    constexpr int kTileABytes = SM::kTileABytes, kTileBBytes = SM::kTileBBytes, kTileOBytes = SM::kTileOBytes, kTileCBytes = SM::kTileCBytes;
    constexpr bool kLo = NSPLIT == 3, kF16 = NSPLIT == 2;
    const CUtensorMap &mAhi = kQ64 ? mp.Ahi64 : mp.Ahi, &mAlo = kQ64 ? mp.Alo64 : mp.Alo;
    const CUtensorMap &mB2hi = kQ64 ? mp.B2hiHalf : mp.B2hi, &mB2lo = kQ64 ? mp.B2loHalf : mp.B2lo;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // accumulator row inside the tile; warp w reads TMEM lane quarter w % 4 (BM = 128: row = lane; BM = 64: row 16 q + i in lane 32 q + i)
    const int row = kQ64 ? (warp & 3) * 16 + (lane & 15) : (warp & 3) * 32 + lane;
    // column group: columns CPT g .. CPT g + CPT - 1 of the tile (BM = 64: threads 16..31 take the 8 columns after those of threads 0..15)
    const int g = kQ64 ? 2 * (warp >> 2) + (lane >> 4) : warp >> 2;
    const uint32_t tq = (uint32_t)((warp & 3) * 32) << 16;  // TMEM lane quarter of the warp (address bits 16..)
    const uint32_t wcol = kQ64 ? (warp >> 2) * 16 : g * CPT;  // first accumulator column a tcgen05.ld of the warp addresses
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
    // split-K over blockIdx.z: this CTA contracts k-blocks [kb0, kb0 + num_kb) and stores its fp32 partial tile to C[.., z]
    const int num_kb = a.kb_per_split ? a.kb_per_split : a.K / kTcBK;
    const int kb0 = a.kb_per_split ? blockIdx.z * num_kb : 0;
    // "spread" form (latency mode, idle SMs available): blockIdx.z replicates the FC1 tile and replica z computes and stores columns
    // [N2 z, N2 z + N2) of the chained product — a CTA's egress (~26 B/clk/SM) is what bounds the 96 KB partial-tile epilogue.
    const bool sliced = a.chain_slices > 1;  // (BM = 64: two slices of kChainN64 columns)
    const int N2 = sliced ? a.chain_n / a.chain_slices : a.chain_n;   // chained columns of this CTA
    const int acc2_cols = (sliced && kLo) ? 2 * N2 : N2;              // sliced + bf16x3: hi*lo term in a second column half
    // dup_ln (spread form of a GEMM with fused LayerNorm): replica 0 stores the fp32 tile, replica 1 the LayerNorm hi tile, replica 2 the lo tile
    const bool do_ln = !kQ64 && a.ln_g != nullptr && (!a.dup_ln || blockIdx.z > 0), do_c = !kQ64 && a.c_on && (!a.dup_ln || blockIdx.z == 0);
    const bool ln_hi = !a.dup_ln || blockIdx.z == 1, ln_lo = kLo && (!a.dup_ln || blockIdx.z == 2);
    // dup_hl (spread form of the QKV scatter): replica 0 stores the bf16 hi tiles, replica 1 the lo tiles
    const bool st_hi = !a.dup_hl || blockIdx.z == 0, st_lo = kLo && (!a.dup_hl || blockIdx.z == 1);
    const int npre = num_kb < kTcStages ? num_kb : kTcStages;
    constexpr uint32_t kAcc1Cols = kLo ? 2 * BN : BN;  // bf16x3 keeps hi*lo in a second column half
    // sliced chain: the hidden tile as a packed bf16 A operand, behind the chained accumulator (BM = 128: 2 x 64, BM = 64: 2 x 96 columns)
    constexpr uint32_t kColA2 = kQ64 ? kAcc1Cols + 2 * kChainN64 : 256;
    const uint32_t tmem_need = a.chain_n == 0 ? kAcc1Cols : ((sliced && kLo) ? kColA2 + 64 : kAcc1Cols + acc2_cols);
    const uint32_t tmem_cols = tmem_need <= 32 ? 32 : (tmem_need <= 64 ? 64 : (tmem_need <= 128 ? 128 : (tmem_need <= 256 ? 256 : 512)));
    bool ok = true;
    TraceRec tr;
    tr.begin(&trace_slot, a.trace, a.trace_id);

    // ---- prologue: independent of the preceding kernel, overlaps its tail under PDL
    if (warp == 0 && elect_one_sync()) {  // (one thread; elect.sync lets the compiler issue the TMA instructions without election loops)
        tma_prefetch_desc(&mAhi), tma_prefetch_desc(&mp.Bhi);
        if (kLo) tma_prefetch_desc(&mAlo), tma_prefetch_desc(&mp.Blo);
        for (int s = 0; s < kTcStages; ++s) mbar_init(&full_bar[s], 1), mbar_init(&empty_bar[s], 1);
        mbar_init(&accum_bar, 1), mbar_init(&resid_bar, 1), mbar_init(&b2_bar, 1), mbar_init(&accum2_bar, 1), mbar_init(&ln_bar, 1);
        fence_barrier_init();
        // LayerNorm exchange: every CTA of the cluster (this one included) sends one float2 per row into ln_part of this CTA
        if (do_ln && cluster_nctarank() > 1) mbar_arrive_expect_tx(&ln_bar, cluster_nctarank() * kTcBM * (uint32_t)sizeof(float2));
        // the weights never depend on the preceding kernel: start streaming them right away
        for (int kb = 0; kb < npre; ++kb) {
            uint8_t* sb = smem + kb * SM::kStageBytes + SM::kParts * kTileABytes;
            mbar_arrive_expect_tx(&full_bar[kb], SM::kStageBytes);
            tma_load_2d(sb, &mp.Bhi, &full_bar[kb], (kb0 + kb) * kTcBK, n0);
            if (kLo) tma_load_2d(sb + kTileBBytes, &mp.Blo, &full_bar[kb], (kb0 + kb) * kTcBK, n0);
        }
        if (a.chain_n) {  // weight slice of the chained GEMM: W2[rows of this CTA][n0 .. n0 + 64), 64-row boxes per precision part
            tma_prefetch_desc(&mB2hi);
            mbar_arrive_expect_tx(&b2_bar, SM::kParts * N2 * 128);
            if (sliced) {  // [W2_hi slice; W2_lo slice] adjacent: one N = 2 N2 B operand
                tma_load_2d(smem + SM::kOffB2, &mB2hi, &b2_bar, n0, blockIdx.z * N2);
                if (kLo) tma_load_2d(smem + SM::kOffB2 + N2 * 128, &mB2lo, &b2_bar, n0, blockIdx.z * N2);
            } else if (!kQ64) {
                for (int r = 0; r < N2; r += 64) {
                    tma_load_2d(smem + SM::kOffB2 + r * 128, &mp.B2hi, &b2_bar, n0, r);
                    if (kLo) tma_load_2d(smem + SM::kOffB2 + SM::kB2PartBytes + r * 128, &mp.B2lo, &b2_bar, n0, r);
                }
            }
        }
        if (a.residual) tma_prefetch_desc(&mp.R);
    }
    if (warp == 1) {
        tmem_alloc(&tmem_base_s, tmem_cols);  // 64 (bf16x3: 128) fp32 accumulator columns (+ N2 for a chained second GEMM)
        tmem_relinquish();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = tmem_base_s;
    // cluster handshake ("this CTA is running, its barriers are initialised and armed"): peers may push LayerNorm partials into its
    // shared memory after the matching wait
    const bool clustered = a.ln_g != nullptr;
    if (clustered) cluster_arrive_release();

    pdl_wait();               // the activations (A, residual) are complete and visible from here on
    if (tid == 0) tr.mark(2);
    pdl_launch_dependents();  // let the next kernel of the chain run its prologue under our main loop
    if (clustered) cluster_wait_acquire();

    uint8_t* sC = smem + SM::kOffC;
    if (warp == 0) {
        if (elect_one_sync()) {  // ---- TMA producer
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % kTcStages;
                uint8_t* st = smem + s * SM::kStageBytes;
                if (kb >= kTcStages) {
                    ok &= mbar_wait(&empty_bar[s], ((kb / kTcStages) - 1) & 1);
                    mbar_arrive_expect_tx(&full_bar[s], SM::kStageBytes);
                    uint8_t* sb = st + SM::kParts * kTileABytes;
                    tma_load_2d(sb, &mp.Bhi, &full_bar[s], (kb0 + kb) * kTcBK, n0);
                    if (kLo) tma_load_2d(sb + kTileBBytes, &mp.Blo, &full_bar[s], (kb0 + kb) * kTcBK, n0);
                }
                if (!kQ64 && a.conv_feat) {  // 3x3 conv: K index = tap * feat + d; A rows are the 16x16 grid of one target
                    const int chunks = a.conv_feat / kTcBK, tap = (kb0 + kb) / chunks, d0 = ((kb0 + kb) % chunks) * kTcBK;
                    const int b = m0 / kNTx, y0 = (m0 % kNTx) / kMap;
                    tma_load_4d(st, &mp.Ahi, &full_bar[s], d0, tap % 3 - 1, y0 + tap / 3 - 1, b);
                    if (kLo) tma_load_4d(st + kTileABytes, &mp.Alo, &full_bar[s], d0, tap % 3 - 1, y0 + tap / 3 - 1, b);
                } else {
                    tma_load_2d(st, &mAhi, &full_bar[s], (kb0 + kb) * kTcBK, m0);
                    if (kLo) tma_load_2d(st + kTileABytes, &mAlo, &full_bar[s], (kb0 + kb) * kTcBK, m0);
                }
                if (!kQ64 && kb == 0 && a.residual) {  // residual rows of this tile (flat [rows][N] fp32), two 128-byte-wide boxes
                    mbar_arrive_expect_tx(&resid_bar, kTileCBytes);
#pragma unroll
                    for (int bx = 0; bx < BN / 32; ++bx) tma_load_2d(sC + bx * (kTcBM * 128), &mp.R, &resid_bar, n0 + 32 * bx, m0);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issuer: one elected lane (elect.sync: the compiler emits tcgen05.mma without a per-thread election loop); descriptors
        // step by one add
        // bf16x3: A_hi x [W_hi; W_lo] as ONE N = 128 UMMA (the two weight parts are adjacent 64-row tiles of the stage) into
        // accumulator columns [0, 64) (hi*hi) and [64, 128) (hi*lo), then A_lo x W_hi (N = 64) into [0, 64); the epilogue adds the
        // two halves.  (tools/probes/probe_umma.cu: an MMA with both operands in shared memory costs ~43 + N / 2 clk — the 4 KB A slice
        // is fetched before the math starts — so N = 128 + N = 64 (107 + 81 clk) beats three N = 64 MMAs (243 clk).)
        constexpr uint32_t idesc = umma_idesc_h<kF16>(BM, BN), idesc2n = umma_idesc_h<kF16>(BM, 2 * BN);
        const uint32_t lo0 = umma_desc_lo(smem_u32(smem));
        if (elect_one_sync()) {
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % kTcStages;
                ok &= mbar_wait(&full_bar[s], (kb / kTcStages) & 1);
                tcgen05_fence_after();
                const uint32_t sa = lo0 + s * (SM::kStageBytes >> 4), sb = sa + (SM::kParts * kTileABytes >> 4);
#pragma unroll
                for (int k = 0; k < kTcBK / 16; ++k) {  // 16 bf16 = 32 bytes inside the 128-byte swizzle row: descriptor + 2
                    const uint64_t dAhi = umma_desc_from_lo(sa + 2 * k), dBhi = umma_desc_from_lo(sb + 2 * k);
                    if (kLo) {
                        umma_bf16(tmem, dAhi, dBhi, idesc2n, (kb | k) != 0);
                        umma_bf16(tmem, umma_desc_from_lo(sa + (kTileABytes >> 4) + 2 * k), dBhi, idesc, 1);
                    } else {
                        umma_bf16(tmem, dAhi, dBhi, idesc, (kb | k) != 0);
                    }
                }
                umma_commit(&empty_bar[s]);  // stage reusable once these MMAs have read it
            }
            umma_commit(&accum_bar);
        }
        __syncwarp();
    }

    // ---- epilogue: thread (row, g) owns 16 accumulator columns of its row
    const int m = m0 + row, nc = n0 + g * CPT;
    // this thread's CPT / 4 16-byte chunks of the fp32 tile: 32-column box (CPT g) / 32, first chunk ((CPT g) % 32) / 4, swizzled
    uint8_t* c_row = sC + ((g * CPT) >> 5) * (BM * 128) + row * 128;
    const int c_chunk0 = ((g * CPT) & 31) >> 2, sw = row & 7;
    const TileRows tr_rows(m0, a.period, a.batch_off);
    int o_which = 0, o_h = 0, o_d = 0;
    if (a.o_mode == 2) {  // QKV: this CTA's 64 columns are one head of Q, K or V
        const int Dm = a.N / 3;
        o_which = n0 / Dm, o_h = (n0 - o_which * Dm) / 64, o_d = (n0 - o_which * Dm) % 64;  // head_dim 64
    }
    float bias_v[CPT];
    if (a.bias) {  // does not depend on the accumulator: fetch while the MMAs run
#pragma unroll
        for (int j = 0; j < CPT; j += 4) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.bias + nc + j));
            bias_v[j] = b4.x, bias_v[j + 1] = b4.y, bias_v[j + 2] = b4.z, bias_v[j + 3] = b4.w;
        }
    } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) bias_v[j] = 0.f;
    }
    ok &= mbar_wait(&accum_bar, 0);
    tcgen05_fence_after();
    if (tid == 0) tr.mark(6);
    auto ld_acc = [&](uint32_t col, float(&x)[CPT]) {  // this thread's CPT accumulator columns from the warp's column `col` on
        if constexpr (kQ64) tmem_ld_16x2(tmem + tq + col, x);
        else tmem_ld_cols(tmem + tq + col, x);
    };
    float v[CPT];
    ld_acc(wcol, v);
    if (kLo) {
        float hl[CPT];
        ld_acc(BN + wcol, hl);
#pragma unroll
        for (int j = 0; j < CPT; ++j) v[j] += hl[j];
    }
#pragma unroll
    for (int j = 0; j < CPT; ++j) v[j] += bias_v[j];
    if (a.gelu) {
#pragma unroll
        for (int j = 0; j < CPT; j += 2) gelu_erf2(v[j], v[j + 1]);
    }
    if (a.relu) {
#pragma unroll
        for (int j = 0; j < CPT; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    if (a.pos) {
        const float* pp = a.pos + (int64_t)(m % a.pos_rows) * a.N + nc;
#pragma unroll
        for (int j = 0; j < CPT; j += 4) {
            const float4 p4 = __ldg(reinterpret_cast<const float4*>(pp + j));
            v[j] += p4.x, v[j + 1] += p4.y, v[j + 2] += p4.z, v[j + 3] += p4.w;
        }
    }
    if (!kQ64 && a.residual) {
        ok &= mbar_wait(&resid_bar, 0);
#pragma unroll
        for (int q = 0; q < CPT / 4; ++q) {
            const float4 r4 = *reinterpret_cast<const float4*>(c_row + (((c_chunk0 + q) ^ sw) << 4));
            v[4 * q] += r4.x, v[4 * q + 1] += r4.y, v[4 * q + 2] += r4.z, v[4 * q + 3] += r4.w;
        }
    }
    if (do_ln) {  // row statistics of this thread's CPT columns; combined per row after the staging barrier below
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < CPT; ++j) s += v[j];
        const float mu = s * (1.f / CPT);
        float m2 = 0.f;
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            const float d = v[j] - mu;
            m2 = fmaf(d, d, m2);
        }
        ln_loc[g][row] = make_float2(s, m2);
    }
    if (tid == 0) tr.mark(4);
    // ---- stage the output tiles in shared memory (the pipeline ring is dead: every MMA has completed)
    if (do_c) {
#pragma unroll
        for (int q = 0; q < CPT / 4; ++q)
            *reinterpret_cast<float4*>(c_row + (((c_chunk0 + q) ^ sw) << 4)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    }
    // sliced chain: the hidden tile goes back into tensor memory as packed bf16 (thread (row, g) = K-step g: 8 columns hi, 8 columns
    // lo), so the chained UMMAs fetch only the weight slice from shared memory
    const bool a_tmem = sliced && kLo && a.o_mode == 3;
    // (BM = 64: K-step warp / 4, threads 0..15 its elements 0..7 in columns +0..3 / +8..11, threads 16..31 elements 8..15 in +4..7 / +12..15)
    if (a_tmem) {
        uint32_t hi[CPT / 2], lo[CPT / 2];
#pragma unroll
        for (int j = 0; j < CPT; j += 2) split2_bf16(v[j], v[j + 1], hi[j >> 1], lo[j >> 1]);
        const uint32_t ta = tmem + tq + kColA2 + (wcol & ~15u);
        if constexpr (kQ64) {
            tmem_st_16x2_x4(ta, hi);
            tmem_st_16x2_x4(ta + 8, lo);
        } else {
            tmem_st_32x8(ta, hi);
            tmem_st_32x8(ta + 8, lo);
        }
        tmem_st_wait();
    } else if (a.o_mode) {  // (o_mode 3: staged only — the tile is the A operand of the chained GEMM)
        if (o_which < 2) {
            stage_split<CPT, kF16, RB>(v, smem + SM::kOffOhi, smem + SM::kOffOlo, row, g, kLo);
        } else {  // V^T: BM / 64 unswizzled [BN d][64 tokens] sub-tiles; lanes are consecutive tokens -> 64-byte contiguous runs
            const int sub = (row >> 6) * (BN * kHalfRows) + (g * CPT) * kHalfRows + (row & 63);
            __nv_bfloat16* th = reinterpret_cast<__nv_bfloat16*>(smem + SM::kOffOhi) + sub;
            __nv_bfloat16* tl = reinterpret_cast<__nv_bfloat16*>(smem + SM::kOffOlo) + sub;
            // (packed cvt.rn.bf16x2: the scalar cvt.rn.bf16.f32 runs on the 16/clk conversion pipe — 32 of them per thread made the V^T
            // tiles finish 0.3 us after the Q / K tiles)
            unsigned short* uh = reinterpret_cast<unsigned short*>(th);
            unsigned short* ul = reinterpret_cast<unsigned short*>(tl);
#pragma unroll
            for (int j = 0; j < CPT; j += 2) {
                uint32_t h2, l2;
                split2_h<kF16>(v[j], v[j + 1], h2, l2);
                uh[j * kHalfRows] = (unsigned short)(h2 & 0xffffu), uh[(j + 1) * kHalfRows] = (unsigned short)(h2 >> 16);
                if (kLo) ul[j * kHalfRows] = (unsigned short)(l2 & 0xffffu), ul[(j + 1) * kHalfRows] = (unsigned short)(l2 >> 16);
            }
        }
    }
    if (a.o_mode == 3) {
        if (a_tmem) tcgen05_fence_before();
        else fence_proxy_async_smem();  // the staged tile is read by the tensor core (async proxy) in the chained GEMM
    }
    __syncthreads();
    if (!kQ64 && do_ln && g == 0) {  // one thread per row: (sum, M2) over the BN columns of this CTA (Chan), sent to every CTA of the cluster
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < kTcColGroups; ++q) s += ln_loc[q][row].x;
        const float mu = s * (1.f / BN);
        float m2 = 0.f;
#pragma unroll
        for (int q = 0; q < kTcColGroups; ++q) {
            const float2 p = ln_loc[q][row];
            const float d = p.x * (1.f / CPT) - mu;
            m2 += p.y + (float)CPT * d * d;
        }
        if (cluster_nctarank() > 1) {
            const uint32_t mine = smem_u32(&ln_part[cluster_ctarank()][row]), bar = smem_u32(&ln_bar);  // (peers are known to run: cluster handshake above)
            for (uint32_t r = 0; r < cluster_nctarank(); ++r) st_async_cluster_f2(cluster_map_shared(mine, r), s, m2, cluster_map_shared(bar, r));
        } else {  // N = BN: the row lives in this CTA alone (launched without a cluster: st.async would be an illegal instruction)
            ln_part[0][row] = make_float2(s, m2);
        }
    }
    if (do_c) {  // split-K partials: plane = blockIdx.z
#pragma unroll
        for (int bx = 0; bx < BN / 32; ++bx)
            tile_to_global<128>(sC + bx * (BM * 128), a.c, (int64_t)(n0 + 32 * bx) * 4, tr_rows, a.c_row_off, 0, a.kb_per_split ? blockIdx.z : 0, tid);
    }
    if (!kQ64 && a.o_mode == 1) {
        if (st_hi) tile_to_global<RB>(smem + SM::kOffOhi, a.o[0], (int64_t)n0 * 2, tr_rows, a.o_row_off, 0, 0, tid);
        if (st_lo) tile_to_global<RB>(smem + SM::kOffOlo, a.o[1], (int64_t)n0 * 2, tr_rows, a.o_row_off, 0, 0, tid);
    } else if (a.o_mode == 2) {  // Q / K: [B][heads][320][64]; V^T: [B][heads][64][320]
        if (o_which < 2) {
            if (st_hi) tile_to_global<RB, BM>(smem + SM::kOffOhi, a.o[2 * o_which], (int64_t)o_d * 2, tr_rows, 0, o_h, 0, tid);
            if (st_lo) tile_to_global<RB, BM>(smem + SM::kOffOlo, a.o[2 * o_which + 1], (int64_t)o_d * 2, tr_rows, 0, o_h, 0, tid);
        } else {
            if (st_hi) vt_tile_to_global<BN, BM / 64>(smem + SM::kOffOhi, a.o[4], tr_rows, o_h, o_d, tid);
            if (st_lo) vt_tile_to_global<BN, BM / 64>(smem + SM::kOffOlo, a.o[5], tr_rows, o_h, o_d, tid);
        }
    }
    if (tid == 0) tr.mark(7);
    if (a.chain_n) {
        // ---- chained GEMM: P_j[BM, N2] = hidden tile (just staged as a 128B-swizzled K-major A operand, bf16 hi / lo) x
        // W2[:, n0 .. n0 + 64)^T.  The hidden activations never travel to global memory; the N / 64 partial results P_j of one row
        // tile are summed in a fixed order by reduce_ln_kernel, which also applies bias, residual and the next LayerNorm.
        if (warp == 1) {
            ok &= mbar_wait(&b2_bar, 0);
            tcgen05_fence_after();
            const uint32_t a_lo = umma_desc_lo(smem_u32(smem + SM::kOffOhi)), b_lo = umma_desc_lo(smem_u32(smem + SM::kOffB2));
            constexpr uint32_t kLoA = kTileOBytes >> 4, kLoB = SM::kB2PartBytes >> 4;
            if (elect_one_sync()) {
                if (kQ64 || (sliced && kLo)) {  // H_hi x [W2_hi; W2_lo] as one UMMA of 2 N2 columns + H_lo x W2_hi (the epilogue adds the halves)
                    const uint32_t idesc2 = umma_idesc_bf16(BM, N2), idesc2n = umma_idesc_bf16(BM, 2 * N2);
#pragma unroll
                    for (int k = 0; k < BN / 16; ++k) {
                        const uint64_t dB = umma_desc_from_lo(b_lo + 2 * k);
                        umma_bf16_ta(tmem + kAcc1Cols, tmem + kColA2 + 16 * k, dB, idesc2n, k != 0);
                        umma_bf16_ta(tmem + kAcc1Cols, tmem + kColA2 + 16 * k + 8, dB, idesc2, 1);
                    }
                } else {
                    const uint32_t idesc2 = kF16 ? umma_idesc_f16(BM, N2) : umma_idesc_bf16(BM, N2);  // K = the 64 hidden columns of this CTA
#pragma unroll
                    for (int k = 0; k < BN / 16; ++k) {
                        const uint64_t dA = umma_desc_from_lo(a_lo + 2 * k), dB = umma_desc_from_lo(b_lo + 2 * k);
                        umma_bf16(tmem + kAcc1Cols, dA, dB, idesc2, k != 0);
                        if (kLo) {
                            umma_bf16(tmem + kAcc1Cols, dA, umma_desc_from_lo(b_lo + kLoB + 2 * k), idesc2, 1);
                            umma_bf16(tmem + kAcc1Cols, umma_desc_from_lo(a_lo + kLoA + 2 * k), dB, idesc2, 1);
                        }
                    }
                }
                umma_commit(&accum2_bar);
            }
        }
        __syncwarp();
        ok &= mbar_wait(&accum2_bar, 0);
        tcgen05_fence_after();
        if (tid == 0) tr.mark(5);
        // fp32 tile staged as N2/32 boxes of [BM rows][128 B], swizzled; stage4 = the 4 columns c.. of this thread's row
        auto stage4 = [&](int c, float x0, float x1, float x2, float x3) {
            *reinterpret_cast<float4*>(smem + SM::kOffP + (c >> 5) * (BM * 128) + row * 128 + ((((c & 31) >> 2) ^ sw) << 4)) = make_float4(x0, x1, x2, x3);
        };
        if constexpr (kQ64) {
            // warp group w / 4 owns the 24 columns 24 (w / 4) .. of the N2 = 96: threads 0..15 columns +0..7 and +16..19, threads
            // 16..31 +8..15 and +20..23; all four loads (hi*hi + lo*hi, hi*lo halves) in flight before the wait
            constexpr int kW = kChainN64 / 4;
            const uint32_t t2 = tmem + tq + kAcc1Cols + (warp >> 2) * kW;
            uint32_t pa[8], pb[4], ha[8], hb[4];
            tmem_ld_16x2_x8_issue(t2, pa), tmem_ld_16x2_x4_issue(t2 + 16, pb);
            tmem_ld_16x2_x8_issue(t2 + kChainN64, ha), tmem_ld_16x2_x4_issue(t2 + kChainN64 + 16, hb);
            tmem_ld_wait(pa), tmem_ld_wait(pb), tmem_ld_wait(ha), tmem_ld_wait(hb);
            float p[12];
#pragma unroll
            for (int j = 0; j < 8; ++j) p[j] = __uint_as_float(pa[j]) + __uint_as_float(ha[j]);
#pragma unroll
            for (int j = 0; j < 4; ++j) p[8 + j] = __uint_as_float(pb[j]) + __uint_as_float(hb[j]);
            const int c0 = (warp >> 2) * kW, h = lane >> 4;
            stage4(c0 + 8 * h, p[0], p[1], p[2], p[3]);
            stage4(c0 + 8 * h + 4, p[4], p[5], p[6], p[7]);
            stage4(c0 + 16 + 4 * h, p[8], p[9], p[10], p[11]);
        } else {
            // thread (row, g) owns columns g * N2/4 .. of its row
            const int cols_per = N2 / kTcColGroups;
            for (int c = g * cols_per; c < (g + 1) * cols_per; c += 16) {
                float p[16];
                tmem_ld_32x16(tmem + tq + kAcc1Cols + c, p);
                if (sliced && kLo) {
                    float hl[16];
                    tmem_ld_32x16(tmem + tq + kAcc1Cols + N2 + c, hl);
#pragma unroll
                    for (int j = 0; j < 16; ++j) p[j] += hl[j];
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) stage4(c + 4 * q, p[4 * q], p[4 * q + 1], p[4 * q + 2], p[4 * q + 3]);
            }
        }
        __syncthreads();
        if (tid == 0) tr.mark(4);
        for (int cb = 0; cb < N2 / 32; ++cb)  // P[j = blockIdx.x][target][row][32 cb ..]
            tile_to_global<128, BM>(smem + SM::kOffP + cb * (BM * 128), a.p, (int64_t)cb * 128 + (sliced ? (int64_t)blockIdx.z * N2 * 4 : 0), tr_rows, 0, 0,
                                blockIdx.x, tid);
    }
    if (!kQ64 && do_ln) {  // ---- fused LayerNorm over the full row (N columns = cluster of N / BN CTAs)
        const uint32_t nct = cluster_nctarank();
        float gam[CPT], bet[CPT];
#pragma unroll
        for (int j = 0; j < CPT; j += 4) {
            const float4 g4 = __ldg(reinterpret_cast<const float4*>(a.ln_g + nc + j)), b4 = __ldg(reinterpret_cast<const float4*>(a.ln_b + nc + j));
            gam[j] = g4.x, gam[j + 1] = g4.y, gam[j + 2] = g4.z, gam[j + 3] = g4.w;
            bet[j] = b4.x, bet[j + 1] = b4.y, bet[j + 2] = b4.z, bet[j + 3] = b4.w;
        }
        // all partials of this CTA's rows have landed (complete_tx bytes); nobody exits before its own ln_part is complete, and a
        // peer only completes after receiving ours, so no CTA of the cluster can disappear under an in-flight store
        if (nct > 1) ok &= mbar_wait(&ln_bar, 0);
        else __syncthreads();
        if (tid == 0) tr.mark(5);
        float tot = 0.f;
        for (uint32_t r = 0; r < nct; ++r) tot += ln_part[r][row].x;
        const float mean = tot / (float)a.N;
        float M2 = 0.f;
        for (uint32_t r = 0; r < nct; ++r) {
            const float2 p = ln_part[r][row];
            const float d = p.x * (1.f / BN) - mean;
            M2 += p.y + (float)BN * d * d;
        }
        const float rstd = 1.f / sqrtf(M2 / (float)a.N + 1e-6f);
        float y[CPT];
#pragma unroll
        for (int j = 0; j < CPT; ++j) y[j] = (v[j] - mean) * rstd * gam[j] + bet[j];
        stage_split<CPT, kF16>(y, smem + SM::kOffLnHi, smem + SM::kOffLnLo, row, g, kLo);
        __syncthreads();
        if (ln_hi) tile_to_global<RB>(smem + SM::kOffLnHi, a.ln_out[0], (int64_t)n0 * 2, tr_rows, a.ln_row_off, 0, 0, tid);
        if (ln_lo) tile_to_global<RB>(smem + SM::kOffLnLo, a.ln_out[1], (int64_t)n0 * 2, tr_rows, a.ln_row_off, 0, 0, tid);
    }
    if (!ok && a.err) atomicExch(a.err, 1);
    tcgen05_fence_before();
    __syncthreads();
    if (tid == 0) tr.mark(3);
    if (warp == 1) tmem_dealloc(tmem, tmem_cols);
}

// ---- host side ------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// tensor [dims...] (dims[0] innermost, contiguous) of 2-byte (bf16) or 4-byte (fp32) elements, box per dim, zero OOB fill
bool tc_make_map_ex(CUtensorMap* out, const void* base, int elem_bytes, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, bool swizzle128) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return false;
    }
    cuuint64_t gd[5], gs[5];
    cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; ++i) gd[i] = dims[i], bx[i] = box[i], es[i] = 1;
    for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
    CUresult r = fn(out, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank,
                    const_cast<void*>(base), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu x %llu)", (int)r, rank, (unsigned long long)dims[0],
                  (unsigned long long)(rank > 1 ? dims[1] : 1));
        return false;
    }
    return true;
}
bool tc_make_map(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box) {
    return tc_make_map_ex(out, base, 2, rank, dims, strides_bytes, box, true);
}

bool tc_make_map_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    const uint64_t dims[2] = {cols, rows}, strides[1] = {cols * 2};
    const uint32_t box[2] = {(uint32_t)kTcBK, box_rows};
    return tc_make_map(out, base, 2, dims, strides, box);
}

// dense [planes][batch][heads][rows][cols] output of elem_bytes-wide elements (planes: split-K / chained partials)
TcOut tc_out(void* base, int elem_bytes, int64_t cols, int rows, int heads, int batch, int planes) {
    (void)planes;
    TcOut o;
    o.base = static_cast<uint8_t*>(base);
    o.row_bytes = cols * elem_bytes;
    o.rows = rows, o.heads = heads, o.batch = batch;
    o.plane_bytes = o.row_bytes * rows * heads * batch;
    return o;
}
// V^T output [batch][heads][64 d][tokens] bf16: rows = tokens (the range check), row_bytes = bytes of one d-row
TcOut tc_out_vt(void* base, int tokens, int heads, int batch) {
    TcOut o;
    o.base = static_cast<uint8_t*>(base);
    o.row_bytes = (int64_t)tokens * 2;
    o.rows = tokens, o.heads = heads, o.batch = batch, o.plane_bytes = 0;
    return o;
}
// flat [rows][cols] fp32 residual tile source (two 32-column boxes per 64-column tile)
bool tc_resid_map(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols) {
    const uint64_t dims[2] = {cols, rows}, strides[1] = {cols * 4};
    const uint32_t box[2] = {32, (uint32_t)kTcBM};
    return tc_make_map_ex(out, base, 4, 2, dims, strides, box, true);
}

// chained second GEMM of plan p: weights W2 [N2][K2] (K2 = N of the first GEMM), partial results P [N/64][batch][rows][N2] fp32
bool tc_plan_chain(TcGemmPlan* p, const __nv_bfloat16* W2hi, const __nv_bfloat16* W2lo, int N2, float* P, uint64_t rows, uint64_t batch) {
    if (N2 % 64 || N2 > kMaxChainN) {
        set_error("chained GEMM needs N2 %% 64 == 0 and N2 <= %d (N2=%d)", kMaxChainN, N2);
        return false;
    }
    const uint64_t K2 = (uint64_t)p->args.N;
    const uint64_t dims[2] = {K2, (uint64_t)N2}, strides[1] = {K2 * 2};
    const uint32_t box[2] = {(uint32_t)kTcBK, 64};  // loaded as 64-row boxes (a CTA of the sliced form takes one of them)
    bool ok = tc_make_map(&p->maps.B2hi, W2hi, 2, dims, strides, box) && tc_make_map(&p->maps.B2lo, W2lo ? W2lo : W2hi, 2, dims, strides, box);
    const uint32_t box_half[2] = {(uint32_t)kTcBK, (uint32_t)N2 / 2};  // one slice of the two-slice form of the 64-row tiles
    ok &= tc_make_map(&p->maps.B2hiHalf, W2hi, 2, dims, strides, box_half) && tc_make_map(&p->maps.B2loHalf, W2lo ? W2lo : W2hi, 2, dims, strides, box_half);
    p->args.p = tc_out(P, 4, N2, rows, 1, batch, K2 / kTcBN);
    p->args.chain_n = N2, p->args.o_mode = 3;
    return ok;
}

bool tc_plan_init(TcGemmPlan* p, const __nv_bfloat16* Ahi, const __nv_bfloat16* Alo, uint64_t a_rows, const __nv_bfloat16* Whi,
                  const __nv_bfloat16* Wlo, int N, int K, int conv_feat, int conv_batch) {
    memset(p, 0, sizeof(*p));
    if (N % kTcBN || K % kTcBK || (conv_feat && conv_feat % kTcBK)) {
        set_error("tcgen05 GEMM needs N %% 64 == 0 and K %% 64 == 0 (N=%d K=%d)", N, K);
        return false;
    }
    bool ok = true;
    if (conv_feat) {  // A = token grid [batch][16][16][feat]
        const uint64_t dims[4] = {(uint64_t)conv_feat, kMap, kMap, (uint64_t)conv_batch};
        const uint64_t strides[3] = {(uint64_t)conv_feat * 2, (uint64_t)conv_feat * 2 * kMap, (uint64_t)conv_feat * 2 * kMap * kMap};
        const uint32_t box[4] = {(uint32_t)kTcBK, kMap, kTcBM / kMap, 1};
        ok &= tc_make_map(&p->maps.Ahi, Ahi, 4, dims, strides, box);
        ok &= tc_make_map(&p->maps.Alo, Alo ? Alo : Ahi, 4, dims, strides, box);
        p->maps.Ahi64 = p->maps.Ahi, p->maps.Alo64 = p->maps.Alo;  // (no 64-row form)
    } else {
        ok &= tc_make_map_2d(&p->maps.Ahi, Ahi, a_rows, K, kTcBM);
        ok &= tc_make_map_2d(&p->maps.Alo, Alo ? Alo : Ahi, a_rows, K, kTcBM);
        ok &= tc_make_map_2d(&p->maps.Ahi64, Ahi, a_rows, K, 64);
        ok &= tc_make_map_2d(&p->maps.Alo64, Alo ? Alo : Ahi, a_rows, K, 64);
    }
    ok &= tc_make_map_2d(&p->maps.Bhi, Whi, N, K, kTcBN);
    ok &= tc_make_map_2d(&p->maps.Blo, Wlo ? Wlo : Whi, N, K, kTcBN);
    // unused output maps must still be valid descriptors (they are never dereferenced when their mode is off)
    p->maps.R = p->maps.B2hi = p->maps.B2lo = p->maps.B2hiHalf = p->maps.B2loHalf = p->maps.Bhi;
    p->args.N = N, p->args.K = K, p->args.conv_feat = conv_feat;
    p->args.pos_rows = 1, p->args.period = 1 << 30;
    return ok;
}

cudaError_t tc_gemm_setup() {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<1, kTcBM>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem<1>::kTotal);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<3, kTcBM>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem<3>::kTotal);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<2, kTcBM>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem<2>::kTotal);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<3, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem<3, 64>::kTotal);
    return e;
}

// the epilogues the 64-row kernel has: the QKV scatter and the chained FC1 with the hidden tile in tensor memory (bf16x3, N2 = 192)
bool tc_gemm_q64_supported(const TcGemmPlan& p, int nsplit) {
    const TcGemmArgs& a = p.args;
    if (nsplit != 3 || a.kb_per_split || a.conv_feat || a.ln_g || a.c_on || a.residual) return false;
    return (a.o_mode == 2 && !a.chain_n) || (a.o_mode == 3 && a.chain_n == kMaxChainN);
}

cudaError_t tc_gemm_launch(const TcGemmPlan& p, int M, int nsplit, cudaStream_t s, bool pdl, bool spread, bool q64) {
    if (M <= 0) return cudaSuccess;
    TcGemmArgs a = p.args;
    a.M = M;
    if (q64) {  // two replicas of every 64-row tile: hi / lo stores of the QKV scatter, or two slices of the chained product
        if (!spread || !tc_gemm_q64_supported(p, nsplit)) return cudaErrorInvalidValue;
        a.chain_slices = a.chain_n ? 2 : 0, a.dup_hl = a.chain_n ? 0 : 1, a.dup_ln = 0;
        const dim3 grid(a.N / kTcBN, (M + 63) / 64, 2);
        return launch_ex(gemm_tc_kernel<3, 64>, grid, dim3(kTcThreads), TcSmem<3, 64>::kTotal, s, pdl, 1, p.maps, a);
    }
    dim3 grid(a.N / kTcBN, (M + kTcBM - 1) / kTcBM, a.kb_per_split ? a.K / kTcBK / a.kb_per_split : 1);
    a.chain_slices = 0, a.dup_hl = 0, a.dup_ln = 0;
    if (spread && !a.kb_per_split && nsplit == 3 && a.ln_g && a.c_on && !a.chain_n && !a.o_mode && grid.x * grid.y * 3 <= (unsigned)kSpreadCtas)
        a.dup_ln = 1, grid.z = 3;  // three replicas of every tile: fp32 tile / LayerNorm hi / LayerNorm lo
    if (spread && !a.kb_per_split && nsplit == 3 && !a.chain_n && !a.ln_g && !a.c_on && (a.o_mode == 1 || a.o_mode == 2) &&
        grid.x * grid.y * 2 <= (unsigned)kSpreadCtas)
        a.dup_hl = 1, grid.z = 2;  // two replicas of every tile, one stores the hi parts and one the lo parts (halves the per-CTA egress)
    // latency mode: replicate the FC1 tiles over idle SMs, each replica computes and stores one 64-column slice of the chained product
    if (spread && !a.kb_per_split && a.chain_n && a.chain_n % (3 * 64) == 0 && grid.x * grid.y * 3 <= (unsigned)kSpreadCtas) a.chain_slices = 3, grid.z = 3;
    // fused LayerNorm: the N / 64 column tiles of a row tile form one cluster
    const int cluster_x = a.ln_g ? a.N / kTcBN : 1;
    if (cluster_x > kMaxLnCluster) return cudaErrorInvalidValue;
    if (nsplit == 2) return launch_ex(gemm_tc_kernel<2, kTcBM>, grid, dim3(kTcThreads), TcSmem<2>::kTotal, s, pdl, cluster_x, p.maps, a);
    if (nsplit == 3) return launch_ex(gemm_tc_kernel<3, kTcBM>, grid, dim3(kTcThreads), TcSmem<3>::kTotal, s, pdl, cluster_x, p.maps, a);
    return launch_ex(gemm_tc_kernel<1, kTcBM>, grid, dim3(kTcThreads), TcSmem<1>::kTotal, s, pdl, cluster_x, p.maps, a);
}

// fp32 -> bf16 (hi, lo) split of a dense buffer
// lo == nullptr: single-pass fp16 operands (hi holds fp16 values)
__global__ void split_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        if (!lo) {
            reinterpret_cast<unsigned short*>(hi)[i] = half_bits(x[i], true);
            continue;
        }
        __nv_bfloat16 h, l;
        split_bf16(x[i], h, l);
        hi[i] = h, lo[i] = l;
    }
}
cudaError_t launch_split_bf16(const float* x, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t n, cudaStream_t s) {
    if (!n) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    split_bf16_kernel<<<(unsigned)blocks, 256, 0, s>>>(x, hi, lo, n);
    return cudaGetLastError();
}

}  // namespace vt

// ---- diagnostics entry: one GEMM on host data through the tensor-core kernel (unit tests) -----------------------------------
extern "C" vt_status vt_debug_gemm(int32_t device, int32_t M, int32_t N, int32_t K, const float* A, const float* W, const float* bias,
                                   int32_t nsplit, int32_t gelu, float* C_out, int32_t* err_out) {
    using namespace vt;
    if (!A || !W || !C_out || M <= 0 || nsplit < 1 || nsplit > 3) return VT_ERR_INVALID;  // 1 bf16, 2 fp16, 3 bf16 hi + lo
    VT_CUDA(cudaSetDevice(device));
    VT_CUDA(tc_gemm_setup());
    float *dA = nullptr, *dW = nullptr, *dB = nullptr, *dC = nullptr;
    __nv_bfloat16 *Ahi = nullptr, *Alo = nullptr, *Whi = nullptr, *Wlo = nullptr;
    int* dErr = nullptr;
    const size_t na = (size_t)M * K, nw = (size_t)N * K;
    VT_CUDA(cudaMalloc(&dA, na * 4)); VT_CUDA(cudaMalloc(&dW, nw * 4)); VT_CUDA(cudaMalloc(&dC, (size_t)M * N * 4));
    VT_CUDA(cudaMalloc(&Ahi, na * 2)); VT_CUDA(cudaMalloc(&Alo, na * 2)); VT_CUDA(cudaMalloc(&Whi, nw * 2)); VT_CUDA(cudaMalloc(&Wlo, nw * 2));
    VT_CUDA(cudaMalloc(&dErr, 4)); VT_CUDA(cudaMemset(dErr, 0, 4));
    VT_CUDA(cudaMemcpy(dA, A, na * 4, cudaMemcpyHostToDevice)); VT_CUDA(cudaMemcpy(dW, W, nw * 4, cudaMemcpyHostToDevice));
    if (bias) {
        VT_CUDA(cudaMalloc(&dB, (size_t)N * 4));
        VT_CUDA(cudaMemcpy(dB, bias, (size_t)N * 4, cudaMemcpyHostToDevice));
    }
    VT_CUDA(cudaMemset(dC, 0, (size_t)M * N * 4));
    VT_CUDA(launch_split_bf16(dA, Ahi, nsplit == 2 ? nullptr : Alo, na, 0)); VT_CUDA(launch_split_bf16(dW, Whi, nsplit == 2 ? nullptr : Wlo, nw, 0));
    TcGemmPlan plan;
    vt_status st = VT_OK;
    if (!tc_plan_init(&plan, Ahi, Alo, M, Whi, Wlo, N, K, 0, 0)) st = VT_ERR_CUDA;
    if (st == VT_OK) {
        plan.args.bias = dB, plan.args.gelu = gelu, plan.args.err = dErr, plan.args.c_on = 1;
        plan.args.c = tc_out(dC, 4, N, M, 1, 1, 1);
    }
    if (st == VT_OK) {
        cudaError_t e = tc_gemm_launch(plan, M, nsplit, 0, false);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            set_error("tcgen05 GEMM failed: %s", cudaGetErrorString(e));
            st = VT_ERR_CUDA;
        }
    }
    if (st == VT_OK) {
        VT_CUDA(cudaMemcpy(C_out, dC, (size_t)M * N * 4, cudaMemcpyDeviceToHost));
        int herr = 0;
        VT_CUDA(cudaMemcpy(&herr, dErr, 4, cudaMemcpyDeviceToHost));
        if (err_out) *err_out = herr;
    }
    cudaFree(dA), cudaFree(dW), cudaFree(dB), cudaFree(dC), cudaFree(Ahi), cudaFree(Alo), cudaFree(Whi), cudaFree(Wlo), cudaFree(dErr);
    return st;
}
