// vit.cu — fp32 CUDA-core kernels of the ViT forward pass and the score-map decode.
//
// These are the numerically-anchoring kernels (fp32 everywhere, oracle-order accumulation
// where it matters).  The tensor-core path (gemm_tcgen05.cu) replaces launch_gemm_simt for the
// dense contractions; LayerNorm / attention softmax / decode stay as warp-shuffle kernels.
// Replaces VitTrack::update's network + decode (call site /root/reference/src/tracker_context.rs:120;
// algorithm: OpenCV TrackerVit, SURVEY.md Appendix A.5-A.6).
#include "vt_internal.h"

namespace vt {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }

// ------------------------------------------------------------------------------------------------
// GEMM  C[M,N] = epi( pro(A)[M,K] * W[N,K]^T + bias )       (fp32 SIMT, BK = 32)
// ------------------------------------------------------------------------------------------------
constexpr int kBK = 32;

__device__ __forceinline__ int map_row(int m, int rows_in, int rows_stride, int row_off) {
    return (m / rows_in) * rows_stride + row_off + (m % rows_in);
}

template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__(256) gemm_simt_kernel(GemmArgs g) {
    static_assert((BM / TM) * (BN / TN) == 256, "256 threads");
    __shared__ float As[kBK][BM + 4];
    __shared__ float Ws[kBK][BN + 4];
    __shared__ float s_mean[BM], s_rstd[BM];

    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);

    // LayerNorm statistics of this CTA's rows (two-pass, like the oracle)
    if (g.ln_g) {
        const int warp = tid >> 5, lane = tid & 31;
        for (int r = warp; r < BM; r += 8) {
            const int m = m0 + r;
            float mean = 0.f, rstd = 0.f;
            if (m < g.M) {
                const float* a = g.A + (int64_t)map_row(m, g.a_rows_in, g.a_rows_stride, g.a_row_off) * g.lda;
                float s = 0.f;
                for (int k = lane; k < g.K; k += 32) s += a[k];
                mean = warp_sum(s) / (float)g.K;
                float v = 0.f;
                for (int k = lane; k < g.K; k += 32) {
                    const float d = a[k] - mean;
                    v += d * d;
                }
                v = warp_sum(v) / (float)g.K;
                rstd = 1.f / sqrtf(v + 1e-6f);
            }
            if (lane == 0) s_mean[r] = mean, s_rstd[r] = rstd;
        }
        __syncthreads();
    }

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < g.K; k0 += kBK) {
        // ---- A tile -> As[k][m]
        for (int v = tid; v < BM * (kBK / 4); v += 256) {
            const int r = v / (kBK / 4), kq = (v % (kBK / 4)) * 4;
            const int m = m0 + r;
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m < g.M) {
                if (g.im2col_feat) {
                    const int feat = g.im2col_feat;
                    const int tap = k0 / feat, d0 = k0 % feat;
                    const int p = m % g.a_rows_in, b = m / g.a_rows_in;
                    const int yy = p / kMap + tap / 3 - 1, xx = p % kMap + tap % 3 - 1;
                    if (yy >= 0 && yy < kMap && xx >= 0 && xx < kMap)
                        a = *reinterpret_cast<const float4*>(g.A + (int64_t)(b * g.a_rows_stride + g.a_row_off + yy * kMap + xx) * g.lda + d0 + kq);
                } else {
                    a = *reinterpret_cast<const float4*>(g.A + (int64_t)map_row(m, g.a_rows_in, g.a_rows_stride, g.a_row_off) * g.lda + k0 + kq);
                    if (g.ln_g) {
                        const float mu = s_mean[r], rs = s_rstd[r];
                        const float4 gg = *reinterpret_cast<const float4*>(g.ln_g + k0 + kq);
                        const float4 bb = *reinterpret_cast<const float4*>(g.ln_b + k0 + kq);
                        a.x = (a.x - mu) * rs * gg.x + bb.x;
                        a.y = (a.y - mu) * rs * gg.y + bb.y;
                        a.z = (a.z - mu) * rs * gg.z + bb.z;
                        a.w = (a.w - mu) * rs * gg.w + bb.w;
                    }
                }
            }
            As[kq + 0][r] = a.x, As[kq + 1][r] = a.y, As[kq + 2][r] = a.z, As[kq + 3][r] = a.w;
        }
        // ---- W tile -> Ws[k][n]
        for (int v = tid; v < BN * (kBK / 4); v += 256) {
            const int r = v / (kBK / 4), kq = (v % (kBK / 4)) * 4;
            const int n = n0 + r;
            float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n < g.N) w = *reinterpret_cast<const float4*>(g.W + (int64_t)n * g.K + k0 + kq);
            Ws[kq + 0][r] = w.x, Ws[kq + 1][r] = w.y, Ws[kq + 2][r] = w.z, Ws[kq + 3][r] = w.w;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kBK; ++kk) {
            float a[TM], w[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; ++j) w[j] = Ws[kk][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int m = m0 + ty * TM + i;
        if (m >= g.M) continue;
        const int64_t row = (int64_t)map_row(m, g.c_rows_in, g.c_rows_stride, g.c_row_off) * g.ldc;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int n = n0 + tx * TN + j;
            if (n >= g.N) continue;
            float v = acc[i][j] + (g.bias ? g.bias[n] : 0.f);
            if (g.gelu) v = gelu_exact(v);
            if (g.relu) v = fmaxf(v, 0.f);
            if (g.pos) v += g.pos[(int64_t)(m % g.c_rows_in) * g.N + n];
            if (g.residual) v += g.C[row + n];
            g.C[row + n] = v;
        }
    }
}

cudaError_t launch_gemm_simt(const GemmArgs& g, cudaStream_t s) {
    if (g.M <= 0 || g.N <= 0) return cudaSuccess;
    if (g.K % kBK != 0 || (g.im2col_feat && g.im2col_feat % kBK != 0)) return cudaErrorInvalidValue;
    // pick the tile that gives the most CTAs up to ~2 waves of 148 SMs
    const long long ctas64 = (long long)((g.M + 63) / 64) * ((g.N + 63) / 64);
    const long long ctas32x64 = (long long)((g.M + 31) / 32) * ((g.N + 63) / 64);
    if (ctas64 >= 296) {
        dim3 grid((g.N + 63) / 64, (g.M + 63) / 64);
        gemm_simt_kernel<64, 64, 4, 4><<<grid, 256, 0, s>>>(g);
    } else if (ctas32x64 >= 148) {
        dim3 grid((g.N + 63) / 64, (g.M + 31) / 32);
        gemm_simt_kernel<32, 64, 2, 4><<<grid, 256, 0, s>>>(g);
    } else {
        dim3 grid((g.N + 31) / 32, (g.M + 31) / 32);
        gemm_simt_kernel<32, 32, 2, 2><<<grid, 256, 0, s>>>(g);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// LayerNorm, one warp per row (two-pass statistics, eps 1e-6)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ g,
                                                        const float* __restrict__ b, float* __restrict__ y, int64_t ldy, int M, int D,
                                                        int rows_in, int rows_stride, int row_off) {
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (m >= M) return;
    const float* r = x + (int64_t)map_row(m, rows_in, rows_stride, row_off) * ldx;
    float s = 0.f;
    for (int k = lane; k < D; k += 32) s += r[k];
    const float mean = warp_sum(s) / (float)D;
    float v = 0.f;
    for (int k = lane; k < D; k += 32) {
        const float d = r[k] - mean;
        v += d * d;
    }
    const float rstd = 1.f / sqrtf(warp_sum(v) / (float)D + 1e-6f);
    for (int k = lane; k < D; k += 32) y[(int64_t)m * ldy + k] = (r[k] - mean) * rstd * g[k] + b[k];
}

cudaError_t launch_layernorm(const float* x, int64_t ldx, const float* g, const float* b, float* y, int64_t ldy, int M, int D,
                             int rows_in, int rows_stride, int row_off, cudaStream_t s) {
    if (M <= 0) return cudaSuccess;
    layernorm_kernel<<<(M + 7) / 8, 256, 0, s>>>(x, ldx, g, b, y, ldy, M, D, rows_in, rows_stride, row_off);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) layernorm_split_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ g,
                                                              const float* __restrict__ b, __nv_bfloat16* __restrict__ hi,
                                                              __nv_bfloat16* __restrict__ lo, int M, int D, int rows_in, int rows_stride,
                                                              int row_off) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (m >= M) return;
    const float* r = x + (int64_t)map_row(m, rows_in, rows_stride, row_off) * ldx;
    float s = 0.f;
    for (int k = lane; k < D; k += 32) s += r[k];
    const float mean = warp_sum(s) / (float)D;
    float v = 0.f;
    for (int k = lane; k < D; k += 32) {
        const float d = r[k] - mean;
        v += d * d;
    }
    const float rstd = 1.f / sqrtf(warp_sum(v) / (float)D + 1e-6f);
    for (int k = lane; k < D; k += 32) {
        const float y = (r[k] - mean) * rstd * g[k] + b[k];
        if (!lo) {  // single-pass fp16 operands
            reinterpret_cast<unsigned short*>(hi)[(int64_t)m * D + k] = operand_bits(y, true);
            continue;
        }
        const __nv_bfloat16 h = __float2bfloat16_rn(y);
        hi[(int64_t)m * D + k] = h;
        lo[(int64_t)m * D + k] = __float2bfloat16_rn(y - __bfloat162float(h));
    }
}

cudaError_t launch_layernorm_split(const float* x, int64_t ldx, const float* g, const float* b, __nv_bfloat16* hi, __nv_bfloat16* lo, int M,
                                   int D, int rows_in, int rows_stride, int row_off, cudaStream_t s, bool pdl) {
    if (M <= 0) return cudaSuccess;
    return launch_ex(layernorm_split_kernel, dim3((M + 7) / 8), dim3(256), 0, s, pdl, 1, x, ldx, g, b, hi, lo, M, D, rows_in, rows_stride, row_off);
}

// ------------------------------------------------------------------------------------------------
// Sum of the split partial GEMM results + bias + addend (residual / pos-embed), fused with the following LayerNorm
// (ReduceLnArgs in vt_internal.h).  One warp per row; lane l owns the column pairs 2 l + 64 i: every partial row is read with
// fully coalesced 8-byte loads, all issued before the first add (one L2 round trip).  The partials are added in index order,
// so the result does not depend on scheduling.
// ------------------------------------------------------------------------------------------------
// Rows (= warps) per CTA.  (Measured: 2 rows per CTA — 160 CTAs instead of 40 for one target — changes nothing; the kernel is bound by
// the L2 round trips of its dependent loads, not by the per-SM read rate.)
constexpr int kReduceRows = 8;
// FRONT (latency mode: the GPU is otherwise idle): every partial-plane load ahead of the first add, see below.  Not in throughput mode:
// there the 110 registers per thread of the 12-plane form cost more resident CTAs than the shorter latency gains (cfg5 -2 %).
template <int NPAIR, int NP, bool FRONT>  // D / 64 column pairs per lane; number of partials (0 = runtime np, batches of 4)
__global__ void __launch_bounds__(32 * kReduceRows) reduce_ln_kernel(const ReduceLnArgs a) {
    constexpr int D = NPAIR * 64;
    const int m = blockIdx.x * kReduceRows + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (m >= a.M) return;
    const int b = m / a.period, t = m - b * a.period;
    const int64_t xrow = (int64_t)b * a.x_rows + t + a.x_row_off;
    const float2* ar = reinterpret_cast<const float2*>(a.add + (a.add_period ? (int64_t)(m % a.add_period) : xrow) * D);
    // LayerNorm gain / bias are fetched with the first batch of loads: a late __ldg would add an L2 round trip behind the reductions.
    // (Measured: issuing the parameter loads BEFORE griddepcontrol.wait makes the kernel 0.7 us slower, so they stay behind it.)
    float2 acc[NPAIR], gam[NPAIR], bet[NPAIR], x2[NPAIR];
#pragma unroll
    for (int i = 0; i < NPAIR; ++i) {
        acc[i] = __ldg(reinterpret_cast<const float2*>(a.bias) + lane + 32 * i), x2[i] = __ldcg(ar + lane + 32 * i);
        gam[i] = __ldg(reinterpret_cast<const float2*>(a.ln_g) + lane + 32 * i), bet[i] = __ldg(reinterpret_cast<const float2*>(a.ln_b) + lane + 32 * i);
    }
    const float2* pr = reinterpret_cast<const float2*>(a.P + (int64_t)m * D);
    const int64_t ps = a.p_stride / 2;
    if (NP > 0) {
        float2 v[NP > 0 ? NP : 1][NPAIR];
#pragma unroll
        for (int j = 0; j < NP; ++j)
#pragma unroll
            for (int i = 0; i < NPAIR; ++i) v[j][i] = __ldcg(pr + j * ps + lane + 32 * i);  // L2 loads: the partials were written by other SMs a moment ago
        // The fence keeps every load above ahead of the first add (ptxas may not sink a load below it).  Without it ptxas (40
        // registers) interleaves the loads with the in-order adds and has only ~12 of the 48 loads of the 12-plane reduce in flight:
        // several dependent L2 round trips instead of one.  (The adds need every load anyway, so waiting for them at the fence costs nothing.)
        if (FRONT) __threadfence_block();
#pragma unroll
        for (int i = 0; i < NPAIR; ++i) acc[i].x = x2[i].x + acc[i].x, acc[i].y = x2[i].y + acc[i].y;  // (x + bias) first, as before
#pragma unroll
        for (int j = 0; j < NP; ++j)
#pragma unroll
            for (int i = 0; i < NPAIR; ++i) acc[i].x += v[j][i].x, acc[i].y += v[j][i].y;
    } else {
#pragma unroll
        for (int i = 0; i < NPAIR; ++i) acc[i].x = x2[i].x + acc[i].x, acc[i].y = x2[i].y + acc[i].y;
        for (int j0 = 0; j0 < a.np; j0 += 4) {
            float2 v[4][NPAIR];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                for (int i = 0; i < NPAIR; ++i) v[jj][i] = j0 + jj < a.np ? __ldcg(pr + (j0 + jj) * ps + lane + 32 * i) : make_float2(0.f, 0.f);
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                for (int i = 0; i < NPAIR; ++i) acc[i].x += v[jj][i].x, acc[i].y += v[jj][i].y;
        }
    }
    float2* xw = reinterpret_cast<float2*>(a.X + xrow * D);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NPAIR; ++i) xw[lane + 32 * i] = acc[i], s += acc[i].x + acc[i].y;
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NPAIR; ++i) {
        const float dx = acc[i].x - mean, dy = acc[i].y - mean;
        q += dx * dx + dy * dy;
    }
    const float rstd = 1.f / sqrtf(warp_sum(q) / (float)D + 1e-6f);
    if (t + a.ln_row_off < 0) return;
    const int64_t orow = (int64_t)b * a.ln_rows + t + a.ln_row_off;
    uint32_t* oh = reinterpret_cast<uint32_t*>(a.ln_hi + orow * D);
    uint32_t* ol = reinterpret_cast<uint32_t*>(a.ln_lo + orow * D);
#pragma unroll
    for (int i = 0; i < NPAIR; ++i) {
        const float2 g2 = gam[i], b2 = bet[i];
        const float y0 = (acc[i].x - mean) * rstd * g2.x + b2.x, y1 = (acc[i].y - mean) * rstd * g2.y + b2.y;
        // packed cvt.rn.bf16x2 (bit-identical to two scalar splits; the scalar conversion runs on the slow 16/clk pipe)
        uint32_t h2, l2;
        if (!a.ln_lo) {  // single-pass fp16 operands
            asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(h2) : "f"(y1), "f"(y0));
            oh[lane + 32 * i] = h2;
            continue;
        }
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h2) : "f"(y1), "f"(y0));
        const float r0 = y0 - __uint_as_float(h2 << 16), r1 = y1 - __uint_as_float(h2 & 0xffff0000u);
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(l2) : "f"(r1), "f"(r0));
        oh[lane + 32 * i] = h2;
        ol[lane + 32 * i] = l2;
    }
}

cudaError_t launch_reduce_ln(const ReduceLnArgs& a, cudaStream_t s, bool pdl, bool front) {
    if (a.M <= 0) return cudaSuccess;
    const dim3 grid((a.M + kReduceRows - 1) / kReduceRows), block(32 * kReduceRows);
#define VT_RL(NPAIR_, NP_) return front ? launch_ex(reduce_ln_kernel<NPAIR_, NP_, true>, grid, block, 0, s, pdl, 1, a) \
                                   : launch_ex(reduce_ln_kernel<NPAIR_, NP_, false>, grid, block, 0, s, pdl, 1, a)
    switch (a.D / 64) {
        case 1:
            if (a.np == 4) VT_RL(1, 4);
            VT_RL(1, 0);
        case 2: VT_RL(2, 0);
        case 3:
            if (a.np == 12) VT_RL(3, 12);
            if (a.np == 4) VT_RL(3, 4);
            if (a.np == 3) VT_RL(3, 3);  // per-head partial proj products of the chained attention form
            VT_RL(3, 0);
        default: return cudaErrorInvalidValue;
    }
#undef VT_RL
}

// ------------------------------------------------------------------------------------------------
// Attention over the joint 320-token sequence: one CTA per (16-query tile, head, target).
// scores -> shared memory, warp-shuffle softmax, P*V from shared memory.
// ------------------------------------------------------------------------------------------------
constexpr int kBQ = 16, kKT = 64;

template <int DH>
__global__ void __launch_bounds__(128) attention_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                        __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, int D) {
    __shared__ float Qs[kBQ][DH];
    __shared__ float S[kBQ][kNTok];
    __shared__ float KV[kKT][DH + 1];
    const int tid = threadIdx.x, q0 = blockIdx.x * kBQ, h = blockIdx.y, b = blockIdx.z;
    const int64_t ld = 3 * (int64_t)D;
    const float* base = qkv + (int64_t)b * kNTok * ld + h * DH;
    const float scale = 1.f / sqrtf((float)DH);

    for (int i = tid; i < kBQ * DH; i += 128) Qs[i / DH][i % DH] = base[(int64_t)(q0 + i / DH) * ld + i % DH];

    // scores
    for (int kt = 0; kt < kNTok; kt += kKT) {
        __syncthreads();
        for (int i = tid; i < kKT * DH; i += 128) KV[i / DH][i % DH] = base[(int64_t)(kt + i / DH) * ld + D + i % DH];
        __syncthreads();
        const int j = tid % kKT, qh = tid / kKT;  // 2 groups of 8 queries
#pragma unroll
        for (int qi = 0; qi < 8; ++qi) {
            const int q = qh * 8 + qi;
            float acc = 0.f;
#pragma unroll
            for (int d = 0; d < DH; ++d) acc = fmaf(Qs[q][d], KV[j][d], acc);
            S[q][kt + j] = acc * scale;
        }
    }
    __syncthreads();
    // softmax: warp w owns rows 4w..4w+3
    {
        const int warp = tid >> 5, lane = tid & 31;
        for (int q = warp * 4; q < warp * 4 + 4; ++q) {
            float mx = -INFINITY;
            for (int j = lane; j < kNTok; j += 32) mx = fmaxf(mx, S[q][j]);
            mx = warp_max(mx);
            float sum = 0.f;
            for (int j = lane; j < kNTok; j += 32) {
                const float e = expf(S[q][j] - mx);
                S[q][j] = e;
                sum += e;
            }
            const float inv = 1.f / warp_sum(sum);
            for (int j = lane; j < kNTok; j += 32) S[q][j] *= inv;
        }
    }
    // O = P V
    constexpr int kGroups = 128 / DH, kQPer = kBQ / kGroups;
    const int d = tid % DH, qg = tid / DH;
    float o[kQPer];
#pragma unroll
    for (int i = 0; i < kQPer; ++i) o[i] = 0.f;
    for (int kt = 0; kt < kNTok; kt += kKT) {
        __syncthreads();
        for (int i = tid; i < kKT * DH; i += 128) KV[i / DH][i % DH] = base[(int64_t)(kt + i / DH) * ld + 2 * D + i % DH];
        __syncthreads();
        for (int j = 0; j < kKT; ++j) {
            const float v = KV[j][d];
#pragma unroll
            for (int i = 0; i < kQPer; ++i) o[i] = fmaf(S[qg * kQPer + i][kt + j], v, o[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < kQPer; ++i) {
        const int64_t idx = ((int64_t)b * kNTok + q0 + qg * kQPer + i) * D + h * DH + d;
        if (out) out[idx] = o[i];
        if (out_hi) {
            if (!out_lo) {  // single-pass fp16 operands
                reinterpret_cast<unsigned short*>(out_hi)[idx] = operand_bits(o[i], true);
                continue;
            }
            const __nv_bfloat16 hh = __float2bfloat16_rn(o[i]);
            out_hi[idx] = hh;
            out_lo[idx] = __float2bfloat16_rn(o[i] - __bfloat162float(hh));
        }
    }
}

cudaError_t launch_attention(const float* qkv, float* out, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, int B, int D, int heads,
                             cudaStream_t s) {
    if (B <= 0) return cudaSuccess;
    const int dh = D / heads;
    dim3 grid(kNTok / kBQ, heads, B);
    switch (dh) {
        case 16: attention_kernel<16><<<grid, 128, 0, s>>>(qkv, out, out_hi, out_lo, D); break;
        case 32: attention_kernel<32><<<grid, 128, 0, s>>>(qkv, out, out_hi, out_lo, D); break;
        case 64: attention_kernel<64><<<grid, 128, 0, s>>>(qkv, out, out_hi, out_lo, D); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

__device__ void decode_finish(TargetState* st, int slot, float threshold, float score, int best, float ox, float oy, float bw, float bh,
                              DeviceResult* res, int decode_window, const int* tc_err);

// ------------------------------------------------------------------------------------------------
// K8 decode: 1x1 conv -> sigmoid -> hann window -> first-maximum argmax -> bbox (App. A.5-A.6).
// One CTA (256 threads = 256 map cells) per target; the winning cell is found with a
// warp-shuffle (value, index) reduction; thread 0 updates rect_last on the device so the next
// frame's crop needs no host round trip.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) decode_kernel(const float* __restrict__ h1, int C, const float* __restrict__ w2,
                                                     const float* __restrict__ b2, const float* __restrict__ hann,
                                                     TargetState* __restrict__ state, const int32_t* __restrict__ slots, float threshold,
                                                     DeviceResult* __restrict__ res, float* __restrict__ maps, unsigned long long* stamps,
                                                     int decode_window) {
    if (stamps && threadIdx.x == 0 && blockIdx.x == 0) stamps[ST_DEC] = device_time_ns();
    __shared__ float s_val[8];
    __shared__ int s_idx[8];
    __shared__ float s_out[4];
    __shared__ float tile[kNTx][33];   // 32-channel slab of the head features, padded: conflict-free row reads
    __shared__ float w2s[5][32];
    const int bi = blockIdx.x, slot = slots[bi], p = threadIdx.x;
    const float* f = h1 + (int64_t)bi * kNTx * C;
    float o[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) o[k] = b2[k];
    for (int c0 = 0; c0 < C; c0 += 32) {
        __syncthreads();
        for (int i = p; i < kNTx * 32; i += 256) tile[i >> 5][i & 31] = f[(int64_t)(i >> 5) * C + c0 + (i & 31)];  // coalesced 128-byte rows
        if (p < 160) w2s[p >> 5][p & 31] = w2[(p >> 5) * C + c0 + (p & 31)];
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const float x = tile[p][j];
#pragma unroll
            for (int k = 0; k < 5; ++k) o[k] = __fadd_rn(o[k], __fmul_rn(x, w2s[k][j]));  // oracle order (c ascending), unfused
        }
    }
    const float conf = 1.f / (1.f + expf(-o[0]));
    const float sw = 1.f / (1.f + expf(-o[1])), sh = 1.f / (1.f + expf(-o[2]));
    const float cw = __fmul_rn(conf, hann[p]);
    float* m = maps + (int64_t)slot * 1280;
    m[p] = cw, m[256 + p] = sw, m[512 + p] = sh, m[768 + p] = o[3], m[1024 + p] = o[4];

    // first row-major maximum
    float bv = cw;
    int bidx = p;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
        if (ov > bv || (ov == bv && oi < bidx)) bv = ov, bidx = oi;
    }
    if ((p & 31) == 0) s_val[p >> 5] = bv, s_idx[p >> 5] = bidx;
    __syncthreads();
    if (p < 32) {
        bv = p < 8 ? s_val[p] : -INFINITY;
        bidx = p < 8 ? s_idx[p] : 0x7fffffff;
#pragma unroll
        for (int off = 4; off > 0; off >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
            if (ov > bv || (ov == bv && oi < bidx)) bv = ov, bidx = oi;
        }
        if (p == 0) s_idx[0] = bidx, s_val[0] = bv;
    }
    __syncthreads();
    const int best = s_idx[0];
    if (p == best) s_out[0] = o[3], s_out[1] = o[4], s_out[2] = sw, s_out[3] = sh;
    __syncthreads();
    if (p == 0) {
        decode_finish(state + slot, slot, threshold, s_val[0], best, s_out[0], s_out[1], s_out[2], s_out[3], res, decode_window, nullptr);
        if (stamps && blockIdx.x == 0) stamps[ST_DEC_END] = device_time_ns();
    }
}

// rect_last update + result record from the winning cell (App. A.6); shared by both decode kernels.
// decode_window (App. A.7): 0 = the crop's own c = ceil(sqrt(w*h)*4) (OpenCV 4.13), 1 = 4*floor(sqrt(w*h)) (older OpenCV).
// tc_err: the tensor-core kernels' error flag of this frame — an expired pipeline wait means the maps are garbage: the frame is reported
// as failed by wait() and rect_last must keep the last good box.
__device__ void decode_finish(TargetState* st, int slot, float threshold, float score, int best, float ox, float oy, float bw, float bh,
                              DeviceResult* res, int decode_window, const int* tc_err) {
    DeviceResult r;
    r.success = 0, r.score = 0.f, r.bbox[0] = r.bbox[1] = r.bbox[2] = r.bbox[3] = 0, r.best = best;
    r.status = VT_OK;
    if (!st->active) {
        r.status = VT_ERR_NOT_INIT;
    } else if (st->crop_err) {
        r.status = VT_ERR_CROP_OUTSIDE;
    } else {
        r.score = score;
        if (r.score >= threshold) {
            const int my = best / kMap, mx = best % kMap;
            const float cx = __fdiv_rn(__fadd_rn((float)mx, ox), 16.f);
            const float cy = __fdiv_rn(__fadd_rn((float)my, oy), 16.f);
            const int lx = st->rect[0], ly = st->rect[1], lw = st->rect[2], lh = st->rect[3];
            const double sq = sqrt((double)((long long)lw * lh));
            const int cwin = decode_window ? 4 * (int)floor(sq) : (int)ceil(__dmul_rn(sq, 4.0));
            const int x0 = lx + (lw - cwin) / 2, y0 = ly + (lh - cwin) / 2;
            const float fc = (float)cwin;
            r.bbox[0] = (int)floorf(__fadd_rn(__fmul_rn(__fsub_rn(cx, __fdiv_rn(bw, 2.f)), fc), (float)x0));
            r.bbox[1] = (int)floorf(__fadd_rn(__fmul_rn(__fsub_rn(cy, __fdiv_rn(bh, 2.f)), fc), (float)y0));
            r.bbox[2] = (int)floorf(__fmul_rn(bw, fc));
            r.bbox[3] = (int)floorf(__fmul_rn(bh, fc));
            r.success = 1;
            if (!(tc_err && *reinterpret_cast<const volatile int*>(tc_err)))
                st->rect[0] = r.bbox[0], st->rect[1] = r.bbox[1], st->rect[2] = r.bbox[2], st->rect[3] = r.bbox[3];
        }
    }
    res[slot] = r;
}

// ------------------------------------------------------------------------------------------------
// K7b + K8 for the tensor-core path: the 3x3 head conv arrives as one fp32 partial per tap (split-K GEMM); this kernel sums
// them (+ bias, ReLU), applies the 1x1 conv, sigmoid and hann window and finds the first row-major maximum.
// grid (16 map rows, targets) x 256 threads: warp w owns cells 2w, 2w+1 of the row, lane l owns channels CPL l .. CPL l + CPL - 1
// (coalesced 16-byte loads, every partial of a cell in flight at once); the 1x1 conv is a warp-shuffle reduction.
// The 16 row candidates of a target are merged by the last CTA to arrive (atomic ticket), in row order -> deterministic.
// ------------------------------------------------------------------------------------------------
template <int N> struct VecOf;
template <> struct VecOf<4> { typedef float4 type; };
template <> struct VecOf<2> { typedef float2 type; };
constexpr int kCandStride = 8;  // floats per row candidate: value, index, off_x, off_y, size_w, size_h
template <int CPL, int NP, bool FRONT>  // channels per lane: head_ch / 32; taps (0 = runtime np, three in flight); FRONT: as reduce_ln_kernel
__global__ void __launch_bounds__(256) head_decode_kernel(const float* __restrict__ P, int np, int64_t p_stride, const float* __restrict__ b1,
                                                          const float* __restrict__ w2, const float* __restrict__ b2,
                                                          const float* __restrict__ hann, TargetState* __restrict__ state,
                                                          const int32_t* __restrict__ slots, float threshold, DeviceResult* __restrict__ res,
                                                          float* __restrict__ maps, float* cand, unsigned* counters, unsigned long long* stamps,
                                                          int decode_window, const int* tc_err) {
    constexpr int C = CPL * 32;
    __shared__ float s_c[16][6];
    __shared__ int s_last;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (stamps && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) stamps[ST_DEC] = device_time_ns();
    const int bi = blockIdx.y, y = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Every load this CTA needs is issued in ONE batch (parameters, hann weights, all taps of both cells): the kernel is a chain of L2
    // round trips (~0.7 us each), not of bytes, so nothing is fetched behind a reduction.
    const int slot = slots[bi];
    float w[5][CPL], bch[CPL], b2v[5], hw[2];
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
        bch[c] = __ldg(b1 + lane * CPL + c);
#pragma unroll
        for (int k = 0; k < 5; ++k) w[k][c] = __ldg(w2 + k * C + lane * CPL + c);
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) b2v[k] = __ldg(b2 + k);
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) hw[cc] = __ldg(hann + y * kMap + 2 * warp + cc);
    using Vec = typename VecOf<CPL>::type;  // float4 / float2: one coalesced load per lane and partial
    float hsum[2][CPL];
    if (NP > 0) {
        Vec v[2][NP > 0 ? NP : 1];
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            const float* pr = P + ((int64_t)bi * kNTx + y * kMap + 2 * warp + cc) * C + lane * CPL;
#pragma unroll
            for (int j = 0; j < NP; ++j) v[cc][j] = *reinterpret_cast<const Vec*>(pr + (int64_t)j * p_stride);
        }
        if (FRONT) __threadfence_block();  // every tap load ahead of the first add (as in reduce_ln_kernel)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
#pragma unroll
            for (int c = 0; c < CPL; ++c) hsum[cc][c] = bch[c];
#pragma unroll
            for (int j = 0; j < NP; ++j)  // taps in index order, as the runtime form
#pragma unroll
                for (int c = 0; c < CPL; ++c) hsum[cc][c] += reinterpret_cast<const float*>(&v[cc][j])[c];
        }
    } else {
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            const float* pr = P + ((int64_t)bi * kNTx + y * kMap + 2 * warp + cc) * C + lane * CPL;
#pragma unroll
            for (int c = 0; c < CPL; ++c) hsum[cc][c] = bch[c];
            for (int j0 = 0; j0 < np; j0 += 3) {  // three taps (one kernel row) in flight per cell
                Vec v[3];
#pragma unroll
                for (int jj = 0; jj < 3; ++jj) v[jj] = j0 + jj < np ? *reinterpret_cast<const Vec*>(pr + (int64_t)(j0 + jj) * p_stride) : Vec{};
#pragma unroll
                for (int jj = 0; jj < 3; ++jj)
#pragma unroll
                    for (int c = 0; c < CPL; ++c) hsum[cc][c] += reinterpret_cast<const float*>(&v[jj])[c];
            }
        }
    }
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
        const int p = y * kMap + 2 * warp + cc;
        float o[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            float d = 0.f;
#pragma unroll
            for (int c = 0; c < CPL; ++c) d = fmaf(fmaxf(hsum[cc][c], 0.f), w[k][c], d);
            o[k] = warp_sum(d) + b2v[k];
        }
        if (lane == 0) {
            const float conf = 1.f / (1.f + expf(-o[0]));
            const float sw = 1.f / (1.f + expf(-o[1])), sh = 1.f / (1.f + expf(-o[2]));
            const float cw = __fmul_rn(conf, hw[cc]);
            float* mm = maps + (int64_t)slot * 1280;
            mm[p] = cw, mm[256 + p] = sw, mm[512 + p] = sh, mm[768 + p] = o[3], mm[1024 + p] = o[4];
            float* sc = s_c[2 * warp + cc];
            sc[0] = cw, sc[1] = o[3], sc[2] = o[4], sc[3] = sw, sc[4] = sh;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int best = 0;
        for (int i = 1; i < 16; ++i)
            if (s_c[i][0] > s_c[best][0]) best = i;  // first maximum of the row
        float* cd = cand + ((int64_t)bi * 16 + y) * kCandStride;
        *reinterpret_cast<float4*>(cd) = make_float4(s_c[best][0], (float)(y * kMap + best), s_c[best][1], s_c[best][2]);
        *reinterpret_cast<float2*>(cd + 4) = make_float2(s_c[best][3], s_c[best][4]);
        __threadfence();
        s_last = atomicAdd(&counters[bi], 1u) == 15u;
    }
    __syncthreads();
    if (s_last && warp == 0) {
        // the last CTA to arrive merges the 16 row candidates: lane i fetches candidate i (all of them in flight at once, L2 loads),
        // then a shuffle arg-max with "lower row wins ties" = first row-major maximum
        __threadfence();
        const float* cd = cand + ((int64_t)bi * 16 + (lane & 15)) * kCandStride;
        const float4 c0 = __ldcg(reinterpret_cast<const float4*>(cd));
        const float2 c1 = __ldcg(reinterpret_cast<const float2*>(cd + 4));
        float bv = c0.x;
        int by = lane & 15;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oy = __shfl_xor_sync(0xffffffffu, by, o);
            if (ov > bv || (ov == bv && oy < by)) bv = ov, by = oy;
        }
        const float f1 = __shfl_sync(0xffffffffu, c0.y, by), f2 = __shfl_sync(0xffffffffu, c0.z, by), f3 = __shfl_sync(0xffffffffu, c0.w, by);
        const float f4 = __shfl_sync(0xffffffffu, c1.x, by), f5 = __shfl_sync(0xffffffffu, c1.y, by);
        if (lane == 0) {
            decode_finish(state + slot, slot, threshold, bv, (int)f1, f2, f3, f4, f5, res, decode_window, tc_err);
            counters[bi] = 0;  // ready for the next frame
            if (stamps && bi == gridDim.y - 1) stamps[ST_DEC_END] = device_time_ns();
        }
    }
}

cudaError_t launch_head_decode(const float* P, int np, int64_t p_stride, int head_ch, const float* b1, const float* w2, const float* b2,
                               const float* hann, TargetState* d_state, const int32_t* d_slots, int n, float threshold, DeviceResult* d_res,
                               float* d_maps, float* d_cand, unsigned* d_counters, unsigned long long* stamps, cudaStream_t s, bool pdl,
                               int decode_window, const int* tc_err, bool front) {
    if (n <= 0) return cudaSuccess;
    const dim3 grid(kMap, n), block(256);
    if (front && head_ch == 128 && np == 9)
        return launch_ex(head_decode_kernel<4, 9, true>, grid, block, 0, s, pdl, 1, P, np, p_stride, b1, w2, b2, hann, d_state, d_slots, threshold, d_res, d_maps, d_cand, d_counters, stamps, decode_window, tc_err);
    if (head_ch == 128 && np == 9)
        return launch_ex(head_decode_kernel<4, 9, false>, grid, block, 0, s, pdl, 1, P, np, p_stride, b1, w2, b2, hann, d_state, d_slots, threshold, d_res, d_maps, d_cand, d_counters, stamps, decode_window, tc_err);
    if (head_ch == 64 && np == 9)
        return launch_ex(head_decode_kernel<2, 9, false>, grid, block, 0, s, pdl, 1, P, np, p_stride, b1, w2, b2, hann, d_state, d_slots, threshold, d_res, d_maps, d_cand, d_counters, stamps, decode_window, tc_err);
    if (head_ch == 128)
        return launch_ex(head_decode_kernel<4, 0, false>, grid, block, 0, s, pdl, 1, P, np, p_stride, b1, w2, b2, hann, d_state, d_slots, threshold, d_res, d_maps, d_cand, d_counters, stamps, decode_window, tc_err);
    if (head_ch == 64)
        return launch_ex(head_decode_kernel<2, 0, false>, grid, block, 0, s, pdl, 1, P, np, p_stride, b1, w2, b2, hann, d_state, d_slots, threshold, d_res, d_maps, d_cand, d_counters, stamps, decode_window, tc_err);
    return cudaErrorInvalidValue;
}

cudaError_t launch_decode(const float* h1, int head_ch, const float* w2, const float* b2, const float* hann, TargetState* d_state,
                          const int32_t* d_slots, int n, float threshold, DeviceResult* d_res, float* d_maps, unsigned long long* stamps,
                          cudaStream_t s, int decode_window) {
    if (n <= 0) return cudaSuccess;
    decode_kernel<<<n, 256, 0, s>>>(h1, head_ch, w2, b2, hann, d_state, d_slots, threshold, d_res, d_maps, stamps, decode_window);
    return cudaGetLastError();
}

}  // namespace vt
