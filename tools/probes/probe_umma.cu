// Probe (diagnostics): how fast does one SM execute tcgen05.mma (kind::f16, bf16 operands, M = 128 or 64, K = 16, cta_group::1) as a function
//   of N (64 / 128 / 160 / 192 / 256), where A comes from (shared memory, 128B-swizzled K-major / tensor memory), and whether consecutive MMAs
//   accumulate into the same TMEM columns or rotate over 2 / 4 accumulators?
// One CTA per SM (grid = number of SMs given on the command line, default 1), one elected lane issues `count` MMAs back to back and
// waits for the commit; reported: clocks per MMA from the difference of a long and a short run (fixed latencies cancel), and the floor
// N / 2 clocks.  Operand contents are irrelevant (zeros).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I gstreamer_vit_tracker_b200/csrc -I include tools/probes/probe_umma.cu -o tools/probes/probe_umma
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "tc_common.cuh"

using namespace vt::tc;

struct Cfg {
    int N, a_tmem, n_acc, pair;  // pair: alternate (N, N / 2) as the bf16x3 K-step does
    int M;
};

__global__ void __launch_bounds__(128, 1) probe(const Cfg c, const int count, long long* out) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    for (int i = threadIdx.x; i < (96 * 1024) / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) mbar_init(&bar, 1), fence_barrier_init();
    if (threadIdx.x < 32) tmem_alloc(&tmem_base_s, 512), tmem_relinquish();
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = tmem_base_s;
    if (threadIdx.x < 32) {
        // A: 4 k-blocks of [128 rows][128 B] (16 KB each) at 0; B: 4 k-blocks of [256 rows][128 B] (32 KB each)... only 2 fit: B walks 2
        const uint32_t a_lo = umma_desc_lo(smem_u32(smem)), b_lo = umma_desc_lo(smem_u32(smem + 32 * 1024));
        const uint32_t idesc = umma_idesc_bf16(c.M, c.N), idesc_h = umma_idesc_bf16(c.M, c.N / 2);
        // accumulators at columns 0, N, 2N, ... (n_acc * N <= 448); TMEM A operand at column 448
        long long t0 = 0, t1 = 0;
        if (elect_one_sync()) {
            t0 = clock64();
            for (int i = 0; i < count; ++i) {
                const int k = i & 3, kb = (i >> 2) & 1;
                const uint32_t acc = tmem + (uint32_t)((i % c.n_acc) * c.N);
                const uint64_t dA = umma_desc_from_lo(a_lo + kb * (16384 >> 4) + 2 * k), dB = umma_desc_from_lo(b_lo + kb * (32768 >> 4) + 2 * k);
                const bool half = c.pair && (i & 1);
                if (c.a_tmem) umma_bf16_ta(acc, tmem + 448 + 8 * k, dB, half ? idesc_h : idesc, 1);
                else umma_bf16(acc, dA, dB, half ? idesc_h : idesc, 1);
            }
            umma_commit(&bar);
        }
        __syncwarp();
        mbar_wait(&bar, 0);
        t1 = clock64();
        if (elect_one_sync() && blockIdx.x == 0) out[0] = t1 - t0;
        __syncwarp();
    }
    tcgen05_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// M = 64 layout check (one CTA, 4 warps).  smem: A [64 rows][128 B] at 0, B [256 rows][128 B] at 16 KB (128B swizzle, K-major).
// A[m][0] = m, A[m][1] = 1; B[n][0] = 256, B[n][1] = n  ->  D[m][n] = 256 m + n (exact in fp32).
// out[0 .. 128 * 4): per TMEM lane, 32x32b column 0, 1, 2, 3 of D;  out[512 .. 640): per thread (warp w, lane l), the first value of its
// 16x32bx2.x8 load (offset 8) at column 0;  out[640]: mismatches of the TS product D2 = P V^T (P from tcgen05.st 16x32bx2, V = B rows)
__device__ __forceinline__ void put_bf16(uint8_t* tile, int row, int k, float v) {
    const int off = (row >> 3) * 1024 + (row & 7) * 128 + ((((k * 2) >> 4) ^ (row & 7)) << 4) + ((k * 2) & 15);
    *reinterpret_cast<__nv_bfloat16*>(tile + off) = __float2bfloat16_rn(v);
}
__global__ void __launch_bounds__(128, 1) layout_probe(float* out) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *sA = smem, *sB = smem + 16 * 1024;
    for (int i = threadIdx.x; i < (48 * 1024) / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (threadIdx.x < 64) put_bf16(sA, threadIdx.x, 0, (float)threadIdx.x), put_bf16(sA, threadIdx.x, 1, 1.f);
    for (int n = threadIdx.x; n < 256; n += blockDim.x) put_bf16(sB, n, 0, 256.f), put_bf16(sB, n, 1, (float)n);
    if (threadIdx.x == 0) mbar_init(&bar, 1), fence_barrier_init();
    if (threadIdx.x < 32) tmem_alloc(&tmem_base_s, 512), tmem_relinquish();
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = tmem_base_s;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    {   // zero columns 0..255 of every lane, so that lanes the MMA does not write read back as 0
        const uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int c = 0; c < 256; c += 8) tmem_st_32x8(lane_addr + c, z);
        tmem_st_wait();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    if (warp == 0 && elect_one_sync()) {
        umma_bf16(tmem, umma_desc_sw128(smem_u32(sA)), umma_desc_sw128(smem_u32(sB)), umma_idesc_bf16(64, 128), 0);
        umma_commit(&bar);
    }
    __syncwarp();
    mbar_wait(&bar, 0);
    tcgen05_fence_after();
    float v[8];
    tmem_ld_32x8(lane_addr, v);
    for (int j = 0; j < 4; ++j) out[(warp * 32 + lane) * 4 + j] = v[j];
    tmem_ld_16x2(lane_addr, v);
    out[512 + threadIdx.x] = v[0];
    // P[m][k] = (m + k) % 7 - 3 (k < 16) as packed bf16 pairs, written like the attention kernel's P: columns 256 .. 263 of the M = 64 layout
    {
        const int m = warp * 16 + (lane & 15), k0 = (lane >> 4) * 8;
        uint32_t pk[4];
        for (int j = 0; j < 4; ++j) {
            const float a = (float)((m + k0 + 2 * j) % 7 - 3), b = (float)((m + k0 + 2 * j + 1) % 7 - 3);
            pk[j] = pack_bf16(__float2bfloat16_rn(a), __float2bfloat16_rn(b));
        }
        tmem_st_16x2_x4(lane_addr + 256, pk);
        tmem_st_wait();
    }
    // V[n][k] = (n + 2 k) % 5 - 2 as the B operand (rows 0..63, K = 16), over the dead A / B tiles
    __syncthreads();
    for (int n = threadIdx.x; n < 64; n += blockDim.x)
        for (int k = 0; k < 64; ++k) put_bf16(sB, n, k, k < 16 ? (float)((n + 2 * k) % 5 - 2) : 0.f);
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    if (warp == 0 && elect_one_sync()) {
        umma_bf16_ta(tmem + 384, tmem + 256, umma_desc_sw128(smem_u32(sB)), umma_idesc_bf16(64, 64), 0);
        umma_commit(&bar);
    }
    __syncwarp();
    mbar_wait(&bar, 1);
    tcgen05_fence_after();
    int bad = 0;
    for (int c = 0; c < 64; c += 8) {
        tmem_ld_16x2(lane_addr + 384 + c, v);  // thread l < 16: columns c .. c + 7 of row 16 w + l; l >= 16: columns c + 8 .. (past 64: skipped)
        const int m = warp * 16 + (lane & 15), n0 = c + (lane >> 4) * 8;
        for (int j = 0; j < 8; ++j) {
            const int n = n0 + j;
            if (n >= 64) continue;
            float ref = 0.f;
            for (int k = 0; k < 16; ++k) ref += (float)((m + k) % 7 - 3) * (float)((n + 2 * k) % 5 - 2);
            bad += v[j] != ref;
        }
    }
    atomicAdd(reinterpret_cast<int*>(out + 640), bad);
    tcgen05_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

int main(int argc, char** argv) {
    const int grid = argc > 1 ? atoi(argv[1]) : 1;
    long long* d_out;
    cudaMalloc(&d_out, 8);
    const size_t smem = 97 * 1024 + 1024;
    cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const Cfg cfgs[] = {{64, 0, 1, 0, 128},  {128, 0, 1, 0, 128}, {192, 0, 1, 0, 128}, {256, 0, 1, 0, 128}, {64, 0, 2, 0, 128},  {64, 0, 4, 0, 128},
                        {128, 0, 2, 0, 128}, {128, 0, 1, 1, 128}, {64, 1, 1, 0, 128},  {128, 1, 1, 0, 128}, {192, 1, 1, 0, 128}, {256, 1, 1, 0, 128},
                        {64, 1, 2, 0, 128},  {64, 1, 4, 0, 128},  {128, 1, 1, 1, 128}, {160, 0, 1, 0, 128}, {160, 0, 2, 0, 128},
                        {64, 0, 1, 0, 64},   {128, 0, 1, 0, 64},  {160, 0, 1, 0, 64},  {256, 0, 1, 0, 64},  {160, 0, 2, 0, 64},  {64, 1, 1, 0, 64},
                        {128, 1, 1, 0, 64},  {128, 1, 1, 1, 64}};
    printf("grid %d CTA(s)\n%4s %5s %6s %5s %5s | %10s %10s | %8s\n", grid, "M", "N", "A", "accs", "pair", "clk/MMA", "floor", "ratio");
    for (const Cfg& c : cfgs) {
        long long t[2] = {0, 0};
        const int counts[2] = {64, 576};
        for (int r = 0; r < 2; ++r) {
            for (int rep = 0; rep < 3; ++rep) {  // last repetition counts (warm)
                probe<<<grid, 128, smem>>>(c, counts[r], d_out);
                cudaError_t e = cudaDeviceSynchronize();
                if (e != cudaSuccess) {
                    printf("CUDA error: %s\n", cudaGetErrorString(e));
                    return 1;
                }
                cudaMemcpy(&t[r], d_out, 8, cudaMemcpyDeviceToHost);
            }
        }
        const double per = (double)(t[1] - t[0]) / (counts[1] - counts[0]);
        // floor: N / 2 clk for M = 128 (the measured M = 128 rate); M = 64 is printed against the same floor
        const double floor_clk = c.pair ? 0.5 * (c.N / 2.0 + c.N / 4.0) : c.N / 2.0;
        printf("%4d %5d %6s %5d %5d | %10.1f %10.1f | %8.2f\n", c.M, c.N, c.a_tmem ? "tmem" : "smem", c.n_acc, c.pair, per, floor_clk, per / floor_clk);
    }
    // ---- M = 64 layout
    float* d_lay;
    cudaMalloc(&d_lay, 641 * sizeof(float));
    cudaMemset(d_lay, 0, 641 * sizeof(float));
    cudaFuncSetAttribute(layout_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 49 * 1024);
    layout_probe<<<1, 128, 49 * 1024>>>(d_lay);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        printf("CUDA error (layout): %s\n", cudaGetErrorString(e));
        return 1;
    }
    std::vector<float> h(641);
    cudaMemcpy(h.data(), d_lay, 641 * sizeof(float), cudaMemcpyDeviceToHost);
    printf("\nM = 64 accumulator, 32x32b read: TMEM lane -> row of D (column 0 = 256 row + 0; '-' = not written); columns 1..3 checked\n");
    int col_bad = 0;
    for (int q = 0; q < 4; ++q) {
        printf("  lanes %3d..%3d:", 32 * q, 32 * q + 31);
        for (int l = 0; l < 32; ++l) {
            const float* x = &h[(32 * q + l) * 4];
            if (x[0] == 0.f && x[1] == 0.f) printf("   -");
            else printf(" %3d", (int)(x[0] / 256.f));
            for (int j = 1; j < 4; ++j)
                if (!(x[0] == 0.f && x[1] == 0.f) && x[j] != x[0] + j) ++col_bad;
        }
        printf("\n");
    }
    printf("  column mismatches: %d\n", col_bad);
    printf("16x32bx2.x8 (offset 8) read at column 0: thread -> (row, column) of its first value\n");
    for (int w = 0; w < 4; ++w) {
        printf("  warp %d:", w);
        for (int l = 0; l < 32; ++l) {
            const int v = (int)h[512 + 32 * w + l];
            printf(" %d/%d", v >> 8, v & 255);
        }
        printf("\n");
    }
    int bad;
    memcpy(&bad, &h[640], 4);
    printf("TS UMMA M = 64, N = 64, A = P from tcgen05.st 16x32bx2 (offset 4): %d mismatches of 4096\n", bad);
    return 0;
}
