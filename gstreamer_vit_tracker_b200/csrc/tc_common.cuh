// tc_common.cuh — sm_100a PTX wrappers for the tensor-core path: mbarrier, TMA (cp.async.bulk.tensor),
// TMEM allocation, tcgen05.mma / commit / ld, UMMA shared-memory and instruction descriptors.
// Encodings follow the PTX ISA as transcribed in the CUTLASS headers shipped with this image
// (cute/arch/mma_sm100_desc.hpp, cute/arch/copy_sm100.hpp); no CUTLASS code is compiled in.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vt {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol error must surface as an error code, never as a hung GPU.
constexpr uint32_t kSpinCap = 1u << 20;
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t i = 0; i < kSpinCap; ++i)
        if (mbar_try_wait(bar, parity)) return true;
    return false;
}

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------
// Every kernel of the per-frame chain is launched with cudaLaunchAttributeProgrammaticStreamSerialization and follows
//   prologue (barrier init, TMEM alloc, descriptor prefetch, weight TMA)  ->  pdl_wait()  ->  pdl_launch_dependents()  ->  work
// pdl_wait() returns when the preceding kernel has completed and its writes are visible.  Triggering the dependents only
// AFTER the wait bounds residency to two kernels of the chain (the running one and the next one's prologue), so a waiting
// prologue can never hold shared memory / TMEM that an earlier kernel still needs.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- device-side timeline (diagnostics; enabled per handle with VT_B200_TRACE=1) -----------------------------------
// trace[0] = record counter; record i = trace[1 + 8 i ..]: {kernel id, t_entry, t_after_pdl_wait, t_end, 4 kernel-specific marks}
// in %globaltimer ns, written by threads of CTA (0,0,0) only.
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
    return t;
}
struct TraceRec {
    unsigned long long** slot;  // shared-memory cell holding the record pointer (null when tracing is off / not CTA 0)
    __device__ __forceinline__ void begin(unsigned long long** shared_slot, unsigned long long* trace, int id) {
        slot = shared_slot;
        if (threadIdx.x == 0) {
            unsigned long long* rec = nullptr;
            // id bit 8 (VT_B200_TRACE_LASTX): trace the CTA with the LAST blockIdx.x instead of the first (e.g. a V^T tile of the QKV GEMM)
            const unsigned bx = (id & 0x100) ? gridDim.x - 1 : 0u;
            if (trace && blockIdx.x == bx && blockIdx.y == 0 && blockIdx.z == 0) {
                const unsigned long long i = atomicAdd(trace, 1ull);
                if (i < 2048) {
                    rec = trace + 1 + 8 * i;
                    rec[0] = (unsigned long long)(id & 0xff), rec[1] = globaltimer_ns();
                }
            }
            *slot = rec;
        }
    }
    // valid after the first __syncthreads() following begin()
    __device__ __forceinline__ void mark(int k) const {
        unsigned long long* rec = *slot;
        if (rec) rec[k] = globaltimer_ns();
    }
};
// Free-form events of the traced CTA (diagnostics; tools/chain_timeline.py --events): any thread appends (code, time) to a small
// shared-memory log (one shared-memory atomic, ~20 clk), thread 0 copies the log into records {256 + code, t, kernel id} of the trace
// buffer at the end of the kernel.
constexpr int kTraceEvents = 96;
struct TraceEvents {
    unsigned long long (*buf)[2];
    unsigned* cnt;
    const TraceRec* tr;
    __device__ __forceinline__ void begin(unsigned long long (*b)[2], unsigned* c, const TraceRec* t) {
        buf = b, cnt = c, tr = t;
        if (threadIdx.x == 0) *c = 0;
    }
    __device__ __forceinline__ void event(int code) const {  // valid after the first __syncthreads()
        if (!*tr->slot) return;
        const unsigned i = atomicAdd(cnt, 1u);
        if (i < (unsigned)kTraceEvents) buf[i][0] = 256ull + (unsigned long long)code, buf[i][1] = globaltimer_ns();
    }
    __device__ __forceinline__ void flush(unsigned long long* trace) const {  // thread 0, after the closing __syncthreads()
        unsigned long long* rec = *tr->slot;
        if (!rec) return;
        const unsigned n = *cnt < (unsigned)kTraceEvents ? *cnt : (unsigned)kTraceEvents;
        const unsigned long long i0 = atomicAdd(trace, (unsigned long long)n);
        for (unsigned i = 0; i < n && i0 + i < 2048; ++i) {
            unsigned long long* r = trace + 1 + 8 * (i0 + i);
            r[0] = buf[i][0], r[1] = buf[i][1], r[2] = rec[0], r[3] = r[4] = r[5] = r[6] = r[7] = 0;
        }
    }
};
constexpr size_t kTraceWords = 1 + 8 * 2048;

// ---- thread-block clusters / distributed shared memory ------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
// address of the same shared-memory variable in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t cluster_map_shared(uint32_t smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_shared_cluster_f2(uint32_t addr, float x, float y) {
    asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(x), "f"(y) : "memory");
}
// asynchronous store into a peer CTA's shared memory that signals the peer's mbarrier with the byte count (no cluster barrier needed:
// the receiver waits for expect_tx bytes on its own mbarrier)
__device__ __forceinline__ void st_async_cluster_f2(uint32_t remote_addr, float x, float y, uint32_t remote_mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(remote_addr), "f"(x), "f"(y),
                 "r"(remote_mbar)
                 : "memory");
}
__device__ __forceinline__ void st_async_cluster_f4(uint32_t remote_addr, float x, float y, float z, float w, uint32_t remote_mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(remote_addr), "f"(x), "f"(y),
                 "f"(z), "f"(w), "r"(remote_mbar)
                 : "memory");
}
__device__ __forceinline__ void st_shared_cluster_f4(uint32_t addr, float x, float y, float z, float w) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
// bulk copy from this CTA's shared memory into a peer's (addresses of the peer: mapa), completion counted on the peer's mbarrier
__device__ __forceinline__ void dsmem_bulk_copy(uint32_t remote_dst, uint32_t local_src, uint32_t bytes, uint32_t remote_mbar) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(remote_dst), "r"(local_src),
                 "r"(bytes), "r"(remote_mbar)
                 : "memory");
}
__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// ---- async-proxy fences ---------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMA -------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// One CTA of a cluster loads the box and the TMA unit delivers it — data and mbarrier complete_tx — to the same shared-memory offsets
// of every CTA in cta_mask: the CTAs of a cluster that need the same activation tile fetch it from L2 once.
__device__ __forceinline__ void tma_load_2d_mcast(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}

// ---- TMEM ------------------------------------------------------------------------------------------
// Must be executed by one full warp; ncols is a power of two in [32, 512].
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- UMMA descriptors ----------------------------------------------------------------------------------
// K-major operand tile stored as rows of 128 bytes (64 bf16) with the 128-byte swizzle, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address        bits [0,14)
    d |= (uint64_t)1 << 16;                         // leading byte offset  bits [16,30) (unused for swizzled K-major)
    d |= (uint64_t)(1024u >> 4) << 32;              // stride byte offset   bits [32,46): next 8-row group
    d |= (uint64_t)1 << 46;                         // descriptor version   bits [46,48) = 1 on sm_100
    d |= (uint64_t)2 << 61;                         // layout type          bits [61,64) = SWIZZLE_128B
    return d;
}
// The same descriptor from its two halves: the high word is constant for every 128B-swizzled K-major tile, the low word is
// (address >> 4) | LBO.  MMA issue loops keep `lo` of a tile in a (uniform) register and step it by 2 per K = 16 slice (32 bytes): one
// add per operand and MMA instead of the shift / mask / or chain of umma_desc_sw128 — the issuing thread's instruction latency, not the
// tensor pipe, paced the MMAs (measured: ~170 clk per UMMA pair step issued against a 96 clk floor).
constexpr uint32_t kUmmaDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t umma_desc_from_lo(uint32_t lo) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(kUmmaDescHi));
    return d;
}
// One lane of the (converged) warp: the compiler knows the guarded region runs in a single thread, so uniform-datapath instructions such
// as tcgen05.mma need no per-thread election loop around them.
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// kind::f16, A = B = bf16, D = fp32, both operands K-major, dense.
// a_format = b_format = F16 (0): same instruction kind, 10 mantissa bits instead of 7 (VT_GEMM_TCGEN05_FP16)
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
template <bool F16>
__host__ __device__ constexpr uint32_t umma_idesc_h(int M, int N);
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4)                    // c_format = F32
           | (1u << 7) | (1u << 10)     // a_format = b_format = BF16
           | ((uint32_t)(N >> 3) << 17) // n_dim
           | ((uint32_t)(M >> 4) << 24);// m_dim
}
template <bool F16>
__host__ __device__ constexpr uint32_t umma_idesc_h(int M, int N) {
    return F16 ? umma_idesc_f16(M, N) : umma_idesc_bf16(M, N);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (128 rows = lanes, two bf16 K-elements per 32-bit column, 8 columns per K = 16 step) is
// read from tensor memory, so the MMA fetches only B from shared memory.
__device__ __forceinline__ void umma_bf16_ta(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// registers -> TMEM: 8 consecutive 32-bit columns of this thread's lane (warp w owns lanes 32 (w % 4) ..)
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Arrives on the mbarrier when all previously issued MMAs of this thread have completed (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// the same arrival delivered to the barrier at this shared-memory offset in every CTA of cta_mask (stages that a multicast load fills
// in all CTAs of a cluster are released cluster-wide)
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}

// TMEM -> registers: 32 lanes (this warp's quarter) x 32 consecutive fp32 columns; thread l gets lane 32*(warp%4)+l.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
    // the registers are written asynchronously: tie them to the wait so that no use can be scheduled above it
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])::"memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

#define VT_TMEM_REGS32(r, o)                                                                                                         \
    "=r"(r[o + 0]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]), "=r"(r[o + 6]), "=r"(r[o + 7]),       \
        "=r"(r[o + 8]), "=r"(r[o + 9]), "=r"(r[o + 10]), "=r"(r[o + 11]), "=r"(r[o + 12]), "=r"(r[o + 13]), "=r"(r[o + 14]),              \
        "=r"(r[o + 15]), "=r"(r[o + 16]), "=r"(r[o + 17]), "=r"(r[o + 18]), "=r"(r[o + 19]), "=r"(r[o + 20]), "=r"(r[o + 21]),            \
        "=r"(r[o + 22]), "=r"(r[o + 23]), "=r"(r[o + 24]), "=r"(r[o + 25]), "=r"(r[o + 26]), "=r"(r[o + 27]), "=r"(r[o + 28]),            \
        "=r"(r[o + 29]), "=r"(r[o + 30]), "=r"(r[o + 31])
#define VT_TMEM_TIE32(r, o)                                                                                                          \
    "+r"(r[o + 0]), "+r"(r[o + 1]), "+r"(r[o + 2]), "+r"(r[o + 3]), "+r"(r[o + 4]), "+r"(r[o + 5]), "+r"(r[o + 6]), "+r"(r[o + 7]),       \
        "+r"(r[o + 8]), "+r"(r[o + 9]), "+r"(r[o + 10]), "+r"(r[o + 11]), "+r"(r[o + 12]), "+r"(r[o + 13]), "+r"(r[o + 14]),              \
        "+r"(r[o + 15]), "+r"(r[o + 16]), "+r"(r[o + 17]), "+r"(r[o + 18]), "+r"(r[o + 19]), "+r"(r[o + 20]), "+r"(r[o + 21]),            \
        "+r"(r[o + 22]), "+r"(r[o + 23]), "+r"(r[o + 24]), "+r"(r[o + 25]), "+r"(r[o + 26]), "+r"(r[o + 27]), "+r"(r[o + 28]),            \
        "+r"(r[o + 29]), "+r"(r[o + 30]), "+r"(r[o + 31])
#define VT_TMEM_LD32_ASM                                                                                         \
    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                    \
    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                    \
    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"

// TMEM -> registers, 64 consecutive fp32 columns of this thread's lane: both loads are in flight before the single wait
__device__ __forceinline__ void tmem_ld_32x64(uint32_t taddr, float (&v)[64]) {
    uint32_t r[64];
    asm volatile(VT_TMEM_LD32_ASM : VT_TMEM_REGS32(r, 0) : "r"(taddr));
    asm volatile(VT_TMEM_LD32_ASM : VT_TMEM_REGS32(r, 32) : "r"(taddr + 32));
    asm volatile("tcgen05.wait::ld.sync.aligned;" : VT_TMEM_TIE32(r, 0)::"memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" : VT_TMEM_TIE32(r, 32)::"memory");
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}
// issue-only / wait-only pair for software-pipelined readers (raw registers; convert after tmem_ld_wait32)
__device__ __forceinline__ void tmem_ld_32x32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(VT_TMEM_LD32_ASM : VT_TMEM_REGS32(r, 0) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait32(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" : VT_TMEM_TIE32(r, 0)::"memory");
}

// TMEM -> registers: 16 consecutive fp32 columns of this thread's lane
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                   "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])::"memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// split form for software pipelining: issue the load of the NEXT block, work on the current one, then wait.  The registers must not be
// read between the two calls (the wait takes them as in/out operands, which orders every later use behind it).
__device__ __forceinline__ void tmem_ld_32x16_issue(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                   "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])::"memory");
}
// TMEM -> registers: 8 consecutive fp32 columns of this thread's lane
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])::"memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[16]) { tmem_ld_32x16(taddr, v); }
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[8]) { tmem_ld_32x8(taddr, v); }

// ---- M = 64 accumulators (cta_group::1): row 16 q + i sits in lane 32 q + i, i < 16 — the first 16 lanes of every lane quarter.
// The 16x32bx2 shapes address those 16 lanes from a whole warp: thread l < 16 accesses lane l of the warp's quarter at columns
// taddr .., thread l >= 16 lane l - 16 at columns taddr + OFF .. (OFF: immediate, in 32-bit columns).
__device__ __forceinline__ void tmem_ld_16x2_x8_issue(uint32_t taddr, uint32_t (&r)[8]) {  // OFF = 8
    asm volatile("tcgen05.ld.sync.aligned.16x32bx2.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8], 8;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[8]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])::"memory");
}
__device__ __forceinline__ void tmem_ld_16x2(uint32_t taddr, float (&v)[8]) {  // OFF = 8
    uint32_t r[8];
    tmem_ld_16x2_x8_issue(taddr, r);
    tmem_ld_wait(r);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_16x2(uint32_t taddr, float (&v)[4]) {  // OFF = 4
    uint32_t r[4];
    asm volatile("tcgen05.ld.sync.aligned.16x32bx2.x4.b32 {%0, %1, %2, %3}, [%4], 4;" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3])::"memory");
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st_16x2_x4(uint32_t taddr, const uint32_t (&r)[4]) {  // OFF = 4
    asm volatile("tcgen05.st.sync.aligned.16x32bx2.x4.b32 [%0], 4, {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
                 : "memory");
}
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- packed fp32 pairs (Blackwell FFMA2 / FMUL2 / FADD2: one issue slot for two lanes; results identical to the scalar .rn ops) ----
__device__ __forceinline__ uint64_t f2_pack(float a, float b) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t f2_bcast(float c) { return f2_pack(c, c); }

// fp32 -> (hi, lo) bf16 split: v ~= hi + lo with ~16 mantissa bits
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(v);
    lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
// two values at once: hi / lo hold (a, b) as packed bf16x2 (a in the low half); bit-identical to two split_bf16 calls
__device__ __forceinline__ void split2_bf16(float a, float b, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const float ra = a - __uint_as_float(hi << 16), rb = b - __uint_as_float(hi & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}
// (a, b) -> packed fp16x2, a in the low half (single-pass fp16 operands: no lo part)
__device__ __forceinline__ uint32_t pack2_f16(float a, float b) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
// operand split by mode: F16 -> hi = fp16 pair, lo unused; otherwise the bf16 (hi, lo) split
template <bool F16>
__device__ __forceinline__ void split2_h(float a, float b, uint32_t& hi, uint32_t& lo) {
    if (F16) hi = pack2_f16(a, b), lo = 0;
    else split2_bf16(a, b, hi, lo);
}
// scalar form for the small kernels: f16 != 0 -> the 16 bits of the fp16 value, else of the bf16 value
__device__ __forceinline__ unsigned short half_bits(float v, bool f16) {
    return f16 ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
__device__ __forceinline__ uint32_t pack_bf16(__nv_bfloat16 a, __nv_bfloat16 b) {
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

}  // namespace tc
}  // namespace vt
