// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Everything the kernels in this directory need from the Blackwell ISA lives here so that the
// kernels read as algorithms.  No CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace omg {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ------------------------------------------------------------------ programmatic dependent launch
// launch_dependents: the next kernel in the stream may start occupying freed SMs; wait: block until the previous
// kernel has completed and its memory is visible (must precede the first dependent global read or write).
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU box (~2 s at 2 GHz).
#ifndef OMG_MBAR_TIMEOUT_CYCLES
#define OMG_MBAR_TIMEOUT_CYCLES (4000000000LL)
#endif
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or ~`ns` have passed, instead
// of coming back after the (short) system default - a polling producer / MMA-issuer warp otherwise issues a try_wait + branch
// every ~80 ns next to the softmax / epilogue warps of its scheduler (ncu: 18 % of all instructions of the attention kernel)
#ifndef OMG_MBAR_SUSPEND_NS
#define OMG_MBAR_SUSPEND_NS 20000
#endif
__device__ __forceinline__ bool mbar_try_wait_long(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)OMG_MBAR_SUSPEND_NS)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    uint32_t spins = 0;
    while (!mbar_try_wait_long(bar, parity)) {
        if ((++spins & 0x3FF) == 0 && clock64() - t0 > OMG_MBAR_TIMEOUT_CYCLES) {
            printf("omg: mbarrier timeout block=(%d,%d,%d) thread=%d bar=%u parity=%u\n", (int)blockIdx.x,
                   (int)blockIdx.y, (int)blockIdx.z, (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// 2^x for x <= 0 on the FMA pipe (degree-3 minimax on the fractional part, rel. error 1.4e-4 < fp16 rounding):
// off-loads the MUFU, which is the bottleneck unit of the softmax at head_dim 64.
__device__ __forceinline__ float poly_exp2(float x) {
    x = fmaxf(x, -126.0f);
    const float t = x + 12582912.0f;             // 1.5 * 2^23: integer part of x lands in the low mantissa bits
    const float f = x - (t - 12582912.0f);       // fractional part in [-0.5, 0.5]
    float p = fmaf(f, 0.055029309f, 0.242256802f);
    p = fmaf(p, f, 0.693253036f);
    p = fmaf(p, f, 0.999951347f);
    const int e = (__float_as_int(t) - 0x4B400000) << 23;
    return __int_as_float(__float_as_int(p) + e);
}

// ------------------------------------------------------------------ packed fp32x2 arithmetic (FFMA2 / FADD2 on sm_100)
// one issue slot for two lanes of work: the softmax of attention at head_dim 64 is issue-slot bound
__device__ __forceinline__ uint64_t pack_f32x2(float a, float b) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& a, float& b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fsub2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// poly_exp2 for two values at once: 2 FMNMX + 3 FADD2 + 3 FFMA2 + 2 IMAD = 5 issue slots per value (scalar: 8)
__device__ __forceinline__ void poly_exp2_x2(float x0, float x1, float& p0, float& p1) {
    const uint64_t magic = pack_f32x2(12582912.0f, 12582912.0f);
    const uint64_t x = pack_f32x2(fmaxf(x0, -126.0f), fmaxf(x1, -126.0f));
    const uint64_t t = fadd2(x, magic);
    const uint64_t f = fsub2(x, fsub2(t, magic));
    uint64_t p = ffma2(f, pack_f32x2(0.055029309f, 0.055029309f), pack_f32x2(0.242256802f, 0.242256802f));
    p = ffma2(p, f, pack_f32x2(0.693253036f, 0.693253036f));
    p = ffma2(p, f, pack_f32x2(0.999951347f, 0.999951347f));
    float t0, t1, q0, q1;
    unpack_f32x2(t, t0, t1);
    unpack_f32x2(p, q0, q1);
    p0 = __int_as_float(__float_as_int(q0) + (__float_as_int(t0) << 23));
    p1 = __int_as_float(__float_as_int(q1) + (__float_as_int(t1) << 23));
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2,
                                             int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------ CTA pairs (cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem offset in the pair's leader CTA (rank bit 24 cleared; CUTLASS
// Sm100MmaPeerBitMask)
__device__ __forceinline__ uint32_t leader_smem_addr(uint32_t a) { return a & 0xFEFFFFFFu; }
// TMA loads of a CTA pair: data lands in the issuing CTA's smem, the transaction bytes are counted on the LEADER's
// mbarrier
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
        "[%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_smem_addr(smem_u32(bar))), "r"(c0),
        "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                                 int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
        "%5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_smem_addr(smem_u32(bar))), "r"(c0),
        "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[both CTAs' smem: 2 x 128 rows] * B[both CTAs' smem: 2 x N/2 rows], issued by the leader
__device__ __forceinline__ void tc_mma_f16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                   uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the mbarrier at this smem offset in BOTH CTAs of the pair when the issued MMAs complete
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}
// arrive on the mbarrier at this smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}

// ------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], fp16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void tc_mma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// All previously issued MMAs of this thread arrive on `bar` when complete (implies fence::before_thread_sync).
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane (taddr.lane + i), columns [col, col+32).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, sm_100):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base_offset | [61,64) layout
// 128B swizzle (layout type 2); the tile is [rows][64 fp16] with 128-byte rows written by TMA SWIZZLE_128B.
//  * K-major operand (rows = M or N index, the 64 contiguous elements are K): 8-row groups are 1024 B apart (SBO).
//  * MN-major operand (rows = K index, the 64 contiguous elements are M/N): 8-row K groups are 1024 B apart (SBO);
//    LBO would step to the next 64-wide MN atom (unused when the MN extent is 64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

// Instruction descriptor, kind::f16, fp16 (or, with bf16 = true, bf16) A/B, fp32 D (cute::UMMA::InstrDescriptor bit layout).
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N, bool a_mn_major, bool b_mn_major, bool bf16 = false) {
    return (1u << 4)                                   // D format f32
           | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10)  // A, B format: 0 f16, 1 bf16
           | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16)
           | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

__device__ __forceinline__ uint32_t pack_bf162(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

// The two 16-bit storage types of the activation paths: fp16 everywhere, bf16 for the VAE decoder with weights whose
// activations exceed the fp16 range.  Both are 2 bytes wide, so TMA boxes, swizzles and vector widths do not change.
template <typename T> struct Pair;
template <> struct Pair<__half> { using type = __half2; };
template <> struct Pair<__nv_bfloat16> { using type = __nv_bfloat162; };
__device__ __forceinline__ float to_float(__half h) { return __half2float(h); }
__device__ __forceinline__ float to_float(__nv_bfloat16 h) { return __bfloat162float(h); }
__device__ __forceinline__ float2 to_float2(__half2 h) { return __half22float2(h); }
__device__ __forceinline__ float2 to_float2(__nv_bfloat162 h) { return __bfloat1622float2(h); }
template <typename T> __device__ __forceinline__ uint32_t pack2(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2<__half>(float a, float b) { return pack_half2(a, b); }
template <> __device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float a, float b) { return pack_bf162(a, b); }

}  // namespace omg
