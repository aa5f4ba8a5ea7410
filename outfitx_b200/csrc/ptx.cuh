// Thin inline-PTX wrappers for the sm_100a features the kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / ld / commit / fences).
// Nothing here is portable to other architectures on purpose.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace ofx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// two fp32 values -> one 32-bit word of 16-bit operands (round to nearest even), T = __nv_bfloat16 or __half
template <class T>
__device__ __forceinline__ uint32_t pack2_16(float a, float b) {
    if constexpr (std::is_same<T, __half>::value) {
        __half2 v = __floats2half2_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&v);
    } else {
        __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&v);
    }
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread for a system-defined time when the phase is not complete)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded spin: a wedged pipeline traps (-> CUDA error at the next sync) instead of hanging
// the GPU box.  ~2^31 polls is minutes of wall clock, far beyond any legitimate wait.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins == 0x40000000u) __trap();
    }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2D tile load: coordinates are (inner = element index along the contiguous dim, outer = row)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar,
                                            int32_t c_inner, int32_t c_outer) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
        "r"(c_inner), "r"(c_outer)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const void* tmap, uint64_t* bar,
                                                 int32_t c_inner, int32_t c_outer,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
        "r"(c_inner), "r"(c_outer), "l"(policy)
        : "memory");
}
// L2 prefetch of one box (no shared-memory destination, no barrier)
__device__ __forceinline__ void tma_prefetch_l2_2d(const void* tmap, int32_t c_inner, int32_t c_outer) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(c_inner), "r"(c_outer)
                 : "memory");
}
// Same encodings CUTLASS uses for TMA::CacheHintSm90
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;

// ---------------------------------------------------------------- explicit address spaces
// Pointers derived from the realigned dynamic-smem base (an integer round trip) or read from
// by-value parameter structs reach ptxas as GENERIC pointers: it then emits LD.E / ST.E, and --
// worse -- cannot reorder a "maybe shared" access against a "maybe global" one, so load batches
// get serialised behind stores.  The hot paths therefore name the state space.
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}
__device__ __forceinline__ void sts64(uint32_t addr, uint2 v) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(v.x), "r"(v.y));
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 ldg128(const float* p) {      // coherent global load
    float4 v;
    asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg128_nc(const float* p) {   // read-only path (data not written by this kernel's other threads)
    float4 v;
    asm("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void stg128(float* p, float4 v) {
    asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---------------------------------------------------------------- TMA store (smem -> global)
// 2D tile store: the box described by `tmap` is read from shared memory (128B-swizzled rows)
// and written to global memory; rows / columns outside the tensor are clipped by the hardware.
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int32_t c_inner,
                                             int32_t c_outer) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(smem_src)), "r"(c_inner), "r"(c_outer)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores of this thread have finished READING shared memory
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... and have completed entirely (writes visible)
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// whole warp; writes the TMEM base address (lane 0, column c) to *smem_slot
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(smem_slot)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 or fp16 inputs (idesc), fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::
                     "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// ---------------------------------------------------------------- CTA pairs (cta_group::2)
// Two CTAs of a cluster (ranks 2i, 2i+1) drive one tensor-core instruction: the even CTA (the
// "leader") issues tcgen05.mma.cta_group::2; each CTA supplies its half of the M rows of A and
// of the N rows of B from its own shared memory and receives its half of the accumulator rows
// in its own TMEM.  Barrier traffic between the two goes through shared::cluster addresses.
__device__ __forceinline__ uint32_t mapa_shared(uint32_t cta_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
    return r;
}
// arrive on a barrier of any CTA of the cluster (address from mapa_shared)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id):
    // a .release.cluster arrive compiles to MEMBAR.ALL.GPU + ERRBAR, ~1-2k cycles per arrive.
    // The operand data never crosses CTAs through the generic proxy here: each CTA's UMMA reads
    // that CTA's own shared memory after the writer's fence.proxy.async.
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// wait with cluster-scope acquire: for barriers that threads of the peer CTA arrive on
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait_cluster(bar, parity)) {
        if (++spins == 0x40000000u) __trap();
    }
}
// TMA tile load whose complete_tx lands on a barrier of either CTA of the pair
// (`bar_cluster_addr` from mapa_shared); the data goes to this CTA's own shared memory.
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap,
                                                 uint32_t bar_cluster_addr, int32_t c_inner,
                                                 int32_t c_outer, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster_addr),
        "r"(c_inner), "r"(c_outer), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(smem_slot)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
// D[tmem of both CTAs] (+)= A * B^T over the pair; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                               uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// As umma_bf16_pair with the A operand in TENSOR MEMORY (lane = row of this CTA's half of M, 32-bit column j =
// K elements 2j (low half) and 2j+1; a K = 16 step reads 8 columns from a_tmem).  Verified against a known answer
// and at the SS issue rate by tools/ubench/umma_ts.cu (M = 256: 128 cycles at N = 256, 64 at N = 128).
__device__ __forceinline__ void umma_bf16_pair_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                                  uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns, registers -> TMEM: thread t of the warp writes lane (base_lane + t)
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
        : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// full proxy fence (generic <-> async, all state spaces): global data written by bulk stores / read by bulk loads
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// ---------------------------------------------------------------- flags in global memory (CTA <-> CTA of other clusters)
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_gpu_add(int* p, int v) {
    asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_relaxed_gpu_add(int* p, int v) {
    asm volatile("red.relaxed.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// bounded spin until *p >= target (traps instead of hanging the GPU if the partner never arrives)
__device__ __forceinline__ void wait_flag_ge(const int* p, int target) {
    uint32_t spins = 0;
    while (ld_acquire_gpu(p) < target) {
        __nanosleep(40);
        if (++spins == 0x4000000u) __trap();
    }
}
// arrives (once all earlier MMAs of this thread retired) on the barrier at this offset in every
// CTA of `mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
            "r"(smem_u32(bar)), "h"(mask)
        : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
          "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
          "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- UMMA descriptors
// K-major operand tile in shared memory, rows of 64 bf16 (128 B) with the 128-byte TMA /
// UMMA swizzle: 8-row groups are 1024 B apart (SBO), LBO is unused for swizzled K-major.
// Field layout: cute/arch/mma_sm100_desc.hpp (SmemDescriptor): start>>4 [0,14), LBO>>4
// [16,30), SBO>>4 [32,46), version=1 [46,48), layout_type [61,64) with SWIZZLE_128B = 2.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>(1) << 16;            // LBO (ignored for SW128 K-major)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;    // SBO = 8 rows * 128 B
    d |= static_cast<uint64_t>(1) << 46;            // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;            // SWIZZLE_128B
    return d;
}
// Instruction descriptor for kind::f16, BF16 x BF16 -> FP32, both operands K-major
// (InstrDescriptor in the same header): c_format=F32 [4,6), a/b_format=BF16 [7,10)/[10,13),
// a/b_major=K (0) [15],[16], N>>3 [17,23), M>>4 [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t m, uint32_t n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// The same for FP16 x FP16 -> FP32: a/b_format = F16 (0)
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t m, uint32_t n) {
    return (1u << 4) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// ... chosen by the 16-bit operand type (__nv_bfloat16 or __half)
template <class T>
__host__ __device__ constexpr uint32_t umma_idesc_16(uint32_t m, uint32_t n) {
    return std::is_same<T, __half>::value ? umma_idesc_f16(m, n) : umma_idesc_bf16(m, n);
}

}  // namespace ofx
