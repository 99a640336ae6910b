// common.cuh — sm_100a device helpers shared by the kernels: mbarrier, TMA (cp.async.bulk.tensor),
// packed fp32x2 math (FFMA2), bf16 unpacking, bounded waits.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vrwkv {

typedef unsigned long long u64;

// ---------------------------------------------------------------------------------------------
// shared-memory addressing / mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
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
// Bounded wait: a protocol bug traps (launch fails with an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}

// ---------------------------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile global -> shared, completion counted in bytes on `bar`.
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
}
// 2-D tile shared -> global (bulk group completion).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(x), "r"(y)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// 1-D bulk copy global -> shared.
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// 1-D bulk copy shared -> global (bulk group completion: tma_store_commit / tma_store_wait*).
__device__ __forceinline__ void bulk_store_1d(void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(dst)),
                 "r"(smem_u32(src)), "r"(bytes)
                 : "memory");
}

// ---------------------------------------------------------------------------------------------
// packed fp32x2 arithmetic (Blackwell FFMA2 / FMUL2 / FADD2)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ u64 fmul2(u64 a, u64 b) {
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 fadd2(u64 a, u64 b) {
    u64 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ float hsum2(u64 v) {
    float lo, hi;
    upk2(v, lo, hi);
    return lo + hi;
}

// ---------------------------------------------------------------------------------------------
// bf16 helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float bf16lo_to_f32(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi_to_f32(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ uint16_t f32_to_bf16_bits(float f) {
    return __bfloat16_as_ushort(__float2bfloat16_rn(f));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    return (uint32_t)f32_to_bf16_bits(lo) | ((uint32_t)f32_to_bf16_bits(hi) << 16);
}

// ---------------------------------------------------------------------------------------------
// predicated (branch-free) global stores
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_pred_b16(void* p, uint16_t v, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.global.b16 [%0], %1;\n\t}" ::"l"(p), "h"(v),
                 "r"((uint32_t)pred)
                 : "memory");
}
__device__ __forceinline__ void st_pred_b32(void* p, uint32_t v, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.global.b32 [%0], %1;\n\t}" ::"l"(p), "r"(v),
                 "r"((uint32_t)pred)
                 : "memory");
}
__device__ __forceinline__ void st_pred_f32(void* p, float v, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.global.f32 [%0], %1;\n\t}" ::"l"(p), "f"(v),
                 "r"((uint32_t)pred)
                 : "memory");
}
__device__ __forceinline__ void st_pred_f32x2(void* p, float a, float b, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\t@p st.global.v2.f32 [%0], {%1, %2};\n\t}" ::"l"(p),
                 "f"(a), "f"(b), "r"((uint32_t)pred)
                 : "memory");
}

}  // namespace vrwkv
