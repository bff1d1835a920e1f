// common.cuh — shared device helpers for the sm_100a scoring kernels.
// Compiled with -fmad=false: every fused multiply-add in this library is an explicit fmaf()/__fmaf_rn(), so the
// NVQ bit tricks and the similarity->score maps round exactly like the reference's scalar code.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define JV_METRIC_EUCLIDEAN 0
#define JV_METRIC_DOT 1
#define JV_METRIC_COSINE 2

namespace jv {

constexpr unsigned FULL = 0xffffffffu;

// base:vector/VectorSimilarityFunction.java:37-69 — similarity -> score, fused into every kernel epilogue
__device__ __forceinline__ float score_map(int metric, float raw)
{
    if (metric == JV_METRIC_EUCLIDEAN) return __fdiv_rn(1.0f, __fadd_rn(1.0f, raw));
    return __fdiv_rn(__fadd_rn(1.0f, raw), 2.0f);
}

// base:util/NumericUtils.java:63-65 + base:graph/NodeQueue.java:125-137
__device__ __forceinline__ int32_t float_to_sortable(float f)
{
    int32_t b = __float_as_int(f);
    return b ^ ((b >> 31) & 0x7fffffff);
}
__device__ __forceinline__ long long topk_key(float score, int32_t node)
{
    return (long long)(((unsigned long long)(uint32_t)float_to_sortable(score) << 32) | (unsigned long long)(uint32_t)(~node));
}
__device__ __forceinline__ float key_score(long long key)
{
    int32_t s = (int32_t)(key >> 32);
    return __int_as_float(s ^ ((s >> 31) & 0x7fffffff));
}
__device__ __forceinline__ int32_t key_node(long long key) { return (int32_t)~(uint32_t)((unsigned long long)key & 0xffffffffull); }

constexpr long long KEY_MIN = (long long)0x8000000000000000ull;

// lanes of the calling thread's WIDTH-wide group (groups never straddle a warp; blocks are 1-D, multiple of 32).
// Sub-warp groups of one warp may sit in different loop iterations, so shuffles name only their own group.
template <int WIDTH>
__device__ __forceinline__ unsigned group_mask()
{
    if (WIDTH == 32) return FULL;
    return ((1u << WIDTH) - 1u) << ((threadIdx.x & 31u) & ~(unsigned)(WIDTH - 1));
}
template <int WIDTH>
__device__ __forceinline__ float group_sum(float v)
{
    const unsigned m = group_mask<WIDTH>();
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(m, v, o, WIDTH));
    return v;
}
template <int WIDTH>
__device__ __forceinline__ int group_sum_int(int v)
{
    const unsigned m = group_mask<WIDTH>();
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o, WIDTH);
    return v;
}

// warp-wide double sum, result in every lane
__device__ __forceinline__ double warp_sum_d(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// 128-bit streaming load that bypasses L1 allocation (rows are touched once per query)
__device__ __forceinline__ float4 ldg_stream(const float4 *p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// bulk DRAM -> L2 prefetch of `bytes` (multiple of 16) at a 16-byte aligned address: cp.async.bulk.prefetch.L2, SASS UBLKPF. The
// bytes are in flight without occupying a register or a byte of shared memory; the demand loads that follow hit L2.
__device__ __forceinline__ void bulk_prefetch_l2(const void *p, unsigned bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// ---- TMA-style bulk async copy global -> shared with an mbarrier (cp.async.bulk; SASS UBLKCP) ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, unsigned phase)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned phase)
{
    while (!mbar_try_wait(bar, phase)) {
    }
}

}  // namespace jv
