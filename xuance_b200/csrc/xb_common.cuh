// Shared device/host helpers for the xb200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "../../include/xb200.h"

#define XB_SM_COUNT_FALLBACK 148
#define XB_MAX_PARTIALS 2048               // scratch doubles (per reduction slot group)
#define XB_SCRATCH_DOUBLES (XB_MAX_PARTIALS * 8 + 8)
#define XB_LOG_SQRT_2PI 0.91893853320467274178   // log(sqrt(2 pi)), the constant of Normal.log_prob

static inline int xb_launch_status() {
    cudaError_t e = cudaPeekAtLastError();
    return e == cudaSuccess ? XB_OK : (int)e;
}

static inline int xb_sm_count() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            cached = XB_SM_COUNT_FALLBACK;
    }
    return cached;
}

static inline bool xb_aligned(const void *p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

// ---------------------------------------------------------------- warp / block reductions
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sums K doubles per thread over the block; result valid in thread 0.  smem: K*32 doubles.
template <int K>
__device__ __forceinline__ void block_sum_d(double (&v)[K], double *smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = warp_sum_d(v[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) smem[k * 32 + warp] = v[k];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            double x = lane < nwarps ? smem[k * 32 + lane] : 0.0;
            v[k] = warp_sum_d(x);
        }
    }
}

// Deterministic grid reduction: every block deposits K partial sums, the last block to arrive (ticket counter)
// adds them in block order and calls fin(total[K]).  scratch layout: [K][XB_MAX_PARTIALS] doubles then the
// int32 ticket at scratch[K_MAX*XB_MAX_PARTIALS] (K_MAX = 8).  gridDim.x <= XB_MAX_PARTIALS.
template <int K, typename Fin>
__device__ __forceinline__ void grid_sum_finalize(double (&v)[K], double *scratch, double *smem, Fin fin) {
    __shared__ bool is_last;
    int *ticket = reinterpret_cast<int *>(scratch + 8 * XB_MAX_PARTIALS);
    block_sum_d<K>(v, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) scratch[k * XB_MAX_PARTIALS + blockIdx.x] = v[k];
        __threadfence();
        int t = atomicAdd(ticket, 1);
        is_last = (t == (int)gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.0;
        // fixed order: thread i takes blocks i, i+blockDim, ... then a block tree -> independent of arrival order
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
#pragma unroll
            for (int k = 0; k < K; ++k) acc[k] += __ldcg(&scratch[k * XB_MAX_PARTIALS + b]);
        }
        __syncthreads();
        block_sum_d<K>(acc, smem);
        if (threadIdx.x == 0) {
            *ticket = 0;  // re-arm for the next launch
            fin(acc);
        }
    }
}

// ---------------------------------------------------------------- mbarrier + 1-D bulk async copy (TMA unit)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy, completion counted on an mbarrier (bytes % 16 == 0, both addresses 16B aligned)
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global bulk copy (bulk async-group completion)
__device__ __forceinline__ void bulk_s2g(void *gdst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// streaming 16B global accesses (read-once / write-once data: keep it out of L1)
__device__ __forceinline__ uint4 ldg_stream16(const void *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream16(void *p, const uint4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}
