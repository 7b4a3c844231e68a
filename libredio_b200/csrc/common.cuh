// common.cuh -- shared host/device helpers for libredio_cuda.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <new>
#include "../../include/libredio_cuda.h"
#include "devbuf.h"

// ---------------------------------------------------------------------------------------------
// context + error plumbing
// ---------------------------------------------------------------------------------------------
struct lrc_ctx {
    int          device;
    int          n_sm;
    cudaStream_t stream;       // default compute stream of the context
    cudaStream_t copy_stream;  // H2D ring copies
    cudaStream_t out_stream;   // D2H of results
    int          numa_node;    // NUMA node the GPU hangs off (sysfs), -1 if unknown
    int          numa_nodes;   // online NUMA nodes of the host
};

void lrc_set_error(const char *fmt, ...);

#define LRC_CUDA(call)                                                                       \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            lrc_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return LRC_ERR_CUDA;                                                             \
        }                                                                                    \
    } while (0)

#define LRC_REQUIRE(cond, code, msg)                                                         \
    do {                                                                                     \
        if (!(cond)) {                                                                       \
            lrc_set_error("%s:%d %s", __FILE__, __LINE__, msg);                              \
            return (code);                                                                   \
        }                                                                                    \
    } while (0)

static inline cudaStream_t lrc_stream(const lrc_ctx *ctx, void *s)
{
    return s ? reinterpret_cast<cudaStream_t>(s) : ctx->stream;
}

// every entry point binds the context's device first: several contexts (one per GPU) may live in
// one process (kpn thread-per-block graphs), and torch may have changed the current device.
#define LRC_BIND(ctx)                                                                        \
    do {                                                                                     \
        LRC_REQUIRE((ctx) != nullptr, LRC_ERR_INVALID, "null context");                      \
        LRC_CUDA(cudaSetDevice((ctx)->device));                                              \
    } while (0)

static inline size_t ceil_div(size_t a, size_t b) { return (a + b - 1) / b; }

// Grid-size multiplier of a kernel family, overridable from the environment for A/B runs (read once per process):
// the resident-CTA count `n_sm * occupancy` times this factor caps the grid.  Measured on B200: pure streaming kernels
// run faster with many short CTAs than with one persistent CTA per slot (unpack 0.87 -> 1.04 of the copy bandwidth).
static inline size_t lrc_grid_mult(const char *env_name, size_t dflt)
{
    const char *e = getenv(env_name);
    if (!e) return dflt;
    const long v = atol(e);
    return v > 0 ? (size_t)v : dflt;
}

// CTAs of `kern` resident on the whole device at `threads` threads and `smem` bytes of dynamic shared memory:
// n_sm * occupancy, occupancy at least 1.  Raises the kernel's dynamic shared-memory limit to `smem` first; with
// above_default_only, only when smem exceeds the 48 KB default (kernels whose size follows the plan, launched per call:
// below the default the limit is left alone and the launch costs no extra driver call).
template <typename Kernel>
static inline cudaError_t lrc_resident_ctas(Kernel kern, int threads, size_t smem, int n_sm, size_t *ctas,
                                            bool above_default_only = false)
{
    int occ = 1;
    cudaError_t e = cudaSuccess;
    if (!above_default_only || smem > 48 * 1024)
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem);
    *ctas = (size_t)n_sm * (occ < 1 ? 1 : occ);
    return e;
}

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// ---- packed f32x2 arithmetic (sm_100: add/mul/fma.rn.f32x2 -> SASS FADD2 / FMUL2 / FFMA2) -----------------
// One packed instruction does the re and the im lane of a complex value: the same FP32-pipe cycles as the
// two scalar instructions it replaces, but ONE issue slot instead of two (tools/ubench/f32x2.cu: 73.9 TFLOP/s
// from 1.99 warp-instructions/clk/SM packed vs 71.3 from 3.83 scalar).  The FFT kernels are issue-bound, not
// pipe-bound, so complex arithmetic is written packed.  ptxas folds the lane swap, per-lane negation and scalar
// broadcast of the helpers below into operand modifiers (R.F32x2.LO_HI, .NP, R.F32): no MOVs are emitted.
__device__ __forceinline__ uint64_t pk2(float lo, float hi)
{
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float2 upk2(uint64_t v)
{
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b)
{
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a.x, a.y)), "l"(pk2(b.x, b.y)));
    return upk2(r);
}
__device__ __forceinline__ float2 sub2(float2 a, float2 b)
{
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a.x, a.y)), "l"(pk2(b.x, b.y)));
    return upk2(r);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b)
{
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a.x, a.y)), "l"(pk2(b.x, b.y)));
    return upk2(r);
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c)
{
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk2(a.x, a.y)), "l"(pk2(b.x, b.y)), "l"(pk2(c.x, c.y)));
    return upk2(r);
}

// complex product in two packed instructions: (a.x b.x - a.y b.y, a.y b.x + a.x b.y)
__device__ __forceinline__ float2 cmulf(float2 a, float2 b)
{
    return fma2(a, make_float2(b.x, b.x), mul2(make_float2(a.y, a.x), make_float2(-b.y, b.y)));
}
__device__ __forceinline__ float2 cmul_conjb(float2 a, float2 b)   // a * conj(b)
{
    return fma2(a, make_float2(b.x, b.x), mul2(make_float2(a.y, a.x), make_float2(b.y, -b.y)));
}

// streaming 128-bit global load that does not allocate in L1 (data is touched once)
__device__ __forceinline__ float4 ldg_stream_f4(const float4 *p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_f4(float4 *p, float4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + TMA (cp.async.bulk, 1-D) -----------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy executed by the TMA engine; bytes, src and dst must be 16-byte aligned.
// Completion is signalled on `bar` as transaction bytes.
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes,
                                            uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// same with an L2 evict-first policy: streaming input that is read exactly once
__device__ __forceinline__ void tma_load_1d_evict_first(void *smem_dst, const void *gmem_src,
                                                        uint32_t bytes, uint64_t *bar)
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}
// Ampere-style asynchronous 4-byte global -> shared copy (LDGSTS); src_bytes = 0 zero-fills without reading
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src, uint32_t src_bytes)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit()
{
    asm volatile("cp.async.commit_group;" ::: "memory");
}
// wait until at most N of this thread's committed groups are still in flight
template <int N>
__device__ __forceinline__ void cp_async_wait_group()
{
    asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory");
}
// order generic-proxy smem accesses before subsequent async-proxy (TMA) writes to the same buffer
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// named barrier among `nthreads` threads (multiple of 32); id 1..15 (0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void named_bar_arrive(int id, int nthreads)
{
    asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

#endif  // __CUDACC__
