// k_fft.cu -- batched FFT (kissfft seam) and the fused window + FFT + |X|^2-average kernel.
//
// Replaces: kissfft::fft block + kiss_fft_alloc/kiss_fft (src/kissfft/src/kissfft.rs:11-31,
// libkissfft/kiss_fft.c:339-388); |X|^2 averaging after tools/psdpng.c:157-178.
//
// Measured and rejected at 1024 points (Gsamples/s, one B200):
//   - the CTA-level TMA-ring kernels (fft_tma_kernel, psd_tma_kernel) that the warp-per-transform kernels replaced:
//     FFT 357.6 and PSD 547.2 (profiles/r1_s3_kernels_table.jsonl) against 422.1 and 657.1 (r1_s8_kernels_table.jsonl);
//   - psd1024_warp_kernel without the L2 prefetch of the next frame (644.0 against 657.0), with an L1 prefetch (657.9,
//     no gain) and bounded for 4 CTAs per SM (624.8 / 623.4) (profiles/r1_s8_grid_sweeps.txt);
//   - psd1024_warp_db_kernel, the next frame double-buffered in registers: 589.0 at 2 CTAs x 4 warps, 566.8 at 1 x 8
//     (r1_s8_grid_sweeps.txt), 519.2 at 3 x 4 (r1_s6_psd_variants.txt);
//   - the folded window and shared-memory accumulators of profiles/r2_psd_variants.txt.
// psd_tma_kernel (512 and 2048 points) also had 2-stage rings at 3 or 4 CTAs per SM and (re^2, im^2) accumulated apart with
// one FFMA2 per bin at 2 CTAs per SM; no recorded measurement put them ahead of 3 stages at 3 CTAs.
#include "fft_core.cuh"
#include <cmath>
#include <vector>

using namespace lrfft;

// mixed-radix path (k_fft_mixed.cu) for sizes that are not powers of two
constexpr int MIXED_MAX_FACTORS = 24;
constexpr int MIXED_MAX_NFFT = 8192;
struct MixedPlan { int nfac; int radix[MIXED_MAX_FACTORS]; };
int lrc_fft_mixed_factor(int n, MixedPlan *mp);
int lrc_fft_mixed_launch(const lrc_ctx *ctx, int nfft, int inverse, const MixedPlan *mp, const float2 *d_tw,
                         const float2 *in, float2 *out, size_t batch, cudaStream_t s);

struct lrc_fft {
    lrc_ctx *ctx;
    int      nfft, log2n, inverse;   // log2n < 0: mixed-radix plan
    DevBuf<float2> d_tw;     // exp(-2 pi j k / nfft), k < nfft (forward table; kernels conjugate for inverse)
    MixedPlan mixed;
};

struct lrc_psd {
    lrc_ctx *ctx;
    int      nfft, log2n;
    DevBuf<float2> d_tw;
    DevBuf<float>  d_win;        // nfft window values (all ones for LRC_WINDOW_NONE)
    DevBuf<float>  d_partial;    // [n_items][nfft] scratch
};

// twiddles exactly as kiss_fft_alloc builds them (kiss_fft.c:357-363): phase in double, cast to float
int lrc_make_twiddles(int nfft, DevBuf<float2> &d_tw)
{
    std::vector<float2> tw(nfft);
    const double pi = 3.141592653589793238462643383279502884197169399375105820974944;
    for (int i = 0; i < nfft; ++i) {
        double ph = -2.0 * pi * i / nfft;
        tw[i] = make_float2((float)cos(ph), (float)sin(ph));
    }
    LRC_CUDA(d_tw.alloc(nfft));
    LRC_CUDA(cudaMemcpy(d_tw, tw.data(), sizeof(float2) * nfft, cudaMemcpyHostToDevice));
    return LRC_OK;
}

int lrc_log2_exact(int n)
{
    int l = 0;
    while ((1 << l) < n) ++l;
    return ((1 << l) == n) ? l : -1;
}

// ---------------------------------------------------------------------------------------------
// batched FFT: G = blockDim/T transforms per CTA, grid-stride over the batch
// ---------------------------------------------------------------------------------------------
template <int LOG2N, bool INV>
__global__ void __launch_bounds__((1 << LOG2N) / 16 > 128 ? (1 << LOG2N) / 16 : 128)
fft_batch_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, size_t batch,
                 const float2 *__restrict__ tw)
{
    using F = CtaFFT<LOG2N, INV>;
    constexpr int N = F::N, E = F::E, T = F::T;
    extern __shared__ float2 sm_all[];
    const int G = blockDim.x / T;
    const int g = threadIdx.x / T, t = threadIdx.x % T;
    float2 *sm = sm_all + (size_t)g * F::SMEM_CPX;
    for (size_t base = (size_t)blockIdx.x * G; base < batch; base += (size_t)gridDim.x * G) {
        const size_t f = base + g;
        const bool active = f < batch;
        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = active ? in[f * N + t + e * T] : make_float2(0.f, 0.f);
        F::run(v, sm, tw, t, SyncCta{});
        if (active) {
#pragma unroll
            for (int e = 0; e < E; ++e) out[f * N + t + e * T] = v[e];
        }
    }
}

// batched FFT with TMA-staged input (N = 512..2048, 16-byte aligned input): each transform group keeps
// FFT_STAGES-1 frame loads in flight in its own shared-memory ring; results go straight from registers to
// global memory in the coalesced "thread t holds X[t + e*T]" layout.
constexpr int FFT_STAGES = 3;

template <int LOG2N, bool INV>
struct FftTmaCfg {
    using F = CtaFFT<LOG2N, INV>;
    static constexpr int THREADS = F::T > 128 ? F::T : 128;
    static constexpr int G = THREADS / F::T;
    static constexpr int FRAME_BYTES = F::N * 8;
    static constexpr int GROUP_BYTES = ((FFT_STAGES * FRAME_BYTES + F::SMEM_CPX * 8 + FFT_STAGES * 8) + 127) / 128 * 128;
    static constexpr int SMEM_BYTES = G * GROUP_BYTES;
};

template <int LOG2N, bool INV>
__global__ void __launch_bounds__(FftTmaCfg<LOG2N, INV>::THREADS)
fft_tma_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, size_t batch, const float2 *__restrict__ tw)
{
    using Cfg = FftTmaCfg<LOG2N, INV>;
    using F = CtaFFT<LOG2N, INV>;
    constexpr int N = F::N, E = F::E, T = F::T, G = Cfg::G;
    extern __shared__ __align__(128) uint8_t fft_smem[];
    const int g = threadIdx.x / T, t = threadIdx.x % T;
    uint8_t *gbase = fft_smem + (size_t)g * Cfg::GROUP_BYTES;
    float2 *stg = reinterpret_cast<float2 *>(gbase);
    float2 *sm = reinterpret_cast<float2 *>(gbase + FFT_STAGES * Cfg::FRAME_BYTES);
    uint64_t *bars = reinterpret_cast<uint64_t *>(gbase + FFT_STAGES * Cfg::FRAME_BYTES + F::SMEM_CPX * 8);
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < FFT_STAGES; ++i) mbar_init(&bars[i], 1);
        mbar_fence_init();
    }
    __syncthreads();
    float2 twr[F::TW_REGS];
    F::load_twiddles(tw, t, twr);
    const size_t stride = (size_t)gridDim.x * G;
    size_t f = (size_t)blockIdx.x * G + g;                 // current frame of this group
    size_t fa = f;                                         // next frame to request
    int requested = 0;
    auto request = [&]() {
        const int stage = requested % FFT_STAGES;
        mbar_expect_tx(&bars[stage], Cfg::FRAME_BYTES);
        tma_load_1d_evict_first(stg + (size_t)stage * N, in + fa * N, Cfg::FRAME_BYTES, &bars[stage]);
        ++requested;
        fa += stride;
    };
    if (t == 0)
        for (int i = 0; i < FFT_STAGES - 1 && fa < batch; ++i) request();
    for (int i = 0; f < batch; ++i, f += stride) {
        const int stage = i % FFT_STAGES;
        if (t == 0 && fa < batch) request();
        mbar_wait(&bars[stage], (uint32_t)((i / FFT_STAGES) & 1));
        float2 v[E];
        const float2 *src = stg + (size_t)stage * N + t;
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = src[e * T];
        F::run_twreg(v, sm, twr, t, SyncNamed{1 + g, T});
        float2 *dst = out + f * N + t;
#pragma unroll
        for (int e = 0; e < E; ++e) __stcs(dst + e * T, v[e]);
    }
}

// N = 1024, one warp per transform (WarpFFT1024): global -> registers -> one exchange -> registers -> global.
// In-place calls are safe: a warp has its whole frame in registers before it stores anything.
constexpr int FFTW_WARPS = 4;
constexpr int FFTW_SMEM_BYTES = (FFTW_WARPS * WarpFFT1024<false>::SMEM_CPX + WarpFFT1024<false>::TW_CPX) * 8;

template <bool INV>
__global__ void __launch_bounds__(FFTW_WARPS * 32, 4)
fft1024_warp_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, size_t batch, const float2 *__restrict__ tw)
{
    using F = WarpFFT1024<INV>;
    extern __shared__ __align__(16) float2 fftw_sm[];
    float2 *tws = fftw_sm + FFTW_WARPS * F::SMEM_CPX;
    F::fill_twiddles(tw, tws);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float2 *xb = fftw_sm + warp * F::SMEM_CPX;
    const size_t stride = (size_t)gridDim.x * FFTW_WARPS;
    for (size_t f = (size_t)blockIdx.x * FFTW_WARPS + warp; f < batch; f += stride) {
        float2 v[32];
        const float2 *src = in + f * 1024 + lane;
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = __ldcs(src + 32 * e);
        if (f + stride < batch) {
            const char *nx = reinterpret_cast<const char *>(in + (f + stride) * 1024) + lane * 256;
            asm volatile("prefetch.global.L2 [%0];" :: "l"(nx));
            asm volatile("prefetch.global.L2 [%0];" :: "l"(nx + 128));
        }
        F::run(v, xb, tws, lane);
        float2 *dst = out + f * 1024 + lane;
#pragma unroll
        for (int e = 0; e < 32; ++e) __stcs(dst + 32 * e, v[e]);
    }
}

// N = 1024 always runs the warp kernel, so launch_fft is never instantiated for it
template <bool INV>
static int launch_fft1024(const lrc_fft *p, const float2 *in, float2 *out, size_t batch, cudaStream_t s)
{
    auto kern = fft1024_warp_kernel<INV>;
    size_t ctas;
    LRC_CUDA(lrc_resident_ctas(kern, FFTW_WARPS * 32, FFTW_SMEM_BYTES, p->ctx->n_sm, &ctas));
    size_t blocks = ceil_div(batch, (size_t)FFTW_WARPS);
    static const size_t gm = lrc_grid_mult("LRC_FFT_GRID", 32);
    const size_t max_blocks = ctas * gm;
    if (blocks > max_blocks) blocks = max_blocks;
    kern<<<(unsigned)blocks, FFTW_WARPS * 32, FFTW_SMEM_BYTES, s>>>(in, out, batch, p->d_tw);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

template <int LOG2N, bool INV>
static int launch_fft(const lrc_fft *p, const float2 *in, float2 *out, size_t batch, cudaStream_t s)
{
    using F = CtaFFT<LOG2N, INV>;
    constexpr int T = F::T;
    if constexpr (T >= 32 && T <= 128) {
        // in-place calls are safe here too: a frame is fully in shared memory before its slot is written
        if (((uintptr_t)in & 15) == 0 && batch >= 64) {
            using Cfg = FftTmaCfg<LOG2N, INV>;
            auto kern = fft_tma_kernel<LOG2N, INV>;
            size_t max_blocks;
            LRC_CUDA(lrc_resident_ctas(kern, Cfg::THREADS, Cfg::SMEM_BYTES, p->ctx->n_sm, &max_blocks));
            size_t blocks = ceil_div(batch, (size_t)Cfg::G);
            if (blocks > max_blocks) blocks = max_blocks;
            kern<<<(unsigned)blocks, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(in, out, batch, p->d_tw);
            LRC_CUDA(cudaGetLastError());
            return LRC_OK;
        }
    }
    const int threads = T > 128 ? T : 128;
    const int G = threads / T;
    const size_t smem = (size_t)G * F::SMEM_CPX * sizeof(float2);
    auto kern = fft_batch_kernel<LOG2N, INV>;
    if (smem > 48 * 1024) LRC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    size_t blocks = ceil_div(batch, (size_t)G);
    const size_t max_blocks = (size_t)p->ctx->n_sm * 16;
    if (blocks > max_blocks) blocks = max_blocks;
    kern<<<(unsigned)blocks, threads, smem, s>>>(in, out, batch, p->d_tw);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

template <bool INV>
static int dispatch_fft(const lrc_fft *p, const float2 *in, float2 *out, size_t batch, cudaStream_t s)
{
    switch (p->log2n) {
        case 1:  return launch_fft<1, INV>(p, in, out, batch, s);
        case 2:  return launch_fft<2, INV>(p, in, out, batch, s);
        case 3:  return launch_fft<3, INV>(p, in, out, batch, s);
        case 4:  return launch_fft<4, INV>(p, in, out, batch, s);
        case 5:  return launch_fft<5, INV>(p, in, out, batch, s);
        case 6:  return launch_fft<6, INV>(p, in, out, batch, s);
        case 7:  return launch_fft<7, INV>(p, in, out, batch, s);
        case 8:  return launch_fft<8, INV>(p, in, out, batch, s);
        case 9:  return launch_fft<9, INV>(p, in, out, batch, s);
        case 10: return launch_fft1024<INV>(p, in, out, batch, s);
        case 11: return launch_fft<11, INV>(p, in, out, batch, s);
        case 12: return launch_fft<12, INV>(p, in, out, batch, s);
        case 13: return launch_fft<13, INV>(p, in, out, batch, s);
    }
    lrc_set_error("nfft=%d not supported", p->nfft);
    return LRC_ERR_UNSUPPORTED;
}

extern "C" int lrc_fft_create(lrc_ctx *ctx, int nfft, int inverse, lrc_fft **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out != nullptr && nfft >= 1, LRC_ERR_INVALID, "lrc_fft_create: bad arguments");
    int l2 = lrc_log2_exact(nfft);
    MixedPlan mp{};
    if (nfft == 1 || l2 > 13) {
        lrc_set_error("lrc_fft_create: nfft=%d: supported sizes are 2..8192", nfft);
        return LRC_ERR_UNSUPPORTED;
    }
    if (l2 < 1) {
        // not a power of two: kissfft's mixed-radix sizes (kf_factor, kiss_fft.c:309-330)
        if (nfft > MIXED_MAX_NFFT || lrc_fft_mixed_factor(nfft, &mp) != 0) {
            lrc_set_error("lrc_fft_create: nfft=%d: sizes that are not powers of two are supported up to %d",
                          nfft, MIXED_MAX_NFFT);
            return LRC_ERR_UNSUPPORTED;
        }
        l2 = -1;
    }
    lrc_fft *p = new (std::nothrow) lrc_fft();
    LRC_REQUIRE(p != nullptr, LRC_ERR_NOMEM, "out of host memory");
    p->ctx = ctx; p->nfft = nfft; p->log2n = l2; p->inverse = inverse ? 1 : 0; p->mixed = mp;
    int rc = lrc_make_twiddles(nfft, p->d_tw);
    if (rc) { lrc_fft_destroy(p); return rc; }
    *out = p;
    return LRC_OK;
}

extern "C" int lrc_fft_destroy(lrc_fft *p)
{
    if (!p) return LRC_OK;
    cudaSetDevice(p->ctx->device);
    delete p;
    return LRC_OK;
}

extern "C" int lrc_fft_run(lrc_fft *p, const float *d_in, float *d_out, size_t batch, void *stream)
{
    LRC_REQUIRE(p != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(p->ctx);
    if (batch == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_out, LRC_ERR_INVALID, "lrc_fft_run: null buffer");
    LRC_REQUIRE(((uintptr_t)d_in & 7) == 0 && ((uintptr_t)d_out & 7) == 0, LRC_ERR_INVALID,
                "lrc_fft_run: buffers must be 8-byte aligned");
    cudaStream_t s = lrc_stream(p->ctx, stream);
    if (p->log2n < 0)
        return lrc_fft_mixed_launch(p->ctx, p->nfft, p->inverse, &p->mixed, p->d_tw, (const float2 *)d_in,
                                    (float2 *)d_out, batch, s);
    return p->inverse ? dispatch_fft<true>(p, (const float2 *)d_in, (float2 *)d_out, batch, s)
                      : dispatch_fft<false>(p, (const float2 *)d_in, (float2 *)d_out, batch, s);
}

extern "C" int lrc_fft_run_host(lrc_fft *p, const float *h_in, float *h_out, size_t n_samples)
{
    LRC_REQUIRE(p != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(p->ctx);
    if (n_samples % (size_t)p->nfft != 0) {
        // assert!(din.len() == block_size)  src/kissfft/src/kissfft.rs:24
        lrc_set_error("lrc_fft_run_host: %zu samples is not a multiple of block_size %d", n_samples, p->nfft);
        return LRC_ERR_LENGTH;
    }
    if (n_samples == 0) return LRC_OK;
    LRC_REQUIRE(h_in && h_out, LRC_ERR_INVALID, "null buffer");
    float *d = nullptr;
    const size_t bytes = n_samples * sizeof(float2);
    LRC_CUDA(cudaMalloc(&d, bytes));
    cudaStream_t s = p->ctx->stream;
    cudaError_t e = cudaMemcpyAsync(d, h_in, bytes, cudaMemcpyHostToDevice, s);
    int rc = LRC_OK;
    if (e == cudaSuccess) rc = lrc_fft_run(p, d, d, n_samples / p->nfft, s);
    if (e == cudaSuccess && rc == LRC_OK) e = cudaMemcpyAsync(h_out, d, bytes, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(d);
    if (e != cudaSuccess) { lrc_set_error("lrc_fft_run_host: %s", cudaGetErrorString(e)); return LRC_ERR_CUDA; }
    return rc;
}

// ---------------------------------------------------------------------------------------------
// window + FFT + |X|^2 accumulate.  Work item = `fpi` consecutive frames inside one row; each
// transform group of a CTA walks its items, accumulating |X|^2 in registers, and writes one
// partial spectrum per item; psd_reduce_kernel sums the partials of a row in fixed order.
// ---------------------------------------------------------------------------------------------
template <int LOG2N>
__global__ void __launch_bounds__((1 << LOG2N) / 16 > 128 ? (1 << LOG2N) / 16 : 128)
psd_kernel(const float2 *__restrict__ in, const float2 *__restrict__ tw, const float *__restrict__ win,
           float *__restrict__ partial, size_t k_avg, size_t fpi, size_t ipr, size_t n_items)
{
    using F = CtaFFT<LOG2N, false>;
    constexpr int N = F::N, E = F::E, T = F::T;
    extern __shared__ float2 sm_all[];
    const int G = blockDim.x / T;
    const int g = threadIdx.x / T, t = threadIdx.x % T;
    float2 *sm = sm_all + (size_t)g * F::SMEM_CPX;
    float w[E];
#pragma unroll
    for (int e = 0; e < E; ++e) w[e] = win[t + e * T];
    float2 twr[F::TW_REGS];                       // this thread's twiddles never change: fetch them once
    F::load_twiddles(tw, t, twr);

    for (size_t item = (size_t)blockIdx.x * G + g; item < n_items; item += (size_t)gridDim.x * G) {
        const size_t row = item / ipr, c = item % ipr;
        const size_t f0 = row * k_avg + c * fpi;
        size_t f1 = f0 + fpi;
        if (f1 > (row + 1) * k_avg) f1 = (row + 1) * k_avg;
        float acc[E];
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = 0.f;
        for (size_t f = f0; f < f1; ++f) {
            float2 v[E];
            const float2 *src = in + f * N + t;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                float2 x = __ldcs(src + e * T);
                v[e] = mul2(x, make_float2(w[e], w[e]));
            }
            if constexpr (T >= 32) {
                F::run_twreg(v, sm, twr, t, SyncNamed{1 + g, T});
            } else {
                const unsigned lane = threadIdx.x & 31;
                const unsigned mask = (T == 32) ? 0xffffffffu : (((1u << T) - 1u) << (lane / T * T));
                F::run_twreg(v, sm, twr, t, SyncWarp{mask});
            }
#pragma unroll
            for (int e = 0; e < E; ++e) acc[e] = fmaf(v[e].x, v[e].x, fmaf(v[e].y, v[e].y, acc[e]));
        }
        float *dst = partial + item * N + t;
#pragma unroll
        for (int e = 0; e < E; ++e) dst[e * T] = acc[e];
    }
}

// Same work, frames staged by the TMA engine: every transform group owns a PSD_STAGES-deep ring of frame
// buffers in shared memory; its leader thread keeps PSD_STAGES-1 bulk copies in flight while the group
// transforms the current frame, so HBM latency is hidden inside the group instead of by occupancy alone.
// Used for N = 512 and 2048 (T = 32 and 128 threads per transform) when the input is 16-byte aligned.
constexpr int PSD_STAGES = 3;

template <int LOG2N>
struct PsdTmaCfg {
    using F = CtaFFT<LOG2N, false>;
    static constexpr int THREADS = F::T > 128 ? F::T : 128;
    static constexpr int G = THREADS / F::T;
    static constexpr int FRAME_BYTES = F::N * 8;
    static constexpr int GROUP_BYTES = ((PSD_STAGES * FRAME_BYTES + F::SMEM_CPX * 8 + PSD_STAGES * 8) + 127) / 128 * 128;
    static constexpr int SMEM_BYTES = G * GROUP_BYTES;
};

template <int LOG2N>
__global__ void __launch_bounds__(PsdTmaCfg<LOG2N>::THREADS, 3)
psd_tma_kernel(const float2 *__restrict__ in, const float2 *__restrict__ tw, const float *__restrict__ win,
               float *__restrict__ partial, size_t k_avg, size_t fpi, size_t ipr, size_t n_items)
{
    using Cfg = PsdTmaCfg<LOG2N>;
    using F = CtaFFT<LOG2N, false>;
    constexpr int N = F::N, E = F::E, T = F::T, G = Cfg::G;
    extern __shared__ __align__(128) uint8_t psd_smem[];
    const int g = threadIdx.x / T, t = threadIdx.x % T;
    uint8_t *gbase = psd_smem + (size_t)g * Cfg::GROUP_BYTES;
    float2 *stg = reinterpret_cast<float2 *>(gbase);
    float2 *sm = reinterpret_cast<float2 *>(gbase + PSD_STAGES * Cfg::FRAME_BYTES);
    uint64_t *bars = reinterpret_cast<uint64_t *>(gbase + PSD_STAGES * Cfg::FRAME_BYTES + F::SMEM_CPX * 8);
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < PSD_STAGES; ++i) mbar_init(&bars[i], 1);
        mbar_fence_init();
    }
    __syncthreads();

    float w[E];
#pragma unroll
    for (int e = 0; e < E; ++e) w[e] = win[t + e * T];
    float2 twr[F::TW_REGS];
    F::load_twiddles(tw, t, twr);

    // the group's frame sequence: items item0, item0 + stride, ...; frames f0..f1-1 inside each
    const size_t stride = (size_t)gridDim.x * G;
    auto item_range = [&](size_t item, size_t &f0, size_t &f1) {
        const size_t row = item / ipr, c = item % ipr;
        f0 = row * k_avg + c * fpi;
        f1 = f0 + fpi;
        if (f1 > (row + 1) * k_avg) f1 = (row + 1) * k_avg;
    };
    struct Cursor { size_t item, f, f1; };
    auto advance = [&](Cursor &c) {
        if (++c.f == c.f1) {
            c.item += stride;
            if (c.item < n_items) item_range(c.item, c.f, c.f1);
        }
    };
    Cursor cur{(size_t)blockIdx.x * G + g, 0, 0};
    if (cur.item >= n_items) return;
    item_range(cur.item, cur.f, cur.f1);
    Cursor ahead = cur;                                   // next frame to request
    int requested = 0;
    auto request = [&]() {                                // leader only
        const int stage = requested % PSD_STAGES;
        mbar_expect_tx(&bars[stage], Cfg::FRAME_BYTES);
        tma_load_1d_evict_first(stg + (size_t)stage * N, in + ahead.f * N, Cfg::FRAME_BYTES, &bars[stage]);
        ++requested;
        advance(ahead);
    };
    if (t == 0)
        for (int i = 0; i < PSD_STAGES - 1 && ahead.item < n_items; ++i) request();

    float acc[E];
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] = 0.f;
    for (int i = 0; cur.item < n_items; ++i) {
        const int stage = i % PSD_STAGES;
        // the stage being refilled now was read (into registers) one iteration ago, and every thread has
        // passed a group barrier of that transform since
        if (t == 0 && ahead.item < n_items) request();
        mbar_wait(&bars[stage], (uint32_t)((i / PSD_STAGES) & 1));
        float2 v[E];
        const float2 *src = stg + (size_t)stage * N + t;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const float2 x = src[e * T];
            v[e] = mul2(x, make_float2(w[e], w[e]));
        }
        F::run_twreg(v, sm, twr, t, SyncNamed{1 + g, T});
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = fmaf(v[e].x, v[e].x, fmaf(v[e].y, v[e].y, acc[e]));
        if (cur.f + 1 == cur.f1) {                        // last frame of the item: hand the partial spectrum out
            float *dst = partial + cur.item * N + t;
#pragma unroll
            for (int e = 0; e < E; ++e) { dst[e * T] = acc[e]; acc[e] = 0.f; }
        }
        advance(cur);
    }
}

// N = 1024, one WARP per transform (WarpFFT1024): frames go straight from global memory into registers (the
// next frame is prefetched into L2 while this one is transformed), one shared-memory exchange per frame, no
// barrier between warps.  Shared-memory traffic per point: 16 B exchange + 4 B window, against 48 B for the
// TMA-staged CTA-level kernel above, which is bound by exactly that.
constexpr int PSDW_WARPS = 4;
constexpr int PSDW_SMEM_BYTES = (PSDW_WARPS * WarpFFT1024<false>::SMEM_CPX + WarpFFT1024<false>::TW_CPX) * 8 + 1024 * 4;

__device__ __forceinline__ void prefetch_l2(const void *p)
{
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
}

__global__ void __launch_bounds__(PSDW_WARPS * 32, 3)
psd1024_warp_kernel(const float2 *__restrict__ in, const float2 *__restrict__ tw, const float *__restrict__ win,
                    float *__restrict__ partial, size_t k_avg, size_t fpi, size_t ipr, size_t n_items)
{
    using F = WarpFFT1024<false>;
    constexpr int N = 1024;
    extern __shared__ __align__(16) float2 psdw_sm[];
    float2 *tws = psdw_sm + PSDW_WARPS * F::SMEM_CPX;
    float *wsm = reinterpret_cast<float *>(tws + F::TW_CPX);
    for (int i = threadIdx.x; i < N; i += blockDim.x) wsm[i] = win[i];
    F::fill_twiddles(tw, tws);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float2 *xb = psdw_sm + warp * F::SMEM_CPX;
    const float *wl = wsm + lane;

    const size_t stride = (size_t)gridDim.x * PSDW_WARPS;
    for (size_t item = (size_t)blockIdx.x * PSDW_WARPS + warp; item < n_items; item += stride) {
        const size_t row = item / ipr, c = item % ipr;
        const size_t f0 = row * k_avg + c * fpi;
        size_t f1 = f0 + fpi;
        if (f1 > (row + 1) * k_avg) f1 = (row + 1) * k_avg;
        // first frame of this warp's next item, for the prefetch issued during the last frame of this one
        size_t fnext_item = 0;
        const bool has_next = item + stride < n_items;
        if (has_next) {
            const size_t it2 = item + stride;
            fnext_item = (it2 / ipr) * k_avg + (it2 % ipr) * fpi;
        }
        float acc[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) acc[e] = 0.f;
        for (size_t f = f0; f < f1; ++f) {
            float2 v[32];
            const float2 *src = in + f * N + lane;
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __ldcs(src + 32 * e);
            {   // next frame -> L2: 8 KB = 64 lines of 128 B, two per lane
                const bool more = f + 1 < f1;
                if (more || has_next) {
                    const char *nx = reinterpret_cast<const char *>(in + (more ? f + 1 : fnext_item) * N) + lane * 256;
                    prefetch_l2(nx); prefetch_l2(nx + 128);
                }
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const float w = wl[32 * e];
                v[e] = mul2(v[e], make_float2(w, w));
            }
            F::run(v, xb, tws, lane);
#pragma unroll
            for (int e = 0; e < 32; ++e) acc[e] = fmaf(v[e].x, v[e].x, fmaf(v[e].y, v[e].y, acc[e]));
        }
        float *dst = partial + item * N + lane;
#pragma unroll
        for (int e = 0; e < 32; ++e) dst[32 * e] = acc[e];
    }
}

__global__ void psd_reduce_kernel(const float *__restrict__ partial, float *__restrict__ rows, int nfft,
                                  size_t ipr, size_t n_rows, float scale, int accumulate)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * (size_t)nfft) return;
    const size_t row = i / nfft, b = i % nfft;
    const float *p = partial + row * ipr * nfft + b;
    float s = 0.f;
    for (size_t c = 0; c < ipr; ++c) s += p[c * nfft];
    s *= scale;
    rows[i] = accumulate ? rows[i] + s : s;
}

template <int LOG2N>
static int launch_psd(lrc_psd *p, const float2 *in, size_t k_avg, size_t fpi, size_t ipr, size_t n_items,
                      cudaStream_t s)
{
    using F = CtaFFT<LOG2N, false>;
    constexpr int T = F::T;
    if constexpr (T >= 32 && T <= 128) {            // N = 512 .. 2048: the ring fits several CTAs per SM
        if (((uintptr_t)in & 15) == 0) {
            if constexpr (LOG2N == 10) {
                auto kern = psd1024_warp_kernel;
                size_t ctas;
                LRC_CUDA(lrc_resident_ctas(kern, PSDW_WARPS * 32, PSDW_SMEM_BYTES, p->ctx->n_sm, &ctas));
                size_t blocks = ceil_div(n_items, (size_t)PSDW_WARPS);
                static const size_t gm = lrc_grid_mult("LRC_PSD_GRID", 16);
                const size_t max_blocks = ctas * gm;
                if (blocks > max_blocks) blocks = max_blocks;
                kern<<<(unsigned)blocks, PSDW_WARPS * 32, PSDW_SMEM_BYTES, s>>>(in, p->d_tw, p->d_win, p->d_partial, k_avg, fpi, ipr, n_items);
                LRC_CUDA(cudaGetLastError());
                return LRC_OK;
            } else {
                using Cfg = PsdTmaCfg<LOG2N>;
                auto kern = psd_tma_kernel<LOG2N>;
                size_t max_blocks;
                LRC_CUDA(lrc_resident_ctas(kern, Cfg::THREADS, Cfg::SMEM_BYTES, p->ctx->n_sm, &max_blocks));
                size_t blocks = ceil_div(n_items, (size_t)Cfg::G);
                if (blocks > max_blocks) blocks = max_blocks;
                kern<<<(unsigned)blocks, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(in, p->d_tw, p->d_win, p->d_partial, k_avg, fpi, ipr, n_items);
                LRC_CUDA(cudaGetLastError());
                return LRC_OK;
            }
        }
    }
    const int threads = T > 128 ? T : 128;
    const int G = threads / T;
    const size_t smem = (size_t)G * F::SMEM_CPX * sizeof(float2);
    auto kern = psd_kernel<LOG2N>;
    size_t max_blocks;
    LRC_CUDA(lrc_resident_ctas(kern, threads, smem, p->ctx->n_sm, &max_blocks, true));
    size_t blocks = ceil_div(n_items, (size_t)G);
    if (blocks > max_blocks) blocks = max_blocks;
    kern<<<(unsigned)blocks, threads, smem, s>>>(in, p->d_tw, p->d_win, p->d_partial, k_avg, fpi, ipr, n_items);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

extern "C" int lrc_psd_create(lrc_ctx *ctx, int nfft, int window, lrc_psd **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out != nullptr, LRC_ERR_INVALID, "lrc_psd_create: null out");
    const int l2 = lrc_log2_exact(nfft);
    if (l2 < 1 || l2 > 13) {
        lrc_set_error("lrc_psd_create: nfft=%d: only powers of two in [2, 8192]", nfft);
        return LRC_ERR_UNSUPPORTED;
    }
    LRC_REQUIRE(window == LRC_WINDOW_NONE || window == LRC_WINDOW_HANN, LRC_ERR_INVALID, "unknown window");
    lrc_psd *p = new (std::nothrow) lrc_psd();
    LRC_REQUIRE(p != nullptr, LRC_ERR_NOMEM, "out of host memory");
    p->ctx = ctx; p->nfft = nfft; p->log2n = l2;
    int rc = lrc_make_twiddles(nfft, p->d_tw);
    if (rc) { lrc_psd_destroy(p); return rc; }
    std::vector<float> w(nfft);
    const double pi = 3.14159265358979323846264338327950288;
    for (int i = 0; i < nfft; ++i)
        w[i] = window == LRC_WINDOW_HANN ? (float)(0.5 - 0.5 * cos(2.0 * pi * i / nfft)) : 1.0f;
    if (p->d_win.alloc(nfft) != cudaSuccess) { lrc_psd_destroy(p); lrc_set_error("cudaMalloc window"); return LRC_ERR_CUDA; }
    rc = lrc_psd_set_window(p, w.data());
    if (rc) { lrc_psd_destroy(p); return rc; }
    *out = p;
    return LRC_OK;
}

extern "C" int lrc_psd_set_window(lrc_psd *p, const float *h_window)
{
    LRC_REQUIRE(p && h_window, LRC_ERR_INVALID, "lrc_psd_set_window: null");
    LRC_BIND(p->ctx);
    LRC_CUDA(cudaMemcpy(p->d_win, h_window, sizeof(float) * p->nfft, cudaMemcpyHostToDevice));
    return LRC_OK;
}

extern "C" int lrc_psd_destroy(lrc_psd *p)
{
    if (!p) return LRC_OK;
    cudaSetDevice(p->ctx->device);
    delete p;
    return LRC_OK;
}

// frames per work item: small enough that items outnumber resident transform groups several times,
// large enough that the 4*nfft-byte partial written per item is noise next to fpi*8*nfft bytes read
size_t lrc_psd_frames_per_item(size_t k_avg) { return k_avg < 16 ? (k_avg ? k_avg : 1) : 16; }

int lrc_psd_reduce(const float *d_partial, float *d_rows, int nfft, size_t ipr, size_t n_rows, float scale,
                   int accumulate, cudaStream_t s)
{
    const size_t n = n_rows * (size_t)nfft;
    psd_reduce_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(d_partial, d_rows, nfft, ipr, n_rows, scale, accumulate);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

extern "C" int lrc_psd_run(lrc_psd *p, const float *d_in, size_t n_frames, size_t k_avg, float *d_rows,
                           void *stream)
{
    LRC_REQUIRE(p != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(p->ctx);
    LRC_REQUIRE(k_avg >= 1, LRC_ERR_INVALID, "lrc_psd_run: k_avg must be >= 1");
    const size_t n_rows = n_frames / k_avg;
    if (n_rows == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_rows, LRC_ERR_INVALID, "lrc_psd_run: null buffer");
    LRC_REQUIRE(((uintptr_t)d_in & 7) == 0, LRC_ERR_INVALID, "lrc_psd_run: input must be 8-byte aligned");
    cudaStream_t s = lrc_stream(p->ctx, stream);
    // the grouping of frames into items is a function of k_avg alone, so results do not depend on the launch
    // or on how a stream is sharded (finer items were measured slower: 16 -> 8 costs 2 %, -> 4 costs 9 %)
    const size_t fpi = lrc_psd_frames_per_item(k_avg);
    const size_t ipr = ceil_div(k_avg, fpi);
    const size_t n_items = n_rows * ipr;
    LRC_CUDA(p->d_partial.ensure(n_items * (size_t)p->nfft));
    int rc;
    const float2 *in = (const float2 *)d_in;
    switch (p->log2n) {
#define PSD_CASE(L) case L: rc = launch_psd<L>(p, in, k_avg, fpi, ipr, n_items, s); break;
        PSD_CASE(1) PSD_CASE(2) PSD_CASE(3) PSD_CASE(4) PSD_CASE(5) PSD_CASE(6) PSD_CASE(7)
        PSD_CASE(8) PSD_CASE(9) PSD_CASE(10) PSD_CASE(11) PSD_CASE(12) PSD_CASE(13)
#undef PSD_CASE
        default: rc = LRC_ERR_UNSUPPORTED;
    }
    if (rc) return rc;
    return lrc_psd_reduce(p->d_partial, d_rows, p->nfft, ipr, n_rows, 1.0f / (float)k_avg, 0, s);
}
