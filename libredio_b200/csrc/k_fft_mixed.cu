// k_fft_mixed.cu -- the rest of the kissfft surface: transform sizes that are not powers of two, and the
// real-input transform pair.
//
//  * any nfft = 2^a 3^b 5^c x (odd primes): kissfft factors 4s, then 2, 3, 5, then the remaining odd
//    primes through its generic butterfly (libkissfft/kiss_fft.c:21-235 kf_bfly2/3/4/5/generic, :309-330
//    kf_factor).  Here: one CTA per transform, the frame lives in two shared-memory buffers and every
//    pass is a Stockham (auto-sort) pass, so input and output are in natural order and d_in == d_out works.
//    Twiddles come from the same length-nfft table kiss_fft_alloc builds (phase in double, cast to float,
//    :357-363).  This is the coverage path (sizes LibRedio's block accepts through kiss_fft_alloc); the
//    power-of-two kernels of k_fft.cu stay the fast path.
//  * kiss_fftr / kiss_fftri (libkissfft/tools/kiss_fftr.c:67-159): nfft real points <-> nfft/2+1 bins via
//    one complex transform of nfft/2 points plus the split/merge butterfly with the "super twiddles"
//    exp(-+ j pi ((k+1)/ncfft + 1/2)) (:57-64).  Unscaled in both directions like the reference.
#include "fft_core.cuh"
#include <cmath>
#include <vector>

using namespace lrfft;

struct lrc_fft;                                   // k_fft.cu

constexpr int MIXED_MAX_FACTORS = 24;
constexpr int MIXED_MAX_NFFT = 8192;              // 2 x nfft x 8 B of shared memory
struct MixedPlan { int nfac; int radix[MIXED_MAX_FACTORS]; };

// kf_factor (kiss_fft.c:309-330): 4s first, then 2, 3, 5, 7, 9...; p*p > n -> n itself
int lrc_fft_mixed_factor(int n, MixedPlan *mp)
{
    int p = 4;
    mp->nfac = 0;
    const double floor_sqrt = floor(sqrt((double)n));
    do {
        while (n % p) {
            switch (p) {
                case 4: p = 2; break;
                case 2: p = 3; break;
                default: p += 2; break;
            }
            if (p > floor_sqrt) p = n;
        }
        n /= p;
        if (mp->nfac >= MIXED_MAX_FACTORS) return -1;
        mp->radix[mp->nfac++] = p;
    } while (n > 1);
    return 0;
}

template <bool INV>
__device__ __forceinline__ float2 tw_get(const float2 *__restrict__ tw, int idx)
{
    float2 w = __ldg(tw + idx);
    if (INV) w.y = -w.y;
    return w;
}

// one Stockham pass of radix P over the frame in `src` -> `dst`.  ns = product of the radices already done.
template <int P, bool INV>
__device__ __forceinline__ void mixed_pass(const float2 *src, float2 *dst, int n, int ns, const float2 *__restrict__ tw)
{
    const int m = n / P;
    const int twstep = n / (ns * P);
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const int k = j % ns;
        float2 v[P];
#pragma unroll
        for (int r = 0; r < P; ++r) {
            v[r] = src[j + r * m];
            if (r && ns > 1) v[r] = cmulf(v[r], tw_get<INV>(tw, r * k * twstep));
        }
        float2 *o = dst + (j - k) * P + k;
        if constexpr (P == 2) {
            o[0] = cadd(v[0], v[1]);
            o[ns] = csub(v[0], v[1]);
        } else if constexpr (P == 4) {
            bfly4<INV>(v[0], v[1], v[2], v[3]);
            o[0] = v[0]; o[ns] = v[1]; o[2 * ns] = v[2]; o[3 * ns] = v[3];
        } else if constexpr (P == 3) {
            constexpr float S = 0.86602540378443864676f;             // sin(2 pi / 3)
            const float2 a = cadd(v[1], v[2]), d = csub(v[1], v[2]);
            const float2 t = make_float2(v[0].x - 0.5f * a.x, v[0].y - 0.5f * a.y);
            // forward: -j S d ; inverse: +j S d
            const float2 u = INV ? make_float2(-S * d.y, S * d.x) : make_float2(S * d.y, -S * d.x);
            o[0] = cadd(v[0], a);
            o[ns] = cadd(t, u);
            o[2 * ns] = csub(t, u);
        } else {   // P == 5
            constexpr float C1 = 0.30901699437494742410f, C2 = -0.80901699437494742410f;   // cos(2pi/5), cos(4pi/5)
            constexpr float S1 = 0.95105651629515357212f, S2 = 0.58778525229247312917f;    // sin(2pi/5), sin(4pi/5)
            const float2 a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
            const float2 b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
            const float2 t1 = make_float2(v[0].x + C1 * a1.x + C2 * a2.x, v[0].y + C1 * a1.y + C2 * a2.y);
            const float2 t2 = make_float2(v[0].x + C2 * a1.x + C1 * a2.x, v[0].y + C2 * a1.y + C1 * a2.y);
            const float2 u1 = make_float2(S1 * b1.x + S2 * b2.x, S1 * b1.y + S2 * b2.y);
            const float2 u2 = make_float2(S2 * b1.x - S1 * b2.x, S2 * b1.y - S1 * b2.y);
            // forward: t -+ j u  (-j u = (u.y, -u.x)); inverse: the other sign
            const float2 ju1 = INV ? make_float2(-u1.y, u1.x) : make_float2(u1.y, -u1.x);
            const float2 ju2 = INV ? make_float2(-u2.y, u2.x) : make_float2(u2.y, -u2.x);
            o[0] = make_float2(v[0].x + a1.x + a2.x, v[0].y + a1.y + a2.y);
            o[ns] = cadd(t1, ju1);
            o[4 * ns] = csub(t1, ju1);
            o[2 * ns] = cadd(t2, ju2);
            o[3 * ns] = csub(t2, ju2);
        }
    }
}

// any other (odd prime) radix, the role of kf_bfly_generic (kiss_fft.c:197-235): one thread per OUTPUT,
// p complex multiply-adds each; the p-th roots of unity are entries (q r mod p) n/p of the same table.
template <bool INV>
__device__ __forceinline__ void mixed_pass_generic(const float2 *src, float2 *dst, int n, int ns, int p,
                                                   const float2 *__restrict__ tw)
{
    const int m = n / p;
    const int twstep = n / (ns * p);
    for (int idx = threadIdx.x; idx < n; idx += blockDim.x) {
        const int q = idx / m, j = idx - q * m;
        const int k = j % ns;
        float2 acc = src[j];
        int qr = 0;
        for (int r = 1; r < p; ++r) {
            qr += q;
            if (qr >= p) qr -= p;
            float2 x = src[j + r * m];
            if (ns > 1) x = cmulf(x, tw_get<INV>(tw, (int)(((long long)r * k * twstep) % n)));
            const float2 y = cmulf(x, tw_get<INV>(tw, qr * m));
            acc.x += y.x; acc.y += y.y;
        }
        dst[(j - k) * p + k + q * ns] = acc;
    }
}

template <bool INV>
__global__ void __launch_bounds__(256)
fft_mixed_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, size_t batch, int n, MixedPlan mp,
                 const float2 *__restrict__ tw)
{
    extern __shared__ float2 mx_smem[];
    for (size_t f = blockIdx.x; f < batch; f += gridDim.x) {
        float2 *a = mx_smem, *b = mx_smem + n;
        for (int i = threadIdx.x; i < n; i += blockDim.x) a[i] = in[f * (size_t)n + i];
        __syncthreads();
        int ns = 1;
        for (int s = 0; s < mp.nfac; ++s) {
            const int p = mp.radix[s];
            switch (p) {
                case 2: mixed_pass<2, INV>(a, b, n, ns, tw); break;
                case 3: mixed_pass<3, INV>(a, b, n, ns, tw); break;
                case 4: mixed_pass<4, INV>(a, b, n, ns, tw); break;
                case 5: mixed_pass<5, INV>(a, b, n, ns, tw); break;
                default: mixed_pass_generic<INV>(a, b, n, ns, p, tw); break;
            }
            __syncthreads();
            float2 *t = a; a = b; b = t;
            ns *= p;
        }
        for (int i = threadIdx.x; i < n; i += blockDim.x) out[f * (size_t)n + i] = a[i];
        __syncthreads();
    }
}

int lrc_fft_mixed_launch(const lrc_ctx *ctx, int nfft, int inverse, const MixedPlan *mp, const float2 *d_tw,
                         const float2 *in, float2 *out, size_t batch, cudaStream_t s)
{
    const size_t smem = (size_t)2 * nfft * sizeof(float2);
    const int threads = nfft >= 1024 ? 256 : (nfft >= 256 ? 128 : 64);
    size_t blocks = batch;
    const size_t cap = (size_t)ctx->n_sm * 8;
    if (blocks > cap) blocks = cap;
    if (inverse) {
        if (smem > 48 * 1024) LRC_CUDA(cudaFuncSetAttribute(fft_mixed_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fft_mixed_kernel<true><<<(unsigned)blocks, threads, smem, s>>>(in, out, batch, nfft, *mp, d_tw);
    } else {
        if (smem > 48 * 1024) LRC_CUDA(cudaFuncSetAttribute(fft_mixed_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fft_mixed_kernel<false><<<(unsigned)blocks, threads, smem, s>>>(in, out, batch, nfft, *mp, d_tw);
    }
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

// ---------------------------------------------------------------------------------------------
// real-input pair
// ---------------------------------------------------------------------------------------------
struct lrc_rfft {
    lrc_ctx *ctx;
    int      nfft, ncfft, inverse;
    lrc_fft *sub;                // complex plan of ncfft points
    DevBuf<float2> d_super;      // ncfft/2 super twiddles
    DevBuf<float2> d_tmp;        // [batch][ncfft] scratch
};

// kiss_fftr.c:93-119: tmp = FFT_ncfft(time data as complex) -> freq[0..ncfft]
__global__ void __launch_bounds__(256)
rfft_split_kernel(const float2 *__restrict__ tmp, float2 *__restrict__ freq, size_t batch, int ncfft,
                  const float2 *__restrict__ super)
{
    const int per = ncfft / 2 + 1;                      // k = 0 .. ncfft/2
    const size_t total = batch * (size_t)per;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t f = i / per;
        const int k = (int)(i - f * per);
        const float2 *t = tmp + f * (size_t)ncfft;
        float2 *o = freq + f * (size_t)(ncfft + 1);
        if (k == 0) {
            const float2 tdc = t[0];
            o[0] = make_float2(tdc.x + tdc.y, 0.f);
            o[ncfft] = make_float2(tdc.x - tdc.y, 0.f);
        } else {
            const float2 fpk = t[k];
            const float2 fpnk = make_float2(t[ncfft - k].x, -t[ncfft - k].y);
            const float2 f1k = cadd(fpk, fpnk), f2k = csub(fpk, fpnk);
            const float2 w = cmulf(f2k, __ldg(super + k - 1));
            o[k] = make_float2(0.5f * (f1k.x + w.x), 0.5f * (f1k.y + w.y));
            o[ncfft - k] = make_float2(0.5f * (f1k.x - w.x), 0.5f * (w.y - f1k.y));
        }
    }
}

// kiss_fftr.c:134-157: freq[0..ncfft] -> tmp, then the inverse complex transform gives the time data
__global__ void __launch_bounds__(256)
rfft_merge_kernel(const float2 *__restrict__ freq, float2 *__restrict__ tmp, size_t batch, int ncfft,
                  const float2 *__restrict__ super)
{
    const int per = ncfft / 2 + 1;
    const size_t total = batch * (size_t)per;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t f = i / per;
        const int k = (int)(i - f * per);
        const float2 *q = freq + f * (size_t)(ncfft + 1);
        float2 *t = tmp + f * (size_t)ncfft;
        if (k == 0) {
            t[0] = make_float2(q[0].x + q[ncfft].x, q[0].x - q[ncfft].x);
        } else {
            const float2 fk = q[k];
            const float2 fnkc = make_float2(q[ncfft - k].x, -q[ncfft - k].y);
            const float2 fek = cadd(fk, fnkc), d = csub(fk, fnkc);
            const float2 fok = cmulf(d, __ldg(super + k - 1));
            const float2 lo = cadd(fek, fok), hi = csub(fek, fok);
            t[k] = lo;
            t[ncfft - k] = make_float2(hi.x, -hi.y);      // for k == ncfft/2 this is the value the reference keeps
        }
    }
}

extern "C" int lrc_rfft_create(lrc_ctx *ctx, int nfft, int inverse, lrc_rfft **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out != nullptr && nfft >= 2, LRC_ERR_INVALID, "lrc_rfft_create: bad arguments");
    if (nfft & 1) {
        lrc_set_error("lrc_rfft_create: nfft=%d: real FFT size must be even (kiss_fftr.c:34-37)", nfft);
        return LRC_ERR_INVALID;
    }
    lrc_rfft *p = new (std::nothrow) lrc_rfft();
    LRC_REQUIRE(p != nullptr, LRC_ERR_NOMEM, "out of host memory");
    p->ctx = ctx; p->nfft = nfft; p->ncfft = nfft / 2; p->inverse = inverse ? 1 : 0;
    int rc = lrc_fft_create(ctx, p->ncfft, inverse, &p->sub);
    if (rc) { lrc_rfft_destroy(p); return rc; }
    const int ns = p->ncfft / 2;
    std::vector<float2> sup(ns > 0 ? ns : 1);
    for (int i = 0; i < ns; ++i) {
        double phase = -3.14159265358979323846264338327 * ((double)(i + 1) / p->ncfft + .5);   // kiss_fftr.c:57-62
        if (inverse) phase *= -1;
        sup[i] = make_float2((float)cos(phase), (float)sin(phase));
    }
    cudaError_t e = p->d_super.alloc(sup.size());
    if (e == cudaSuccess) e = cudaMemcpy(p->d_super, sup.data(), sup.size() * sizeof(float2), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        lrc_set_error("lrc_rfft_create: %s", cudaGetErrorString(e));
        lrc_rfft_destroy(p);
        return LRC_ERR_CUDA;
    }
    *out = p;
    return LRC_OK;
}

extern "C" int lrc_rfft_destroy(lrc_rfft *p)
{
    if (!p) return LRC_OK;
    cudaSetDevice(p->ctx->device);
    lrc_fft_destroy(p->sub);
    delete p;
    return LRC_OK;
}

extern "C" int lrc_rfft_run(lrc_rfft *p, const float *d_in, float *d_out, size_t batch, void *stream)
{
    LRC_REQUIRE(p != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(p->ctx);
    if (batch == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_out && d_in != d_out, LRC_ERR_INVALID, "lrc_rfft_run: null or aliased buffers");
    LRC_REQUIRE(((uintptr_t)d_in & 7) == 0 && ((uintptr_t)d_out & 7) == 0, LRC_ERR_INVALID,
                "lrc_rfft_run: buffers must be 8-byte aligned");
    cudaStream_t s = lrc_stream(p->ctx, stream);
    const size_t need = batch * (size_t)p->ncfft;
    LRC_CUDA(p->d_tmp.ensure(need));
    const size_t items = batch * (size_t)(p->ncfft / 2 + 1);
    size_t blocks = ceil_div(items, 256);
    const size_t cap = (size_t)p->ctx->n_sm * 16;
    if (blocks > cap) blocks = cap;
    if (!p->inverse) {
        // nfft reals == ncfft complex samples, frames contiguous (kiss_fftr.c:84)
        int rc = lrc_fft_run(p->sub, d_in, (float *)p->d_tmp.get(), batch, s);
        if (rc) return rc;
        rfft_split_kernel<<<(unsigned)blocks, 256, 0, s>>>(p->d_tmp, (float2 *)d_out, batch, p->ncfft, p->d_super);
        LRC_CUDA(cudaGetLastError());
        return LRC_OK;
    }
    rfft_merge_kernel<<<(unsigned)blocks, 256, 0, s>>>((const float2 *)d_in, p->d_tmp, batch, p->ncfft, p->d_super);
    LRC_CUDA(cudaGetLastError());
    return lrc_fft_run(p->sub, (const float *)p->d_tmp.get(), d_out, batch, s);
}

extern "C" int lrc_rfft_run_host(lrc_rfft *p, const float *h_in, float *h_out, size_t batch)
{
    LRC_REQUIRE(p != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(p->ctx);
    if (batch == 0) return LRC_OK;
    LRC_REQUIRE(h_in && h_out, LRC_ERR_INVALID, "null buffer");
    const size_t time_b = batch * (size_t)p->nfft * sizeof(float);
    const size_t freq_b = batch * (size_t)(p->ncfft + 1) * sizeof(float2);
    const size_t in_b = p->inverse ? freq_b : time_b, out_b = p->inverse ? time_b : freq_b;
    DevBuf<float> d_a, d_b;
    LRC_CUDA(d_a.alloc(in_b / sizeof(float)));
    if (d_b.alloc(out_b / sizeof(float)) != cudaSuccess) { lrc_set_error("lrc_rfft_run_host: cudaMalloc"); return LRC_ERR_CUDA; }
    cudaStream_t s = p->ctx->stream;
    cudaError_t e = cudaMemcpyAsync(d_a, h_in, in_b, cudaMemcpyHostToDevice, s);
    int rc = LRC_OK;
    if (e == cudaSuccess) rc = lrc_rfft_run(p, d_a, d_b, batch, s);
    if (e == cudaSuccess && rc == LRC_OK) e = cudaMemcpyAsync(h_out, d_b, out_b, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { lrc_set_error("lrc_rfft_run_host: %s", cudaGetErrorString(e)); return LRC_ERR_CUDA; }
    return rc;
}
