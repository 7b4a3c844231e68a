// k_fastfir.cu -- long FIR by FFT overlap-save ("overlap-scrap"), one kernel per call.
//
// Replaces kiss_fastfir_alloc / kiss_fastfir (libkissfft/tools/kiss_fastfir.c:65-245):
//   H = FFT(h rotated left by nh-1) / nfft                      (:148-169)
//   per block b: out[b*ngood .. +ngood) = IFFT(FFT(in[b*ngood .. +nfft)) .* H)[0 .. ngood)   (:173-204)
//   flush: the remainder zero-padded to nfft, ngood - zpad outputs kept               (:208-226)
// One CTA owns one block at a time: forward FFT, spectrum multiply and inverse FFT all happen in
// registers/shared memory (the forward output layout "thread t holds bin t + e*T" is exactly the
// inverse input layout), so HBM sees nfft reads and ngood writes per block and nothing else.
//
// Measured and rejected (round 1, one B200, 4096 taps): fastfir_kernel<13>, the register-resident CTA-level kernel, for
// 8192-point blocks: 50 300 Msamples/s against 99 400 for fastfir8k_kernel (DESIGN.md, overlap-save rows; SASS in
// profiles/sass/r1_fastfir_8192.sass and r1_fastfir8k.sass).
#include "fft_core.cuh"
#include <cmath>
#include <utility>
#include <vector>

using namespace lrfft;

int lrc_make_twiddles(int nfft, float2 **d_tw);
int lrc_log2_exact(int n);
// k_fastfir16k.cu (16384-point blocks)
void lrc_fastfir16k_permute_H(const float2 *H, float2 *Hq);
int lrc_fastfir16k_prepare(void);
int lrc_fastfir16k_launch(int n_sm, const float2 *in, size_t n_in, float2 *out, size_t full, size_t nblk, size_t ngood,
                          size_t keep, const float2 *d_tw16k, const float2 *d_tw1k, const float2 *d_Hp, cudaStream_t s);

struct lrc_fastfir {
    lrc_ctx *ctx;
    size_t   nh, nfft, ngood;   // nfft/ngood: the block size that fixes the OUTPUT LENGTH (kiss_fastfir's, or the caller's)
    int      log2n;
    float2  *d_tw;
    float2  *d_H;
    float2  *d_Hc;     // 8192-point kernel: H in the order fastfir8k_kernel uses; 16384-point kernel: Hq (k_fastfir16k.cu)
    float2  *d_tw1k;   // 16384-point kernel: W_1024^k for the warp-level sub-transforms
    bool     compute16k;        // blocks are COMPUTED 16384 points at a time whatever nfft says (see lrc_fastfir_create)
};

// host-side f64 radix-2 FFT (forward), used only to build H for block sizes our own FFT plans do not cover
static void host_fft_f64(std::vector<double> &re, std::vector<double> &im)
{
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) { std::swap(re[i], re[j]); std::swap(im[i], im[j]); }
    }
    const double pi = 3.14159265358979323846264338327950288;
    for (size_t len = 2; len <= n; len <<= 1) {
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < len / 2; ++k) {
                const double a = -2.0 * pi * (double)k / (double)len, c = cos(a), s = sin(a);
                const size_t u = i + k, v = i + k + len / 2;
                const double tr = re[v] * c - im[v] * s, ti = re[v] * s + im[v] * c;
                re[v] = re[u] - tr; im[v] = im[u] - ti;
                re[u] += tr; im[u] += ti;
            }
    }
}

template <int LOG2N>
__global__ void __launch_bounds__(CtaFFT<LOG2N, false>::T)
fastfir_kernel(const float2 *__restrict__ in, size_t n_in, float2 *__restrict__ out, size_t n_blocks_full,
               size_t n_blocks, size_t ngood, size_t flush_keep, const float2 *__restrict__ tw,
               const float2 *__restrict__ H)
{
    using FF = CtaFFT<LOG2N, false>;
    using FI = CtaFFT<LOG2N, true>;
    constexpr int N = FF::N, E = FF::E, T = FF::T;
    extern __shared__ float2 sm[];
    const int t = threadIdx.x;
    for (size_t b = blockIdx.x; b < n_blocks; b += gridDim.x) {
        const size_t s0 = b * ngood;
        const size_t avail = n_in - s0;              // < N only for the flush block
        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const size_t i = (size_t)t + (size_t)e * T;
            v[e] = (i < avail) ? __ldcs(in + s0 + i) : make_float2(0.f, 0.f);
        }
        FF::run(v, sm, tw, t, SyncCta{});
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = t + e * T;
            v[e] = cmulf(v[e], __ldg(H + i));        // C_MUL(freqbuf[i], fir_freq_resp[i])  :180-184
        }
        FI::run(v, sm, tw, t, SyncCta{});
        const size_t keep = (b < n_blocks_full) ? ngood : flush_keep;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const size_t i = (size_t)t + (size_t)e * T;
            if (i < keep) __stcs(out + s0 + i, v[e]);
        }
    }
}


// ---------------------------------------------------------------------------------------------
// nfft = 8192 (kiss_fastfir's automatic size for 2048 < nh <= 4096, the config-5 shape): in-place
// shared-memory variant.  The register-resident Stockham kernel above fills half the register file
// with one transform, so only one CTA fits an SM and every barrier and global load is exposed.  Here
// the block lives in shared memory (68 KB), a thread only ever holds one butterfly, and two CTAs per
// SM cover each other's barriers and loads.
//
//   8192 = 16 x 16 x 32.  Forward = decimation in frequency, in place:
//     P1  radix 16, stride 512, inputs straight from global memory, twiddle W_8192^(q j)
//     P2  radix 16 inside each 512-block, stride 32, twiddle W_512^(q j)
//     MID the 256 contiguous 32-point sub-blocks: DFT32 -> .* H -> IDFT32 in registers
//   and the inverse mirrors it as decimation in time (P2', then P1' whose outputs go straight to
//   global memory), so the digit-reversed order produced by the DIF passes is never undone: H is
//   stored in that order instead (position 512 b + 32 q2 + k2 holds bin b + 16 q2 + 256 k2).
//   Shared-memory index i is padded to i + 2 (i / 32): the strided passes stay conflict-free and
//   the contiguous 32-point blocks of MID start 17 x 16 bytes apart (conflict-free LDS.128).
// ---------------------------------------------------------------------------------------------
namespace ff8k {
constexpr int N = 8192, NT = 256;
constexpr int DATA_CPX = N + 2 * (N / 32);                 // 8704 float2
constexpr int TW1_CPX = 15 * 256, TW2_CPX = 15 * 32;
constexpr int SMEM_BYTES = (DATA_CPX + TW1_CPX + TW2_CPX) * 8;
__host__ __device__ constexpr int pad(int i) { return i + 2 * (i >> 5); }

// exp(-2 pi j n / 32), n < 16
__device__ __forceinline__ float2 w32(int n)
{
    constexpr float C[16] = {1.f, 0.98078528040323044913f, 0.92387953251128675613f, 0.83146961230254523708f,
                             0.70710678118654752440f, 0.55557023301960222474f, 0.38268343236508977173f,
                             0.19509032201612826785f, 0.f, -0.19509032201612826785f, -0.38268343236508977173f,
                             -0.55557023301960222474f, -0.70710678118654752440f, -0.83146961230254523708f,
                             -0.92387953251128675613f, -0.98078528040323044913f};
    constexpr float S[16] = {0.f, 0.19509032201612826785f, 0.38268343236508977173f, 0.55557023301960222474f,
                             0.70710678118654752440f, 0.83146961230254523708f, 0.92387953251128675613f,
                             0.98078528040323044913f, 1.f, 0.98078528040323044913f, 0.92387953251128675613f,
                             0.83146961230254523708f, 0.70710678118654752440f, 0.55557023301960222474f,
                             0.38268343236508977173f, 0.19509032201612826785f};
    return make_float2(C[n], -S[n]);
}
}  // namespace ff8k

__global__ void __launch_bounds__(ff8k::NT, 2)
fastfir8k_kernel(const float2 *__restrict__ in, size_t n_in, float2 *__restrict__ out, size_t n_blocks_full,
                 size_t n_blocks, size_t ngood, size_t flush_keep, const float2 *__restrict__ tw,
                 const float2 *__restrict__ Hc)
{
    using namespace ff8k;
    extern __shared__ __align__(16) float2 ff8k_smem[];
    float2 *sd = ff8k_smem;
    float2 *tw1 = ff8k_smem + DATA_CPX;            // [q-1][j], j < 256 : W_8192^(q j)
    float2 *tw2 = tw1 + TW1_CPX;             // [q-1][j], j < 32  : W_512^(q j)
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int i = t; i < TW1_CPX; i += NT) tw1[i] = __ldg(tw + ((i >> 8) + 1) * (i & 255));
    for (int i = t; i < TW2_CPX; i += NT) tw2[i] = __ldg(tw + 16 * ((i >> 5) + 1) * (i & 31));
    __syncthreads();

    // P1 forward of one column j of block `blk`: inputs from global memory, results into the column's
    // 16 shared-memory slots (no other thread touches column j during the P1 phases)
    auto p1_load = [&](size_t blk, int j, float2 *v) {
        const size_t s0 = blk * ngood, avail = n_in - s0;        // avail < N only for the flush block
        const float2 *src = in + s0;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const size_t i = (size_t)(j + 512 * r);
            v[r] = i < avail ? __ldg(src + i) : make_float2(0.f, 0.f);
        }
    };
    auto p1_forward = [&](int h, float2 *v) {
        RegFFT<16, false>::run(v);
        float2 *dst = sd + pad(t + 256 * h);         // pad(j + 512 q) = pad(j) + 544 q
        dst[0] = v[0];
#pragma unroll
        for (int q = 1; q < 16; ++q) {
            float2 w = tw1[(q - 1) * 256 + t];
            if (h) w = cmulf(w, w32(q));                 // W_8192^(256 q) = W_32^q
            dst[544 * q] = cmulf(v[q], w);
        }
    };

    size_t b = blockIdx.x;
    if (b < n_blocks) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float2 v[16];
            p1_load(b, t + 256 * h, v);
            p1_forward(h, v);
        }
    }
    for (; b < n_blocks; b += gridDim.x) {
        // the next block's input (512 lines) is asked into L2 now; its P1 loads come four phases later
        if (b + gridDim.x < n_blocks) {
            const char *nsrc = reinterpret_cast<const char *>(in + (b + gridDim.x) * ngood);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const size_t off = (size_t)(t + 256 * k) * 128;
                if ((b + gridDim.x) * ngood * 8 + off < n_in * 8)
                    asm volatile("prefetch.global.L2 [%0];" :: "l"(nsrc + off));
            }
        }
        // first half of this thread's H values (an L2 round trip): in flight across the whole P2 phase
        float2 hv[16];
#pragma unroll
        for (int m = 0; m < 16; ++m) hv[m] = __ldg(Hc + m * 256 + t);
        __syncthreads();
        // ---- P2 forward: (block bb, j = lane), bb = warp and warp + 8 ---------------------------------
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float2 *p = sd + 544 * (warp + 8 * h) + lane;    // pad(512 bb + j + 32 r) = 544 bb + 34 r + j
            float2 v[16];
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = p[34 * r];
            RegFFT<16, false>::run(v);
            p[0] = v[0];
#pragma unroll
            for (int q = 1; q < 16; ++q) p[34 * q] = cmulf(v[q], tw2[(q - 1) * 32 + lane]);
        }
        // ---- MID: sub-block t, 32 contiguous points: DFT32, .* H, IDFT32 --------------------------------
        {
            float4 *p4 = reinterpret_cast<float4 *>(sd + 34 * t);
            __syncthreads();
            float2 u[32];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float4 x = p4[i];
                u[2 * i] = make_float2(x.x, x.y);
                u[2 * i + 1] = make_float2(x.z, x.w);
            }
#pragma unroll
            for (int n = 0; n < 16; ++n) {
                const float2 a = cadd(u[n], u[n + 16]);
                const float2 d = csub(u[n], u[n + 16]);
                u[n] = a;
                u[n + 16] = n ? cmulf(d, w32(n)) : d;
            }
            RegFFT<16, false>::run(u);                   // u[m]      = X2[2 m]
#pragma unroll
            for (int m = 0; m < 16; ++m) u[m] = cmulf(u[m], hv[m]);               // C_MUL  :180-184
#pragma unroll
            for (int m = 0; m < 16; ++m) hv[m] = __ldg(Hc + (16 + m) * 256 + t);
            RegFFT<16, true>::run(u);
            RegFFT<16, false>::run(u + 16);              // u[16 + m] = X2[2 m + 1]
#pragma unroll
            for (int m = 0; m < 16; ++m) u[16 + m] = cmulf(u[16 + m], hv[m]);
            RegFFT<16, true>::run(u + 16);
#pragma unroll
            for (int n = 0; n < 16; ++n) {
                const float2 c = n ? cmul_conjb(u[n + 16], w32(n)) : u[n + 16];
                const float2 a = u[n];
                u[n] = cadd(a, c);
                u[n + 16] = csub(a, c);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) p4[i] = make_float4(u[2 * i].x, u[2 * i].y, u[2 * i + 1].x, u[2 * i + 1].y);
        }
        // column t of the CTA's next block: requested now, used after this block's P1 inverse of column t
        const size_t nb = b + gridDim.x;
        const bool more = nb < n_blocks;
        float2 nx0[16];
        if (more) p1_load(nb, t, nx0);
        __syncthreads();
        // ---- P2 inverse ------------------------------------------------------------------------------
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float2 *p = sd + 544 * (warp + 8 * h) + lane;
            float2 v[16];
            v[0] = p[0];
#pragma unroll
            for (int q = 1; q < 16; ++q) v[q] = cmul_conjb(p[34 * q], tw2[(q - 1) * 32 + lane]);
            RegFFT<16, true>::run(v);
#pragma unroll
            for (int r = 0; r < 16; ++r) p[34 * r] = v[r];
        }
        __syncthreads();
        // ---- P1 inverse of this block, column by column, fused with P1 forward of the CTA's next block:
        // the next block's column is requested from global memory first, the inverse butterfly of the
        // current column runs while those loads are in flight, and the forward results then reuse the
        // column's slots -- no barrier between the two blocks' P1 phases.
        const size_t s0 = b * ngood;
        const size_t keep = (b < n_blocks_full) ? ngood : flush_keep;
        float2 *dstg = out + s0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = t + 256 * h;
            float2 nx[16];
            if (h == 0) {
#pragma unroll
                for (int r = 0; r < 16; ++r) nx[r] = nx0[r];
            } else if (more) {
                p1_load(nb, j, nx);
            }
            {
                const float2 *p = sd + pad(j);
                float2 v[16];
                v[0] = p[0];
#pragma unroll
                for (int q = 1; q < 16; ++q) {
                    float2 w = tw1[(q - 1) * 256 + t];
                    if (h) w = cmulf(w, w32(q));
                    v[q] = cmul_conjb(p[544 * q], w);
                }
                RegFFT<16, true>::run(v);
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const size_t i = (size_t)(j + 512 * r);
                    if (i < keep) __stcs(dstg + i, v[r]);
                }
            }
            if (more) p1_forward(h, nx);
        }
    }
}

// H (natural order, already scaled by 1/nfft) -> the order fastfir8k_kernel's MID stage meets it in:
// Hc[m * 256 + s], s = 16 b + q2 the 32-point sub-block, m the register index after the split DFT32
// (m < 16: k2 = 2 m, else k2 = 2 (m - 16) + 1), bin = b + 16 q2 + 256 k2.
static void fastfir8k_permute_H(const std::vector<float2> &H, std::vector<float2> &Hc)
{
    Hc.resize(8192);
    for (int s = 0; s < 256; ++s)
        for (int m = 0; m < 32; ++m) {
            const int bb = s >> 4, q2 = s & 15, k2 = m < 16 ? 2 * m : 2 * (m - 16) + 1;
            Hc[m * 256 + s] = H[bb + 16 * q2 + 256 * k2];
        }
}

extern "C" int lrc_fastfir_create(lrc_ctx *ctx, const float *h_taps_cpx, size_t nh, size_t nfft_arg, lrc_fastfir **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && h_taps_cpx && nh >= 1, LRC_ERR_INVALID, "lrc_fastfir_create: bad arguments");
    size_t nfft = nfft_arg;
    if (nfft == 0) {
        // kiss_fastfir.c:81-93: next power of two at least twice the impulse response, at least 1024
        size_t i = nh - 1;
        nfft = 2;
        do { nfft <<= 1; } while (i >>= 1);
        if (nfft < 1024) nfft = 1024;
    }
    const bool automatic = nfft_arg == 0;
    const int l2 = lrc_log2_exact((int)nfft);
    if (l2 < 1 || l2 > 14) {
        lrc_set_error("lrc_fastfir_create: nfft=%zu: only powers of two in [2, 16384] (nh <= 8192 with the "
                      "automatic size)", nfft);
        return LRC_ERR_UNSUPPORTED;
    }
    LRC_REQUIRE(nfft >= nh, LRC_ERR_INVALID, "lrc_fastfir_create: nfft shorter than the impulse response");
    // Overlap-save gives the same y[k] whatever the block size; the block size only fixes how many outputs a call
    // without flush produces (kff_nocopy :199-204 stops at the last FULL block).  So `nfft` keeps that meaning, and
    // long filters are COMPUTED in 16384-point blocks: 12289 of 16384 outputs kept per block for 4096 taps instead of
    // 4097 of 8192.  An explicit nfft < 16384 is honoured for the arithmetic as well (A/B runs, golden tests of that size).
    const bool c16 = nfft == 16384 || (automatic && nh > 1024);
    lrc_fastfir *f = new (std::nothrow) lrc_fastfir{ctx, nh, nfft, nfft - nh + 1, l2, nullptr, nullptr, nullptr, nullptr, c16};
    LRC_REQUIRE(f != nullptr, LRC_ERR_NOMEM, "out of host memory");
    if (c16) {
        const size_t n16 = 16384;
        int rc16 = lrc_make_twiddles(16384, &f->d_tw);
        if (!rc16) rc16 = lrc_make_twiddles(1024, &f->d_tw1k);
        if (!rc16) rc16 = lrc_fastfir16k_prepare();
        if (rc16) { lrc_fastfir_destroy(f); return rc16; }
        // H = FFT(h rotated) / nfft in f64 on the host (:148-169), rounded once to f32
        const float2 *h16 = reinterpret_cast<const float2 *>(h_taps_cpx);
        std::vector<double> re(n16, 0.0), im(n16, 0.0);
        re[0] = h16[nh - 1].x; im[0] = h16[nh - 1].y;
        for (size_t i = 0; i + 1 < nh; ++i) { re[n16 - nh + 1 + i] = h16[i].x; im[n16 - nh + 1 + i] = h16[i].y; }
        host_fft_f64(re, im);
        std::vector<float2> H(n16), Hq(n16);
        for (size_t i = 0; i < n16; ++i) H[i] = make_float2((float)(re[i] / (double)n16), (float)(im[i] / (double)n16));
        lrc_fastfir16k_permute_H(H.data(), Hq.data());
        cudaError_t e16 = cudaMalloc(&f->d_H, n16 * sizeof(float2));
        if (e16 == cudaSuccess) e16 = cudaMemcpy(f->d_H, H.data(), n16 * sizeof(float2), cudaMemcpyHostToDevice);
        if (e16 == cudaSuccess) e16 = cudaMalloc(&f->d_Hc, n16 * sizeof(float2));
        if (e16 == cudaSuccess) e16 = cudaMemcpy(f->d_Hc, Hq.data(), n16 * sizeof(float2), cudaMemcpyHostToDevice);
        if (e16 != cudaSuccess) {
            lrc_set_error("lrc_fastfir_create: %s", cudaGetErrorString(e16));
            lrc_fastfir_destroy(f);
            return LRC_ERR_CUDA;
        }
        *out = f;
        return LRC_OK;
    }
    int rc = lrc_make_twiddles((int)nfft, &f->d_tw);
    if (rc) { delete f; return rc; }
    // rotated impulse response (:148-154), transformed with our own FFT kernel, scaled by 1/nfft (:159-169)
    const float2 *h = reinterpret_cast<const float2 *>(h_taps_cpx);
    std::vector<float2> rot(nfft, make_float2(0.f, 0.f));
    rot[0] = h[nh - 1];
    for (size_t i = 0; i + 1 < nh; ++i) rot[nfft - nh + 1 + i] = h[i];
    lrc_fft *plan = nullptr;
    rc = lrc_fft_create(ctx, (int)nfft, 0, &plan);
    cudaError_t e = cudaSuccess;
    if (!rc) e = cudaMalloc(&f->d_H, nfft * sizeof(float2));
    if (!rc && e == cudaSuccess) e = cudaMemcpy(f->d_H, rot.data(), nfft * sizeof(float2), cudaMemcpyHostToDevice);
    if (!rc && e == cudaSuccess) rc = lrc_fft_run(plan, (const float *)f->d_H, (float *)f->d_H, 1, ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaMemcpy(rot.data(), f->d_H, nfft * sizeof(float2), cudaMemcpyDeviceToHost);
    if (!rc && e == cudaSuccess) {
        const float scale = (float)(1.0 / (double)nfft);
        for (size_t i = 0; i < nfft; ++i) { rot[i].x *= scale; rot[i].y *= scale; }
        e = cudaMemcpy(f->d_H, rot.data(), nfft * sizeof(float2), cudaMemcpyHostToDevice);
        if (e == cudaSuccess && nfft == 8192) {
            std::vector<float2> hc;
            fastfir8k_permute_H(rot, hc);
            e = cudaMalloc(&f->d_Hc, nfft * sizeof(float2));
            if (e == cudaSuccess) e = cudaMemcpy(f->d_Hc, hc.data(), nfft * sizeof(float2), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(fastfir8k_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ff8k::SMEM_BYTES);
        }
    }
    lrc_fft_destroy(plan);
    if (rc || e != cudaSuccess) {
        if (e != cudaSuccess) { lrc_set_error("lrc_fastfir_create: %s", cudaGetErrorString(e)); rc = LRC_ERR_CUDA; }
        lrc_fastfir_destroy(f);
        return rc;
    }
    *out = f;
    return LRC_OK;
}

extern "C" int lrc_fastfir_destroy(lrc_fastfir *f)
{
    if (!f) return LRC_OK;
    cudaSetDevice(f->ctx->device);
    cudaFree(f->d_tw); cudaFree(f->d_H); cudaFree(f->d_Hc); cudaFree(f->d_tw1k);
    delete f;
    return LRC_OK;
}

extern "C" size_t lrc_fastfir_nfft(const lrc_fastfir *f) { return f ? f->nfft : 0; }

static void fastfir_counts(const lrc_fastfir *f, size_t n_in, int flush, size_t *full, size_t *flush_keep)
{
    // kff_nocopy :199-204: while (n >= nfft) { ...; n -= ngood; }
    *full = n_in >= f->nfft ? (n_in - f->nfft) / f->ngood + 1 : 0;
    const size_t rem = n_in - *full * f->ngood;
    // kff_flush :213-225: zpad = nfft - rem; keep ngood - zpad = rem - (nh - 1) samples (none if negative)
    *flush_keep = (flush && rem + 1 > f->nh) ? rem + 1 - f->nh : 0;
}

extern "C" size_t lrc_fastfir_out_len(const lrc_fastfir *f, size_t n_in, int flush)
{
    if (!f) return 0;
    size_t full, keep;
    fastfir_counts(f, n_in, flush, &full, &keep);
    return full * f->ngood + keep;
}

template <int LOG2N>
static int launch_fastfir(lrc_fastfir *f, const float2 *in, size_t n_in, float2 *out, size_t full, size_t nblk,
                          size_t keep, cudaStream_t s)
{
    using FF = CtaFFT<LOG2N, false>;
    const int threads = FF::T;
    const size_t smem = (size_t)FF::SMEM_CPX * sizeof(float2);
    auto kern = fastfir_kernel<LOG2N>;
    if (smem > 48 * 1024) LRC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    LRC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
    if (occ < 1) occ = 1;
    size_t blocks = (size_t)f->ctx->n_sm * occ;
    if (blocks > nblk) blocks = nblk;
    kern<<<(unsigned)blocks, threads, smem, s>>>(in, n_in, out, full, nblk, f->ngood, keep, f->d_tw, f->d_H);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

extern "C" int lrc_fastfir_run(lrc_fastfir *f, const float *d_in, size_t n_in, float *d_out, int flush,
                               size_t *n_out, void *stream)
{
    LRC_REQUIRE(f != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(f->ctx);
    size_t full, keep;
    fastfir_counts(f, n_in, flush, &full, &keep);
    if (n_out) *n_out = full * f->ngood + keep;
    const size_t nblk = full + (keep ? 1 : 0);
    if (nblk == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_out && d_in != d_out, LRC_ERR_INVALID, "lrc_fastfir_run: null or aliased buffers");
    LRC_REQUIRE(((uintptr_t)d_in & 7) == 0 && ((uintptr_t)d_out & 7) == 0, LRC_ERR_INVALID, "lrc_fastfir_run: misaligned");
    cudaStream_t s = lrc_stream(f->ctx, stream);
    const float2 *in = (const float2 *)d_in;
    float2 *out = (float2 *)d_out;
    if (f->compute16k) {
        // the same full * ngood + keep outputs, cut into 16384-point blocks: every output k < n_total only needs
        // x[k .. k + nh - 1], which the call holds; the last block keeps the remainder and reads zeros past the input
        const size_t n_total = full * f->ngood + keep, ngood16 = 16384 - f->nh + 1;
        const size_t full16 = n_total / ngood16, keep16 = n_total % ngood16;
        return lrc_fastfir16k_launch(f->ctx->n_sm, in, n_in, out, full16, full16 + (keep16 ? 1 : 0), ngood16, keep16, f->d_tw,
                                     f->d_tw1k, f->d_Hc, s);
    }
    if (f->log2n == 13) {                 // 8192-point blocks: the plan holds d_Hc for fastfir8k_kernel
        size_t blocks = (size_t)f->ctx->n_sm * 2;
        if (blocks > nblk) blocks = nblk;
        fastfir8k_kernel<<<(unsigned)blocks, ff8k::NT, ff8k::SMEM_BYTES, s>>>(in, n_in, out, full, nblk, f->ngood, keep,
                                                                             f->d_tw, f->d_Hc);
        LRC_CUDA(cudaGetLastError());
        return LRC_OK;
    }
    switch (f->log2n) {
#define FF_CASE(L) case L: return launch_fastfir<L>(f, in, n_in, out, full, nblk, keep, s);
        FF_CASE(1) FF_CASE(2) FF_CASE(3) FF_CASE(4) FF_CASE(5) FF_CASE(6) FF_CASE(7)
        FF_CASE(8) FF_CASE(9) FF_CASE(10) FF_CASE(11) FF_CASE(12)
#undef FF_CASE
    }
    return LRC_ERR_UNSUPPORTED;
}
