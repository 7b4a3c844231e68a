// k_fastfir.cu -- long FIR by FFT overlap-save ("overlap-scrap"), one kernel per call.
//
// Replaces kiss_fastfir_alloc / kiss_fastfir (libkissfft/tools/kiss_fastfir.c:65-245):
//   H = FFT(h rotated left by nh-1) / nfft                      (:148-169)
//   per block b: out[b*ngood .. +ngood) = IFFT(FFT(in[b*ngood .. +nfft)) .* H)[0 .. ngood)   (:173-204)
//   flush: the remainder zero-padded to nfft, ngood - zpad outputs kept               (:208-226)
// One CTA owns one block at a time: forward FFT, spectrum multiply and inverse FFT all happen in
// registers/shared memory (the forward output layout "thread t holds bin t + e*T" is exactly the
// inverse input layout), so HBM sees nfft reads and ngood writes per block and nothing else.
// Plans with nh > 1024 or nfft >= 8192 compute in 16384-point blocks instead (k_fastfir16k.cu).
//
// Measured and rejected (one B200, 4096 taps):
//   - fastfir_kernel<13>, the register-resident CTA-level kernel, for 8192-point blocks (round 1): 50 300 Msamples/s
//     against 99 400 for the shared-memory kernel of the next item (DESIGN.md, overlap-save rows; SASS in
//     profiles/sass/r1_fastfir_8192.sass).
//   - fastfir8k_kernel, 8192-point blocks in place in shared memory, two CTAs per SM: 100.2 against 121.0 Gsamples/s
//     for the 16384-point kernel in the same process (profiles/r1_s8_fastfir16k_check.json), 99.9 against 121.3 in
//     round 2 (profiles/r2_a_ff16k_v1_check.json); the 16384-point kernel has since reached 145.3.  SASS and ncu keys
//     in profiles/sass/r1_fastfir8k.sass and profiles/r1_s3_fastfir8k_v4_ncu_keys.txt.
//
// Streaming (lrc_fastfir_stream_*): every channel carries the samples of its row that no complete compute block has
// consumed yet (fewer than one compute block) in a device carry buffer; a push runs the STREAM instance of the plan's
// kernel over every (channel, block) whose window is complete, reading [carry | chunk] in place (fastfir.cuh), then
// copies the new tail into the other carry buffer of a ping-pong pair.  Blocks sit at multiples of ngood from the start
// of the stream and see the same window and zero padding as in one lrc_fastfir_run over the whole stream, so the outputs
// are bitwise those of that call whatever the push sizes.
#include "fastfir.cuh"
#include "fft_core.cuh"
#include <cmath>
#include <utility>
#include <vector>

using namespace lrfft;

int lrc_make_twiddles(int nfft, DevBuf<float2> &d_tw);
int lrc_log2_exact(int n);

struct lrc_fastfir {
    lrc_ctx *ctx;
    size_t   nh, nfft, ngood;   // nfft/ngood: the block size that fixes the OUTPUT LENGTH (kiss_fastfir's, or the caller's)
    int      log2n;             // log2(nfft): the fastfir_kernel instance when !compute16k
    DevBuf<float2> d_tw;        // twiddles of the compute block size (nfft, or 16384)
    DevBuf<float2> d_H;         // FFT(h rotated) / compute block size, in the order the plan's kernel reads it
    DevBuf<float2> d_tw1k;      // 16384-point kernel: W_1024^k for the warp-level sub-transforms
    bool     compute16k;        // blocks are COMPUTED 16384 points at a time whatever nfft says (see lrc_fastfir_create)
};

// host-side f64 radix-2 FFT (forward): the only H builder, for every compute block size
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

// STREAM: n_blocks counts (channel, block) items of a stream push, n_blocks_full the full blocks per channel (fastfir.cuh)
template <int LOG2N, bool STREAM>
__global__ void __launch_bounds__(CtaFFT<LOG2N, false>::T)
fastfir_kernel(const float2 *__restrict__ in, size_t n_in, float2 *__restrict__ out, size_t n_blocks_full,
               size_t n_blocks, size_t ngood, size_t flush_keep, const float2 *__restrict__ tw,
               const float2 *__restrict__ H, FfStreamArgs sa)
{
    using FF = CtaFFT<LOG2N, false>;
    using FI = CtaFFT<LOG2N, true>;
    constexpr int N = FF::N, E = FF::E, T = FF::T;
    extern __shared__ float2 sm[];
    const int t = threadIdx.x;
    for (size_t w = blockIdx.x; w < n_blocks; w += gridDim.x) {
        size_t b = w;
        const float2 *src = in;
        float2 *dst = out;
        if constexpr (STREAM) {
            const size_t c = (unsigned)w / (unsigned)sa.nblk;
            b = w - c * sa.nblk;
            src = in + c * sa.in_stride;
            dst = out + c * sa.out_stride;
        }
        const size_t s0 = b * ngood;
        const size_t avail = n_in - s0;              // < N only for the flush block
        float2 v[E];
        if constexpr (STREAM) {
            if (s0 >= sa.held) {                     // the block lies in the chunk (CTA-uniform)
                src += s0 - sa.held;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const size_t i = (size_t)t + (size_t)e * T;
                    v[e] = (i < avail) ? __ldcs(src + i) : make_float2(0.f, 0.f);
                }
            } else {                                 // straddles the carried history
                const float2 *crow = sa.carry + ((unsigned)w / (unsigned)sa.nblk) * sa.carry_pitch;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const size_t i = s0 + (size_t)t + (size_t)e * T;
                    v[e] = i < sa.held ? __ldg(crow + i) : i < n_in ? __ldcs(src + (i - sa.held)) : make_float2(0.f, 0.f);
                }
            }
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const size_t i = (size_t)t + (size_t)e * T;
                v[e] = (i < avail) ? __ldcs(in + s0 + i) : make_float2(0.f, 0.f);
            }
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
            if (i < keep) __stcs(dst + s0 + i, v[e]);
        }
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
    const int l2 = lrc_log2_exact((int)nfft);
    if (l2 < 1 || l2 > 14) {
        lrc_set_error("lrc_fastfir_create: nfft=%zu: only powers of two in [2, 16384] (nh <= 8192 with the "
                      "automatic size)", nfft);
        return LRC_ERR_UNSUPPORTED;
    }
    LRC_REQUIRE(nfft >= nh, LRC_ERR_INVALID, "lrc_fastfir_create: nfft shorter than the impulse response");
    // Overlap-save gives the same y[k] whatever the block size; the block size only fixes how many outputs a call
    // without flush produces (kff_nocopy :199-204 stops at the last FULL block).  So `nfft` keeps that meaning, and
    // long filters and large blocks are COMPUTED in 16384-point blocks: 12289 of 16384 outputs kept per block for 4096
    // taps instead of 4097 of 8192.
    const bool c16 = nh > 1024 || nfft >= 8192;
    const size_t nc = c16 ? 16384 : nfft;        // the compute block size
    lrc_fastfir *f = new (std::nothrow) lrc_fastfir();
    LRC_REQUIRE(f != nullptr, LRC_ERR_NOMEM, "out of host memory");
    f->ctx = ctx; f->nh = nh; f->nfft = nfft; f->ngood = nfft - nh + 1; f->log2n = l2; f->compute16k = c16;
    int rc = lrc_make_twiddles((int)nc, f->d_tw);
    if (!rc && c16) rc = lrc_make_twiddles(1024, f->d_tw1k);
    if (!rc && c16) rc = lrc_fastfir16k_prepare();
    if (rc) { lrc_fastfir_destroy(f); return rc; }
    // H = FFT(h rotated left by nh-1) / nc (:148-169) in f64 on the host, rounded once to f32
    const float2 *h = reinterpret_cast<const float2 *>(h_taps_cpx);
    std::vector<double> re(nc, 0.0), im(nc, 0.0);
    re[0] = h[nh - 1].x; im[0] = h[nh - 1].y;
    for (size_t i = 0; i + 1 < nh; ++i) { re[nc - nh + 1 + i] = h[i].x; im[nc - nh + 1 + i] = h[i].y; }
    host_fft_f64(re, im);
    std::vector<float2> H(nc);
    for (size_t i = 0; i < nc; ++i) H[i] = make_float2((float)(re[i] / (double)nc), (float)(im[i] / (double)nc));
    if (c16) {
        const std::vector<float2> Hn(H);
        lrc_fastfir16k_permute_H(Hn.data(), H.data());
    }
    cudaError_t e = f->d_H.alloc(nc);
    if (e == cudaSuccess) e = cudaMemcpy(f->d_H, H.data(), nc * sizeof(float2), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        lrc_set_error("lrc_fastfir_create: %s", cudaGetErrorString(e));
        lrc_fastfir_destroy(f);
        return LRC_ERR_CUDA;
    }
    *out = f;
    return LRC_OK;
}

extern "C" int lrc_fastfir_destroy(lrc_fastfir *f)
{
    if (!f) return LRC_OK;
    cudaSetDevice(f->ctx->device);
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

template <int LOG2N, bool STREAM>
static int launch_fastfir(lrc_fastfir *f, const float2 *in, size_t n_in, float2 *out, size_t full, size_t nblk,
                          size_t keep, const FfStreamArgs &sa, cudaStream_t s)
{
    using FF = CtaFFT<LOG2N, false>;
    const int threads = FF::T;
    const size_t smem = (size_t)FF::SMEM_CPX * sizeof(float2);
    auto kern = fastfir_kernel<LOG2N, STREAM>;
    size_t blocks;
    LRC_CUDA(lrc_resident_ctas(kern, threads, smem, f->ctx->n_sm, &blocks, true));
    if (blocks > nblk) blocks = nblk;
    kern<<<(unsigned)blocks, threads, smem, s>>>(in, n_in, out, full, nblk, f->ngood, keep, f->d_tw, f->d_H, sa);
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
                                     f->d_tw1k, f->d_H, nullptr, s);
    }
    switch (f->log2n) {
#define FF_CASE(L) case L: return launch_fastfir<L, false>(f, in, n_in, out, full, nblk, keep, FfStreamArgs{}, s);
        FF_CASE(1) FF_CASE(2) FF_CASE(3) FF_CASE(4) FF_CASE(5) FF_CASE(6) FF_CASE(7)
        FF_CASE(8) FF_CASE(9) FF_CASE(10) FF_CASE(11) FF_CASE(12)
#undef FF_CASE
    }
    return LRC_ERR_UNSUPPORTED;
}

// ---- streaming ---------------------------------------------------------------------------------
struct lrc_fastfir_stream {
    lrc_fastfir *ff;
    size_t       n_ch;
    size_t       nc, ngood;     // the compute block (nfft, or 16384) and its advance nc - nh + 1
    size_t       held;          // samples every channel carries, < nc
    DevBuf<float2> d_carry[2];  // [n_ch][nc] each, ping-pong; d_carry[cur] holds the history
    int          cur;
};

extern "C" int lrc_fastfir_stream_create(lrc_fastfir *f, size_t n_ch, lrc_fastfir_stream **out)
{
    LRC_REQUIRE(f && out && n_ch >= 1, LRC_ERR_INVALID, "lrc_fastfir_stream_create: bad arguments");
    LRC_BIND(f->ctx);
    lrc_fastfir_stream *st = new (std::nothrow) lrc_fastfir_stream();
    LRC_REQUIRE(st != nullptr, LRC_ERR_NOMEM, "out of host memory");
    st->ff = f; st->n_ch = n_ch;
    st->nc = f->compute16k ? 16384 : f->nfft;
    st->ngood = st->nc - f->nh + 1;
    st->held = 0; st->cur = 0;
    for (auto &p : st->d_carry) {
        const cudaError_t e = p.alloc(n_ch * st->nc);
        if (e != cudaSuccess) {
            lrc_set_error("lrc_fastfir_stream_create: %s", cudaGetErrorString(e));
            lrc_fastfir_stream_destroy(st);
            return LRC_ERR_CUDA;
        }
    }
    *out = st;
    return LRC_OK;
}

extern "C" int lrc_fastfir_stream_destroy(lrc_fastfir_stream *st)
{
    if (!st) return LRC_OK;
    cudaSetDevice(st->ff->ctx->device);
    delete st;
    return LRC_OK;
}

extern "C" int lrc_fastfir_stream_reset(lrc_fastfir_stream *st)
{
    LRC_REQUIRE(st != nullptr, LRC_ERR_INVALID, "null stream");
    st->held = 0; st->cur = 0;
    return LRC_OK;
}

// complete compute blocks of a row of held + n samples and, with flush, the outputs of the zero-padded remainder
static void stream_counts(const lrc_fastfir_stream *st, size_t n, int flush, size_t *full, size_t *flush_keep)
{
    const size_t total = st->held + n;
    *full = total >= st->nc ? (total - st->nc) / st->ngood + 1 : 0;
    const size_t rem = total - *full * st->ngood;
    *flush_keep = (flush && rem + 1 > st->ff->nh) ? rem + 1 - st->ff->nh : 0;
}

extern "C" size_t lrc_fastfir_stream_next_out_len(const lrc_fastfir_stream *st, size_t n, int flush)
{
    if (!st) return 0;
    size_t full, keep;
    stream_counts(st, n, flush, &full, &keep);
    return full * st->ngood + keep;
}

// `rows` rows of `width` bytes; one row needs no pitch (a one-channel stream may have any chunk_stride)
static cudaError_t copy_rows(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width, size_t rows,
                             cudaStream_t s)
{
    if (rows == 1) return cudaMemcpyAsync(dst, src, width, cudaMemcpyDeviceToDevice, s);
    return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, cudaMemcpyDeviceToDevice, s);
}

extern "C" int lrc_fastfir_stream_push(lrc_fastfir_stream *st, const float *d_chunk, size_t n, size_t chunk_stride,
                                       float *d_out, size_t out_stride, int flush, size_t *n_out, void *stream)
{
    LRC_REQUIRE(st && n_out, LRC_ERR_INVALID, "lrc_fastfir_stream_push: null argument");
    lrc_fastfir *f = st->ff;
    LRC_BIND(f->ctx);
    *n_out = 0;
    const size_t n_ch = st->n_ch, es = sizeof(float2);
    size_t full, keep;
    stream_counts(st, n, flush, &full, &keep);
    const size_t no = full * st->ngood + keep, nblk = full + (keep ? 1 : 0);
    if (n > 0) {
        LRC_REQUIRE(d_chunk != nullptr && chunk_stride >= n, LRC_ERR_INVALID, "lrc_fastfir_stream_push: bad chunk");
        LRC_REQUIRE(((uintptr_t)d_chunk & 7) == 0, LRC_ERR_INVALID, "lrc_fastfir_stream_push: misaligned chunk");
    }
    if (no > 0) {
        LRC_REQUIRE(d_out != nullptr && ((uintptr_t)d_out & 7) == 0, LRC_ERR_INVALID,
                    "lrc_fastfir_stream_push: null or misaligned output");
        LRC_REQUIRE(out_stride >= no, LRC_ERR_CAPACITY, "lrc_fastfir_stream_push: out_stride shorter than the outputs");
        if (n > 0) {
            const uintptr_t c0 = (uintptr_t)d_chunk, c1 = c0 + ((n_ch - 1) * chunk_stride + n) * es;
            const uintptr_t o0 = (uintptr_t)d_out, o1 = o0 + ((n_ch - 1) * out_stride + no) * es;
            LRC_REQUIRE(o1 <= c0 || c1 <= o0, LRC_ERR_INVALID, "lrc_fastfir_stream_push: output overlaps the chunk");
        }
        LRC_REQUIRE(n_ch * nblk <= 0xffffffffull, LRC_ERR_UNSUPPORTED, "lrc_fastfir_stream_push: more than 2^32 blocks");
    }
    cudaStream_t s = lrc_stream(f->ctx, stream);
    const float2 *chunk = (const float2 *)d_chunk;
    float2 *carry = st->d_carry[st->cur];
    if (nblk > 0) {
        const FfStreamArgs sa{carry, st->nc, st->held, chunk_stride, out_stride, nblk, 0, 0};
        const size_t total = st->held + n;
        float2 *out = (float2 *)d_out;
        int rc = LRC_ERR_UNSUPPORTED;
        if (f->compute16k) {
            rc = lrc_fastfir16k_launch(f->ctx->n_sm, chunk, total, out, full, n_ch * nblk, st->ngood, keep, f->d_tw,
                                       f->d_tw1k, f->d_H, &sa, s);
        } else {
            switch (f->log2n) {
#define FF_CASE(L) case L: rc = launch_fastfir<L, true>(f, chunk, total, out, full, n_ch * nblk, keep, sa, s); break;
                FF_CASE(1) FF_CASE(2) FF_CASE(3) FF_CASE(4) FF_CASE(5) FF_CASE(6) FF_CASE(7)
                FF_CASE(8) FF_CASE(9) FF_CASE(10) FF_CASE(11) FF_CASE(12)
#undef FF_CASE
            }
        }
        if (rc) return rc;
    }
    if (flush) {
        st->held = 0;                                    // back at the initial state
    } else if (full == 0) {
        // no block completed: the chunk goes behind the history
        if (n > 0)
            LRC_CUDA(copy_rows(carry + st->held, st->nc * es, chunk, chunk_stride * es, n * es, n_ch, s));
        st->held += n;
    } else {
        // the new history is row[consumed .. held + n), into the other buffer of the pair
        const size_t consumed = full * st->ngood;
        float2 *next = st->d_carry[st->cur ^ 1];
        size_t at = 0;
        if (consumed < st->held) {
            at = st->held - consumed;
            LRC_CUDA(copy_rows(next, st->nc * es, carry + consumed, st->nc * es, at * es, n_ch, s));
        }
        const size_t skip = consumed > st->held ? consumed - st->held : 0;
        if (n > skip)
            LRC_CUDA(copy_rows(next + at, st->nc * es, chunk + skip, chunk_stride * es, (n - skip) * es, n_ch, s));
        st->held = st->held + n - consumed;
        st->cur ^= 1;
    }
    *n_out = no;
    return LRC_OK;
}
