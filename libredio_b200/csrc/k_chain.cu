// k_chain.cu -- the headline chain as ONE kernel:
//   cf32 -> FIR(64 taps)/10 (dsputils::convolve, dsputils.rs:30-32, + decimation)
//        -> frames of 1024 -> window -> FFT (kiss_fft, kiss_fft.c:238-388) -> |X|^2 averaged
//           over k_avg frames (tools/psdpng.c:165-177).
// The decimated signal and the spectra never touch HBM: per 1024-point frame the kernel reads
// 10294 input samples (82 KB, one TMA bulk copy) and writes nothing until a partial spectrum
// (4 KB) per work item of up to 16 frames.
//
// CTA layout (224 threads, 2 CTAs per SM):
//   warps 0-4  FIR producers : wait for the TMA tile, register-blocked FIR (fir_core.cuh, R = 7
//                              outputs per thread), hand the 1024 outputs over in shared memory,
//                              re-arm the TMA for the next frame
//   warps 5-6  FFT consumers : pull the frame into registers (x window), Stockham FFT
//                              (fft_core.cuh), accumulate |X|^2 in registers
// so the FFT of frame i overlaps the FIR of frame i+1, and the TMA of one CTA overlaps the
// arithmetic of the other CTA on the SM.
#include "fir_core.cuh"
#include "fft_core.cuh"
#include "unpack.cuh"
#include "chain_generic.cuh"
#include <vector>
#include <cmath>

using namespace lrfft;

int    lrc_make_twiddles(int nfft, DevBuf<float2> &d_tw);
int    lrc_log2_exact(int n);
size_t lrc_psd_frames_per_item(size_t k_avg);
int    lrc_psd_reduce(const float *d_partial, float *d_rows, int nfft, size_t ipr, size_t n_rows, float scale,
                      int accumulate, cudaStream_t s);

struct lrc_chain {
    lrc_ctx *ctx;
    int      ntaps, decim, nfft, log2n, window;
    bool     fused;            // the BASELINE instance chain_kernel<64,10,10,7> (cf32 and u8 input)
    bool     fused_generic;    // an instance of chain_gen_kernel (chain_generic.cuh): ntaps <= 128, decim in {4,5,8,10,16}, nfft in {512,1024,2048}
    std::vector<float> taps;
    DevBuf<float2> d_tw;
    DevBuf<float>  d_win;
    DevBuf<float>  d_partial;
    // unfused fallback for shapes without a fused instance
    lrc_fir *fir; lrc_psd *psd;
    DevBuf<float>  d_tmp;                      // decimated signal
    // host ring (lrc_chain_run_host)
    DevBuf<float>  d_ring[2];                  // cf32
    DevBuf<uint8_t> d_ring_u8[2];              // u8 IQ staging of lrc_chain_run_host_u8 (2 bytes per sample)
    DevEvent ev_ready[2], ev_free[2];
    DevBuf<float>  d_rows;
    DevBuf<float>  d_u8tmp;                    // lrc_chain_run_u8 without a fused instance: unpacked input (cf32)
};

template <int NTAPS, int DECIM, int LOG2N, int R>
struct ChainCfg {
    using Tile = FirTile<NTAPS, DECIM, R>;
    using FFT = CtaFFT<LOG2N, false>;
    static constexpr int N = 1 << LOG2N;
    static constexpr int FRAME_ADV = N * DECIM;                         // input samples between frames
    static constexpr int TILE_IN = (N - 1) * DECIM + NTAPS;             // input samples a frame needs
    static constexpr int NFIR = (N + R - 1) / R;                        // threads doing FIR work
    static constexpr int NFIR_T = (NFIR + 31) / 32 * 32;                // FIR warps, whole
    static constexpr int NFFT_T = FFT::T;                               // FFT threads (64 for N = 1024)
    static constexpr int NT = NFIR_T + NFFT_T;
    static constexpr int TILE_SAMPLES = (NFIR - 1) * Tile::STEP + Tile::WIN;   // last thread's window end
    static constexpr uint32_t TMA_BYTES = TILE_IN * 8;
    // u8 instance: the raw IQ tile (2 B per sample) lands at the END of the cf32 tile buffer and is expanded in place
    static constexpr uint32_t RAW_BYTES = TILE_IN * 2;
    static constexpr uint32_t RAW_TMA_BYTES = RAW_BYTES & ~15u;                   // bulk part; the < 16-byte rest by hand
    static constexpr int RAW_WORDS = (RAW_BYTES + 3) / 4;                         // two samples per word
    static constexpr int RAW_OFF = (TILE_SAMPLES * 8 - (int)((RAW_BYTES + 15) & ~15u)) & ~15;
    static constexpr int RAW_PER_THREAD = (RAW_WORDS + NFIR_T - 1) / NFIR_T;
    static_assert(RAW_BYTES % 4 == 0, "whole words");
    static_assert((RAW_BYTES - RAW_TMA_BYTES) / 4 <= NFIR_T, "the rest words fall into the last two words of their owners");
    static constexpr int OFF_HAND = TILE_SAMPLES * 8;                   // FIR -> FFT hand-over buffer
    static constexpr int OFF_XCHG = OFF_HAND + FFT::SMEM_CPX * 8;       // FFT pass exchange buffer
    static constexpr int OFF_BAR = OFF_XCHG + FFT::SMEM_CPX * 8;
    static constexpr int SMEM_BYTES = OFF_BAR + 16;
    static_assert(TMA_BYTES % 16 == 0 && (FRAME_ADV * 8) % 16 == 0, "TMA alignment");
    static_assert(NFFT_T % 32 == 0, "FFT threads must be whole warps");
};

enum { BAR_FULL = 1, BAR_EMPTY = 2, BAR_TILE = 3, BAR_FFT = 4 };

// IS_U8: `in` points at rtlsdr u8 I,Q (2 bytes per sample, rtlsdr.rs:160-162).  The producers expand the raw tile to cf32
// IN SHARED MEMORY with the one device definition of i2f (unpack.cuh: the reference's division and subtraction, bit-exact),
// then run the very same FIR code on it, so the rows equal unpack-then-chain bit for bit while HBM (and PCIe, through
// lrc_chain_run_host_u8) carries 2 bytes per sample instead of 8 and no separate unpack launch exists.
template <int NTAPS, int DECIM, int LOG2N, int R, bool IS_U8>
__global__ void __launch_bounds__(ChainCfg<NTAPS, DECIM, LOG2N, R>::NT, 2)
chain_kernel(const float2 *__restrict__ in, const float2 *__restrict__ tw, const float *__restrict__ win,
             float *__restrict__ partial, size_t k_avg, size_t fpi, size_t ipr, size_t n_items,
             const __grid_constant__ FirTaps<NTAPS> taps)
{
    using Cfg = ChainCfg<NTAPS, DECIM, LOG2N, R>;
    using Tile = typename Cfg::Tile;
    using FFT = typename Cfg::FFT;
    constexpr int N = Cfg::N, E = FFT::E, T = FFT::T;
    extern __shared__ __align__(128) uint8_t smem[];
    float2 *tile = reinterpret_cast<float2 *>(smem);
    float2 *hand = reinterpret_cast<float2 *>(smem + Cfg::OFF_HAND);
    float2 *xchg = reinterpret_cast<float2 *>(smem + Cfg::OFF_XCHG);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + Cfg::OFF_BAR);
    const int tid = threadIdx.x;
    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    __syncthreads();
    if ((size_t)blockIdx.x >= n_items) return;

    // both roles walk the same (item, frame) schedule
    auto item_range = [&](size_t item, size_t &f0, size_t &f1) {
        const size_t row = item / ipr, c = item % ipr;
        f0 = row * k_avg + c * fpi;
        f1 = f0 + fpi;
        if (f1 > (row + 1) * k_avg) f1 = (row + 1) * k_avg;
    };

    if (tid < Cfg::NFIR_T) {
        // ================= FIR producers =================
        uint32_t phase = 0;
        bool first = true;
        size_t item = blockIdx.x, f0, f1;
        item_range(item, f0, f1);
        size_t f = f0;
        const uint8_t *in8 = reinterpret_cast<const uint8_t *>(in);
        uint8_t *raw = smem + Cfg::RAW_OFF;
        auto load_frame = [&](size_t fr) {                       // thread 0
            if (IS_U8) {
                mbar_expect_tx(bar, Cfg::RAW_TMA_BYTES);
                tma_load_1d_evict_first(raw, in8 + fr * (size_t)Cfg::FRAME_ADV * 2, Cfg::RAW_TMA_BYTES, bar);
            } else {
                mbar_expect_tx(bar, Cfg::TMA_BYTES);
                tma_load_1d_evict_first(tile, in + fr * Cfg::FRAME_ADV, Cfg::TMA_BYTES, bar);
            }
        };
        if (tid == 0) load_frame(f);
        while (true) {
            if (IS_U8) {
                // the last < 16 bytes of the raw tile are not a whole TMA unit: their owners fetch them with plain loads,
                // issued before the wait (they can only fall into a thread's last two words)
                constexpr int TMA_WORDS = (int)(Cfg::RAW_TMA_BYTES / 4), KL = Cfg::RAW_PER_THREAD;
                uint32_t rest[2] = {0u, 0u};
#pragma unroll
                for (int k = KL - 2; k < KL; ++k) {
                    const int i = tid + k * Cfg::NFIR_T;
                    if (k >= 0 && i >= TMA_WORDS && i < Cfg::RAW_WORDS)
                        rest[k - (KL - 2)] = *reinterpret_cast<const uint32_t *>(in8 + f * (size_t)Cfg::FRAME_ADV * 2 + 4 * (size_t)i);
                }
                mbar_wait(bar, phase);
                // expand in place: every producer first takes its share of the raw words into registers, then (barrier)
                // writes them back as cf32 -- the cf32 tile grows over the raw bytes only after all of them were read
                uint32_t wv[Cfg::RAW_PER_THREAD];
                const uint32_t *rw = reinterpret_cast<const uint32_t *>(raw);
#pragma unroll
                for (int k = 0; k < KL; ++k) {
                    const int i = tid + k * Cfg::NFIR_T;
                    wv[k] = i < TMA_WORDS ? rw[i] : (k >= KL - 2 ? rest[k - (KL - 2)] : 0u);
                }
                named_bar_sync(BAR_TILE, Cfg::NFIR_T);
                float4 *t4 = reinterpret_cast<float4 *>(tile);
#pragma unroll
                for (int k = 0; k < Cfg::RAW_PER_THREAD; ++k) {
                    const int i = tid + k * Cfg::NFIR_T;
                    if (i < Cfg::RAW_WORDS)
                        t4[i] = make_float4(lr_i2f_byte(wv[k], 0), lr_i2f_byte(wv[k], 1), lr_i2f_byte(wv[k], 2), lr_i2f_byte(wv[k], 3));
                }
                named_bar_sync(BAR_TILE, Cfg::NFIR_T);
            } else {
                mbar_wait(bar, phase);
            }
            phase ^= 1;
            float2 acc[R];
            if (tid < Cfg::NFIR) Tile::run_cf32(tile + (size_t)tid * Tile::STEP, taps, acc);
            // next frame of this CTA
            size_t nf = f + 1, nitem = item, nf1 = f1;
            if (nf == f1) {
                nitem = item + gridDim.x;
                if (nitem < n_items) item_range(nitem, nf, nf1);
            }
            const bool has_next = nitem < n_items;
            // every FIR thread is done with the tile -> re-arm the TMA for the next frame
            named_bar_sync(BAR_TILE, Cfg::NFIR_T);
            if (tid == 0 && has_next) load_frame(nf);
            // hand-over buffer free? (the FFT warps arrive on EMPTY once they hold the previous frame)
            if (!first) named_bar_sync(BAR_EMPTY, Cfg::NT);
            first = false;
            if (tid < Cfg::NFIR) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int o = tid * R + r;
                    if (o < N) hand[FFT::pad(o)] = acc[r];
                }
            }
            __threadfence_block();
            named_bar_arrive(BAR_FULL, Cfg::NT);
            if (!has_next) break;
            item = nitem; f = nf; f1 = nf1;
        }
    } else {
        // ================= FFT consumers =================
        const int t = tid - Cfg::NFIR_T;
        float w[E], acc[E];
#pragma unroll
        for (int e = 0; e < E; ++e) { w[e] = win[t + e * T]; acc[e] = 0.f; }
        size_t item = blockIdx.x, f0, f1;
        item_range(item, f0, f1);
        size_t f = f0;
        while (true) {
            size_t nf = f + 1, nitem = item, nf1 = f1;
            if (nf == f1) {
                nitem = item + gridDim.x;
                if (nitem < n_items) item_range(nitem, nf, nf1);
            }
            const bool has_next = nitem < n_items;
            named_bar_sync(BAR_FULL, Cfg::NT);
            float2 v[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const float2 x = hand[FFT::pad(t + e * T)];
                v[e] = make_float2(x.x * w[e], x.y * w[e]);
            }
            if (has_next) named_bar_arrive(BAR_EMPTY, Cfg::NT);
            FFT::run(v, xchg, tw, t, SyncNamed{BAR_FFT, T});
#pragma unroll
            for (int e = 0; e < E; ++e) acc[e] = fmaf(v[e].x, v[e].x, fmaf(v[e].y, v[e].y, acc[e]));
            const bool item_done = (f + 1 == f1);
            if (item_done) {
                float *dst = partial + item * N + t;
#pragma unroll
                for (int e = 0; e < E; ++e) { dst[e * T] = acc[e]; acc[e] = 0.f; }
            }
            if (!has_next) break;
            item = nitem; f = nf; f1 = nf1;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static const size_t SEG_FRAMES = 400;     // host ring: frames per H2D segment (~33 MB of cf32 at 64/10/1024)

extern "C" int lrc_chain_create(lrc_ctx *ctx, const float *h_taps, int ntaps, int decim, int nfft, int window,
                                lrc_chain **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && h_taps && ntaps >= 1 && decim >= 1, LRC_ERR_INVALID, "lrc_chain_create: bad arguments");
    const int l2 = lrc_log2_exact(nfft);
    if (l2 < 1 || l2 > 13) {
        lrc_set_error("lrc_chain_create: nfft=%d: only powers of two in [2, 8192]", nfft);
        return LRC_ERR_UNSUPPORTED;
    }
    lrc_chain *c = new (std::nothrow) lrc_chain();
    LRC_REQUIRE(c != nullptr, LRC_ERR_NOMEM, "out of host memory");
    c->ctx = ctx; c->ntaps = ntaps; c->decim = decim; c->nfft = nfft; c->log2n = l2; c->window = window;
    c->taps.assign(h_taps, h_taps + ntaps);
    c->fused = (ntaps == 64 && decim == 10 && nfft == 1024);
    c->fused_generic = false;
    // A/B knobs: LRC_CHAIN_NO_GENERIC=1 forces the unfused path, LRC_CHAIN_GENERIC_ALL=1 the fused instance for every shape that
    // has one (by default only where it measured faster than the unfused kernels, chain_generic.cuh: prefer_fused)
    if (!c->fused && !getenv("LRC_CHAIN_NO_GENERIC")) {
        c->fused_generic = lrc_chaing_has(ntaps, decim, l2, getenv("LRC_CHAIN_GENERIC_ALL") != nullptr);
    }
    int rc = lrc_fir_create(ctx, h_taps, ntaps, decim, &c->fir);       // also validates the taps
    if (!rc) rc = lrc_psd_create(ctx, nfft, window, &c->psd);
    if (!rc) rc = lrc_make_twiddles(nfft, c->d_tw);
    if (!rc) {
        std::vector<float> w(nfft);
        const double pi = 3.14159265358979323846264338327950288;
        for (int i = 0; i < nfft; ++i)
            w[i] = window == LRC_WINDOW_HANN ? (float)(0.5 - 0.5 * cos(2.0 * pi * i / nfft)) : 1.0f;
        if (c->d_win.alloc(nfft) != cudaSuccess ||
            cudaMemcpy(c->d_win, w.data(), sizeof(float) * nfft, cudaMemcpyHostToDevice) != cudaSuccess) {
            lrc_set_error("lrc_chain_create: %s", cudaGetErrorString(cudaGetLastError()));
            rc = LRC_ERR_CUDA;
        }
    }
    if (rc) { lrc_chain_destroy(c); return rc; }
    *out = c;
    return LRC_OK;
}

extern "C" int lrc_chain_destroy(lrc_chain *c)
{
    if (!c) return LRC_OK;
    cudaSetDevice(c->ctx->device);
    lrc_fir_destroy(c->fir); lrc_psd_destroy(c->psd);
    delete c;
    return LRC_OK;
}

extern "C" size_t lrc_chain_frames(const lrc_chain *c, size_t n_in)
{
    if (!c) return 0;
    const size_t tile_in = (size_t)(c->nfft - 1) * c->decim + c->ntaps;
    if (n_in < tile_in) return 0;
    return (n_in - tile_in) / ((size_t)c->nfft * c->decim) + 1;
}

extern "C" int lrc_chain_kind(const lrc_chain *c)
{
    if (!c) return 0;
    return c->fused ? 1 : (c->fused_generic ? 2 : 0);
}

template <bool IS_U8>
static int chain_launch_fused(lrc_chain *c, const void *d_in, size_t k_local, size_t fpi, size_t ipr, size_t n_items, cudaStream_t s)
{
    using Cfg = ChainCfg<64, 10, 10, 7>;
    auto kern = chain_kernel<64, 10, 10, 7, IS_U8>;
    size_t ctas;
    LRC_CUDA(lrc_resident_ctas(kern, Cfg::NT, Cfg::SMEM_BYTES, c->ctx->n_sm, &ctas));
    static const size_t gm = lrc_grid_mult("LRC_CHAIN_GRID", 1);
    size_t blocks = ctas * gm;
    if (blocks > n_items) blocks = n_items;
    FirTaps<64> taps;
    for (int i = 0; i < 64; ++i) taps.h[i] = c->taps[i];
    kern<<<(unsigned)blocks, Cfg::NT, Cfg::SMEM_BYTES, s>>>((const float2 *)d_in, c->d_tw, c->d_win, c->d_partial,
                                                           k_local, fpi, ipr, n_items, taps);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

// rows_local rows of k_local frames each, starting at d_in (cf32, or u8 I,Q when input_is_u8 -- fused instance only);
// rows[r] (op)= scale * sum |X|^2
static int chain_launch(lrc_chain *c, const void *d_in_any, int input_is_u8, size_t rows_local, size_t k_local, float *d_rows,
                        float scale, int accumulate, cudaStream_t s)
{
    const float *d_in = (const float *)d_in_any;
    if (rows_local == 0 || k_local == 0) return LRC_OK;
    const size_t fpi = lrc_psd_frames_per_item(k_local);
    const size_t ipr = ceil_div(k_local, fpi);
    const size_t n_items = rows_local * ipr;
    LRC_CUDA(c->d_partial.ensure(n_items * (size_t)c->nfft));
    int rc;
    if (c->fused) {
        rc = input_is_u8 ? chain_launch_fused<true>(c, d_in_any, k_local, fpi, ipr, n_items, s)
                         : chain_launch_fused<false>(c, d_in_any, k_local, fpi, ipr, n_items, s);
        if (rc) return rc;
        return lrc_psd_reduce(c->d_partial, d_rows, c->nfft, ipr, rows_local, scale, accumulate, s);
    }
    LRC_REQUIRE(!input_is_u8, LRC_ERR_INVALID, "chain_launch: u8 input without a fused instance");
    if (c->fused_generic) {
        chaing::Args a;
        a.in = (const float2 *)d_in_any; a.tw = c->d_tw; a.win = c->d_win; a.taps = c->taps.data(); a.partial = c->d_partial;
        a.k_avg = k_local; a.fpi = fpi; a.ipr = ipr; a.n_items = n_items; a.ntaps = c->ntaps; a.n_sm = c->ctx->n_sm; a.stream = s;
        const int grc = lrc_chaing_launch(a, c->decim, c->log2n);
        if (grc > 0) return grc;
        if (grc == 0) return lrc_psd_reduce(c->d_partial, d_rows, c->nfft, ipr, rows_local, scale, accumulate, s);
        // grc < 0 cannot happen for a plan whose fused_generic is set; fall through to the unfused kernels
    }
    // unfused fallback: FIR into a scratch signal, then the PSD kernel
    const size_t n_frames = rows_local * k_local;
    const size_t n_dec = n_frames * (size_t)c->nfft;
    const size_t n_in = (n_dec - 1) * (size_t)c->decim + c->ntaps;
    LRC_CUDA(c->d_tmp.ensure(n_dec * 2 + (size_t)c->nfft * rows_local));
    rc = lrc_fir_run_cf32(c->fir, d_in, 1, n_in, n_in, c->d_tmp, n_dec, s);
    if (rc) return rc;
    float *rows_tmp = c->d_tmp + n_dec * 2;
    rc = lrc_psd_run(c->psd, c->d_tmp, n_frames, k_local, rows_tmp, s);
    if (rc) return rc;
    // rows (op)= scale*k_local * rows_tmp  (lrc_psd_run already divided by k_local)
    return lrc_psd_reduce(rows_tmp, d_rows, c->nfft, 1, rows_local, scale * (float)k_local, accumulate, s);
}

extern "C" int lrc_chain_run(lrc_chain *c, const float *d_in, size_t n_in, size_t k_avg, float *d_rows,
                             size_t *n_rows, void *stream)
{
    LRC_REQUIRE(c != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(c->ctx);
    LRC_REQUIRE(k_avg >= 1, LRC_ERR_INVALID, "lrc_chain_run: k_avg must be >= 1");
    const size_t rows = lrc_chain_frames(c, n_in) / k_avg;
    if (n_rows) *n_rows = rows;
    if (rows == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_rows, LRC_ERR_INVALID, "lrc_chain_run: null buffer");
    LRC_REQUIRE(((uintptr_t)d_in & 15) == 0, LRC_ERR_INVALID, "lrc_chain_run: input must be 16-byte aligned");
    return chain_launch(c, d_in, 0, rows, k_avg, d_rows, 1.0f / (float)k_avg, 0, lrc_stream(c->ctx, stream));
}

// device-resident rtlsdr u8 I,Q input: the fused instance expands the tile on chip; other shapes unpack into a scratch
// buffer first (lrc_unpack_u8_cf32) and run the cf32 path
extern "C" int lrc_chain_run_u8(lrc_chain *c, const uint8_t *d_iq, size_t n_in, size_t k_avg, float *d_rows,
                                size_t *n_rows, void *stream)
{
    LRC_REQUIRE(c != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(c->ctx);
    LRC_REQUIRE(k_avg >= 1, LRC_ERR_INVALID, "lrc_chain_run_u8: k_avg must be >= 1");
    const size_t rows = lrc_chain_frames(c, n_in) / k_avg;
    if (n_rows) *n_rows = rows;
    if (rows == 0) return LRC_OK;
    LRC_REQUIRE(d_iq && d_rows, LRC_ERR_INVALID, "lrc_chain_run_u8: null buffer");
    cudaStream_t s = lrc_stream(c->ctx, stream);
    if (c->fused) {
        LRC_REQUIRE(((uintptr_t)d_iq & 15) == 0, LRC_ERR_INVALID, "lrc_chain_run_u8: input must be 16-byte aligned");
        return chain_launch(c, d_iq, 1, rows, k_avg, d_rows, 1.0f / (float)k_avg, 0, s);
    }
    const size_t need = (rows * k_avg - 1) * (size_t)c->nfft * c->decim + (size_t)(c->nfft - 1) * c->decim + c->ntaps;
    LRC_CUDA(c->d_u8tmp.ensure(need * 2));
    const int urc = lrc_unpack_u8_cf32(c->ctx, d_iq, need * 2, c->d_u8tmp, s);
    if (urc) return urc;
    return chain_launch(c, c->d_u8tmp, 0, rows, k_avg, d_rows, 1.0f / (float)k_avg, 0, s);
}

static int chain_run_host_impl(lrc_chain *c, const void *h_in_any, int input_is_u8, size_t n_in, size_t k_avg,
                               float *h_rows, size_t *n_rows)
{
    const float *h_in = (const float *)h_in_any;
    const uint8_t *h_in_u8 = (const uint8_t *)h_in_any;
    LRC_REQUIRE(c != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(c->ctx);
    LRC_REQUIRE(k_avg >= 1, LRC_ERR_INVALID, "lrc_chain_run_host: k_avg must be >= 1");
    const size_t rows = lrc_chain_frames(c, n_in) / k_avg;
    if (n_rows) *n_rows = rows;
    if (rows == 0) return LRC_OK;
    LRC_REQUIRE(h_in && h_rows, LRC_ERR_INVALID, "lrc_chain_run_host: null buffer");
    const size_t adv = (size_t)c->nfft * c->decim;                      // input samples per frame
    const size_t tile_in = (size_t)(c->nfft - 1) * c->decim + c->ntaps;  // input samples one frame reads
    const size_t tail = (size_t)c->ntaps > (size_t)c->decim ? (size_t)c->ntaps - c->decim : 0;  // samples past the last frame's advance
    // segment plan: whole rows per segment when rows are short, slices of one row otherwise
    const bool slice_rows = k_avg > SEG_FRAMES;
    const size_t seg_frames = slice_rows ? SEG_FRAMES / 16 * 16 : (SEG_FRAMES / k_avg) * k_avg;
    const size_t slot_samples = seg_frames * adv + tail + 8;
    const bool direct_u8 = input_is_u8 && c->fused;     // the fused u8 instance reads the raw slot itself
    for (int i = 0; i < 2; ++i) {
        if (!direct_u8) LRC_CUDA(c->d_ring[i].ensure(slot_samples * 2));
        if (input_is_u8) LRC_CUDA(c->d_ring_u8[i].ensure(slot_samples * 2));
    }
    LRC_CUDA(c->d_rows.ensure(rows * (size_t)c->nfft));
    for (int i = 0; i < 2; ++i) {
        LRC_CUDA(c->ev_ready[i].ensure());
        LRC_CUDA(c->ev_free[i].ensure());
    }
    cudaStream_t cs = c->ctx->copy_stream, ks = c->ctx->stream;
    const size_t total_frames = rows * k_avg;
    const float scale = 1.0f / (float)k_avg;
    size_t seg = 0;
    for (size_t f = 0; f < total_frames; ++seg) {
        size_t nfr = seg_frames;
        if (slice_rows) {
            const size_t row_end = (f / k_avg + 1) * k_avg;            // slices never cross a row
            if (f + nfr > row_end) nfr = row_end - f;
        }
        if (f + nfr > total_frames) nfr = total_frames - f;
        const int b = (int)(seg & 1);
        // exactly what the segment's last frame reaches: (nfr-1)*adv + tile_in.  With decim > ntaps that is LESS than
        // nfr*adv, and lrc_chain_frames guarantees the caller's buffer no further than this.
        const size_t ns = (nfr - 1) * adv + tile_in;
        if (seg >= 2) LRC_CUDA(cudaStreamWaitEvent(cs, c->ev_free[b], 0));
        if (input_is_u8)      // 2 bytes per sample over PCIe; rtlsdr::data_to_samples runs on the device
            LRC_CUDA(cudaMemcpyAsync(c->d_ring_u8[b], h_in_u8 + 2 * f * adv, ns * 2, cudaMemcpyHostToDevice, cs));
        else
            LRC_CUDA(cudaMemcpyAsync(c->d_ring[b], h_in + 2 * f * adv, ns * sizeof(float2), cudaMemcpyHostToDevice, cs));
        LRC_CUDA(cudaEventRecord(c->ev_ready[b], cs));
        LRC_CUDA(cudaStreamWaitEvent(ks, c->ev_ready[b], 0));
        if (input_is_u8 && !direct_u8) {
            const int urc = lrc_unpack_u8_cf32(c->ctx, c->d_ring_u8[b], ns * 2, c->d_ring[b], ks);
            if (urc) return urc;
        }
        const void *seg_in = direct_u8 ? (const void *)c->d_ring_u8[b].get() : (const void *)c->d_ring[b].get();
        int rc;
        if (slice_rows) {
            const size_t row = f / k_avg;
            rc = chain_launch(c, seg_in, direct_u8, 1, nfr, c->d_rows + row * c->nfft, scale, (f % k_avg) != 0, ks);
        } else {
            rc = chain_launch(c, seg_in, direct_u8, nfr / k_avg, k_avg, c->d_rows + (f / k_avg) * c->nfft, scale, 0, ks);
        }
        if (rc) return rc;
        LRC_CUDA(cudaEventRecord(c->ev_free[b], ks));
        f += nfr;
    }
    LRC_CUDA(cudaMemcpyAsync(h_rows, c->d_rows, rows * (size_t)c->nfft * sizeof(float), cudaMemcpyDeviceToHost, ks));
    LRC_CUDA(cudaStreamSynchronize(ks));
    return LRC_OK;
}

extern "C" int lrc_chain_run_host(lrc_chain *c, const float *h_in, size_t n_in, size_t k_avg, float *h_rows,
                                  size_t *n_rows)
{
    return chain_run_host_impl(c, h_in, 0, n_in, k_avg, h_rows, n_rows);
}

extern "C" int lrc_chain_run_host_u8(lrc_chain *c, const uint8_t *h_iq, size_t n_in, size_t k_avg, float *h_rows,
                                     size_t *n_rows)
{
    return chain_run_host_impl(c, h_iq, 1, n_in, k_avg, h_rows, n_rows);
}
