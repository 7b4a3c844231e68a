// chain_generic.cuh -- the fused chain (k_chain.cu) for shapes other than the BASELINE one:
//   cf32 -> FIR(ntaps <= NTAPS)/DECIM (dsputils::convolve, dsputils.rs:30-32, + decimation)
//        -> frames of N = 2^LOG2N -> window -> FFT (kiss_fft.c:238-388) -> |X|^2 averaged (psdpng.c:165-177)
// one kernel, the decimated signal and the spectra never in HBM -- same warp-specialised layout as chain_kernel
// (FIR producer warps, FFT consumer warps, named barriers between them, mbarrier for the TMA), with three
// generalisations:
//
//  * ntaps is a RUN-TIME value <= NTAPS: the taps are zero-padded to NTAPS (a zero tap adds +-0 to the
//    accumulator: the sum is the ntaps-tap sum), the TMA brings exactly the (N-1) DECIM + ntaps samples
//    lrc_chain_frames promises, and the rest of the tile is zeroed once per CTA so the padded taps only ever meet zeros.
//
//  * the tile is written by the TMA in CHUNKS of STEP = R DECIM samples (one thread window advance), chunk c at byte
//    c (8 STEP + PADB): when 8 STEP is an even multiple of 16 bytes -- every power-of-two DECIM -- the thread windows of a
//    dense tile would start in the same one or two bank groups and the FIR's LDS.128 would run 4 to 8 ways conflicted
//    (the BASELINE shape escapes with R = 7, DECIM = 10: 560 bytes = 35 x 16); PADB = 16 makes the window pitch an odd
//    multiple of 16 bytes again.  A thread's sample j sits at 8 j + PADB (j / STEP) from its window start: compile-time
//    offsets after unrolling.  FIR thread t issues the bulk copy of chunk t, so the 70-300 copies of a tile are issued
//    in parallel, all completing on one mbarrier.
//
//  * N in {512, 1024, 2048}; a frame is produced in 1, 2 or 4 sub-tiles (GenCfg below), so every one of the 30 shapes fits
//    shared memory and the ones that only fit one CTA per SM overlap their own loads through a two-stage tile ring.
#pragma once
#include "fir_core.cuh"
#include "fft_core.cuh"

namespace chaing {
using namespace lrfft;

template <int NTAPS, int DECIM, int R>
struct GenTile {
    static constexpr int STEP = R * DECIM;
    static_assert(STEP % 2 == 0, "thread windows must start 16-byte aligned");
    static constexpr int WIN = (R - 1) * DECIM + NTAPS;
    static constexpr int WINL = (WIN + 1) & ~1;                       // loaded as pairs; a pad sample meets no tap
    static constexpr int PADB = ((STEP / 2) % 2 == 0) ? 16 : 0;
    static constexpr int PITCH = STEP * 8 + PADB;                      // bytes between thread windows = between chunks
    __host__ __device__ static constexpr int off(int j) { return j * 8 + PADB * (j / STEP); }

    __device__ __forceinline__ static void run(const uint8_t *wb, const FirTaps<NTAPS> &taps, float2 *acc)
    {
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < WINL; j += 2) {
            const float4 x = *reinterpret_cast<const float4 *>(wb + off(j));
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int k0 = j - r * DECIM, k1 = k0 + 1;
                // one packed FFMA2 per sample and tap (re and im lanes, the tap broadcast from a uniform register): the
                // shapes with a small decimation are FP32-issue bound, not HBM bound
                if (k0 >= 0 && k0 < NTAPS) acc[r] = fma2(make_float2(x.x, x.y), make_float2(taps.h[k0], taps.h[k0]), acc[r]);
                if (k1 >= 0 && k1 < NTAPS) acc[r] = fma2(make_float2(x.z, x.w), make_float2(taps.h[k1], taps.h[k1]), acc[r]);
            }
        }
    }
};

// sub-tiling: a frame's N outputs are produced in SUBT sub-tiles of NS = N / SUBT outputs, each from its own TMA tile.
//   SUBT = 1, one tile buffer : the whole frame from one tile (the BASELINE instance's scheme; with two or more CTAs per SM the
//                               TMA of one CTA overlaps the arithmetic of the others);
//   SUBT = 2 or 4, two buffers: a two-stage ring of half- or quarter-frame tiles: sub-tile g + 2 is on its way while g + 1 is
//                               filtered.  This is how 2048 x 16 (a 262 KB frame tile) fits at all.
template <int NTAPS, int DECIM, int LOG2N, int R, int SUBT_>
struct GenLayout {
    using Tile = GenTile<NTAPS, DECIM, R>;
    using FFT = CtaFFT<LOG2N, false>;
    static constexpr int N = 1 << LOG2N, SUBT = SUBT_, NBUF = SUBT == 1 ? 1 : 2;
    static constexpr int NS = N / SUBT;                                  // outputs per sub-tile
    static constexpr int TILE_IN_MAX = (NS - 1) * DECIM + NTAPS;
    static constexpr int NFIR = (NS + R - 1) / R;
    static constexpr int N_CHUNKS_MAX = (TILE_IN_MAX + Tile::STEP - 1) / Tile::STEP;
    static constexpr int WIN_END = (NFIR - 1) * Tile::PITCH + Tile::off(Tile::WINL - 1) + 16;   // last byte a FIR thread reads
    static constexpr int CHUNK_END = N_CHUNKS_MAX * Tile::PITCH;
    static constexpr int TILE_BYTES = ((WIN_END > CHUNK_END ? WIN_END : CHUNK_END) + 127) / 128 * 128;
    static constexpr int SMEM_BYTES = NBUF * TILE_BYTES + 2 * FFT::SMEM_CPX * 8 + 32;
};

template <int NTAPS, int DECIM, int LOG2N, int R>
struct GenCfg {
    using L1 = GenLayout<NTAPS, DECIM, LOG2N, R, 1>;
    using L2 = GenLayout<NTAPS, DECIM, LOG2N, R, 2>;
    // Measured (profiles/r2_p_chain_generic.jsonl): for shapes that fit ONE CTA per SM the two-stage ring with half-frame
    // sub-tiles is slower than the whole-frame tile (64/16/1024: 0.71 vs 0.89 of HBM, 64/10/2048: 0.63 vs 0.74) -- half the
    // producer threads, and only one 66-82 KB sub-tile in flight while the other is filtered, where the whole-frame load
    // keeps 130-160 KB in flight.  So sub-tiling is used only where the whole-frame tile does not fit at all (2048 x 16).
    static constexpr int SUBT = (L1::SMEM_BYTES + 1024 <= 227 * 1024) ? 1 : (L2::SMEM_BYTES <= 227 * 1024 ? 2 : 4);
    using L = GenLayout<NTAPS, DECIM, LOG2N, R, SUBT>;
    using Tile = typename L::Tile;
    using FFT = typename L::FFT;
    static constexpr int N = L::N, NS = L::NS, NBUF = L::NBUF;
    static constexpr int FRAME_ADV = N * DECIM;
    static constexpr int SUB_ADV = NS * DECIM;                           // input samples between sub-tiles
    static constexpr int NFIR = L::NFIR;
    static constexpr int NFIR_T = (NFIR + 31) / 32 * 32;
    static constexpr int NFFT_T = FFT::T;
    static constexpr int NT = NFIR_T + NFFT_T;
    static constexpr int TILE_BYTES = L::TILE_BYTES;
    static constexpr int OFF_HAND = NBUF * TILE_BYTES;
    static constexpr int OFF_XCHG = OFF_HAND + FFT::SMEM_CPX * 8;
    static constexpr int OFF_BAR = OFF_XCHG + FFT::SMEM_CPX * 8;
    static constexpr int SMEM_BYTES = OFF_BAR + 32;
    static constexpr bool FITS = SMEM_BYTES <= 227 * 1024 && NT <= 1024;
    // as many CTAs per SM as shared memory and a 128-register thread (the 16-point-per-thread FFT needs that) allow
    // (decim 4 / 5 are FP32-bound in the FIR producers, which need ~40 registers: there the budget is 96 registers -- the FFT warps
    // still fit without spilling and the producers get a third CTA per SM: 64/4/1024 0.835 -> 0.716 ms, 64/5/1024 0.752 -> 0.607;
    // 80 registers, four CTAs and 56 bytes of spill measured the same)
    static constexpr int REG_BUDGET = DECIM <= 5 ? 96 : 128;
    static constexpr int BY_SMEM = (227 * 1024) / (SMEM_BYTES + 1024), BY_REGS = 65536 / (NT * REG_BUDGET);
    static constexpr int MIN_CTAS_RAW = BY_SMEM < BY_REGS ? BY_SMEM : BY_REGS;
    static constexpr int MIN_CTAS = MIN_CTAS_RAW < 1 ? 1 : (MIN_CTAS_RAW > 8 ? 8 : MIN_CTAS_RAW);
    static_assert((FRAME_ADV * 8) % 16 == 0 && (SUB_ADV * 8) % 16 == 0 && (Tile::STEP * 8) % 16 == 0, "TMA alignment");
    static_assert(NFFT_T % 32 == 0, "FFT threads must be whole warps");
    static_assert(N % SUBT == 0, "whole sub-tiles");
};

enum { BAR_FULL = 1, BAR_EMPTY = 2, BAR_TILE = 3, BAR_FFT = 4 };

template <int NTAPS, int DECIM, int LOG2N, int R>
__global__ void __launch_bounds__(GenCfg<NTAPS, DECIM, LOG2N, R>::NT, GenCfg<NTAPS, DECIM, LOG2N, R>::MIN_CTAS)
chain_gen_kernel(const float2 *__restrict__ in, const float2 *__restrict__ tw, const float *__restrict__ win,
                 float *__restrict__ partial, size_t k_avg, size_t fpi, size_t ipr, size_t n_items, int ntaps_rt,
                 const __grid_constant__ FirTaps<NTAPS> taps)
{
    using Cfg = GenCfg<NTAPS, DECIM, LOG2N, R>;
    using Tile = typename Cfg::Tile;
    using FFT = typename Cfg::FFT;
    constexpr int N = Cfg::N, E = FFT::E, T = FFT::T, SUBT = Cfg::SUBT, NBUF = Cfg::NBUF, NS = Cfg::NS;
    extern __shared__ __align__(128) uint8_t smem[];
    float2 *hand = reinterpret_cast<float2 *>(smem + Cfg::OFF_HAND);
    float2 *xchg = reinterpret_cast<float2 *>(smem + Cfg::OFF_XCHG);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + Cfg::OFF_BAR);
    const int tid = threadIdx.x;
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < NBUF; ++i) mbar_init(bar + i, 1);
        mbar_fence_init();
    }
    // the padded taps (ntaps_rt..NTAPS-1 are zero) must only ever meet finite values: zero the tiles once
    for (int i = tid; i < NBUF * Cfg::TILE_BYTES / 16; i += Cfg::NT) reinterpret_cast<float4 *>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_proxy_async();                                   // ... before the TMA (async proxy) writes over them
    __syncthreads();
    if ((size_t)blockIdx.x >= n_items) return;

    auto item_range = [&](size_t item, size_t &f0, size_t &f1) {
        const size_t row = item / ipr, c = item % ipr;
        f0 = row * k_avg + c * fpi;
        f1 = f0 + fpi;
        if (f1 > (row + 1) * k_avg) f1 = (row + 1) * k_avg;
    };

    if (tid < Cfg::NFIR_T) {
        // ================= FIR producers =================
        const int tile_in = (NS - 1) * DECIM + ntaps_rt;                // samples of a sub-tile that exist in the input
        const int n_chunks = (tile_in + Tile::STEP - 1) / Tile::STEP;
        const int tma_samples = tile_in & ~1;                           // bulk copies move whole 16-byte units ...
        // the CTA's schedule as a cursor over (item, frame, sub-tile); two cursors walk it: `cur` (being filtered) and
        // `ld` (being loaded, NBUF sub-tiles ahead)
        struct Cursor { size_t item, f, f1; int s; bool ok; };
        auto start = [&]() { Cursor c; c.item = blockIdx.x; size_t f0; item_range(c.item, f0, c.f1); c.f = f0; c.s = 0; c.ok = true; return c; };
        auto advance = [&](Cursor &c) {
            if (++c.s < SUBT) return;
            c.s = 0;
            if (++c.f < c.f1) return;
            c.item += gridDim.x;
            if (c.item < n_items) { size_t f0; item_range(c.item, f0, c.f1); c.f = f0; }
            else c.ok = false;
        };
        auto load_sub = [&](const Cursor &c, int buf) {                 // every producer thread: its chunk(s)
            const float2 *src = in + c.f * (size_t)Cfg::FRAME_ADV + (size_t)c.s * Cfg::SUB_ADV;
            uint8_t *tile = smem + (size_t)buf * Cfg::TILE_BYTES;
            if (tid == 0) mbar_expect_tx(bar + buf, (uint32_t)tma_samples * 8u);
            for (int ch = tid; ch < n_chunks; ch += Cfg::NFIR_T) {
                const int s0 = ch * Tile::STEP;
                int ns = tma_samples - s0;
                if (ns > Tile::STEP) ns = Tile::STEP;
                if (ns > 0) tma_load_1d_evict_first(tile + (size_t)ch * Tile::PITCH, src + s0, (uint32_t)ns * 8u, bar + buf);
                // ... and an odd last sample goes by hand; a BAR_TILE barrier lies between this store and the sub-tile's use
                if ((tile_in & 1) && s0 + Tile::STEP >= tile_in && s0 < tile_in)
                    *reinterpret_cast<float2 *>(tile + (size_t)ch * Tile::PITCH + (size_t)(tile_in - 1 - s0) * 8) = __ldg(src + tile_in - 1);
            }
        };
        Cursor cur = start(), ld = cur;
#pragma unroll
        for (int i = 0; i < NBUF; ++i)
            if (ld.ok) { load_sub(ld, i); advance(ld); }
        named_bar_sync(BAR_TILE, Cfg::NFIR_T);                          // hand-copied samples of the first sub-tiles
        uint32_t g = 0;                                                  // sub-tiles done by this CTA
        bool first = true;
        while (true) {
            const int buf = (int)(g % NBUF);
            mbar_wait(bar + buf, (g / NBUF) & 1u);
            float2 acc[R];
            if (tid < Cfg::NFIR) Tile::run(smem + (size_t)buf * Cfg::TILE_BYTES + (size_t)tid * Tile::PITCH, taps, acc);
            // every FIR thread is done with the tile -> the chunks of the sub-tile NBUF ahead go into it
            named_bar_sync(BAR_TILE, Cfg::NFIR_T);
            if (ld.ok) { load_sub(ld, buf); advance(ld); }
            // a new frame starts: is the hand-over buffer free? (the FFT warps arrive on EMPTY once they hold the previous frame)
            if (cur.s == 0) {
                if (!first) named_bar_sync(BAR_EMPTY, Cfg::NT);
                first = false;
            }
            if (tid < Cfg::NFIR) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int o = tid * R + r;
                    if (o < NS) hand[FFT::pad(cur.s * NS + o)] = acc[r];
                }
            }
            const bool frame_done = cur.s == SUBT - 1;
            advance(cur);
            if (frame_done) {
                __threadfence_block();
                named_bar_arrive(BAR_FULL, Cfg::NT);
            }
            if (!cur.ok) break;
            if (NBUF == 1 && (tile_in & 1)) named_bar_sync(BAR_TILE, Cfg::NFIR_T);   // the hand-copied sample, single buffer
            ++g;
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
            if (f + 1 == f1) {
                float *dst = partial + item * N + t;
#pragma unroll
                for (int e = 0; e < E; ++e) { dst[e * T] = acc[e]; acc[e] = 0.f; }
            }
            if (!has_next) break;
            item = nitem; f = nf; f1 = nf1;
        }
    }
}

// what a launch needs besides the template arguments
struct Args {
    const float2 *in, *tw;
    const float *win, *taps;     // taps: host pointer, ntaps values
    float *partial;
    size_t k_avg, fpi, ipr, n_items;
    int ntaps, n_sm;
    cudaStream_t stream;
};

// LRC_OK = launched, -1 = no instance for this shape (caller runs unfused), > 0 = LRC error
template <int NTAPS, int DECIM, int LOG2N, int R>
static int launch_one(const Args &a)
{
    using Cfg = GenCfg<NTAPS, DECIM, LOG2N, R>;
    if constexpr (!Cfg::FITS) {
        return -1;
    } else {
        auto kern = chain_gen_kernel<NTAPS, DECIM, LOG2N, R>;
        size_t blocks;
        LRC_CUDA(lrc_resident_ctas(kern, Cfg::NT, Cfg::SMEM_BYTES, a.n_sm, &blocks));
        if (blocks > a.n_items) blocks = a.n_items;
        FirTaps<NTAPS> taps;
        for (int i = 0; i < NTAPS; ++i) taps.h[i] = i < a.ntaps ? a.taps[i] : 0.0f;
        kern<<<(unsigned)blocks, Cfg::NT, Cfg::SMEM_BYTES, a.stream>>>(a.in, a.tw, a.win, a.partial, a.k_avg, a.fpi, a.ipr,
                                                                      a.n_items, a.ntaps, taps);
        LRC_CUDA(cudaGetLastError());
        return 0;
    }
}

// R per decimation: window advance R DECIM of 28..64 samples (enough producer threads, 2-3x shared-memory read amplification)
template <int DECIM> struct RFor;
template <> struct RFor<4>  { static constexpr int R = 8; };
template <> struct RFor<5>  { static constexpr int R = 8; };
template <> struct RFor<8>  { static constexpr int R = 7; };
template <> struct RFor<10> { static constexpr int R = 7; };
template <> struct RFor<16> { static constexpr int R = 4; };

template <int NTAPS, int DECIM>
static int launch_decim_n(const Args &a, int log2n)
{
    constexpr int R = RFor<DECIM>::R;
    switch (log2n) {
        case 9:  return launch_one<NTAPS, DECIM, 9, R>(a);
        case 10: return launch_one<NTAPS, DECIM, 10, R>(a);
        case 11: return launch_one<NTAPS, DECIM, 11, R>(a);
        default: return -1;
    }
}

// Which shapes a plan runs fused.  Every instance FITS; whether it is the faster path was measured against the unfused one
// (FIR tile kernel -> HBM -> PSD kernel, itself at 0.8 of the HBM roofline since the FIR got tile instances for these shapes too,
// profiles/r2_w_chain_generic_vs_unfused.txt): fused wins 1.03-1.22x when two or more CTAs fit an SM (the TMA of one overlaps the
// arithmetic of the other) and the producers are not starved (decim >= 8; decim 4 / 5 up to 64 taps and nfft 1024, where the
// 96-register budget gives them a third CTA); it ties or loses (1.01-0.74x) for the one-CTA shapes (whole-frame tile: load and
// filter serialise) and for 128 taps at decim 4 / 5 (FP32-bound producers with 18 warps per SM against the stand-alone FIR's 24).
// all = true (LRC_CHAIN_GENERIC_ALL=1, what the parity tests use) selects every fitting instance.
template <int NTAPS, int DECIM, int LOG2N>
static constexpr bool prefer_fused()
{
    using C = GenCfg<NTAPS, DECIM, LOG2N, RFor<DECIM>::R>;
    return C::FITS && C::BY_SMEM >= 2 && (DECIM >= 8 || LOG2N <= 9 || (LOG2N == 10 && NTAPS <= 64));
}

template <int DECIM>
static bool has_decim(int ntaps, int log2n, bool all)
{
    constexpr int R = RFor<DECIM>::R;
    if (ntaps < 1 || ntaps > 128 || log2n < 9 || log2n > 11) return false;
    if (ntaps <= 64) {
        if (log2n == 9)  return GenCfg<64, DECIM, 9, R>::FITS && (all || prefer_fused<64, DECIM, 9>());
        if (log2n == 10) return GenCfg<64, DECIM, 10, R>::FITS && (all || prefer_fused<64, DECIM, 10>());
        return GenCfg<64, DECIM, 11, R>::FITS && (all || prefer_fused<64, DECIM, 11>());
    }
    if (log2n == 9)  return GenCfg<128, DECIM, 9, R>::FITS && (all || prefer_fused<128, DECIM, 9>());
    if (log2n == 10) return GenCfg<128, DECIM, 10, R>::FITS && (all || prefer_fused<128, DECIM, 10>());
    return GenCfg<128, DECIM, 11, R>::FITS && (all || prefer_fused<128, DECIM, 11>());
}

}  // namespace chaing

// Translation units: the three nfft instances of a (decimation, 64-tap) pair share one (k_chaing_d*_n64.cu); a 128-tap instance
// is a minute or more of compilation on its own, so each has its own (k_chaing_d*_n128_l*.cu) -- a fresh build is then bounded by
// the core count, not by one file.
#define LRC_CHAING_DECL(D_, NT_) int lrc_chaing_launch_d##D_##_n##NT_(const chaing::Args &a, int log2n)
#define LRC_CHAING_DEFINE(D_, NT_) LRC_CHAING_DECL(D_, NT_) { return chaing::launch_decim_n<NT_, D_>(a, log2n); }
#define LRC_CHAING_DECL1(D_, NT_, L_) int lrc_chaing_launch_d##D_##_n##NT_##_l##L_(const chaing::Args &a)
#define LRC_CHAING_DEFINE1(D_, NT_, L_) \
    LRC_CHAING_DECL1(D_, NT_, L_) { return chaing::launch_one<NT_, D_, L_, chaing::RFor<D_>::R>(a); }
LRC_CHAING_DECL(4, 64); LRC_CHAING_DECL(5, 64); LRC_CHAING_DECL(8, 64); LRC_CHAING_DECL(10, 64); LRC_CHAING_DECL(16, 64);
#define LRC_CHAING_DECL3(D_) LRC_CHAING_DECL1(D_, 128, 9); LRC_CHAING_DECL1(D_, 128, 10); LRC_CHAING_DECL1(D_, 128, 11)
LRC_CHAING_DECL3(4); LRC_CHAING_DECL3(5); LRC_CHAING_DECL3(8); LRC_CHAING_DECL3(10); LRC_CHAING_DECL3(16);
int  lrc_chaing_launch(const chaing::Args &a, int decim, int log2n);     // k_chaing.cu: dispatch
bool lrc_chaing_has(int ntaps, int decim, int log2n, bool all);
