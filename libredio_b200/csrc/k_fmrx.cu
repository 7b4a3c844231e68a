// k_fmrx.cu -- BASELINE config 3 as ONE kernel per chunk:
//   rtlsdr u8 IQ (rtlsdr.rs:159-162) -> FIR 64 taps / 10 (dsputils.rs:30-32 + decimation) -> quadrature discriminator
//   (north-star stage) -> 1/5 polyphase resampler (samplerate.rs:59-87, our definition) -> 48 kHz f32 audio.
// HBM sees the 2 B/sample of raw IQ once and the 0.08 B/sample of audio once; the 240 kHz complex baseband and the
// 240 kHz discriminator output (2 x 8 B + 2 x 4 B per baseband sample in the three-launch pipeline) stay on chip.
//
// Work item = (channel PAIR, segment of the call's audio outputs).  A 256-thread CTA walks a segment in rounds:
//   round    : one TMA bulk copy per channel of the 6454 raw samples that 640 baseband samples need (double buffered);
//              threads 0-127 filter channel A, 128-255 channel B, 5 outputs each (FirTile<64,10,5>::run_u8, the same
//              packed FFMA2 chain as the stand-alone kernel: bit-identical baseband), the sample before a thread's
//              first comes from the left lane by shuffle (warp seams through 8 shared words), then x[n] conj(x[n-1])
//              -> atan2 (fm_core.cuh) -> the discriminator ring in shared memory, channels A and B INTERLEAVED as
//              {dA[i], dB[i]} pairs;
//   tile     : after 4 rounds (2560 new samples per channel) every thread computes 2 audio outputs of BOTH channels with
//              the packed window loop of the stand-alone decimator (RsDec2Steps<5,2>: one LDS.128 = two samples of
//              both channels, one FFMA2 per tap advances both accumulators), then the last 320 ring entries move to
//              the front as the next tile's history;
//   segment  : starts with one priming round that only fills that history (5-13 % extra FIR work per segment is the price
//              of having more work items than CTA slots; a segment is sized so that it stays near 5 %).
// Every audio sample is the same operation sequence wherever it falls in a tile, segment or call, so the stream is
// bit-identical however it is chunked; the carried state between calls is just raw input: the last <= 6.7 k samples.
//
// Measured and rejected (one B200): the three stand-alone stages for this shape, 752 200 Msamples/s in round 1 against
// 765 400 for this kernel in round 2 (DESIGN.md, config 3); they stay the path for every other shape.  fmrx_kernel bounded
// for 2 CTAs per SM (128 registers) instead of 3, timed against it in tools/runs/r2h.sh; the 3-CTA captures of that run are
// profiles/r2_r2h_fmrx3_ncu_keys.txt and r2_r2h_fmrx3_ncu_phases.txt.
#include "fir_core.cuh"
#include "fm_core.cuh"
#include <cmath>
#include <vector>

namespace fmrx {
constexpr int NTAPS = 64, DECIM = 10, M = 5;
constexpr int TPP = 2 * 32 * M + 1, HIST = TPP - 1;       // 321 resampler taps, 320 samples of history
constexpr int NT = 256, HALF = NT / 2;
constexpr int RF = 5;                                     // FIR outputs per thread and round
constexpr int ROUND_Z = RF * HALF;                        // 640 baseband samples per channel and round
constexpr int ROUNDS = 4;
constexpr int TILE_D = ROUND_Z * ROUNDS;                  // 2560 new discriminator samples per tile
// Measured and rejected (round 2, profiles/r2_r_fmrx_r2x8_ncu.txt): the resampler phase with R2 = 8 outputs on 64 threads and a
// padded ring (RsDec2Steps' STEPP/PADP form) -- 3.7x fewer shared-memory wavefronts in the phase, but six of the CTA's eight warps
// then wait at the barrier behind two (barrier stall 0.59 -> 3.2 per issue, instruction-fetch stalls on the 3 k-instruction
// straight-line block): 0.382 ms against 0.321 ms.  The kernel is issue-bound by its FIR phase (158 M of 218 M warp-instructions).
constexpr int R2 = 2;                                     // audio outputs per thread and tile (per channel)
constexpr int TILE_A = TILE_D / M;                        // 512
static_assert(TILE_A == R2 * NT, "every thread resamples");
constexpr int RING = HIST + TILE_D;                       // pairs
constexpr int ROUND_X = (ROUND_Z - 1) * DECIM + NTAPS;    // raw samples a round reads per channel
constexpr int RAW_BYTES = (ROUND_X * 2 + 15) / 16 * 16 + 16;   // + the 0..12 byte alignment shift
constexpr int OFF_RING = 2 * 2 * RAW_BYTES;
constexpr int OFF_ZL = OFF_RING + RING * 8;
constexpr int OFF_BAR = OFF_ZL + 4 * 2 * 4 * 8;
constexpr int SMEM_BYTES = OFF_BAR + 16;
constexpr int WIN2 = ((R2 - 1) * M + TPP + 1) / 2 * 2;    // 326
static_assert((NT - 1) * R2 * M + WIN2 <= RING, "resampler windows stay inside the ring");
using Fir = FirTile<NTAPS, DECIM, RF>;

struct Args {
    const uint8_t *carry; size_t carry_stride;            // [n_ch][carry_stride bytes]: the `held` samples before the chunk
    const uint8_t *chunk; size_t chunk_stride;            // bytes between channel rows
    long long held, n;                                    // samples in the carry / in the chunk
    long long row_abs0;                                   // absolute stream index of carry[0]
    long long m0, n_out;                                  // first audio output of the call, outputs per channel
    float *out; size_t out_stride;
    long long n_ch, tiles_per_pair, total_tiles;          // tiles of one channel pair this call, tiles of all pairs
    int last_rounds;                                      // rounds the (partial) last tile of a pair needs
    int use_tma;
};

// The rounds a CTA works through.  All tiles of the call, pair-major, are cut into gridDim.x contiguous ranges of equal
// length (+-1 tile): no tail wave, whatever the channel count.  A range starts with a priming round (history of its first
// tile) and primes again wherever it crosses into the next channel pair.
struct RoundIter {
    int g, g_end;                                         // current global tile, end of the range
    int q, nq;                                            // round within the tile (-1 = priming round), rounds of the tile
    int pair, ti;                                         // channel pair, tile within the pair
    __device__ void load(const Args &a)
    {
        pair = g / (int)a.tiles_per_pair;
        ti = g - pair * (int)a.tiles_per_pair;
        nq = ti == a.tiles_per_pair - 1 ? a.last_rounds : ROUNDS;
    }
    __device__ void init(const Args &a, int g0, int g1) { g = g0; g_end = g1; q = -1; nq = ROUNDS; pair = ti = 0; if (g < g_end) load(a); }
    __device__ bool valid() const { return g < g_end; }
    __device__ void next(const Args &a)
    {
        if (q < 0) { q = 0; return; }
        if (++q == nq) {
            ++g;
            if (g < g_end) { load(a); q = ti == 0 ? -1 : 0; }
        }
    }
    __device__ bool last_of_segment(const Args &a) const { return q == nq - 1 && (g + 1 == g_end || ti + 1 == a.tiles_per_pair); }
    __device__ long long m_tile0(const Args &a) const { return a.m0 + (long long)ti * TILE_A; }
    __device__ long long nz0(const Args &a) const { return M * m_tile0(a) + (long long)ROUND_Z * q; }   // first baseband index
};
}  // namespace fmrx

__global__ void __launch_bounds__(fmrx::NT, 3)
fmrx_kernel(const __grid_constant__ fmrx::Args a, const __grid_constant__ FirTaps<fmrx::NTAPS> taps127,
            const __grid_constant__ RsTaps<fmrx::TPP> rtaps)
{
    using namespace fmrx;
    extern __shared__ __align__(128) uint8_t fmrx_smem[];
    float2 *ring = reinterpret_cast<float2 *>(fmrx_smem + OFF_RING);
    float2 *zl = reinterpret_cast<float2 *>(fmrx_smem + OFF_ZL);           // [round & 3][channel][warp]: a slot is rewritten
                                                                           // three rounds later, two barriers after its last reader
    uint64_t *bar = reinterpret_cast<uint64_t *>(fmrx_smem + OFF_BAR);
    const int t = threadIdx.x, lane = t & 31, ch = t >> 7, tt = t & (HALF - 1), w = tt >> 5;
    if (t == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_fence_init(); }
    __syncthreads();

    // where a round's raw bytes of one channel live: virtual row [carry | chunk], byte offsets; returns the shift of
    // the round's first byte inside the (16-byte aligned) shared buffer
    const long long HB = 2 * a.held, LB = 2 * (a.held + a.n);
    auto span = [&](long long nz0, long long *lo, long long *hi, long long *a0) {
        const long long vb0 = 2 * (DECIM * nz0 - a.row_abs0);
        *a0 = vb0 & ~15ll;                                               // floors for negative values too
        long long a1 = (vb0 + 2 * ROUND_X + 15) & ~15ll;
        *lo = *a0 < 0 ? 0 : *a0;
        *hi = a1 > LB ? LB : a1;
        return (int)(vb0 - *a0);
    };
    auto issue = [&](const RoundIter &it, int stage) {                   // one thread
        long long lo, hi, a0;
        span(it.nz0(a), &lo, &hi, &a0);
        uint32_t total = 0;
        long long c_lo = lo, c_hi = hi < HB ? hi : HB, k_lo = lo > HB ? lo : HB, k_hi = hi;
        const uint32_t nc = c_hi > c_lo ? (uint32_t)(c_hi - c_lo) : 0u, nk = k_hi > k_lo ? (uint32_t)(k_hi - k_lo) : 0u;
        int live = 0;
        for (int c = 0; c < 2; ++c) live += (2 * (long long)it.pair + c < a.n_ch);
        total = (nc + nk) * live;
        mbar_expect_tx(&bar[stage], total);
        for (int c = 0; c < 2; ++c) {
            const long long chn = 2 * (long long)it.pair + c;
            if (chn >= a.n_ch) continue;
            uint8_t *dst = fmrx_smem + (stage * 2 + c) * RAW_BYTES;
            if (nc) tma_load_1d(dst + (c_lo - a0), a.carry + chn * a.carry_stride + c_lo, nc, &bar[stage]);
            if (nk) tma_load_1d(dst + (k_lo - a0), a.chunk + chn * a.chunk_stride + (k_lo - HB), nk, &bar[stage]);
        }
    };
    // unaligned rows: the CTA copies the round itself, sample by sample (2-byte units), synchronously
    auto fill_sync = [&](const RoundIter &it, int stage) {
        long long lo, hi, a0;
        span(it.nz0(a), &lo, &hi, &a0);
        for (int c = 0; c < 2; ++c) {
            const long long chn = 2 * (long long)it.pair + c;
            if (chn >= a.n_ch) continue;
            uint16_t *dst = reinterpret_cast<uint16_t *>(fmrx_smem + (stage * 2 + c) * RAW_BYTES);
            const uint8_t *crow = a.carry + chn * a.carry_stride, *krow = a.chunk + chn * a.chunk_stride;
            for (long long v = lo + 2 * t; v < hi; v += 2 * NT) {
                const uint8_t *p = v < HB ? crow + v : krow + (v - HB);
                dst[(v - a0) >> 1] = (uint16_t)p[0] | ((uint16_t)p[1] << 8);
            }
        }
    };

    RoundIter cur, ld;
    {
        const long long g0 = a.total_tiles * blockIdx.x / gridDim.x, g1 = a.total_tiles * (blockIdx.x + 1) / gridDim.x;
        cur.init(a, (int)g0, (int)g1);
        ld.init(a, (int)g0, (int)g1);
    }
    if (a.use_tma) {
        for (int s = 0; s < 2; ++s) {
            if (ld.valid()) {
                if (t == 0) issue(ld, s);
                ld.next(a);
            }
        }
    }
    // Software pipeline: iteration g filters round g AND runs the discriminator of round g-1 (whose five samples stayed in
    // registers) in the same straight-line block, so the discriminator's dependent chain (x conj(x'), reciprocal, degree-6
    // polynomial) fills issue slots between the FIR's packed FMAs instead of standing alone between two barriers -- as a
    // phase of its own it took 30 % of the kernel for 13 % of its instructions (profiles/r2_fmrx_v1_ncu_phases.txt).
    struct Pend { bool valid, tile_end, seg_end; int base, k0, k0o, pair; } pend;
    pend.valid = pend.tile_end = pend.seg_end = false; pend.base = 0; pend.k0 = RF + 1; pend.k0o = 0; pend.pair = 0;
    float2 zp[RF];
#pragma unroll
    for (int r = 0; r < RF; ++r) zp[r] = make_float2(0.f, 0.f);
    float *rp = reinterpret_cast<float *>(ring) + ch;
    for (unsigned g = 0; cur.valid() || pend.valid; ++g) {
        const bool have = cur.valid();
        const int stage = g & 1;
        long long nz0 = 0;
        int shift = 0;
        if (have) {
            long long lo, hi, a0;
            nz0 = cur.nz0(a);
            shift = span(nz0, &lo, &hi, &a0);
            if (a.use_tma) {
                mbar_wait(&bar[stage], (g >> 1) & 1);
            } else {
                fill_sync(cur, stage);
                __syncthreads();
            }
        }
        // the sample before this thread's first of round g-1: left lane, or the warp-seam words of rounds g-1 / g-2
        float2 prev = make_float2(__shfl_up_sync(0xffffffffu, zp[RF - 1].x, 1), __shfl_up_sync(0xffffffffu, zp[RF - 1].y, 1));
        if (lane == 0) prev = w ? zl[(((g - 1) & 3) * 2 + ch) * 4 + w - 1] : zl[(((g - 2) & 3) * 2 + ch) * 4 + 3];
        // ---- FIR of round g (garbage from a stale buffer in the drain iteration, never used) ... -------------------
        float2 z[RF];
        const uint32_t *sw = reinterpret_cast<const uint32_t *>(fmrx_smem + (stage * 2 + ch) * RAW_BYTES + shift) + tt * (Fir::STEP / 2);
        // ---- ... with the discriminator of round g-1 threaded through it: sample r after filter step 20 r ---------
        auto side = [&](int j) {
            if (j % 20 == 0 && j / 20 < RF) {
                const int r = j / 20;
                // stream start: x[-1] = 0 (the stand-alone discriminator's initial state), d[n < 0] = 0 (the resampler's)
                const float2 pz = r == pend.k0 ? make_float2(0.f, 0.f) : (r ? zp[r - 1] : prev);
                const float2 zz = fm_mul_conj(zp[r], pz);
                const float d = r >= pend.k0 ? lr_atan2(zz.y, zz.x) : 0.f;
                if (pend.valid && pend.base + r >= 0) rp[2 * (pend.base + r)] = d;
            }
        };
        Fir::template run_u8_with<decltype(side), false>(sw, taps127, z, side);
        if (have && lane == 31) zl[((g & 3) * 2 + ch) * 4 + w] = z[RF - 1];
#pragma unroll
        for (int r = 0; r < RF; ++r) zp[r] = z[r];
        __syncthreads();                                  // raw buffer consumed, ring and warp-seam samples visible
        if (a.use_tma && have && ld.valid()) {
            if (t == 0) issue(ld, stage);
            ld.next(a);
        }
        // ---- round g-1 completed a tile: 2 audio samples per thread and channel --------------------------------
        if (pend.valid && pend.tile_end) {
            float2 acc[R2];
#pragma unroll
            for (int r = 0; r < R2; ++r) acc[r] = make_float2(0.f, 0.f);
            RsDec2Steps<M, R2, TPP, 0, WIN2>::run(ring + t * (R2 * M), rtaps, acc);
            const long long k0o = pend.k0o + R2 * t;                                // index into the call's output
            const long long chA = 2 * (long long)pend.pair, chB = chA + 1;
#pragma unroll
            for (int r = 0; r < R2; ++r) {
                if (k0o + r < a.n_out) {
                    a.out[chA * a.out_stride + k0o + r] = acc[r].x;
                    if (chB < a.n_ch) a.out[chB * a.out_stride + k0o + r] = acc[r].y;
                }
            }
            __syncthreads();                              // before the next iteration's discriminator writes the ring
            if (!pend.seg_end)
                for (int i = t; i < HIST; i += NT) ring[i] = ring[TILE_D + i];
        }
        pend.valid = have;
        if (have) {
            // where round g's samples go in the ring (the priming round keeps its last 320 at the front), and which of this
            // thread's five is absolute sample 0 (anywhere else: outside 0..4)
            const long long n_abs0 = nz0 + RF * tt;
            pend.k0 = n_abs0 > 0 ? -1 : (n_abs0 < -(long long)RF ? RF + 1 : (int)(-n_abs0));
            pend.base = cur.q < 0 ? RF * tt - (ROUND_Z - HIST) : HIST + ROUND_Z * cur.q + RF * tt;
            pend.tile_end = cur.q == cur.nq - 1;
            pend.seg_end = cur.last_of_segment(a);
            pend.k0o = cur.ti * TILE_A;
            pend.pair = cur.pair;
            cur.next(a);
        }
    }
}

// next[c][i] = row[c][from + i], i < keep samples; row = [carry | chunk].  One V per copy: 16 bytes when the carry/chunk
// seam, `from` and both buffers are 16-byte aligned (a vector then never straddles the seam), else one sample (2 bytes).
template <typename V>
__global__ void fmrx_carry_kernel(const uint8_t *__restrict__ carry, size_t carry_stride, long long held_b,
                                  const uint8_t *__restrict__ chunk, size_t chunk_stride, long long from_b,
                                  long long keep_b, uint8_t *__restrict__ next, long long n_ch)
{
    const long long per = (keep_b + (long long)sizeof(V) - 1) / (long long)sizeof(V), total = n_ch * per;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long c = i / per, k = (i % per) * (long long)sizeof(V), v = from_b + k;
        const uint8_t *p = v < held_b ? carry + c * carry_stride + v : chunk + c * chunk_stride + (v - held_b);
        *reinterpret_cast<V *>(next + c * carry_stride + k) = *reinterpret_cast<const V *>(p);
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct lrc_fmrx {
    lrc_ctx *ctx;
    size_t   n_ch, max_chunk;
    bool     fused;
    // fused instance (64 taps / 10, ratio 1/5)
    FirTaps<fmrx::NTAPS> taps127;
    RsTaps<fmrx::TPP>    rtaps;
    DevBuf<uint8_t> d_carry[2]; int cur; size_t carry_stride;    // bytes per channel row
    long long held, n_raw, m_next;
    // composition for every other shape: the three stand-alone stages with their own carried state
    lrc_fir *fir; lrc_fir_stream *fs; lrc_resampler *rs;
    DevBuf<float> d_bb, d_fm, d_state;                    // [n_ch][bb_stride] cf32, [n_ch][bb_stride] f32, [n_ch] cf32
    size_t   bb_stride;
    int      decim, ntaps, rs_L, rs_M;
};

static const size_t FMRX_CARRY_CAP = 6912;                // samples: 6400 (priming round) + 63 + 50 + alignment slack

extern "C" int lrc_fmrx_create(lrc_ctx *ctx, const float *h_taps, int ntaps, int decim, double ratio, size_t n_ch,
                               size_t max_chunk, lrc_fmrx **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && h_taps && ntaps >= 1 && decim >= 1 && n_ch >= 1 && max_chunk >= 1, LRC_ERR_INVALID,
                "lrc_fmrx_create: bad arguments");
    lrc_fmrx *f = new (std::nothrow) lrc_fmrx();
    LRC_REQUIRE(f != nullptr, LRC_ERR_NOMEM, "out of host memory");
    f->ctx = ctx; f->n_ch = n_ch; f->max_chunk = max_chunk; f->decim = decim; f->ntaps = ntaps;
    f->fused = ntaps == fmrx::NTAPS && decim == fmrx::DECIM && fabs(ratio - 0.2) < 1e-15;
    // both forms need the plans: the fused one takes its taps from them (one designer, one rounding)
    int rc = lrc_fir_create(ctx, h_taps, ntaps, decim, &f->fir);           // validates the taps (finite)
    const size_t bb_max = (ntaps + max_chunk) / decim + 2;
    if (!rc) rc = lrc_resampler_create(ctx, ratio, n_ch, bb_max, &f->rs);
    if (!rc) rc = lrc_resampler_get_taps(f->rs, nullptr, 0, nullptr, &f->rs_L, &f->rs_M);
    if (rc) { lrc_fmrx_destroy(f); return rc; }
    if (f->fused) {
        for (int i = 0; i < fmrx::NTAPS; ++i) f->taps127.h[i] = (float)((double)h_taps[i] / 127.0);
        std::vector<double> h(fmrx::TPP);
        size_t nt = 0; int L = 0, Mq = 0;
        rc = lrc_resampler_get_taps(f->rs, h.data(), h.size(), &nt, &L, &Mq);
        if (rc || nt != (size_t)fmrx::TPP || L != 1 || Mq != fmrx::M) {
            lrc_set_error("lrc_fmrx_create: resampler prototype does not match the fused instance");
            lrc_fmrx_destroy(f);
            return rc ? rc : LRC_ERR_UNSUPPORTED;
        }
        for (int i = 0; i < fmrx::TPP; ++i) f->rtaps.g[i] = (float)h[fmrx::TPP - 1 - i];      // reversed: correlation form
        f->carry_stride = FMRX_CARRY_CAP * 2;
        for (int i = 0; i < 2; ++i) {
            if (f->d_carry[i].alloc(n_ch * f->carry_stride) != cudaSuccess) {
                lrc_set_error("lrc_fmrx_create: %s", cudaGetErrorString(cudaGetLastError()));
                lrc_fmrx_destroy(f);
                return LRC_ERR_CUDA;
            }
        }
        cudaError_t e = cudaFuncSetAttribute(fmrx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fmrx::SMEM_BYTES);
        if (e != cudaSuccess) { lrc_set_error("lrc_fmrx_create: %s", cudaGetErrorString(e)); lrc_fmrx_destroy(f); return LRC_ERR_CUDA; }
    } else {
        rc = lrc_fir_stream_create(f->fir, n_ch, max_chunk, 1, &f->fs);
        if (!rc) {
            f->bb_stride = bb_max;
            if (f->d_bb.alloc(n_ch * bb_max * 2) != cudaSuccess || f->d_fm.alloc(n_ch * bb_max) != cudaSuccess ||
                f->d_state.alloc(n_ch * 2) != cudaSuccess ||
                cudaMemset(f->d_state, 0, n_ch * sizeof(float2)) != cudaSuccess) {
                lrc_set_error("lrc_fmrx_create: %s", cudaGetErrorString(cudaGetLastError()));
                rc = LRC_ERR_CUDA;
            }
        }
        if (rc) { lrc_fmrx_destroy(f); return rc; }
    }
    *out = f;
    return LRC_OK;
}

extern "C" int lrc_fmrx_destroy(lrc_fmrx *f)
{
    if (!f) return LRC_OK;
    cudaSetDevice(f->ctx->device);
    lrc_fir_stream_destroy(f->fs); lrc_resampler_destroy(f->rs); lrc_fir_destroy(f->fir);
    delete f;
    return LRC_OK;
}

extern "C" int lrc_fmrx_is_fused(const lrc_fmrx *f) { return f && f->fused ? 1 : 0; }

// audio frames the next push of n samples per channel produces (every channel the same)
static long long fmrx_m_end(const lrc_fmrx *f, long long n_raw)
{
    const long long n_bb = n_raw >= f->ntaps ? (n_raw - f->ntaps) / f->decim + 1 : 0;    // lrc_fir_out_len
    if (n_bb < 1) return 0;
    return (n_bb * f->rs_L - 1) / f->rs_M + 1;                                           // all m with floor(m M / L) <= n_bb - 1
}

extern "C" size_t lrc_fmrx_next_out_len(const lrc_fmrx *f, size_t n)
{
    if (!f) return 0;
    // the same count in both forms: the stages emit what has become computable
    return (size_t)(fmrx_m_end(f, f->n_raw + (long long)n) - f->m_next);
}

extern "C" int lrc_fmrx_push(lrc_fmrx *f, const uint8_t *d_iq, size_t n, size_t chunk_stride, float *d_audio,
                             size_t out_stride, size_t *n_out, void *stream)
{
    LRC_REQUIRE(f && n_out, LRC_ERR_INVALID, "lrc_fmrx_push: null argument");
    LRC_BIND(f->ctx);
    *n_out = 0;
    if (n == 0) return LRC_OK;
    LRC_REQUIRE(n <= f->max_chunk, LRC_ERR_CAPACITY, "lrc_fmrx_push: chunk longer than max_chunk");
    LRC_REQUIRE(d_iq && chunk_stride >= n, LRC_ERR_INVALID, "lrc_fmrx_push: bad input");
    cudaStream_t s = lrc_stream(f->ctx, stream);
    if (!f->fused) {
        size_t n_bb = 0, n_a = 0;
        f->n_raw += (long long)n;
        int rc = lrc_fir_stream_push(f->fs, d_iq, n, chunk_stride, f->d_bb, f->bb_stride, &n_bb, s);
        if (rc || n_bb == 0) return rc;
        rc = lrc_fmdemod_run(f->ctx, f->d_bb, f->n_ch, n_bb, f->bb_stride, f->d_state, f->d_fm, f->bb_stride, s);
        if (rc) return rc;
        const size_t want = lrc_resampler_next_out_len(f->rs, n_bb);
        LRC_REQUIRE(want == 0 || (d_audio && out_stride >= want), LRC_ERR_CAPACITY, "lrc_fmrx_push: output too small");
        rc = lrc_resampler_process(f->rs, f->d_fm, n_bb, f->bb_stride, d_audio, out_stride, &n_a, s);
        f->m_next += (long long)n_a;
        *n_out = n_a;
        return rc;
    }
    using namespace fmrx;
    const long long n_raw1 = f->n_raw + (long long)n;
    const long long m_end = fmrx_m_end(f, n_raw1);
    const long long no = m_end - f->m_next;
    if (no > 0) {
        LRC_REQUIRE(d_audio && out_stride >= (size_t)no, LRC_ERR_CAPACITY, "lrc_fmrx_push: output too small");
        Args a;
        a.carry = f->d_carry[f->cur]; a.carry_stride = f->carry_stride;
        a.chunk = d_iq; a.chunk_stride = chunk_stride * 2;
        a.held = f->held; a.n = (long long)n; a.row_abs0 = f->n_raw - f->held;
        a.m0 = f->m_next; a.n_out = no; a.out = d_audio; a.out_stride = out_stride;
        a.n_ch = (long long)f->n_ch;
        a.tiles_per_pair = (no + TILE_A - 1) / TILE_A;
        const long long outs_last = no - (a.tiles_per_pair - 1) * TILE_A;         // outputs of a pair's last tile
        a.last_rounds = (int)((M * (outs_last - 1) + 1 + ROUND_Z - 1) / ROUND_Z);
        const long long pairs = ((long long)f->n_ch + 1) / 2, slots = (long long)f->ctx->n_sm * 3;    // 3 CTAs per SM
        a.total_tiles = pairs * a.tiles_per_pair;
        // TMA needs 16-byte aligned rows and piece boundaries: held and n multiples of 8 samples, aligned bases / strides
        a.use_tma = (f->held % 8 == 0) && (n % 8 == 0) && (((uintptr_t)d_iq & 15) == 0) && (a.chunk_stride % 16 == 0) &&
                    (a.row_abs0 % 8 == 0);
        long long blocks = slots < a.total_tiles ? slots : a.total_tiles;
        fmrx_kernel<<<(unsigned)blocks, NT, SMEM_BYTES, s>>>(a, f->taps127, f->rtaps);
        LRC_CUDA(cudaGetLastError());
    }
    // carry for the next call: everything from the start of the next segment's priming round, floored to 8 samples
    long long from_abs = (long long)DECIM * (M * m_end - ROUND_Z);
    if (from_abs < 0) from_abs = 0;
    from_abs &= ~7ll;
    const long long row_abs0 = f->n_raw - f->held;
    if (from_abs < row_abs0) from_abs = row_abs0;            // (never asks for more history than it kept)
    const long long keep = n_raw1 - from_abs;
    LRC_REQUIRE(keep <= (long long)FMRX_CARRY_CAP, LRC_ERR_CAPACITY, "lrc_fmrx_push: internal carry overflow");
    if (keep > 0) {
        const long long held_b = 2 * f->held, from_b = 2 * (from_abs - row_abs0), keep_b = 2 * keep;
        const bool vec = held_b % 16 == 0 && from_b % 16 == 0 && keep_b % 16 == 0 && ((uintptr_t)d_iq & 15) == 0 &&
                         (chunk_stride * 2) % 16 == 0;
        long long blocks = (f->n_ch * (keep_b / (vec ? 16 : 2)) + 255) / 256;
        if (blocks > 8192) blocks = 8192;
        if (blocks < 1) blocks = 1;
        if (vec)
            fmrx_carry_kernel<uint4><<<(unsigned)blocks, 256, 0, s>>>(f->d_carry[f->cur], f->carry_stride, held_b, d_iq, chunk_stride * 2,
                                                                     from_b, keep_b, f->d_carry[f->cur ^ 1], (long long)f->n_ch);
        else
            fmrx_carry_kernel<uint16_t><<<(unsigned)blocks, 256, 0, s>>>(f->d_carry[f->cur], f->carry_stride, held_b, d_iq,
                                                                        chunk_stride * 2, from_b, keep_b, f->d_carry[f->cur ^ 1],
                                                                        (long long)f->n_ch);
        LRC_CUDA(cudaGetLastError());
        f->cur ^= 1;
    }
    f->held = keep > 0 ? keep : 0;
    f->n_raw = n_raw1;
    f->m_next = m_end;
    *n_out = (size_t)(no > 0 ? no : 0);
    return LRC_OK;
}

extern "C" int lrc_fmrx_reset(lrc_fmrx *f)
{
    LRC_REQUIRE(f != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(f->ctx);
    f->held = f->n_raw = f->m_next = 0;
    if (!f->fused) {
        // rebuild the carried state of the three stages
        lrc_fir_stream_destroy(f->fs); f->fs = nullptr;
        int rc = lrc_fir_stream_create(f->fir, f->n_ch, f->max_chunk, 1, &f->fs);
        if (rc) return rc;
        LRC_CUDA(cudaMemset(f->d_state, 0, f->n_ch * sizeof(float2)));
        return lrc_resampler_reset(f->rs);
    }
    return LRC_OK;
}
