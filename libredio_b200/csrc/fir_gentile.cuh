// fir_gentile.cuh -- FIR + decimate (dsputils::convolve, dsputils.rs:30-32, + decimation) for the shapes that have no
// dedicated tile instance: ntaps <= 128 (run-time, zero-padded to 64 / 128), decim in {4, 5, 8, 10, 16}, cf32 input.
// Before round 2 every shape but 64 taps / 10 went to the one-thread-per-output kernel (fir_generic_kernel), which
// re-reads each sample ntaps / decim times from L1/L2: 6-11x slower than a tile kernel (profiles/r2_p_chain_generic.jsonl,
// the "unfused" column).  This is the register-blocked tile of the generic fused chain (chain_generic.cuh: GenTile --
// chunked TMA tile with 16 bytes of padding per thread-window advance where that keeps LDS.128 conflict-free, packed
// FFMA2 with the tap broadcast from a uniform register) as a stand-alone multi-channel kernel: many short CTAs,
// several per SM, one TMA tile each.
#pragma once
#include "chain_generic.cuh"

namespace firg {
using namespace chaing;

template <int NTAPS, int DECIM, int R, int NT>
struct Cfg {
    using Tile = GenTile<NTAPS, DECIM, R>;
    static constexpr int TILE_OUT = R * NT;
    static constexpr int TILE_IN_MAX = (TILE_OUT - 1) * DECIM + NTAPS;
    static constexpr int N_CHUNKS_MAX = (TILE_IN_MAX + Tile::STEP - 1) / Tile::STEP;
    static constexpr int WIN_END = (NT - 1) * Tile::PITCH + Tile::off(Tile::WINL - 1) + 16;
    static constexpr int CHUNK_END = N_CHUNKS_MAX * Tile::PITCH;
    static constexpr int TILE_BYTES = ((WIN_END > CHUNK_END ? WIN_END : CHUNK_END) + 127) / 128 * 128;
    static constexpr int SMEM_BYTES = TILE_BYTES + 16;
};

template <int NTAPS, int DECIM, int R, int NT>
__global__ void __launch_bounds__(NT)
fir_gentile_kernel(const float2 *__restrict__ in, size_t n_ch, size_t n_in, size_t in_stride, float2 *__restrict__ out,
                   size_t n_out, size_t out_stride, int use_tma, const __grid_constant__ FirTaps<NTAPS> taps)
{
    using C = Cfg<NTAPS, DECIM, R, NT>;
    using Tile = typename C::Tile;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + C::TILE_BYTES);
    const int t = threadIdx.x;
    if (t == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    // zero-padded taps and the ragged last tile of a channel must only ever meet finite values
    for (int i = t; i < C::TILE_BYTES / 16; i += NT) reinterpret_cast<float4 *>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_proxy_async();
    __syncthreads();
    uint32_t phase = 0;
    const size_t tiles_per_ch = (n_out + C::TILE_OUT - 1) / C::TILE_OUT;
    const size_t n_tiles = tiles_per_ch * n_ch;
    for (size_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const size_t c = tile / tiles_per_ch, o0 = (tile % tiles_per_ch) * C::TILE_OUT;
        const size_t s0 = o0 * DECIM;
        size_t avail = n_in - s0;                              // samples of the channel row from s0 (all readable)
        const int need = avail > (size_t)C::TILE_IN_MAX ? C::TILE_IN_MAX : (int)avail;
        const float2 *src = in + c * in_stride + s0;
        const int n_chunks = (need + Tile::STEP - 1) / Tile::STEP;
        if (use_tma) {
            const int tma_samples = need & ~1;                 // bulk copies move whole 16-byte units, an odd last sample goes by hand
            if (t == 0) mbar_expect_tx(bar, (uint32_t)tma_samples * 8u);
            for (int ch = t; ch < n_chunks; ch += NT) {
                const int c0 = ch * Tile::STEP;
                int ns = tma_samples - c0;
                if (ns > Tile::STEP) ns = Tile::STEP;
                if (ns > 0) tma_load_1d(smem + (size_t)ch * Tile::PITCH, src + c0, (uint32_t)ns * 8u, bar);
                if ((need & 1) && c0 + Tile::STEP >= need && c0 < need)
                    *reinterpret_cast<float2 *>(smem + (size_t)ch * Tile::PITCH + (size_t)(need - 1 - c0) * 8) = __ldg(src + need - 1);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {
            // unaligned rows: cooperative copy into the same padded layout
            for (int i = t; i < need; i += NT)
                *reinterpret_cast<float2 *>(smem + (size_t)(i / Tile::STEP) * Tile::PITCH + (size_t)(i % Tile::STEP) * 8) = __ldg(src + i);
        }
        // ragged last tile of a channel: what lies behind the channel's last sample is left over from an earlier tile; the
        // zero-padded taps reach up to NTAPS - 1 samples into it, so clear that much (a stale NaN times a zero tap is a NaN)
        if (need < C::TILE_IN_MAX)
            for (int i = need + t; i < need + NTAPS && i < C::TILE_IN_MAX; i += NT)
                *reinterpret_cast<float2 *>(smem + (size_t)(i / Tile::STEP) * Tile::PITCH + (size_t)(i % Tile::STEP) * 8) = make_float2(0.f, 0.f);
        __syncthreads();
        float2 acc[R];
        Tile::run(smem + (size_t)t * Tile::PITCH, taps, acc);
        float2 *dst = out + c * out_stride + o0 + (size_t)t * R;
        const size_t left = n_out - o0;
#pragma unroll
        for (int r = 0; r < R; ++r)
            if ((size_t)(t * R + r) < left) dst[r] = acc[r];
        __syncthreads();                                       // tile consumed before the next load
    }
}

template <int NTAPS, int DECIM>
static int launch(int n_sm, const float *h_taps, int ntaps, const float *d_in, size_t n_ch, size_t n_in, size_t in_stride,
                  float *d_out, size_t n_out, size_t out_stride, cudaStream_t s)
{
    constexpr int R = RFor<DECIM>::R, NT = 128;
    using C = Cfg<NTAPS, DECIM, R, NT>;
    auto kern = fir_gentile_kernel<NTAPS, DECIM, R, NT>;
    size_t ctas;
    LRC_CUDA(lrc_resident_ctas(kern, NT, C::SMEM_BYTES, n_sm, &ctas));
    const size_t n_tiles = ceil_div(n_out, (size_t)C::TILE_OUT) * n_ch;
    static const size_t gm = lrc_grid_mult("LRC_FIR_GRID", 1024);
    size_t blocks = ctas * gm;
    if (blocks > n_tiles) blocks = n_tiles;
    // TMA needs 16-byte aligned sources: base, and the channel stride when there is more than one channel row
    const int use_tma = (((uintptr_t)d_in & 15) == 0) && (n_ch == 1 || in_stride % 2 == 0);
    FirTaps<NTAPS> taps;
    for (int i = 0; i < NTAPS; ++i) taps.h[i] = i < ntaps ? h_taps[i] : 0.0f;
    kern<<<(unsigned)blocks, NT, C::SMEM_BYTES, s>>>((const float2 *)d_in, n_ch, n_in, in_stride, (float2 *)d_out, n_out,
                                                    out_stride, use_tma, taps);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}
}  // namespace firg

// one translation unit per (NTAPS, DECIM) instance (k_firg_n*_d*.cu): the fully unrolled 128-tap windows take a minute each to compile
#define LRC_FIRG_DECL(NT_, D_) \
    int lrc_firg_launch_n##NT_##_d##D_(int n_sm, const float *h_taps, int ntaps, const float *d_in, size_t n_ch, size_t n_in, \
                                       size_t in_stride, float *d_out, size_t n_out, size_t out_stride, cudaStream_t s)
#define LRC_FIRG_DEFINE(NT_, D_) \
    LRC_FIRG_DECL(NT_, D_) { return firg::launch<NT_, D_>(n_sm, h_taps, ntaps, d_in, n_ch, n_in, in_stride, d_out, n_out, out_stride, s); }
LRC_FIRG_DECL(64, 4); LRC_FIRG_DECL(64, 5); LRC_FIRG_DECL(64, 8); LRC_FIRG_DECL(64, 10); LRC_FIRG_DECL(64, 16);
LRC_FIRG_DECL(128, 4); LRC_FIRG_DECL(128, 5); LRC_FIRG_DECL(128, 8); LRC_FIRG_DECL(128, 10); LRC_FIRG_DECL(128, 16);
