// k_fm_resample.cu -- quadrature FM discriminator and rational polyphase resampler.
//
// FM discriminator: absent from the reference (north-star stage): d[n] = arg(x[n] conj(x[n-1])).
// Resampler: replaces samplerate::resample (src/samplerate/src/samplerate.rs:59-87), whose arithmetic
// lives in libsamplerate (un-vendored, un-pinned -> parity UNPINNED).  Our definition, mirrored in f64
// by oracle/defined_f64.py:
//     ratio = L/M;  prototype h: ntaps = 2*32*max(L,M)+1, sinc(2 fc (i-c)) * kaiser(beta=12),
//     fc = 0.45/max(L,M), sum(h) = L;
//     y[m] = sum_j h[(mM mod L) + jL] * x[floor(mM/L) - j],  x[<0] = 0   (streaming-causal).
//
// Measured and rejected for the packed decimator at M = 5 (the BASELINE 240 kHz -> 48 kHz shape, 1024 channels x 240 k
// samples, profiles/r1_s8_rs_configs.txt, Gsamples/s): 128 threads (380), and a second cp.async stage that fills the next
// tile pair while this one is filtered, at 64 threads (359) and at 128 (351), against 64 threads and one stage (387).
// The second stage halves the resident CTAs and loses more than the hidden fill gains.
#include "fm_core.cuh"
#include <cmath>
#include <cstdlib>
#include <vector>

// ---------------------------------------------------------------------------------------------
// FM discriminator
// ---------------------------------------------------------------------------------------------
// blockIdx.y = channel; each thread turns two consecutive samples (one 128-bit load) into two phases
__global__ void __launch_bounds__(256)
fmdemod_kernel(const float2 *__restrict__ in, size_t n, size_t in_stride, const float2 *__restrict__ state,
               float *__restrict__ out, size_t out_stride, int vec_ok)
{
    const size_t c = blockIdx.y;
    const float2 *x = in + c * in_stride;
    float *y = out + c * out_stride;
    const float2 first_prev = state ? state[c] : make_float2(0.f, 0.f);
    // main loop: a thread owns 4 consecutive samples (two 128-bit loads, one 128-bit store); the sample before
    // its first comes from the left neighbour's registers by shuffle, only lane 0 re-reads it (an L1/L2 hit).
    // Two quads per thread are in flight per iteration so that enough bytes are outstanding per SM.
    const size_t n_quads = vec_ok ? n / 4 : 0;
    const size_t n_pairs = n_quads * 2;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const unsigned lane = threadIdx.x & 31;
    const float4 *x4 = reinterpret_cast<const float4 *>(x);
    for (size_t q0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;; q0 += 2 * stride) {
        // whole warps stay in the loop together (shuffles); out-of-range quads are masked
        const size_t qa = q0, qb = q0 + stride;
        const bool oka = qa < n_quads, okb = qb < n_quads;
        if (__all_sync(0xffffffffu, !oka && !okb)) break;
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, b0 = a0, b1 = a0;
        if (oka) { a0 = ldg_stream_f4(x4 + 2 * qa); a1 = ldg_stream_f4(x4 + 2 * qa + 1); }
        if (okb) { b0 = ldg_stream_f4(x4 + 2 * qb); b1 = ldg_stream_f4(x4 + 2 * qb + 1); }
        float2 pa = make_float2(__shfl_up_sync(0xffffffffu, a1.z, 1), __shfl_up_sync(0xffffffffu, a1.w, 1));
        float2 pb = make_float2(__shfl_up_sync(0xffffffffu, b1.z, 1), __shfl_up_sync(0xffffffffu, b1.w, 1));
        if (lane == 0) {
            if (oka) pa = qa ? x[4 * qa - 1] : first_prev;
            if (okb) pb = qb ? x[4 * qb - 1] : first_prev;
        }
        if (oka) {
            const float2 s0 = make_float2(a0.x, a0.y), s1 = make_float2(a0.z, a0.w), s2 = make_float2(a1.x, a1.y), s3 = make_float2(a1.z, a1.w);
            const float2 z0 = fm_mul_conj(s0, pa), z1 = fm_mul_conj(s1, s0), z2 = fm_mul_conj(s2, s1), z3 = fm_mul_conj(s3, s2);
            stg_stream_f4(reinterpret_cast<float4 *>(y) + qa, make_float4(lr_atan2(z0.y, z0.x), lr_atan2(z1.y, z1.x),
                                                                          lr_atan2(z2.y, z2.x), lr_atan2(z3.y, z3.x)));
        }
        if (okb) {
            const float2 s0 = make_float2(b0.x, b0.y), s1 = make_float2(b0.z, b0.w), s2 = make_float2(b1.x, b1.y), s3 = make_float2(b1.z, b1.w);
            const float2 z0 = fm_mul_conj(s0, pb), z1 = fm_mul_conj(s1, s0), z2 = fm_mul_conj(s2, s1), z3 = fm_mul_conj(s3, s2);
            stg_stream_f4(reinterpret_cast<float4 *>(y) + qb, make_float4(lr_atan2(z0.y, z0.x), lr_atan2(z1.y, z1.x),
                                                                          lr_atan2(z2.y, z2.x), lr_atan2(z3.y, z3.x)));
        }
    }
    // odd tail, or the whole row when it is not 16-byte aligned
    for (size_t k = 2 * n_pairs + (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) {
        const float2 prev = k ? x[k - 1] : first_prev;
        const float2 z = fm_mul_conj(x[k], prev);
        y[k] = lr_atan2(z.y, z.x);
    }
}

__global__ void fmdemod_state_kernel(const float2 *__restrict__ in, size_t n_ch, size_t n, size_t in_stride,
                                     float2 *__restrict__ state)
{
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_ch) state[c] = in[c * in_stride + n - 1];
}

extern "C" int lrc_fmdemod_run(lrc_ctx *ctx, const float *d_in, size_t n_ch, size_t n, size_t in_stride,
                               float *d_state, float *d_out, size_t out_stride, void *stream)
{
    LRC_BIND(ctx);
    if (n_ch == 0 || n == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_out, LRC_ERR_INVALID, "lrc_fmdemod_run: null buffer");
    LRC_REQUIRE(in_stride >= n && out_stride >= n, LRC_ERR_INVALID, "lrc_fmdemod_run: stride shorter than length");
    LRC_REQUIRE(((uintptr_t)d_in & 7) == 0, LRC_ERR_INVALID, "lrc_fmdemod_run: input must be 8-byte aligned");
    cudaStream_t s = lrc_stream(ctx, stream);
    LRC_REQUIRE(n_ch <= 65535, LRC_ERR_UNSUPPORTED, "lrc_fmdemod_run: more than 65535 channels per call");
    size_t bx = ceil_div(ceil_div(n, 8), 256);
    // many short CTAs: 0.89 -> 0.97 of the copy bandwidth against 16 CTAs per SM looping (profiles/r1_s8_grid_sweeps.txt)
    static const size_t capf = lrc_grid_mult("LRC_FM_CAP", 128);
    const size_t cap = ceil_div((size_t)ctx->n_sm * capf, n_ch);
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    // 128-bit loads and stores need every row start aligned
    const int vec_ok = (((uintptr_t)d_in & 15) == 0) && (in_stride % 2 == 0) && (((uintptr_t)d_out & 15) == 0) && (out_stride % 4 == 0);
    fmdemod_kernel<<<dim3((unsigned)bx, (unsigned)n_ch), 256, 0, s>>>((const float2 *)d_in, n, in_stride,
                                                                    (const float2 *)d_state, d_out, out_stride, vec_ok);
    LRC_CUDA(cudaGetLastError());
    if (d_state) {
        fmdemod_state_kernel<<<(unsigned)ceil_div(n_ch, 256), 256, 0, s>>>((const float2 *)d_in, n_ch, n, in_stride,
                                                                         (float2 *)d_state);
        LRC_CUDA(cudaGetLastError());
    }
    return LRC_OK;
}

// ---------------------------------------------------------------------------------------------
// resampler
// ---------------------------------------------------------------------------------------------
static const int    RS_ZERO_CROSSINGS = 32;
static const double RS_KAISER_BETA = 12.0;
static const double RS_BANDWIDTH = 0.9;
static const int    RS_MAX_DEN = 4096;

struct lrc_resampler {
    lrc_ctx *ctx;
    int      L, M;
    size_t   n_ch, max_chunk, tpp, ntaps, cap;   // cap: floats per staging row
    std::vector<double> h;                       // prototype (f64)
    DevBuf<float> d_hp;                          // [L][tpp] polyphase rows, f32
    DevBuf<float> d_carry[2];                    // [n_ch][tpp] x2: the tpp-1 samples before the next chunk (ping-pong)
    int      cur;                                // which carry buffer is current
    DevBuf<float> d_hin, d_hout;                 // staging for the host entry point
    unsigned long long n_total, m_next;          // inputs consumed / next output index (same for all channels)
};

static double bessel_i0(double x)
{
    double s = 1.0, t = 1.0;
    const double q = x * x / 4.0;
    for (int k = 1; k < 500; ++k) {
        t *= q / ((double)k * (double)k);
        s += t;
        if (t < 1e-18 * s) break;
    }
    return s;
}

// best rational approximation with bounded denominator (continued fractions, as Fraction.limit_denominator)
static bool rational(double x, int max_den, int *num, int *den)
{
    if (!(x > 0) || !std::isfinite(x)) return false;
    long long p0 = 0, q0 = 1, p1 = 1, q1 = 0;
    double r = x;
    for (int it = 0; it < 64; ++it) {
        const double fl = floor(r);
        if (fl > 1e15) break;
        const long long a = (long long)fl;
        const long long p2 = a * p1 + p0, q2 = a * q1 + q0;
        if (q2 > max_den || p2 > max_den) break;
        p0 = p1; q0 = q1; p1 = p2; q1 = q2;
        const double frac = r - fl;
        if (frac < 1e-15) break;
        r = 1.0 / frac;
    }
    if (q1 <= 0 || p1 <= 0) return false;
    if (fabs((double)p1 / (double)q1 - x) > 1e-12 * x) return false;
    *num = (int)p1; *den = (int)q1;
    return true;
}

// The stream a kernel sees is the virtual row [carry (tpp-1 samples of history) | chunk]: no staging copy of
// the chunk is ever made, the first window of a channel simply starts inside the carry buffer.
struct RsRow {
    const float *carry; size_t hist;          // carry + c*tpp, tpp - 1
    const float *in; size_t n_in;             // in + c*in_stride
    __device__ __forceinline__ float at(size_t v) const
    {
        return v < hist ? carry[v] : (v - hist < n_in ? __ldg(in + (v - hist)) : 0.f);
    }
};

template <int UNROLL>
__global__ void __launch_bounds__(256)
resample_kernel(const float *__restrict__ carry, const float *__restrict__ in, size_t n_in, size_t in_stride,
                size_t n_ch, const float *__restrict__ hp, int L, int M,
                int tpp, unsigned long long n_total, unsigned long long m_next, size_t n_out,
                float *__restrict__ out, size_t out_stride)
{
    const size_t total = n_ch * n_out;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / n_out, k = i % n_out;
        const unsigned long long t = (m_next + k) * (unsigned long long)M;
        const unsigned long long base = t / (unsigned long long)L;
        const int phase = (int)(t % (unsigned long long)L);
        // virtual index of x[base]: the row starts at global input index n_total - (tpp - 1)
        const RsRow row{carry + c * (size_t)tpp, (size_t)(tpp - 1), in + c * in_stride, n_in};
        const size_t v0 = (size_t)(base - n_total) + (size_t)(tpp - 1);
        const float *h = hp + (size_t)phase * tpp;
        float acc[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) acc[u] = 0.f;
        int j = 0;
        if (v0 >= (size_t)(tpp - 1) + row.hist) {
            // whole window inside the chunk (every output but the first few of a call): plain pointer walk
            const float *x = row.in + (v0 - row.hist);
            for (; j + UNROLL <= tpp; j += UNROLL) {
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) acc[u] = fmaf(__ldg(h + j + u), x[-(j + u)], acc[u]);
            }
            for (; j < tpp; ++j) acc[0] = fmaf(__ldg(h + j), x[-j], acc[0]);
        } else {
            for (; j + UNROLL <= tpp; j += UNROLL) {
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) acc[u] = fmaf(__ldg(h + j + u), row.at(v0 - (size_t)(j + u)), acc[u]);
            }
            for (; j < tpp; ++j) acc[0] = fmaf(__ldg(h + j), row.at(v0 - (size_t)j), acc[0]);
        }
        float s = 0.f;
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) s += acc[u];
        out[c * out_stride + k] = s;
    }
}

// next history = the last tpp-1 samples of [carry | chunk], written to the other carry buffer
__global__ void rs_carry_kernel(const float *__restrict__ carry, float *__restrict__ next, const float *__restrict__ in,
                                size_t n_in, size_t in_stride, size_t n_ch, int tpp)
{
    const size_t hist = (size_t)(tpp - 1);
    const size_t total = n_ch * hist;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / hist, k = i % hist;
        const RsRow row{carry + c * (size_t)tpp, hist, in + c * in_stride, n_in};
        next[c * (size_t)tpp + k] = row.at(n_in + k);
    }
}

// ---------------------------------------------------------------------------------------------
// L == 1 (pure decimation by M, e.g. 240 kHz -> 48 kHz): y[m] = sum_i g[i] x[m M + i], g = reversed h.
// Same register-blocked shared-memory scheme as the FIR tile (fir_core.cuh) on real samples: a thread owns
// R consecutive outputs, streams its window once through LDS.128 (4 samples each) and feeds every sample to
// the accumulators it belongs to; taps are kernel parameters (constant bank).  R*M*4 bytes is an odd
// multiple of 16 bytes, so the eight threads of an LDS.128 phase hit eight distinct bank groups.
// ---------------------------------------------------------------------------------------------

template <int M, int R, int NT>
struct RsDecCfg {
    static constexpr int TPP = 2 * RS_ZERO_CROSSINGS * M + 1;             // taps (L = 1)
    static constexpr int WIN = (R - 1) * M + TPP;
    static constexpr int WIN4 = (WIN + 3) / 4 * 4;                         // whole LDS.128s
    static constexpr int STEP = R * M;                                     // samples between thread windows
    static constexpr int TILE_OUT = R * NT;
    static constexpr int TILE_IN = (NT - 1) * STEP + WIN4;                 // floats a tile reads
    static constexpr int SMEM_BYTES = TILE_IN * 4;
    static_assert((STEP * 4) % 16 == 0, "thread windows must start 16-byte aligned");
};

template <int M, int R, int NT>
__global__ void __launch_bounds__(NT)
resample_dec_kernel(const float *__restrict__ carry, const float *__restrict__ in, size_t n_in, size_t in_stride,
                    size_t n_ch, size_t s0, size_t n_out,
                    float *__restrict__ out, size_t out_stride, const __grid_constant__ RsTaps<2 * RS_ZERO_CROSSINGS * M + 1> taps)
{
    using Cfg = RsDecCfg<M, R, NT>;
    extern __shared__ __align__(16) float rs_tile[];
    const int t = threadIdx.x;
    const size_t tiles_per_ch = (n_out + Cfg::TILE_OUT - 1) / Cfg::TILE_OUT;
    const size_t n_tiles = tiles_per_ch * n_ch;
    for (size_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const size_t c = tile / tiles_per_ch, o0 = (tile % tiles_per_ch) * Cfg::TILE_OUT;
        const size_t first = s0 + o0 * M;                                   // window of output o0 starts here (virtual row)
        const RsRow row{carry + c * (size_t)Cfg::TPP, (size_t)(Cfg::TPP - 1), in + c * in_stride, n_in};
        if (first >= row.hist) {                                            // every tile but a channel's first
            const float *src = row.in + (first - row.hist);
            const size_t avail = n_in - (first - row.hist);
            for (int i = t; i < Cfg::TILE_IN; i += NT) rs_tile[i] = (size_t)i < avail ? __ldg(src + i) : 0.f;
        } else {
            for (int i = t; i < Cfg::TILE_IN; i += NT) rs_tile[i] = row.at(first + (size_t)i);
        }
        __syncthreads();
        float acc[R];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = 0.f;
        const float *sx = rs_tile + t * Cfg::STEP;
#pragma unroll
        for (int j = 0; j < Cfg::WIN4; j += 4) {
            const float4 x = *reinterpret_cast<const float4 *>(sx + j);
            const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int k = j + u - r * M;
                    if (k >= 0 && k < Cfg::TPP) acc[r] = fmaf(xs[u], taps.g[k], acc[r]);
                }
        }
        float *dst = out + c * out_stride + o0 + (size_t)t * R;
        const size_t left = n_out - o0;
#pragma unroll
        for (int r = 0; r < R; ++r)
            if ((size_t)(t * R + r) < left) dst[r] = acc[r];
        __syncthreads();
    }
}

template <int M, int R>
static int launch_resample_dec(lrc_resampler *r, const float *d_in, size_t n_in, size_t in_stride, size_t no, float *d_out,
                               size_t out_stride, cudaStream_t s)
{
    constexpr int NT = 128;
    using Cfg = RsDecCfg<M, R, NT>;
    auto kern = resample_dec_kernel<M, R, NT>;
    size_t blocks;
    LRC_CUDA(lrc_resident_ctas(kern, NT, Cfg::SMEM_BYTES, r->ctx->n_sm, &blocks));
    const size_t n_tiles = ceil_div(no, (size_t)Cfg::TILE_OUT) * r->n_ch;
    if (blocks > n_tiles) blocks = n_tiles;
    RsTaps<Cfg::TPP> taps;
    for (int i = 0; i < Cfg::TPP; ++i) taps.g[i] = (float)r->h[Cfg::TPP - 1 - i];      // reversed: correlation form
    // buffer index of x[m_next*M - (TPP-1)]: the row starts at global input index n_total - (TPP-1)
    const size_t s0 = (size_t)(r->m_next * (unsigned long long)M - r->n_total);
    kern<<<(unsigned)blocks, NT, Cfg::SMEM_BYTES, s>>>(r->d_carry[r->cur], d_in, n_in, in_stride, r->n_ch, s0, no, d_out, out_stride, taps);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

// ---------------------------------------------------------------------------------------------
// Packed variant of the decimator: the scalar kernel above is FP32-ISSUE bound (82 % issue-active, 73 % of the
// instructions FFMA), not pipe bound.  Here a CTA works on TWO tiles at once (neighbouring work items: two tiles of a
// channel, or the last tile of one channel and the first of the next), stored INTERLEAVED in shared memory as
// {A[i], B[i]} pairs, so one LDS.128 yields two consecutive samples of both tiles and one FFMA2 (tap broadcast to
// both lanes) advances an accumulator of tile A and the matching one of tile B: half the issue slots per FMA.
// Every output is still the same ascending-tap fmaf chain, so results are bit-identical to the scalar kernel.
// R is chosen so that the per-thread stride R*M*8 bytes is an odd multiple of 16 bytes (conflict-free LDS.128).
// ---------------------------------------------------------------------------------------------
template <int M, int R, int NT>
struct RsDec2Cfg {
    static constexpr int TPP = 2 * RS_ZERO_CROSSINGS * M + 1;
    static constexpr int WIN = (R - 1) * M + TPP;
    static constexpr int WIN2 = (WIN + 1) / 2 * 2;                         // whole LDS.128s (2 samples of 2 tiles)
    static constexpr int STEP = R * M;
    static constexpr int TILE_OUT = R * NT;
    static constexpr int TILE_IN = (NT - 1) * STEP + WIN2;                 // float2 pairs a tile pair reads
    static constexpr int SMEM_BYTES = TILE_IN * 8;
    static_assert((STEP * 8) % 16 == 0, "thread windows must start 16-byte aligned");
    static_assert(((STEP * 8) / 16) % 2 == 1, "thread stride must be an odd number of 16-byte bank groups");
};

// one tile of one channel as a source of samples: i -> x[first + i] of the virtual row [carry | chunk].  addr() is
// branch-free: it yields the address of sample i (inside the carry buffer or inside the chunk) and the number of
// bytes an asynchronous copy may read there (4, or 0 = zero-fill: past the end of the row, or no such tile).
struct RsTileSrc {
    RsRow row; size_t first; bool active;
    __device__ __forceinline__ const float *addr(int i, uint32_t *nbytes) const
    {
        const size_t v = first + (size_t)i;
        const bool in_carry = v < row.hist;
        const size_t k = v - row.hist;                       // index into the chunk when !in_carry
        const bool ok = active && (in_carry || k < row.n_in);
        *nbytes = ok ? 4u : 0u;
        return ok ? (in_carry ? row.carry + v : row.in + k) : row.in;
    }
};

template <int M, int R, int NT>
__global__ void __launch_bounds__(NT)
resample_dec2_kernel(const float *__restrict__ carry, const float *__restrict__ in, size_t n_in, size_t in_stride,
                     size_t n_ch, size_t s0, size_t n_out,
                     float *__restrict__ out, size_t out_stride, const __grid_constant__ RsTaps<2 * RS_ZERO_CROSSINGS * M + 1> taps)
{
    using Cfg = RsDec2Cfg<M, R, NT>;
    extern __shared__ __align__(16) float2 rs_tile2[];           // TILE_IN pairs
    const int t = threadIdx.x;
    const size_t tiles_per_ch = (n_out + Cfg::TILE_OUT - 1) / Cfg::TILE_OUT;
    const size_t n_tiles = tiles_per_ch * n_ch;
    const size_t n_pairs = (n_tiles + 1) / 2;
    auto tile_src = [&](size_t w, size_t *c, size_t *o0) {
        RsTileSrc s;
        s.active = w < n_tiles;
        *c = s.active ? w / tiles_per_ch : 0;
        *o0 = s.active ? (w % tiles_per_ch) * Cfg::TILE_OUT : 0;
        s.first = s0 + *o0 * M;
        s.row = RsRow{carry + *c * (size_t)Cfg::TPP, (size_t)(Cfg::TPP - 1), in + *c * in_stride, n_in};
        return s;
    };
    // Fill the tile with the tile pair `pair`: asynchronous 4-byte copies (LDGSTS) straight into the interleaved
    // tile, zero-filled past the end of a row, one commit group per fill.  All loads of a thread are in flight at
    // once and nothing is staged in registers (a register-staged fill exposed one HBM round trip per 16 loads and
    // took 27-60 % of the kernel).  Three paths, cheapest first: both windows inside their rows (no predicates),
    // both windows past the carry (one compare each), anything else (a channel's first tile starts in the carry).
    auto fill = [&](size_t pair, float2 *buf) {
        size_t c_, o_;
        const RsTileSrc A = tile_src(2 * pair, &c_, &o_), B = tile_src(2 * pair + 1, &c_, &o_);
        const size_t h = A.row.hist;
        if (A.first >= h && B.active && B.first >= h) {
            const float *pa = A.row.in + (A.first - h), *pb = B.row.in + (B.first - h);
            const size_t na = n_in - (A.first - h), nb = n_in - (B.first - h);
            if (na >= (size_t)Cfg::TILE_IN && nb >= (size_t)Cfg::TILE_IN) {
#pragma unroll 4
                for (int i = t; i < Cfg::TILE_IN; i += NT) {
                    cp_async4(&buf[i].x, pa + i, 4u);
                    cp_async4(&buf[i].y, pb + i, 4u);
                }
            } else {
                for (int i = t; i < Cfg::TILE_IN; i += NT) {
                    const size_t k = (size_t)i;
                    cp_async4(&buf[i].x, pa + (k < na ? k : 0), k < na ? 4u : 0u);
                    cp_async4(&buf[i].y, pb + (k < nb ? k : 0), k < nb ? 4u : 0u);
                }
            }
        } else {
            for (int i = t; i < Cfg::TILE_IN; i += NT) {
                uint32_t ba, bb;
                const float *pa = A.addr(i, &ba), *pb = B.addr(i, &bb);
                cp_async4(&buf[i].x, pa, ba);
                cp_async4(&buf[i].y, pb, bb);
            }
        }
        cp_async_commit();
    };

    for (size_t pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
        fill(pair, rs_tile2);
        cp_async_wait_group<0>();
        __syncthreads();
        float2 acc[R];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = make_float2(0.f, 0.f);
        const float2 *sx = rs_tile2 + t * Cfg::STEP;
        RsDec2Steps<M, R, Cfg::TPP, 0, Cfg::WIN2>::run(sx, taps, acc);
        size_t cA, oA, cB, oB;
        tile_src(2 * pair, &cA, &oA);
        const bool activeB = tile_src(2 * pair + 1, &cB, &oB).active;
        float *dA = out + cA * out_stride + oA + (size_t)t * R;
        const size_t leftA = n_out - oA;
#pragma unroll
        for (int r = 0; r < R; ++r)
            if ((size_t)(t * R + r) < leftA) dA[r] = acc[r].x;
        if (activeB) {
            float *dB = out + cB * out_stride + oB + (size_t)t * R;
            const size_t leftB = n_out - oB;
#pragma unroll
            for (int r = 0; r < R; ++r)
                if ((size_t)(t * R + r) < leftB) dB[r] = acc[r].y;
        }
        __syncthreads();                                       // tile consumed before it is refilled
    }
}

template <int M, int R, int NT>
static int launch_resample_dec2(lrc_resampler *r, const float *d_in, size_t n_in, size_t in_stride, size_t no, float *d_out,
                                size_t out_stride, cudaStream_t s)
{
    using Cfg = RsDec2Cfg<M, R, NT>;
    constexpr int SMEM = Cfg::SMEM_BYTES;
    auto kern = resample_dec2_kernel<M, R, NT>;
    size_t ctas;
    LRC_CUDA(lrc_resident_ctas(kern, NT, SMEM, r->ctx->n_sm, &ctas));
    const size_t n_pairs = (ceil_div(no, (size_t)Cfg::TILE_OUT) * r->n_ch + 1) / 2;
    static const size_t gm = lrc_grid_mult("LRC_RS_GRID", 1024);
    size_t blocks = ctas * gm;
    if (blocks > n_pairs) blocks = n_pairs;
    RsTaps<Cfg::TPP> taps;
    for (int i = 0; i < Cfg::TPP; ++i) taps.g[i] = (float)r->h[Cfg::TPP - 1 - i];      // reversed: correlation form
    const size_t s0 = (size_t)(r->m_next * (unsigned long long)M - r->n_total);
    kern<<<(unsigned)blocks, NT, SMEM, s>>>(r->d_carry[r->cur], d_in, n_in, in_stride, r->n_ch, s0, no, d_out, out_stride, taps);
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

extern "C" int lrc_resampler_create(lrc_ctx *ctx, double ratio, size_t n_ch, size_t max_chunk, lrc_resampler **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && n_ch >= 1 && max_chunk >= 1, LRC_ERR_INVALID, "lrc_resampler_create: bad arguments");
    int L = 0, M = 0;
    if (!rational(ratio, RS_MAX_DEN, &L, &M)) {
        lrc_set_error("lrc_resampler_create: ratio %.17g is not L/M with L, M <= %d (libsamplerate accepts any "
                      "ratio in [1/256, 256])", ratio, RS_MAX_DEN);
        return LRC_ERR_UNSUPPORTED;
    }
    lrc_resampler *r = new (std::nothrow) lrc_resampler();
    LRC_REQUIRE(r != nullptr, LRC_ERR_NOMEM, "out of host memory");
    r->ctx = ctx; r->L = L; r->M = M; r->n_ch = n_ch; r->max_chunk = max_chunk;
    const int q = L > M ? L : M;
    r->ntaps = (size_t)2 * RS_ZERO_CROSSINGS * q + 1;
    r->tpp = (r->ntaps + L - 1) / L;
    r->h.resize(r->ntaps);
    const double pi = 3.14159265358979323846264338327950288;
    const double c = (double)(r->ntaps - 1) / 2.0, fc = 0.5 * RS_BANDWIDTH / q, i0b = bessel_i0(RS_KAISER_BETA);
    double sum = 0.0;
    for (size_t i = 0; i < r->ntaps; ++i) {
        const double u = 2.0 * fc * ((double)i - c);
        const double snc = (u == 0.0) ? 1.0 : sin(pi * u) / (pi * u);
        const double a = 2.0 * (double)i / (double)(r->ntaps - 1) - 1.0;
        const double arg = 1.0 - a * a;
        const double kw = bessel_i0(RS_KAISER_BETA * sqrt(arg > 0 ? arg : 0.0)) / i0b;
        r->h[i] = snc * kw;
        sum += r->h[i];
    }
    for (size_t i = 0; i < r->ntaps; ++i) r->h[i] *= (double)L / sum;
    std::vector<float> hp((size_t)L * r->tpp, 0.f);
    for (int p = 0; p < L; ++p)
        for (size_t j = 0; j < r->tpp; ++j) {
            const size_t idx = (size_t)p + j * (size_t)L;
            if (idx < r->ntaps) hp[(size_t)p * r->tpp + j] = (float)r->h[idx];
        }
    r->cap = (r->tpp + max_chunk + 3) / 4 * 4;
    if (r->d_hp.alloc(hp.size()) != cudaSuccess || r->d_carry[0].alloc(n_ch * r->tpp) != cudaSuccess ||
        r->d_carry[1].alloc(n_ch * r->tpp) != cudaSuccess ||
        cudaMemcpy(r->d_hp, hp.data(), hp.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
        lrc_set_error("lrc_resampler_create: %s", cudaGetErrorString(cudaGetLastError()));
        lrc_resampler_destroy(r);
        return LRC_ERR_CUDA;
    }
    const int rc = lrc_resampler_reset(r);
    if (rc) { lrc_resampler_destroy(r); return rc; }
    *out = r;
    return LRC_OK;
}

extern "C" int lrc_resampler_destroy(lrc_resampler *r)
{
    if (!r) return LRC_OK;
    cudaSetDevice(r->ctx->device);
    delete r;
    return LRC_OK;
}

extern "C" int lrc_resampler_reset(lrc_resampler *r)
{
    LRC_REQUIRE(r != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(r->ctx);
    r->n_total = 0; r->m_next = 0;
    r->cur = 0;
    LRC_CUDA(cudaMemsetAsync(r->d_carry[0], 0, r->n_ch * r->tpp * sizeof(float), r->ctx->stream));   // x[<0] = 0
    LRC_CUDA(cudaStreamSynchronize(r->ctx->stream));
    return LRC_OK;
}

extern "C" int lrc_resampler_get_taps(const lrc_resampler *r, double *h_taps, size_t cap, size_t *ntaps, int *L, int *M)
{
    LRC_REQUIRE(r != nullptr, LRC_ERR_INVALID, "null plan");
    if (ntaps) *ntaps = r->ntaps;
    if (L) *L = r->L;
    if (M) *M = r->M;
    if (h_taps) {
        LRC_REQUIRE(cap >= r->ntaps, LRC_ERR_CAPACITY, "lrc_resampler_get_taps: buffer too small");
        memcpy(h_taps, r->h.data(), r->ntaps * sizeof(double));
    }
    return LRC_OK;
}

extern "C" size_t lrc_resampler_next_out_len(const lrc_resampler *r, size_t n_in)
{
    if (!r || n_in == 0) return 0;
    // all m with floor(mM/L) <= N-1  <=>  m <= (N L - 1)/M
    const unsigned long long N = r->n_total + n_in;
    const unsigned long long m_end = (N * (unsigned long long)r->L - 1) / (unsigned long long)r->M + 1;
    return (size_t)(m_end - r->m_next);
}

extern "C" int lrc_resampler_process(lrc_resampler *r, const float *d_in, size_t n_in, size_t in_stride,
                                     float *d_out, size_t out_stride, size_t *n_out, void *stream)
{
    LRC_REQUIRE(r && n_out, LRC_ERR_INVALID, "lrc_resampler_process: null argument");
    LRC_BIND(r->ctx);
    *n_out = 0;
    if (n_in == 0) return LRC_OK;
    LRC_REQUIRE(n_in <= r->max_chunk, LRC_ERR_CAPACITY, "lrc_resampler_process: chunk longer than max_chunk");
    LRC_REQUIRE(d_in && in_stride >= n_in, LRC_ERR_INVALID, "lrc_resampler_process: bad input");
    cudaStream_t s = lrc_stream(r->ctx, stream);
    const size_t hist = r->tpp - 1;
    const size_t no = lrc_resampler_next_out_len(r, n_in);
    if (no) {
        LRC_REQUIRE(d_out && out_stride >= no, LRC_ERR_CAPACITY, "lrc_resampler_process: output too small "
                    "(the reference sizes it ratio*len + 1, samplerate.rs:64)");
        int rc = -1;
        // LRC_RS_VARIANT=0 keeps the scalar one-tile kernel (tuning / A-B measurements); default: packed two-tile
        static const int variant = getenv("LRC_RS_VARIANT") ? atoi(getenv("LRC_RS_VARIANT")) : 1;
        if (r->L == 1 && variant == 1) {       // packed (FFMA2) two-tile decimators
            switch (r->M) {
                case 2: rc = launch_resample_dec2<2, 7, 128>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                case 3: rc = launch_resample_dec2<3, 6, 128>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                // 64 threads at M = 5, the BASELINE shape: 387 Gsamples/s against 380 at 128 and 333 for the scalar
                // one-tile kernel (profiles/r1_s8_rs_configs.txt)
                case 5: rc = launch_resample_dec2<5, 6, 64>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                case 6: rc = launch_resample_dec2<6, 5, 128>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                default: break;                // M = 4: no conflict-free R, the scalar tile kernel below
            }
        }
        if (rc < 0 && r->L == 1) {             // decimators with a register-blocked tile instance
            switch (r->M) {
                case 2: rc = launch_resample_dec<2, 6>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                case 3: rc = launch_resample_dec<3, 4>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                case 4: rc = launch_resample_dec<4, 5>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                case 5: rc = launch_resample_dec<5, 4>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                case 6: rc = launch_resample_dec<6, 6>(r, d_in, n_in, in_stride, no, d_out, out_stride, s); break;
                default: break;
            }
        }
        if (rc > 0) return rc;
        if (rc < 0) {                          // general L/M: one thread per output
            size_t blocks = ceil_div(r->n_ch * no, 256);
            const size_t cap = (size_t)r->ctx->n_sm * 16;
            if (blocks > cap) blocks = cap;
            resample_kernel<4><<<(unsigned)blocks, 256, 0, s>>>(r->d_carry[r->cur], d_in, n_in, in_stride, r->n_ch, r->d_hp, r->L,
                                                               r->M, (int)r->tpp, r->n_total, r->m_next, no, d_out, out_stride);
            LRC_CUDA(cudaGetLastError());
        }
    }
    // new history = the last tpp-1 samples of [history | chunk], into the other carry buffer
    if (hist) {
        size_t blocks = ceil_div(r->n_ch * hist, 256);
        if (blocks > 4096) blocks = 4096;
        rs_carry_kernel<<<(unsigned)blocks, 256, 0, s>>>(r->d_carry[r->cur], r->d_carry[r->cur ^ 1], d_in, n_in, in_stride, r->n_ch,
                                                        (int)r->tpp);
        LRC_CUDA(cudaGetLastError());
        r->cur ^= 1;
    }
    r->n_total += n_in;
    r->m_next += no;
    *n_out = no;
    return LRC_OK;
}

extern "C" int lrc_resampler_process_host(lrc_resampler *r, const float *h_in, size_t n_in, float *h_out,
                                          size_t out_cap, size_t *n_out)
{
    LRC_REQUIRE(r && n_out, LRC_ERR_INVALID, "lrc_resampler_process_host: null argument");
    LRC_BIND(r->ctx);
    *n_out = 0;
    if (n_in == 0) return LRC_OK;
    LRC_REQUIRE(h_in != nullptr, LRC_ERR_INVALID, "lrc_resampler_process_host: null input");
    const size_t no = lrc_resampler_next_out_len(r, n_in);
    LRC_REQUIRE(no == 0 || (h_out && out_cap >= no), LRC_ERR_CAPACITY, "lrc_resampler_process_host: output too small");
    LRC_CUDA(r->d_hin.ensure(r->n_ch * n_in));
    LRC_CUDA(r->d_hout.ensure(r->n_ch * (no + 1)));
    cudaStream_t s = r->ctx->stream;
    LRC_CUDA(cudaMemcpyAsync(r->d_hin, h_in, r->n_ch * n_in * sizeof(float), cudaMemcpyHostToDevice, s));
    size_t got = 0;
    int rc = lrc_resampler_process(r, r->d_hin, n_in, n_in, r->d_hout, no + 1, &got, s);
    if (rc) return rc;
    if (got)
        LRC_CUDA(cudaMemcpy2DAsync(h_out, out_cap * sizeof(float), r->d_hout, (no + 1) * sizeof(float), got * sizeof(float),
                                   r->n_ch, cudaMemcpyDeviceToHost, s));
    LRC_CUDA(cudaStreamSynchronize(s));
    *n_out = got;
    return LRC_OK;
}
