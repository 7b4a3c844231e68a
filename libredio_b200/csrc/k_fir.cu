// k_fir.cu -- FIR + decimate (dsputils::convolve + north-star decimation), batch and streaming.
//
//   z[c][k] = sum_{j<ntaps} x[c][k*decim + j] * taps[j]      (src/dsputils/src/dsputils.rs:30-32)
//
// Two code paths, same arithmetic order (j ascending, fused multiply-add):
//   * fir_tile_kernel<64,10,...>: TMA-staged shared-memory tile, register-blocked (fir_core.cuh)
//   * fir_gentile_kernel (k_fir_gentile.cu): cf32, ntaps <= 128, decim in {4,5,8,10,16}: padded-chunk TMA tile, packed FFMA2
//   * fir_generic_kernel: any other (ntaps, decim) and u8 input of those, one thread per output straight from global/L1
#include "fir_core.cuh"
#include <vector>

bool lrc_fir_gentile_has(int ntaps, int decim);
int  lrc_fir_gentile_launch(int n_sm, const float *h_taps, int ntaps, int decim, const float *d_in, size_t n_ch, size_t n_in,
                            size_t in_stride, float *d_out, size_t n_out, size_t out_stride, cudaStream_t s);

struct lrc_fir {
    lrc_ctx *ctx;
    int      ntaps, decim;
    std::vector<float> taps;      // host copy
    DevBuf<float> d_taps;         // device copy (generic path)
    DevBuf<float> d_taps127;      // taps / 127 (u8 generic path)
};

struct lrc_fir_stream {
    lrc_fir *fir;
    size_t   n_ch, max_chunk, cap;   // cap: samples per channel row of the staging buffer
    int      is_u8;
    size_t   esize;                  // bytes per sample (8 or 2)
    size_t   held;                   // samples carried at the row fronts
    size_t   skip;                   // samples of future input to drop (only when decim > ntaps)
    DevBuf<uint8_t> d_buf;           // [n_ch][cap] staging rows: carry followed by the new chunk
    DevBuf<uint8_t> d_carry;         // [n_ch][ntaps + decim] scratch for the carry move
};

// ---------------------------------------------------------------------------------------------
// tile kernel
// ---------------------------------------------------------------------------------------------
template <int NTAPS, int DECIM, int R, int NT, bool IS_U8>
struct FirTileCfg {
    using Tile = FirTile<NTAPS, DECIM, R>;
    static constexpr int TILE_OUT = R * NT;                                  // outputs per tile
    static constexpr int TILE_IN = (TILE_OUT - 1) * DECIM + NTAPS;           // samples per tile
    static constexpr int ESIZE = IS_U8 ? 2 : 8;
    static constexpr int TILE_BYTES = ((TILE_IN * ESIZE + 15) / 16) * 16;
    static constexpr int SMEM_BYTES = TILE_BYTES + 16;                       // + mbarrier
};

template <int NTAPS, int DECIM, int R, int NT, bool IS_U8>
__global__ void __launch_bounds__(NT)
fir_tile_kernel(const uint8_t *__restrict__ in, size_t n_ch, size_t n_in, size_t in_stride,
                float2 *__restrict__ out, size_t n_out, size_t out_stride, int use_tma,
                const __grid_constant__ FirTaps<NTAPS> taps)
{
    using Cfg = FirTileCfg<NTAPS, DECIM, R, NT, IS_U8>;
    using Tile = typename Cfg::Tile;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + Cfg::TILE_BYTES);
    const int t = threadIdx.x;
    if (t == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    __syncthreads();
    uint32_t phase = 0;

    const size_t tiles_per_ch = (n_out + Cfg::TILE_OUT - 1) / Cfg::TILE_OUT;
    const size_t n_tiles = tiles_per_ch * n_ch;
    for (size_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const size_t c = tile / tiles_per_ch, ti = tile % tiles_per_ch;
        const size_t o0 = ti * Cfg::TILE_OUT;                  // first output of the tile
        const size_t s0 = o0 * DECIM;                          // first input sample
        size_t ns = n_in - s0;                                 // samples available from s0
        if (ns > (size_t)Cfg::TILE_IN) ns = Cfg::TILE_IN;
        const uint8_t *src = in + (c * in_stride + s0) * Cfg::ESIZE;
        const uint32_t bytes = (uint32_t)(ns * Cfg::ESIZE);
        if (use_tma) {
            const uint32_t bulk = bytes & ~15u;
            if (t == 0) {
                mbar_expect_tx(bar, bulk);
                if (bulk) tma_load_1d(smem, src, bulk, bar);
            }
            // the < 16-byte remainder of a ragged last tile
            if (t < (int)(bytes - bulk)) smem[bulk + t] = src[bulk + t];
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {
            // unaligned source: cooperative element-wise copy
            for (uint32_t i = t; i < bytes / Cfg::ESIZE; i += NT) {
                if (IS_U8) reinterpret_cast<uint16_t *>(smem)[i] = reinterpret_cast<const uint16_t *>(src)[i];
                else       reinterpret_cast<float2 *>(smem)[i] = reinterpret_cast<const float2 *>(src)[i];
            }
        }
        __syncthreads();

        float2 acc[R];
        if (IS_U8) Tile::run_u8(reinterpret_cast<const uint32_t *>(smem) + (size_t)t * Tile::STEP / 2, taps, acc);
        else       Tile::run_cf32(reinterpret_cast<const float2 *>(smem) + (size_t)t * Tile::STEP, taps, acc);

        float2 *dst = out + c * out_stride + o0 + (size_t)t * R;
        const size_t left = n_out - o0;                        // outputs remaining in this channel
#pragma unroll
        for (int r = 0; r < R; ++r)
            if ((size_t)(t * R + r) < left) dst[r] = acc[r];
        __syncthreads();                                       // tile consumed before the next load
    }
}

// ---------------------------------------------------------------------------------------------
// generic kernel (any ntaps / decim): one thread per output
// ---------------------------------------------------------------------------------------------
template <bool IS_U8>
__global__ void __launch_bounds__(256)
fir_generic_kernel(const uint8_t *__restrict__ in, size_t n_ch, size_t in_stride, float2 *__restrict__ out,
                   size_t n_out, size_t out_stride, const float *__restrict__ taps, int ntaps, int decim)
{
    const size_t total = n_ch * n_out;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / n_out, k = i % n_out;
        float ar = 0.f, ai = 0.f;
        if (IS_U8) {
            const uchar2 *x = reinterpret_cast<const uchar2 *>(in) + c * in_stride + k * decim;
            for (int j = 0; j < ntaps; ++j) {
                const uchar2 b = x[j];
                const float h = __ldg(taps + j);          // taps / 127
                ar = fmaf((float)((int)b.x - 127), h, ar);
                ai = fmaf((float)((int)b.y - 127), h, ai);
            }
        } else {
            const float2 *x = reinterpret_cast<const float2 *>(in) + c * in_stride + k * decim;
            for (int j = 0; j < ntaps; ++j) {
                const float2 v = x[j];
                const float h = __ldg(taps + j);
                ar = fmaf(v.x, h, ar);
                ai = fmaf(v.y, h, ai);
            }
        }
        out[c * out_stride + k] = make_float2(ar, ai);
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
extern "C" int lrc_fir_create(lrc_ctx *ctx, const float *h_taps, int ntaps, int decim, lrc_fir **out)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(out && h_taps && ntaps >= 1 && decim >= 1, LRC_ERR_INVALID, "lrc_fir_create: bad arguments");
    for (int i = 0; i < ntaps; ++i)
        if (!(h_taps[i] == h_taps[i]) || h_taps[i] - h_taps[i] != 0.0f) {
            lrc_set_error("lrc_fir_create: tap %d is not finite (dsputils::lpf yields NaN taps because "
                          "dsputils::window is broken, dsputils.rs:49; supply finite taps)", i);
            return LRC_ERR_INVALID;
        }
    lrc_fir *f = new (std::nothrow) lrc_fir();
    LRC_REQUIRE(f != nullptr, LRC_ERR_NOMEM, "out of host memory");
    f->ctx = ctx; f->ntaps = ntaps; f->decim = decim;
    f->taps.assign(h_taps, h_taps + ntaps);
    std::vector<float> t127(ntaps);
    for (int i = 0; i < ntaps; ++i) t127[i] = (float)((double)h_taps[i] / 127.0);
    if (f->d_taps.alloc(ntaps) != cudaSuccess || f->d_taps127.alloc(ntaps) != cudaSuccess ||
        cudaMemcpy(f->d_taps, h_taps, sizeof(float) * ntaps, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(f->d_taps127, t127.data(), sizeof(float) * ntaps, cudaMemcpyHostToDevice) != cudaSuccess) {
        lrc_set_error("lrc_fir_create: %s", cudaGetErrorString(cudaGetLastError()));
        lrc_fir_destroy(f);
        return LRC_ERR_CUDA;
    }
    *out = f;
    return LRC_OK;
}

extern "C" int lrc_fir_destroy(lrc_fir *f)
{
    if (!f) return LRC_OK;
    cudaSetDevice(f->ctx->device);
    delete f;
    return LRC_OK;
}

extern "C" size_t lrc_fir_out_len(const lrc_fir *f, size_t n_in)
{
    if (!f || n_in < (size_t)f->ntaps) return 0;
    return (n_in - f->ntaps) / f->decim + 1;
}

template <bool IS_U8>
static int fir_launch(lrc_fir *f, const void *d_in, size_t n_ch, size_t n_in, size_t in_stride, float *d_out,
                      size_t out_stride, cudaStream_t s)
{
    const size_t n_out = lrc_fir_out_len(f, n_in);
    if (n_out == 0 || n_ch == 0) return LRC_OK;
    LRC_REQUIRE(d_in && d_out, LRC_ERR_INVALID, "fir: null buffer");
    LRC_REQUIRE(in_stride >= n_in && out_stride >= n_out, LRC_ERR_INVALID, "fir: stride shorter than length");
    LRC_REQUIRE(((uintptr_t)d_out & 7) == 0 && ((uintptr_t)d_in & (IS_U8 ? 1 : 7)) == 0, LRC_ERR_INVALID,
                "fir: misaligned buffer");
    constexpr size_t ES = IS_U8 ? 2 : 8;
    if (f->ntaps == 64 && f->decim == 10) {
        constexpr int R = 7, NT = 128;
        using Cfg = FirTileCfg<64, 10, R, NT, IS_U8>;
        auto kern = fir_tile_kernel<64, 10, R, NT, IS_U8>;
        size_t ctas;
        LRC_CUDA(lrc_resident_ctas(kern, NT, Cfg::SMEM_BYTES, f->ctx->n_sm, &ctas));
        const size_t n_tiles = ceil_div(n_out, (size_t)Cfg::TILE_OUT) * n_ch;
        static const size_t gm = lrc_grid_mult(IS_U8 ? "LRC_FIRU8_GRID" : "LRC_FIR_GRID", IS_U8 ? 16 : 1024);
        size_t blocks = ctas * gm;
        if (blocks > n_tiles) blocks = n_tiles;
        // TMA needs 16-byte aligned sources: base, channel stride and (always true) tile stride
        const int use_tma = (((uintptr_t)d_in & 15) == 0) && (n_ch == 1 || (in_stride * ES) % 16 == 0);
        FirTaps<64> taps;
        for (int i = 0; i < 64; ++i) taps.h[i] = IS_U8 ? (float)((double)f->taps[i] / 127.0) : f->taps[i];
        kern<<<(unsigned)blocks, NT, Cfg::SMEM_BYTES, s>>>((const uint8_t *)d_in, n_ch, n_in, in_stride,
                                                          (float2 *)d_out, n_out, out_stride, use_tma, taps);
    } else if (!IS_U8 && lrc_fir_gentile_has(f->ntaps, f->decim) && !getenv("LRC_FIR_NO_GENTILE")) {
        // cf32, ntaps <= 128, decim in {4,5,8,10,16}: the generic tile kernel (k_fir_gentile.cu); LRC_FIR_NO_GENTILE=1 is the A/B knob
        return lrc_fir_gentile_launch(f->ctx->n_sm, f->taps.data(), f->ntaps, f->decim, (const float *)d_in, n_ch, n_in, in_stride,
                                      d_out, n_out, out_stride, s);
    } else {
        size_t blocks = ceil_div(n_ch * n_out, 256);
        const size_t cap = (size_t)f->ctx->n_sm * 8;
        if (blocks > cap) blocks = cap;
        fir_generic_kernel<IS_U8><<<(unsigned)blocks, 256, 0, s>>>(
            (const uint8_t *)d_in, n_ch, in_stride, (float2 *)d_out, n_out, out_stride,
            IS_U8 ? f->d_taps127 : f->d_taps, f->ntaps, f->decim);
    }
    LRC_CUDA(cudaGetLastError());
    return LRC_OK;
}

extern "C" int lrc_fir_run_cf32(lrc_fir *f, const float *d_in, size_t n_ch, size_t n_in, size_t in_stride,
                                float *d_out, size_t out_stride, void *stream)
{
    LRC_REQUIRE(f != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(f->ctx);
    return fir_launch<false>(f, d_in, n_ch, n_in, in_stride, d_out, out_stride, lrc_stream(f->ctx, stream));
}

extern "C" int lrc_fir_run_u8(lrc_fir *f, const uint8_t *d_in, size_t n_ch, size_t n_in, size_t in_stride,
                              float *d_out, size_t out_stride, void *stream)
{
    LRC_REQUIRE(f != nullptr, LRC_ERR_INVALID, "null plan");
    LRC_BIND(f->ctx);
    return fir_launch<true>(f, d_in, n_ch, n_in, in_stride, d_out, out_stride, lrc_stream(f->ctx, stream));
}

// ---- streaming ---------------------------------------------------------------------------------
extern "C" int lrc_fir_stream_create(lrc_fir *f, size_t n_ch, size_t max_chunk, int input_is_u8,
                                     lrc_fir_stream **out)
{
    LRC_REQUIRE(f && out && n_ch >= 1 && max_chunk >= 1, LRC_ERR_INVALID, "lrc_fir_stream_create: bad arguments");
    LRC_BIND(f->ctx);
    lrc_fir_stream *st = new (std::nothrow) lrc_fir_stream();
    LRC_REQUIRE(st != nullptr, LRC_ERR_NOMEM, "out of host memory");
    st->fir = f; st->n_ch = n_ch; st->max_chunk = max_chunk; st->is_u8 = input_is_u8 ? 1 : 0;
    st->esize = input_is_u8 ? 2 : 8;
    st->held = 0; st->skip = 0;
    // a row holds at most ntaps-1 carried samples plus one chunk; rows are 16-byte multiples so
    // every row start stays TMA-aligned
    st->cap = ((size_t)f->ntaps + max_chunk + 7) / 8 * 8;
    if (st->d_buf.alloc(n_ch * st->cap * st->esize) != cudaSuccess ||
        st->d_carry.alloc(n_ch * (size_t)(f->ntaps + 8) * st->esize) != cudaSuccess) {
        lrc_set_error("lrc_fir_stream_create: %s", cudaGetErrorString(cudaGetLastError()));
        lrc_fir_stream_destroy(st);
        return LRC_ERR_CUDA;
    }
    *out = st;
    return LRC_OK;
}

extern "C" int lrc_fir_stream_destroy(lrc_fir_stream *st)
{
    if (!st) return LRC_OK;
    cudaSetDevice(st->fir->ctx->device);
    delete st;
    return LRC_OK;
}

extern "C" int lrc_fir_stream_push(lrc_fir_stream *st, const void *d_chunk, size_t n, size_t chunk_stride,
                                   float *d_out, size_t out_stride, size_t *n_out, void *stream)
{
    LRC_REQUIRE(st && n_out, LRC_ERR_INVALID, "lrc_fir_stream_push: null argument");
    lrc_fir *f = st->fir;
    LRC_BIND(f->ctx);
    LRC_REQUIRE(n <= st->max_chunk, LRC_ERR_CAPACITY, "lrc_fir_stream_push: chunk longer than max_chunk");
    *n_out = 0;
    if (n == 0) return LRC_OK;
    LRC_REQUIRE(d_chunk != nullptr && chunk_stride >= n, LRC_ERR_INVALID, "lrc_fir_stream_push: bad chunk");
    cudaStream_t s = lrc_stream(f->ctx, stream);
    const size_t es = st->esize, row = st->cap * es;
    if (st->skip) {                                   // decim > ntaps: inputs between windows are unused
        const size_t k = st->skip < n ? st->skip : n;
        st->skip -= k; n -= k;
        d_chunk = (const uint8_t *)d_chunk + k * es;
        if (n == 0) return LRC_OK;
    }
    // append the chunk behind the carried samples of every channel row
    LRC_CUDA(cudaMemcpy2DAsync(st->d_buf + st->held * es, row, d_chunk, chunk_stride * es, n * es, st->n_ch,
                               cudaMemcpyDeviceToDevice, s));
    const size_t total = st->held + n;
    const size_t no = lrc_fir_out_len(f, total);
    if (no > 0) {
        LRC_REQUIRE(d_out != nullptr && out_stride >= no, LRC_ERR_CAPACITY, "lrc_fir_stream_push: output too small");
        int rc = st->is_u8 ? fir_launch<true>(f, st->d_buf, st->n_ch, total, st->cap, d_out, out_stride, s)
                           : fir_launch<false>(f, st->d_buf, st->n_ch, total, st->cap, d_out, out_stride, s);
        if (rc) return rc;
        // keep the samples the next output (index `no`) starts at: [no*decim, total)
        const size_t consumed = no * (size_t)f->decim;
        const size_t carry = total > consumed ? total - consumed : 0;
        if (carry) {
            const size_t crow = (size_t)(f->ntaps + 8) * es;
            LRC_CUDA(cudaMemcpy2DAsync(st->d_carry, crow, st->d_buf + consumed * es, row, carry * es, st->n_ch,
                                       cudaMemcpyDeviceToDevice, s));
            LRC_CUDA(cudaMemcpy2DAsync(st->d_buf, row, st->d_carry, crow, carry * es, st->n_ch,
                                       cudaMemcpyDeviceToDevice, s));
        }
        st->held = carry;
        st->skip = consumed > total ? consumed - total : 0;
    } else {
        st->held = total;
    }
    *n_out = no;
    return LRC_OK;
}
