// k_unpack.cu -- u8 IQ -> interleaved complex f32, bit-exact with rtlsdr::i2f
// (src/rtlsdr/src/rtlsdr.rs:159-162):  i2f(b) = fl(fl(b)/127) - 1.
//
// HBM-bound: 2 B in, 8 B out per sample; 6 full-rate instructions per value (unpack.cuh).
//
// Measured and rejected (round 1, profiles/r1_s8_grid_sweeps.txt, grid capped at 16 CTAs per SM, Gsamples/s): the
// streaming st.global.L1::no_allocate store (562.6) and st.global.cs (563.1) against plain stores (571.1), and a register
// bound for 8 resident CTAs per SM (539.7 / 542.5 / 540.5 for the three store forms) against 4.
#include "common.cuh"
#include "unpack.cuh"

// One 32-bit word (two samples) per lane per step: the warp reads 128 contiguous bytes and writes 512
// contiguous bytes with one STG.128 per lane, so both directions are perfectly coalesced; UNROLL steps are
// issued back to back to keep enough loads in flight.
constexpr int UNPACK_UNROLL = 8;

__global__ void __launch_bounds__(256, 4)
unpack_kernel(const uint8_t *__restrict__ in, float *__restrict__ out, size_t n_bytes)
{
    const size_t n_words = n_bytes / 4;
    const uint32_t *src = reinterpret_cast<const uint32_t *>(in);
    float4 *dst = reinterpret_cast<float4 *>(out);
    const size_t chunk = (size_t)blockDim.x * UNPACK_UNROLL;
    for (size_t base = (size_t)blockIdx.x * chunk; base < n_words; base += (size_t)gridDim.x * chunk) {
        uint32_t w[UNPACK_UNROLL];
#pragma unroll
        for (int u = 0; u < UNPACK_UNROLL; ++u) {
            const size_t i = base + (size_t)u * blockDim.x + threadIdx.x;
            w[u] = i < n_words ? __ldcs(src + i) : 0u;
        }
#pragma unroll
        for (int u = 0; u < UNPACK_UNROLL; ++u) {
            const size_t i = base + (size_t)u * blockDim.x + threadIdx.x;
            if (i < n_words) {
                const float4 v = make_float4(lr_i2f_byte(w[u], 0), lr_i2f_byte(w[u], 1),
                                             lr_i2f_byte(w[u], 2), lr_i2f_byte(w[u], 3));
                dst[i] = v;
            }
        }
    }
    // tail (< 4 bytes) and unaligned buffers are handled by the scalar kernel below
}

__global__ void unpack_scalar_kernel(const uint8_t *__restrict__ in, float *__restrict__ out, size_t first,
                                     size_t n_bytes)
{
    const size_t i = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_bytes) out[i] = lr_i2f(in[i]);
}

extern "C" int lrc_unpack_u8_cf32(lrc_ctx *ctx, const uint8_t *d_iq, size_t n_bytes, float *d_out, void *stream)
{
    LRC_BIND(ctx);
    if (n_bytes & 1) {
        lrc_set_error("lrc_unpack_u8_cf32: %zu bytes is odd; the reference indexes i[1] out of bounds and "
                      "panics (rtlsdr.rs:161)", n_bytes);
        return LRC_ERR_ODD_LENGTH;
    }
    if (n_bytes == 0) return LRC_OK;
    LRC_REQUIRE(d_iq && d_out, LRC_ERR_INVALID, "lrc_unpack_u8_cf32: null buffer");
    cudaStream_t s = lrc_stream(ctx, stream);
    size_t vec_bytes = 0;
    if (((uintptr_t)d_iq & 3) == 0 && ((uintptr_t)d_out & 15) == 0) {
        vec_bytes = n_bytes / 4 * 4;
        if (vec_bytes) {
            size_t blocks = ceil_div(vec_bytes / 4, (size_t)256 * UNPACK_UNROLL);
            // one 8 KB-in / 32 KB-out chunk per CTA and no grid cap: 0.87 -> 1.04 of the copy bandwidth against 16
            // looping CTAs per SM (profiles/r1_s8_grid_sweeps.txt).  LRC_UNPACK_CAP = CTAs per SM cap
            static const size_t capf = lrc_grid_mult("LRC_UNPACK_CAP", (size_t)1 << 20);
            const size_t cap = (size_t)ctx->n_sm * capf;
            if (blocks > cap) blocks = cap;
            if (blocks > 0x7fffffffu) blocks = 0x7fffffffu;
            unpack_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_iq, d_out, vec_bytes);
            LRC_CUDA(cudaGetLastError());
        }
    }
    if (vec_bytes < n_bytes) {
        const size_t rest = n_bytes - vec_bytes;
        unpack_scalar_kernel<<<(unsigned)ceil_div(rest, 256), 256, 0, s>>>(d_iq, d_out, vec_bytes, n_bytes);
        LRC_CUDA(cudaGetLastError());
    }
    return LRC_OK;
}
