// k_psdpng.cu -- the spectrogram rows of libkissfft/tools/psdpng.c (transform_signal, :120-185):
//
//   16-bit PCM, mono or stereo (L + R summed, :141-146) -> frames of nfft reals
//   -> optional removal of the frame mean (-a, :156-161) -> kiss_fftr (:164)
//   -> mag2buf[i] += re^2 + im^2 over navg frames (:166-167)
//   -> row[i] = 10 log10(mag2buf[i] / navg + 1) for the nfft/2+1 bins (:169-176)
//
// A trailing partial frame and a trailing partial row are dropped exactly as the reference's read loop
// drops them (:141-152, :169).  Three launches: frames (convert + mean), the real FFT of k_fft_mixed.cu,
// rows (|X|^2 average + log).  The PNG colour mapping (:68-118) stays on the host: it is display code.
#include "common.cuh"

struct lrc_rfft;

// one CTA per frame: int16 -> f32 (stereo: l + r in float like the reference's `tbuf[i] = inbuf[2*i] + inbuf[2*i+1]`
// -- an int sum converted to float), then tbuf[i] -= avg
__global__ void __launch_bounds__(256)
psdpng_frames_kernel(const int16_t *__restrict__ pcm, float *__restrict__ frames, int nfft, int stereo, int remove_dc)
{
    const size_t f = blockIdx.x;
    const int16_t *src = pcm + f * (size_t)nfft * (stereo ? 2 : 1);
    float *dst = frames + f * (size_t)nfft;
    __shared__ float red[8];
    __shared__ float avg_s;
    float part = 0.f;
    for (int i = threadIdx.x; i < nfft; i += blockDim.x) {
        const float v = stereo ? (float)((int)src[2 * i] + (int)src[2 * i + 1]) : (float)src[i];
        dst[i] = v;
        part += v;
    }
    if (!remove_dc) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
        avg_s = s / (float)nfft;                                           // avg /= nfft  :159
    }
    __syncthreads();
    const float avg = avg_s;
    for (int i = threadIdx.x; i < nfft; i += blockDim.x) dst[i] -= avg;     // own writes, same thread
}

__global__ void __launch_bounds__(256)
psdpng_rows_kernel(const float2 *__restrict__ freq, float *__restrict__ rows, size_t n_rows, int nfreqs, int navg)
{
    const size_t total = n_rows * (size_t)nfreqs;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / nfreqs;
        const int b = (int)(i - r * nfreqs);
        const float2 *p = freq + (r * navg) * (size_t)nfreqs + b;
        float acc = 0.f;
        for (int f = 0; f < navg; ++f) {
            const float2 x = p[(size_t)f * nfreqs];
            acc += x.x * x.x + x.y * x.y;                                   // mag2buf[i] += r*r + i*i  :167
        }
        rows[i] = 10.0f * log10f(acc / (float)navg + 1.0f);                 // :174
    }
}

extern "C" int lrc_psdpng_rows(lrc_ctx *ctx, const int16_t *d_pcm, size_t n_samples, int nfft, int navg,
                               int remove_dc, int stereo, float *d_rows, size_t *n_rows, void *stream)
{
    LRC_BIND(ctx);
    LRC_REQUIRE(nfft >= 4 && navg >= 1 && n_rows, LRC_ERR_INVALID, "lrc_psdpng_rows: bad arguments");
    const size_t n_frames = n_samples / (size_t)nfft;                       // a short last read ends the loop :141-152
    const size_t rows = n_frames / (size_t)navg;
    *n_rows = rows;
    if (rows == 0) return LRC_OK;
    LRC_REQUIRE(d_pcm && d_rows, LRC_ERR_INVALID, "lrc_psdpng_rows: null buffer");
    const size_t use = rows * (size_t)navg;
    const int nfreqs = nfft / 2 + 1;
    cudaStream_t s = lrc_stream(ctx, stream);
    lrc_rfft *plan = nullptr;
    int rc = lrc_rfft_create(ctx, nfft, 0, &plan);                          // kiss_fftr_alloc(nfft,0,0,0)  :131
    if (rc) return rc;
    DevBuf<float> d_frames;
    DevBuf<float2> d_freq;
    cudaError_t e = d_frames.alloc(use * (size_t)nfft);
    if (e == cudaSuccess) e = d_freq.alloc(use * (size_t)nfreqs);
    if (e == cudaSuccess) {
        psdpng_frames_kernel<<<(unsigned)use, 256, 0, s>>>(d_pcm, d_frames, nfft, stereo ? 1 : 0, remove_dc ? 1 : 0);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) rc = lrc_rfft_run(plan, d_frames, (float *)d_freq.get(), use, s);
    if (e == cudaSuccess && rc == LRC_OK) {
        size_t blocks = ceil_div(rows * (size_t)nfreqs, 256);
        const size_t cap = (size_t)ctx->n_sm * 16;
        if (blocks > cap) blocks = cap;
        psdpng_rows_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_freq, d_rows, rows, nfreqs, navg);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);                     // scratch is freed on return
    lrc_rfft_destroy(plan);
    if (e != cudaSuccess) { lrc_set_error("lrc_psdpng_rows: %s", cudaGetErrorString(e)); return LRC_ERR_CUDA; }
    return rc;
}
