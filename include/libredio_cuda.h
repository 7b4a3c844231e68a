/*
 * libredio_cuda.h -- C ABI of libredio_cuda.so, the B200 (sm_100a) implementation of LibRedio's
 * sample-stream DSP hot path.  Plain pointers and sizes only; no C++/torch types cross this line.
 *
 * Each entry point names the reference interface it replaces (paths relative to the LibRedio tree).
 * The kpn-shaped blocks that call it live in kpn/gpu_blocks.hpp (C++) and rust/kpn-gpu (source only);
 * INTEGRATION.md shows the bindings.
 *
 * Conventions
 *   - every function returns an int status (LRC_OK == 0); lrc_last_error() gives the detail text of the
 *     most recent failure on the calling thread.  The reference's convention is unwrap()/panic
 *     (src/kpn/src/kpn.rs:18-28, src/samplerate/src/samplerate.rs:77-83); the kpn wrappers turn a
 *     non-zero status into exactly that.
 *   - pointers prefixed d_ are device pointers on the context's GPU, h_ are host pointers.
 *   - `stream` is a cudaStream_t passed as void*; NULL means the context's own stream.  Calls are
 *     asynchronous on that stream unless stated otherwise.
 *   - complex samples are interleaved f32 {re, im} exactly like num::Complex<f32> / kiss_fft_cpx
 *     (src/kissfft/src/kissfft.rs:14, libkissfft/kiss_fft.h:51-54).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with LRC_ERR_CUDA.
 */
#ifndef LIBREDIO_CUDA_H
#define LIBREDIO_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRC_VERSION 100

enum {
    LRC_OK = 0,
    LRC_ERR_INVALID = 1,      /* bad argument (NULL, zero size, ...) */
    LRC_ERR_CUDA = 2,         /* CUDA runtime/driver error, see lrc_last_error() */
    LRC_ERR_UNSUPPORTED = 3,  /* valid for the reference but not implemented here (e.g. nfft > 8192) */
    LRC_ERR_NOMEM = 4,
    LRC_ERR_CAPACITY = 5,     /* caller-provided output capacity too small */
    LRC_ERR_ODD_LENGTH = 6,   /* odd byte count into the u8-IQ unpack (the reference panics) */
    LRC_ERR_LENGTH = 7        /* frame length != block_size (the reference asserts, kissfft.rs:24) */
};

typedef struct lrc_ctx lrc_ctx;

int         lrc_version(void);
const char *lrc_strerror(int status);
const char *lrc_last_error(void);

/* one context per GPU (one process per GPU under torch.distributed / one thread per GPU otherwise) */
int lrc_ctx_create(int device, lrc_ctx **ctx);
int lrc_ctx_destroy(lrc_ctx *ctx);
int lrc_ctx_sync(lrc_ctx *ctx);                       /* cudaStreamSynchronize of the context stream */
int lrc_ctx_sm_count(lrc_ctx *ctx, int *n_sm);
/* NUMA node of the GPU (-1 if sysfs does not say) and the number of online nodes of the host */
int lrc_ctx_numa_node(lrc_ctx *ctx, int *node, int *n_nodes);
/* pin the calling thread to the CPUs of the GPU's NUMA node (no-op on a single-node host); *n_cpus = CPUs bound to */
int lrc_ctx_bind_thread(lrc_ctx *ctx, int *n_cpus);
/* pinned host memory for the ring / *_host entry points, placed on the GPU's NUMA node when the host has several.
 * A plan object (lrc_fir_stream, lrc_psd, lrc_chain, lrc_resampler, lrc_fmrx, lrc_ook, ...) owns scratch and carried
 * state: use it from ONE thread / stream at a time.  Different plans of one context are independent. */
int lrc_host_alloc(lrc_ctx *ctx, size_t bytes, void **h_ptr);
int lrc_host_free(lrc_ctx *ctx, void *h_ptr);
/* device memory, streams and asynchronous copies for FFI hosts that carry no CUDA bindings of their own (rust/kpn-gpu):
 * together with lrc_host_alloc they are what a KPN block needs to run a pinned, double-buffered ring around the plan entry
 * points (copy in, launch, copy out on the block's stream, an event per ring slot to know when its batch is out).
 * `stream` NULL = the context's own stream. */
int lrc_dev_alloc(lrc_ctx *ctx, size_t bytes, void **d_ptr);
int lrc_dev_free(lrc_ctx *ctx, void *d_ptr);
int lrc_dev_memset(lrc_ctx *ctx, void *d_ptr, int value, size_t bytes, void *stream);
int lrc_stream_create(lrc_ctx *ctx, void **stream);
int lrc_stream_destroy(lrc_ctx *ctx, void *stream);
int lrc_stream_sync(lrc_ctx *ctx, void *stream);
/* completion of one ring slot's batch when several slots share a stream */
int lrc_event_create(lrc_ctx *ctx, void **event);
int lrc_event_destroy(lrc_ctx *ctx, void *event);
int lrc_event_record(lrc_ctx *ctx, void *event, void *stream);
int lrc_event_sync(lrc_ctx *ctx, void *event);
int lrc_copy_h2d_async(lrc_ctx *ctx, void *d_dst, const void *h_src, size_t bytes, void *stream);
int lrc_copy_d2h_async(lrc_ctx *ctx, void *h_dst, const void *d_src, size_t bytes, void *stream);
/* synchronous device -> host copy (for the debug views below and bindings without a CUDA runtime) */
int lrc_copy_to_host(lrc_ctx *ctx, void *h_dst, const void *d_src, size_t bytes);

/* ------------------------------------------------------------------------------------------------
 * (1) u8 IQ -> complex f32.   Replaces rtlsdr::i2f / rtlsdr::data_to_samples
 *     (src/rtlsdr/src/rtlsdr.rs:159-162):  out[k] = { b[2k]/127 - 1, b[2k+1]/127 - 1 }, bit-exact.
 *     n_bytes odd -> LRC_ERR_ODD_LENGTH (the reference indexes out of bounds and panics).
 * ---------------------------------------------------------------------------------------------- */
int lrc_unpack_u8_cf32(lrc_ctx *ctx, const uint8_t *d_iq, size_t n_bytes, float *d_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (2) FIR + decimation.   Replaces dsputils::convolve (src/dsputils/src/dsputils.rs:30-32) applied to
 *     the re and im planes with real taps (valid-mode correlation, taps NOT reversed), followed by the
 *     north-star-defined decimation z[k] = y[k*decim]:
 *         z[k] = sum_{j<ntaps} x[k*decim + j] * taps[j],   k in [0, floor((n - ntaps)/decim)].
 *     Streaming (lrc_fir_stream_*) is seam-exact: the concatenated outputs equal one call over the
 *     concatenated input, whatever the chunking.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_fir lrc_fir;
int    lrc_fir_create(lrc_ctx *ctx, const float *h_taps, int ntaps, int decim, lrc_fir **fir);
int    lrc_fir_destroy(lrc_fir *fir);
size_t lrc_fir_out_len(const lrc_fir *fir, size_t n_in);   /* 0 if n_in < ntaps */
/* n_ch independent channels; channel c starts at d_in + c*in_stride (stride in SAMPLES) */
int lrc_fir_run_cf32(lrc_fir *fir, const float *d_in, size_t n_ch, size_t n_in, size_t in_stride,
                     float *d_out, size_t out_stride, void *stream);
/* fused (1)+(2): input is u8 IQ (2 bytes per sample) */
int lrc_fir_run_u8(lrc_fir *fir, const uint8_t *d_in, size_t n_ch, size_t n_in, size_t in_stride,
                   float *d_out, size_t out_stride, void *stream);

typedef struct lrc_fir_stream lrc_fir_stream;
int lrc_fir_stream_create(lrc_fir *fir, size_t n_ch, size_t max_chunk, int input_is_u8,
                          lrc_fir_stream **st);
int lrc_fir_stream_destroy(lrc_fir_stream *st);
/* push n new samples per channel (device memory, channel stride in samples); writes the outputs that
 * became computable to d_out (+ c*out_stride) and their per-channel count to *n_out (host).
 * Synchronous with respect to the host for the count only (it is arithmetic, no device readback). */
int lrc_fir_stream_push(lrc_fir_stream *st, const void *d_chunk, size_t n, size_t chunk_stride,
                        float *d_out, size_t out_stride, size_t *n_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (3) FFT.   Replaces the kissfft binding: kiss_fft_alloc / kiss_fft (src/kissfft/src/kissfft.rs:11-31,
 *     libkissfft/kiss_fft.c:339-388).  Unscaled, forward e^{-j..}, inverse e^{+j..} also unscaled.
 *     nfft in [2, 8192]: powers of two run the register/shared-memory Stockham kernels, every other
 *     size (kissfft's mixed radix 2/3/4/5 + generic odd primes, kiss_fft.c:309-330) a shared-memory
 *     mixed-radix kernel; larger sizes: LRC_ERR_UNSUPPORTED.  `batch` frames of nfft samples,
 *     contiguous.  d_in == d_out is allowed (kiss_fft.c:373-379).
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_fft lrc_fft;
int lrc_fft_create(lrc_ctx *ctx, int nfft, int inverse, lrc_fft **fft);
int lrc_fft_destroy(lrc_fft *fft);
int lrc_fft_run(lrc_fft *fft, const float *d_in, float *d_out, size_t batch, void *stream);
/* host-buffer convenience with the reference block's contract: n_samples must be a multiple of
 * block_size (LRC_ERR_LENGTH otherwise, the assert of kissfft.rs:24). Synchronous. */
int lrc_fft_run_host(lrc_fft *fft, const float *h_in, float *h_out, size_t n_samples);

/* real-input pair.   Replaces kiss_fftr_alloc / kiss_fftr / kiss_fftri (libkissfft/tools/kiss_fftr.c:
 *     28-66, 67-119, 121-159).  nfft even (odd: LRC_ERR_INVALID, the reference prints "Real FFT
 *     optimization must be even" and returns NULL).  Forward (inverse == 0): `batch` frames of nfft f32
 *     -> batch frames of nfft/2+1 complex bins.  Inverse: nfft/2+1 bins -> nfft f32, unscaled (a round
 *     trip multiplies by nfft, README:105).  nfft/2 follows lrc_fft_create's size rules. */
typedef struct lrc_rfft lrc_rfft;
int lrc_rfft_create(lrc_ctx *ctx, int nfft, int inverse, lrc_rfft **rfft);
int lrc_rfft_destroy(lrc_rfft *rfft);
int lrc_rfft_run(lrc_rfft *rfft, const float *d_in, float *d_out, size_t batch, void *stream);
int lrc_rfft_run_host(lrc_rfft *rfft, const float *h_in, float *h_out, size_t batch);

/* window + |X|^2 averaging (north-star stage; nearest reference code tools/psdpng.c:157-178):
 *     rows[r][b] = (1/k_avg) * sum_{f<k_avg} | FFT(w .* frame[r*k_avg + f]) [b] |^2
 * window: LRC_WINDOW_NONE (psdpng) or LRC_WINDOW_HANN (periodic Hann 0.5-0.5cos(2 pi n/N)), or a
 * caller-supplied table via lrc_psd_set_window. */
enum { LRC_WINDOW_NONE = 0, LRC_WINDOW_HANN = 1 };
typedef struct lrc_psd lrc_psd;
int lrc_psd_create(lrc_ctx *ctx, int nfft, int window, lrc_psd **psd);
int lrc_psd_set_window(lrc_psd *psd, const float *h_window /* nfft */);
int lrc_psd_destroy(lrc_psd *psd);
/* n_frames frames at d_in; k_avg frames per row; writes floor(n_frames/k_avg) rows of nfft f32 */
int lrc_psd_run(lrc_psd *psd, const float *d_in, size_t n_frames, size_t k_avg, float *d_rows,
                void *stream);

/* spectrogram rows of tools/psdpng.c (transform_signal, :120-185): 16-bit PCM, mono or interleaved
 * stereo (channels summed, :141-146); n_samples counts samples PER CHANNEL.  Every nfft samples make a
 * frame; optional frame-mean removal (the -a switch, :156-161); kiss_fftr; |X|^2 summed over navg frames;
 * row[b] = 10 log10(sum/navg + 1), b < nfft/2+1 (:169-176).  Partial trailing frames/rows are dropped as
 * the reference's read loop drops them.  *n_rows rows of nfft/2+1 f32 are written.  Synchronous. */
int lrc_psdpng_rows(lrc_ctx *ctx, const int16_t *d_pcm, size_t n_samples, int nfft, int navg,
                    int remove_dc, int stereo, float *d_rows, size_t *n_rows, void *stream);

/* ------------------------------------------------------------------------------------------------
 * headline chain, one fused kernel: cf32 -> FIR(ntaps)/decim -> frames of nfft -> window -> FFT ->
 * |X|^2 averaged over k_avg frames.  Frame f covers inputs [f*nfft*decim, f*nfft*decim +
 * (nfft-1)*decim + ntaps).  The intermediate FIR output never touches HBM.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_chain lrc_chain;
int    lrc_chain_create(lrc_ctx *ctx, const float *h_taps, int ntaps, int decim, int nfft, int window,
                        lrc_chain **chain);
int    lrc_chain_destroy(lrc_chain *chain);
size_t lrc_chain_frames(const lrc_chain *chain, size_t n_in);       /* whole frames in n_in samples */
/* which kernel the plan runs: 0 = unfused (FIR kernel -> HBM -> PSD kernel), 1 = the fused BASELINE instance
 * (64 taps / 10 / 1024, cf32 and u8 input), 2 = a fused generic instance (ntaps <= 128, decim in {4,5,8,10,16},
 * nfft in {512,1024,2048}, tile fits shared memory).  Results are the same chain either way (FIR to float rounding). */
int    lrc_chain_kind(const lrc_chain *chain);
int    lrc_chain_run(lrc_chain *chain, const float *d_in, size_t n_in, size_t k_avg, float *d_rows,
                     size_t *n_rows, void *stream);
/* same with rtlsdr u8 I,Q on the DEVICE (2 bytes per sample; rtlsdr::data_to_samples, rtlsdr.rs:160-162, folded into the
 * kernel's tile load for the fused 64/10/1024 instance: HBM carries 2 B/sample, rows equal unpack-then-chain bit for bit) */
int    lrc_chain_run_u8(lrc_chain *chain, const uint8_t *d_iq, size_t n_in, size_t k_avg, float *d_rows,
                        size_t *n_rows, void *stream);
/* same through HOST buffers (pinned recommended): chunked H2D on a copy stream overlapped with the
 * kernel through a double-buffered device ring, rows copied back; synchronous. */
int    lrc_chain_run_host(lrc_chain *chain, const float *h_in, size_t n_in, size_t k_avg, float *h_rows,
                          size_t *n_rows);
/* same with the rtlsdr wire format as host input: n_in samples of interleaved u8 I,Q (2 bytes per sample over
 * PCIe instead of 8); rtlsdr::data_to_samples (rtlsdr.rs:160-162) runs on the device: inside the chain kernel's tile load
 * for the fused instance, as a separate launch in front of the chain otherwise. */
int    lrc_chain_run_host_u8(lrc_chain *chain, const uint8_t *h_iq, size_t n_in, size_t k_avg, float *h_rows,
                             size_t *n_rows);

/* ------------------------------------------------------------------------------------------------
 * long FIR by FFT overlap-save.   Replaces kiss_fastfir_alloc / kiss_fastfir
 * (libkissfft/tools/kiss_fastfir.c:65-245): true convolution with the nh-1 transient removed,
 *     y[k] = sum_j h[j] * x[k + nh - 1 - j].
 * nfft = 0 -> next power of two >= 2*nh, at least 1024 (:81-93).  Blocks advance by ngood = nfft-nh+1.
 * nfft fixes the output length; the library chooses the block size it computes in.
 * lrc_fastfir_run processes every full block of the n samples (kff_nocopy :192-206) and, if flush,
 * the zero-padded remainder (kff_flush :208-226); *n_out receives the number of outputs.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_fastfir lrc_fastfir;
int    lrc_fastfir_create(lrc_ctx *ctx, const float *h_taps_cpx, size_t nh, size_t nfft, lrc_fastfir **ff);
int    lrc_fastfir_destroy(lrc_fastfir *ff);
size_t lrc_fastfir_nfft(const lrc_fastfir *ff);
size_t lrc_fastfir_out_len(const lrc_fastfir *ff, size_t n_in, int flush);
int    lrc_fastfir_run(lrc_fastfir *ff, const float *d_in, size_t n_in, float *d_out, int flush,
                       size_t *n_out, void *stream);

/* Streaming form of lrc_fastfir_run over n_ch channels (kiss_fastfir(cfg, inbuf, outbuf, n_new, &offset), :228-245):
 * every channel carries its own history on the device, and all channels of a push go through one launch.
 * Outputs come in whole compute blocks: a push emits every output whose compute block is complete.  Blocks sit at
 * multiples of the compute block's ngood from the start of the stream, and the compute block is nfft points
 * (ngood = nfft - nh + 1) for plans with nh <= 1024 and nfft < 8192, 16384 points (ngood = 16385 - nh) otherwise.  So for
 * the first kind the per-push counts are kiss_fastfir's; for the second they come in units of 16385 - nh, while the
 * values and the flushed total are the same.  For every channel and every way of cutting the input into pushes, the
 * outputs concatenated, with flush on the last push, equal lrc_fastfir_run(whole input, flush = 1) bit for bit; after a
 * push without flush they are a bitwise prefix of it.  The carried history is always shorter than one compute block. */
typedef struct lrc_fastfir_stream lrc_fastfir_stream;
/* n_ch channels through the plan `ff` (borrowed: it must outlive the stream), each from the initial state (no history) */
int    lrc_fastfir_stream_create(lrc_fastfir *ff, size_t n_ch, lrc_fastfir_stream **st);
int    lrc_fastfir_stream_destroy(lrc_fastfir_stream *st);
int    lrc_fastfir_stream_reset(lrc_fastfir_stream *st);
/* outputs per channel that the next push of n samples (and flush) will write; host arithmetic */
size_t lrc_fastfir_stream_next_out_len(const lrc_fastfir_stream *st, size_t n, int flush);
/* n new samples per channel (n may be 0), channel c at d_chunk + c*chunk_stride (samples, >= n), cf32, 8-byte aligned;
 * outputs to d_out + c*out_stride (out_stride >= next_out_len, else LRC_ERR_CAPACITY; d_out must not overlap the
 * chunk); *n_out = outputs per channel (host arithmetic, no readback).  flush: after the chunk, also emit the
 * zero-padded remainder as kff_flush does (kiss_fastfir with n_new == 0, :228-245); the stream is then back at its
 * initial state, and a flush with fewer than nh samples held emits nothing more.  Asynchronous on `stream`; the pushes
 * of one stream must be ordered on the device (one CUDA stream, or synchronised between pushes). */
int    lrc_fastfir_stream_push(lrc_fastfir_stream *st, const float *d_chunk, size_t n, size_t chunk_stride,
                               float *d_out, size_t out_stride, int flush, size_t *n_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (4a) quadrature FM discriminator (north-star stage, absent from the reference):
 *     d[n] = atan2(Im z, Re z), z = x[n] * conj(x[n-1]); x[-1] comes from d_state (one cf32 per
 *     channel, zero at stream start) which is updated to the last sample of the chunk.
 * ---------------------------------------------------------------------------------------------- */
int lrc_fmdemod_run(lrc_ctx *ctx, const float *d_in, size_t n_ch, size_t n, size_t in_stride,
                    float *d_state /* n_ch cf32, may be NULL = stateless, x[-1] = 0 */,
                    float *d_out, size_t out_stride, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (4b) rational polyphase resampler.   Replaces samplerate::resample (src/samplerate/src/
 *     samplerate.rs:59-87: src_new(SRC_SINC_MEDIUM_QUALITY, 1 channel) + src_process per chunk).
 *     ratio = out_rate/in_rate must equal L/M with L, M <= 4096 (else LRC_ERR_UNSUPPORTED).
 *     Streaming-causal definition (DESIGN.md; libsamplerate parity is UNPINNED):
 *         y[m] = sum_j h[(mM mod L) + jL] * x[floor(mM/L) - j],  x[<0] = 0.
 *     State (input history + output phase) is carried per channel across process() calls.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_resampler lrc_resampler;
int    lrc_resampler_create(lrc_ctx *ctx, double ratio, size_t n_ch, size_t max_chunk, lrc_resampler **rs);
int    lrc_resampler_destroy(lrc_resampler *rs);
int    lrc_resampler_reset(lrc_resampler *rs);
int    lrc_resampler_get_taps(const lrc_resampler *rs, double *h_taps, size_t cap, size_t *ntaps, int *L, int *M);
/* outputs produced by the next process() of n_in frames (same for every channel) */
size_t lrc_resampler_next_out_len(const lrc_resampler *rs, size_t n_in);
int    lrc_resampler_process(lrc_resampler *rs, const float *d_in, size_t n_in, size_t in_stride,
                             float *d_out, size_t out_stride, size_t *n_out, void *stream);
/* host-buffer variant with the calling convention of src_process (samplerate.rs:66-84): channel-major
 * host input, caller-allocated host output of `out_cap` frames per channel; synchronous */
int    lrc_resampler_process_host(lrc_resampler *rs, const float *h_in, size_t n_in, float *h_out,
                                  size_t out_cap, size_t *n_out);

/* ------------------------------------------------------------------------------------------------
 * (1)+(2)+(4a)+(4b) as one streaming receiver (BASELINE config 3): rtlsdr u8 IQ chunks -> FIR(ntaps)/decim ->
 *     quadrature discriminator -> resampler(ratio) -> f32 audio, n_ch independent channels, state carried across
 *     pushes so the audio stream does not depend on how the input is chunked.  Replaces the chain
 *     rtlsdr::data_to_samples (rtlsdr.rs:160-162) -> dsputils::convolve (dsputils.rs:30-32) + decimation ->
 *     discriminator -> samplerate::resample (samplerate.rs:59-87) of a KPN FM-receiver graph.
 *     The BASELINE shape (64 taps / 10, ratio 1/5) runs as ONE kernel per push (HBM sees 2 B/sample in and the audio
 *     out, nothing else); any other shape runs the three stand-alone stages behind the same interface.
 *     Each stage's arithmetic is the stand-alone stage's, so the tolerances of (2), (4a), (4b) apply.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_fmrx lrc_fmrx;
int    lrc_fmrx_create(lrc_ctx *ctx, const float *h_taps, int ntaps, int decim, double ratio, size_t n_ch,
                       size_t max_chunk, lrc_fmrx **rx);
int    lrc_fmrx_destroy(lrc_fmrx *rx);
int    lrc_fmrx_reset(lrc_fmrx *rx);
int    lrc_fmrx_is_fused(const lrc_fmrx *rx);
/* audio frames per channel the next push of n samples will produce */
size_t lrc_fmrx_next_out_len(const lrc_fmrx *rx, size_t n);
/* n new samples per channel (u8 I,Q interleaved; channel c at d_iq + 2*c*chunk_stride bytes); writes the audio that
 * became computable to d_audio (+ c*out_stride) and its per-channel count to *n_out (host arithmetic, no readback) */
int    lrc_fmrx_push(lrc_fmrx *rx, const uint8_t *d_iq, size_t n, size_t chunk_stride, float *d_audio,
                     size_t out_stride, size_t *n_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (5) OOK packet decode, bit-exact.   Replaces, per stream, the chain of src/ratpak.rs:60-111:
 *     rtlsdr::data_to_samples (rtlsdr.rs:160) -> |x| (ratpak.rs:64-68) -> bitfount::trigger
 *     (bitfount.rs:36-85, 512-sample blocks) -> bitfount::discretize (:87-96) -> kpn::rle (kpn.rs:17-29)
 *     -> kpn::dle (:32-38) -> the two pulse-pair matchers (ratpak.rs:88-97) -> kpn::shaper_optional
 *     36 / 24 (kpn.rs:266-275).  Input: n_streams finite captures of n_blocks*1024 bytes of u8 IQ,
 *     stream s at d_iq + s*stream_stride_bytes; every stream starts from the reference's initial
 *     state.  Output: packets of proto A (36 bits) and proto B (24 bits), one byte per bit.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_ook lrc_ook;
typedef struct {
    uint32_t stream;       /* stream index */
    uint32_t proto;        /* 0 = A (36 bits), 1 = B (24 bits) */
    uint32_t seq;          /* packet ordinal within (stream, proto) */
    uint32_t nbits;        /* 36 or 24 */
    uint8_t  bits[40];     /* MSB-first bit values 0/1, as kpn::b2d consumes them (kpn.rs:111-113) */
} lrc_ook_packet;
int lrc_ook_create(lrc_ctx *ctx, size_t n_streams, size_t n_blocks, unsigned sample_rate,
                   size_t max_runs_per_stream, size_t max_packets_per_stream, lrc_ook **ook);
int lrc_ook_destroy(lrc_ook *ook);
/* runs the whole chain on the device (asynchronous) */
int lrc_ook_decode(lrc_ook *ook, const uint8_t *d_iq, size_t stream_stride_bytes, void *stream);
/* synchronises, copies the packets back ordered by (stream, proto, seq); LRC_ERR_CAPACITY if a stream
 * overflowed max_runs/max_packets or cap is too small (then *n_packets = required) */
int lrc_ook_fetch_packets(lrc_ook *ook, lrc_ook_packet *h_packets, size_t cap, size_t *n_packets);
/* intermediate products for stage-by-stage parity (device pointers owned by the plan):
 * block sums f32 [n_streams][n_blocks]; per-stream run counts u32 [n_streams]; runs as
 * (value<<31 | length) u32 [n_streams][max_runs] */
int lrc_ook_debug_ptrs(lrc_ook *ook, const float **d_block_sums, const uint32_t **d_run_counts,
                       const uint32_t **d_runs, const uint32_t **d_n_bits);
/* Streaming form of the same chain, for a live receiver that delivers the capture a few blocks at a time.
 * Every stream carries the state the reference's blocks hold between two messages (trigger threshold and counter,
 * the burst still being collected, the open run of rle, the matchers' pending pulse and partial packet), so the
 * packets emitted after any push are exactly those the reference emits on the concatenation of all pushes so far,
 * whatever the push sizes.  The blocks of a burst still open at the end of a push are kept in a per-stream carry of
 * max_carry_blocks blocks (0 = the trigger's OOM guard + 1 = 50 001 blocks, 51 MB per stream: exact for every
 * input); a smaller carry is a memory choice, and a burst that outgrows it is reported (LRC_ERR_CAPACITY naming the
 * stream, no packet from it), never decoded wrongly.  LRC_OOK_TEST_GUARD_BLOCKS is read at create, as for lrc_ook. */
typedef struct lrc_ook_stream lrc_ook_stream;
int lrc_ook_stream_create(lrc_ctx *ctx, size_t n_streams, size_t max_push_blocks, unsigned sample_rate,
                          size_t max_carry_blocks, size_t max_runs_per_push, size_t max_packets_per_fetch,
                          lrc_ook_stream **st);
int lrc_ook_stream_destroy(lrc_ook_stream *st);
/* back to the reference's initial state (every stream; packet sequence numbers restart at 0) */
int lrc_ook_stream_reset(lrc_ook_stream *st);
/* n_blocks (1..max_push_blocks, may differ from push to push) new blocks per stream, stream s at
 * d_iq + s*stream_stride_bytes; 16-byte aligned like lrc_ook_decode.  Asynchronous. */
int lrc_ook_stream_push(lrc_ook_stream *st, const uint8_t *d_iq, size_t n_blocks, size_t stream_stride_bytes,
                        void *stream);
/* synchronises; the packets completed since the previous fetch, ordered by (stream, proto, seq), seq counting from
 * create/reset.  LRC_ERR_CAPACITY if cap is too small (then *n_packets = required and nothing is consumed), and
 * naming the stream if one overflowed max_carry_blocks, max_runs_per_push, max_packets_per_fetch or its bursts per
 * push: then no packet is returned and every push and fetch fails until lrc_ook_stream_reset. */
int lrc_ook_stream_fetch_packets(lrc_ook_stream *st, lrc_ook_packet *h_packets, size_t cap, size_t *n_packets);
/* stage-by-stage parity for the last push, as lrc_ook_debug_ptrs: its block sums [n_streams][n_blocks of that push],
 * the number of runs it completed, those runs (value<<31 | length, the first one including its length before the
 * push), and the bits it emitted; bit positions count from the start of the push */
int lrc_ook_stream_debug_ptrs(lrc_ook_stream *st, const float **d_block_sums, const uint32_t **d_run_counts,
                              const uint32_t **d_runs, const uint32_t **d_n_bits);
/* kpn::eat (kpn.rs:116-124): split MSB-first bit fields; pure host helper for the wrappers */
int lrc_eat(const uint8_t *bits, size_t nbits, const size_t *widths, size_t n_widths, size_t *out);
/* |i2f(b0) + j*i2f(b1)| for all 65536 byte pairs computed ON THE DEVICE with the envelope routine the
 * OOK kernels use (exhaustive parity hook); d_table is 65536 f32, index b0*256 + b1 */
int lrc_ook_envelope_table(lrc_ctx *ctx, float *d_table, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (e) Output gather across GPUs over NVLink (SURVEY 8e).  The reference moves results between blocks by
 *     sending the Vec down an mpsc channel (src/kpn/src/kpn.rs:127-131, e.g. `v.send(x).unwrap()` kpn.rs:27);
 *     when the producer blocks are sharded over several GPUs this is that send: every rank pushes its
 *     output block into block `rank` of every peer's receive buffer with the copy engines (no SMs, no
 *     collective, overlaps the next kernel).  One process per GPU: exchange lrc_gather_export() blobs
 *     (any host transport, e.g. torch.distributed all_gather_object) and lrc_gather_connect(); several
 *     contexts in ONE process (kpn thread-per-block graphs): lrc_gather_connect_local().
 *     Receive buffer of a slot: `world` blocks, block r at  *d_ptr + r * *block_stride  (lrc_gather_buffer).
 *     SPMD contract: every rank pushes a given slot the same number of times; before a slot is pushed again
 *     its readers must be done with it (the application's flow control -- `slots` steps of slack or a
 *     consumer-side handshake; the kpn wrapper uses one slot per in-flight batch).
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrc_gather lrc_gather;
int    lrc_gather_create(lrc_ctx *ctx, int rank, int world, size_t bytes_per_rank, int slots, lrc_gather **g);
/* the same gather into HOST memory shared by the ranks of one node: POSIX shared memory `shm_name` ("/name"), created by rank
 * `root` and opened by the others (they retry for up to 30 s), page-locked and mapped by every rank.  A push is one D2H copy over
 * the pushing GPU's own PCIe link plus the flag write; lrc_gather_wait on the root orders a stream behind the arrival flags;
 * lrc_gather_buffer returns a HOST pointer.  For graphs whose consumer block runs on the CPU (the reference's vidsink / psdpng):
 * no GPU's HBM or NVLink port sees another rank's rows (inbound peer writes cost a bandwidth-bound kernel 4.7 % at 8 GPUs).
 * export / connect / set_root do not apply. */
int    lrc_gather_create_host(lrc_ctx *ctx, int rank, int world, size_t bytes_per_rank, int slots, const char *shm_name,
                              int root, lrc_gather **g);
int    lrc_gather_destroy(lrc_gather *g);
/* root = -1 (default): every rank receives every rank's block (all-gather); root = r: only rank r receives (gather) --
 * pushes then send one block per rank instead of world-1, and lrc_gather_wait is a no-op on the other ranks;
 * root = LRC_GATHER_ROTATE: the receiver rotates, push n (1-based) of slot s lands on rank (n - 1 + s) % world.
 * Same value on every rank, before the first push. */
#define LRC_GATHER_ALL (-1)
#define LRC_GATHER_ROTATE (-2)
int    lrc_gather_set_root(lrc_gather *g, int root);
size_t lrc_gather_handle_bytes(void);
int    lrc_gather_export(lrc_gather *g, void *h_handle, size_t cap);
/* h_handles: `world` handles of lrc_gather_handle_bytes() each, ordered by rank (own entry ignored) */
int    lrc_gather_connect(lrc_gather *g, const void *h_handles);
int    lrc_gather_connect_local(lrc_gather *g, lrc_gather *const *all /* world objects, all[r]->rank == r */);
/* after the work queued on `stream` (the producer of d_src) completes, copy bytes_per_rank bytes from d_src to
 * every rank's receive slot and raise their arrival flags; asynchronous */
int    lrc_gather_push(lrc_gather *g, int slot, const void *d_src, void *stream);
/* order `stream` behind this rank's previous push from `slot` having READ its source buffer (so the buffer
 * may be overwritten by work queued on `stream` afterwards) */
int    lrc_gather_wait_sent(lrc_gather *g, int slot, void *stream);
/* order `stream` behind the ARRIVAL of every rank's latest push into this rank's `slot` */
int    lrc_gather_wait(lrc_gather *g, int slot, void *stream);
/* host gather only: block the calling CPU thread until every rank's latest push into `slot` has arrived, at most timeout_ms
 * (LRC_ERR_CAPACITY on timeout) -- for consumer blocks that run on the CPU and have no stream to order behind the flags */
int    lrc_gather_wait_host(lrc_gather *g, int slot, unsigned timeout_ms);
int    lrc_gather_buffer(lrc_gather *g, int slot, void **d_ptr, size_t *block_stride);

#ifdef __cplusplus
}
#endif
#endif /* LIBREDIO_CUDA_H */
