// gpu_blocks.hpp -- GPU blocks with the reference's block signatures, over the C ABI of
// include/libredio_cuda.h.  Each block keeps the shape `fn(Receiver<In>, Sender<Out>, params...)`
// (src/kpn/src/kpn.rs:127-131) so it drops into an existing Kahn-process-network graph in place of the
// CPU block it names; internally it batches whatever has already queued up on its input port (and, for
// the *_multi blocks, many channels) into pinned, double-buffered host slots before touching the device.
//
//   reference block                               GPU block here
//   rtlsdr::data_to_samples   rtlsdr.rs:160       kpn_gpu::data_to_samples
//   kissfft::fft              kissfft.rs:18-31    kpn_gpu::fft
//   samplerate::resample      samplerate.rs:59    kpn_gpu::resample
//   dsputils::convolve (+/D)  dsputils.rs:30      kpn_gpu::fir_decimate, fir_decimate_multi (channel ring)
//   kiss_fastfir (streaming)  kiss_fastfir.c:228  kpn_gpu::fast_fir_multi (channel ring, long FIR by overlap-save)
//   (north-star) discriminator                    kpn_gpu::fm_demod
//   (north-star) FIR->FFT->|X|^2 chain            kpn_gpu::chain_psd
//   (north-star) config-3 FM receiver, N channels  kpn_gpu::fm_receiver_multi (lrc_fmrx: one kernel per batch)
//   trigger..shaper_optional  ratpak.rs:60-111    kpn_gpu::ook_decode, kpn_gpu::ook_decode_stream (live, message by message)
//
// Errors: a non-zero status of the C ABI is thrown as std::runtime_error -- the analogue of the
// reference's `panic!(src_strerror(..))` (samplerate.rs:77-83); spawn() lets the thread die, which drops
// the block's ports and tears the graph down like any other panic.  There is no CPU fallback.
#pragma once
#include <cuda_runtime_api.h>
#include <algorithm>
#include <complex>
#include <cstdint>
#include <cstring>
#include <string>
#include "../include/libredio_cuda.h"
#include "kpn.hpp"

namespace kpn_gpu {

using cf32 = std::complex<float>;
using kpn::Receiver;
using kpn::Sender;

inline void check(int rc, const char *what)
{
    if (rc != LRC_OK) throw std::runtime_error(std::string(what) + ": " + lrc_strerror(rc) + " [" + lrc_last_error() + "]");
}
inline void cuda_check(cudaError_t e, const char *what)
{
    if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

// one per GPU; blocks sharing a Gpu share its context (their own plans carry their own state)
struct Gpu {
    lrc_ctx *ctx = nullptr;
    int device;
    explicit Gpu(int dev = 0) : device(dev) { check(lrc_ctx_create(dev, &ctx), "lrc_ctx_create"); }
    Gpu(const Gpu &) = delete;
    ~Gpu() { lrc_ctx_destroy(ctx); }
    void bind() const { cuda_check(cudaSetDevice(device), "cudaSetDevice"); }
};

// pinned host + device buffer pair with its own stream: one slot of a ring
struct Slot {
    void *h = nullptr, *d = nullptr;
    size_t bytes = 0;
    void reserve(const Gpu &g, size_t n)
    {
        if (n <= bytes) return;
        release(g);
        check(lrc_host_alloc(g.ctx, n, &h), "lrc_host_alloc");
        cuda_check(cudaMalloc(&d, n), "cudaMalloc");
        bytes = n;
    }
    void release(const Gpu &g)
    {
        if (h) lrc_host_free(g.ctx, h);
        if (d) cudaFree(d);
        h = d = nullptr; bytes = 0;
    }
};

struct Stream {
    cudaStream_t s = nullptr;
    Stream() { cuda_check(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "cudaStreamCreate"); }
    ~Stream() { if (s) cudaStreamDestroy(s); }
    void sync() const { cuda_check(cudaStreamSynchronize(s), "cudaStreamSynchronize"); }
};

// ---- rtlsdr::data_to_samples ------------------------------------------------------------------------
inline void data_to_samples(Gpu &g, Receiver<std::vector<uint8_t>> u, Sender<std::vector<cf32>> v)
{
    g.bind();
    Stream st; Slot in, out;
    for (;;) {
        std::vector<uint8_t> data = u.recv();
        // data[0..].chunks(2) ... i[1]: an odd length indexes out of bounds and panics (rtlsdr.rs:161)
        in.reserve(g, data.size() + 16); out.reserve(g, data.size() * 4 + 16);
        std::memcpy(in.h, data.data(), data.size());
        cuda_check(cudaMemcpyAsync(in.d, in.h, data.size(), cudaMemcpyHostToDevice, st.s), "H2D");
        check(lrc_unpack_u8_cf32(g.ctx, (const uint8_t *)in.d, data.size(), (float *)out.d, st.s), "lrc_unpack_u8_cf32");
        cuda_check(cudaMemcpyAsync(out.h, out.d, data.size() * 4, cudaMemcpyDeviceToHost, st.s), "D2H");
        st.sync();
        const cf32 *p = (const cf32 *)out.h;
        v.send(std::vector<cf32>(p, p + data.size() / 2));
    }
}

// ---- kissfft::fft(pin, cout, block_size, inv) ---------------------------------------------------------
// One frame per message like the reference, but every frame already waiting on `pin` (up to max_batch) goes
// to the device in ONE launch.
inline void fft(Gpu &g, Receiver<std::vector<cf32>> pin, Sender<std::vector<cf32>> cout, uint32_t block_size,
                uint32_t inv, size_t max_batch = 4096)
{
    g.bind();
    lrc_fft *plan = nullptr;
    check(lrc_fft_create(g.ctx, (int)block_size, (int)inv, &plan), "lrc_fft_create");     // kiss_fft_alloc once, :19
    Stream st; Slot buf;
    const size_t fb = (size_t)block_size * sizeof(cf32);
    try {
        for (;;) {
            std::vector<std::vector<cf32>> frames;
            frames.push_back(pin.recv());
            while (frames.size() < max_batch) {
                auto more = pin.try_recv();
                if (!more) break;
                frames.push_back(std::move(*more));
            }
            buf.reserve(g, frames.size() * fb);
            for (size_t k = 0; k < frames.size(); ++k) {
                if (frames[k].size() != block_size)                    // assert!(din.len() == block_size) :24
                    throw std::logic_error("assertion failed: din.len() == block_size");
                std::memcpy((char *)buf.h + k * fb, frames[k].data(), fb);
            }
            cuda_check(cudaMemcpyAsync(buf.d, buf.h, frames.size() * fb, cudaMemcpyHostToDevice, st.s), "H2D");
            check(lrc_fft_run(plan, (const float *)buf.d, (float *)buf.d, frames.size(), st.s), "lrc_fft_run");
            cuda_check(cudaMemcpyAsync(buf.h, buf.d, frames.size() * fb, cudaMemcpyDeviceToHost, st.s), "D2H");
            st.sync();
            for (size_t k = 0; k < frames.size(); ++k) {
                std::memcpy(frames[k].data(), (char *)buf.h + k * fb, fb);
                cout.send(std::move(frames[k]));
            }
        }
    } catch (...) { lrc_fft_destroy(plan); buf.release(g); throw; }
}

// ---- FIR + decimate, one channel, seam-exact across messages -----------------------------------------
inline void fir_decimate(Gpu &g, Receiver<std::vector<cf32>> u, Sender<std::vector<cf32>> v, std::vector<float> taps,
                         size_t decim, size_t max_chunk = 1 << 20)
{
    g.bind();
    lrc_fir *fir = nullptr; lrc_fir_stream *fs = nullptr;
    check(lrc_fir_create(g.ctx, taps.data(), (int)taps.size(), (int)decim, &fir), "lrc_fir_create");
    check(lrc_fir_stream_create(fir, 1, max_chunk, 0, &fs), "lrc_fir_stream_create");
    Stream st; Slot in, out;
    try {
        for (;;) {
            std::vector<cf32> x = u.recv();
            if (x.size() > max_chunk) throw std::length_error("fir_decimate: chunk longer than max_chunk");
            const size_t cap = (taps.size() + x.size()) / decim + 2;
            in.reserve(g, x.size() * sizeof(cf32) + 16); out.reserve(g, cap * sizeof(cf32));
            std::memcpy(in.h, x.data(), x.size() * sizeof(cf32));
            cuda_check(cudaMemcpyAsync(in.d, in.h, x.size() * sizeof(cf32), cudaMemcpyHostToDevice, st.s), "H2D");
            size_t n_out = 0;
            check(lrc_fir_stream_push(fs, in.d, x.size(), x.size(), (float *)out.d, cap, &n_out, st.s), "lrc_fir_stream_push");
            cuda_check(cudaMemcpyAsync(out.h, out.d, n_out * sizeof(cf32), cudaMemcpyDeviceToHost, st.s), "D2H");
            st.sync();
            const cf32 *p = (const cf32 *)out.h;
            v.send(std::vector<cf32>(p, p + n_out));
        }
    } catch (...) { lrc_fir_stream_destroy(fs); lrc_fir_destroy(fir); in.release(g); out.release(g); throw; }
}

// ---- FIR + decimate over MANY channels: the channel ring --------------------------------------------
// One chunk (chunk_len samples) is taken from every channel's port, packed channel-major into a pinned
// slot, and the whole batch goes through ONE kernel launch.  Two slots alternate: while slot A's batch is
// on the device (H2D -> kernel -> D2H on the ring stream) the block is already packing slot B from the
// ports, and A's outputs are scattered to the senders when the block comes back to A.
inline void fir_decimate_multi(Gpu &g, std::vector<Receiver<std::vector<cf32>>> u, std::vector<Sender<std::vector<cf32>>> v,
                               std::vector<float> taps, size_t decim, size_t chunk_len)
{
    g.bind();
    const size_t n_ch = u.size();
    if (v.size() != n_ch || n_ch == 0) throw std::invalid_argument("fir_decimate_multi: port count mismatch");
    lrc_fir *fir = nullptr; lrc_fir_stream *fs = nullptr;
    check(lrc_fir_create(g.ctx, taps.data(), (int)taps.size(), (int)decim, &fir), "lrc_fir_create");
    check(lrc_fir_stream_create(fir, n_ch, chunk_len, 0, &fs), "lrc_fir_stream_create");
    Stream st;
    const size_t cap = (taps.size() + chunk_len) / decim + 2;
    struct RingSlot { Slot in, out; cudaEvent_t done = nullptr; size_t n_out = 0; bool busy = false; } ring[2];
    for (auto &r : ring) {
        r.in.reserve(g, n_ch * chunk_len * sizeof(cf32)); r.out.reserve(g, n_ch * cap * sizeof(cf32));
        cuda_check(cudaEventCreateWithFlags(&r.done, cudaEventDisableTiming), "cudaEventCreate");
    }
    auto drain = [&](RingSlot &r) {
        if (!r.busy) return;
        cuda_check(cudaEventSynchronize(r.done), "cudaEventSynchronize");
        const cf32 *p = (const cf32 *)r.out.h;
        for (size_t c = 0; c < n_ch; ++c) v[c].send(std::vector<cf32>(p + c * cap, p + c * cap + r.n_out));
        r.busy = false;
    };
    try {
        for (size_t it = 0;; ++it) {
            RingSlot &r = ring[it & 1];
            drain(r);                                          // slot reuse: its previous batch must be out
            for (size_t c = 0; c < n_ch; ++c) {
                std::vector<cf32> x = u[c].recv();
                if (x.size() != chunk_len) throw std::length_error("fir_decimate_multi: chunk length != chunk_len");
                std::memcpy((cf32 *)r.in.h + c * chunk_len, x.data(), chunk_len * sizeof(cf32));
            }
            cuda_check(cudaMemcpyAsync(r.in.d, r.in.h, n_ch * chunk_len * sizeof(cf32), cudaMemcpyHostToDevice, st.s), "H2D");
            check(lrc_fir_stream_push(fs, r.in.d, chunk_len, chunk_len, (float *)r.out.d, cap, &r.n_out, st.s),
                  "lrc_fir_stream_push");
            cuda_check(cudaMemcpyAsync(r.out.h, r.out.d, n_ch * cap * sizeof(cf32), cudaMemcpyDeviceToHost, st.s), "D2H");
            cuda_check(cudaEventRecord(r.done, st.s), "cudaEventRecord");
            r.busy = true;
            drain(ring[(it + 1) & 1]);                         // hand out the batch submitted one step ago
        }
    } catch (...) {
        try { drain(ring[0]); drain(ring[1]); } catch (...) {}
        lrc_fir_stream_destroy(fs); lrc_fir_destroy(fir);
        for (auto &r : ring) { r.in.release(g); r.out.release(g); if (r.done) cudaEventDestroy(r.done); }
        throw;
    }
}

// ---- long FIR by overlap-save over MANY channels: kiss_fastfir with a carried offset ----------------------
// The channel ring of fir_decimate_multi over lrc_fastfir_stream: one chunk (chunk_len samples) from every channel's port
// per batch, one push per batch.  Outputs come as whole compute blocks complete (a batch that completes none sends
// nothing); concatenated per channel they are a prefix of lrc_fastfir_run over the channel's whole input.  The block never
// flushes: the reference's ports never end (a closed port tears the graph down).
inline void fast_fir_multi(Gpu &g, std::vector<Receiver<std::vector<cf32>>> u, std::vector<Sender<std::vector<cf32>>> v,
                           std::vector<cf32> h, size_t nfft, size_t chunk_len)
{
    g.bind();
    const size_t n_ch = u.size();
    if (v.size() != n_ch || n_ch == 0) throw std::invalid_argument("fast_fir_multi: port count mismatch");
    lrc_fastfir *ff = nullptr; lrc_fastfir_stream *fs = nullptr;
    check(lrc_fastfir_create(g.ctx, (const float *)h.data(), h.size(), nfft, &ff), "lrc_fastfir_create");
    check(lrc_fastfir_stream_create(ff, n_ch, &fs), "lrc_fastfir_stream_create");
    Stream st;
    const size_t cap = chunk_len + 16384;                  // the history is shorter than one compute block (<= 16384)
    struct RingSlot { Slot in, out; cudaEvent_t done = nullptr; size_t n_out = 0; bool busy = false; } ring[2];
    for (auto &r : ring) {
        r.in.reserve(g, n_ch * chunk_len * sizeof(cf32)); r.out.reserve(g, n_ch * cap * sizeof(cf32));
        cuda_check(cudaEventCreateWithFlags(&r.done, cudaEventDisableTiming), "cudaEventCreate");
    }
    auto drain = [&](RingSlot &r) {
        if (!r.busy) return;
        cuda_check(cudaEventSynchronize(r.done), "cudaEventSynchronize");
        const cf32 *p = (const cf32 *)r.out.h;
        if (r.n_out)
            for (size_t c = 0; c < n_ch; ++c) v[c].send(std::vector<cf32>(p + c * cap, p + c * cap + r.n_out));
        r.busy = false;
    };
    try {
        for (size_t it = 0;; ++it) {
            RingSlot &r = ring[it & 1];
            drain(r);                                          // slot reuse: its previous batch must be out
            for (size_t c = 0; c < n_ch; ++c) {
                std::vector<cf32> x = u[c].recv();
                if (x.size() != chunk_len) throw std::length_error("fast_fir_multi: chunk length != chunk_len");
                std::memcpy((cf32 *)r.in.h + c * chunk_len, x.data(), chunk_len * sizeof(cf32));
            }
            cuda_check(cudaMemcpyAsync(r.in.d, r.in.h, n_ch * chunk_len * sizeof(cf32), cudaMemcpyHostToDevice, st.s), "H2D");
            check(lrc_fastfir_stream_push(fs, (const float *)r.in.d, chunk_len, chunk_len, (float *)r.out.d, cap, 0, &r.n_out,
                                          st.s), "lrc_fastfir_stream_push");
            if (r.n_out)
                cuda_check(cudaMemcpy2DAsync(r.out.h, cap * sizeof(cf32), r.out.d, cap * sizeof(cf32), r.n_out * sizeof(cf32),
                                             n_ch, cudaMemcpyDeviceToHost, st.s), "D2H");
            cuda_check(cudaEventRecord(r.done, st.s), "cudaEventRecord");
            r.busy = true;
            drain(ring[(it + 1) & 1]);                         // hand out the batch submitted one step ago
        }
    } catch (...) {
        try { drain(ring[0]); drain(ring[1]); } catch (...) {}
        lrc_fastfir_stream_destroy(fs); lrc_fastfir_destroy(ff);
        for (auto &r : ring) { r.in.release(g); r.out.release(g); if (r.done) cudaEventDestroy(r.done); }
        throw;
    }
}

// ---- quadrature FM discriminator ----------------------------------------------------------------------
inline void fm_demod(Gpu &g, Receiver<std::vector<cf32>> u, Sender<std::vector<float>> v)
{
    g.bind();
    Stream st; Slot in, out;
    float *d_state = nullptr;
    cuda_check(cudaMalloc((void **)&d_state, sizeof(cf32)), "cudaMalloc");
    cuda_check(cudaMemset(d_state, 0, sizeof(cf32)), "cudaMemset");        // x[-1] = 0 at stream start
    try {
        for (;;) {
            std::vector<cf32> x = u.recv();
            in.reserve(g, x.size() * sizeof(cf32) + 16); out.reserve(g, x.size() * sizeof(float) + 16);
            std::memcpy(in.h, x.data(), x.size() * sizeof(cf32));
            cuda_check(cudaMemcpyAsync(in.d, in.h, x.size() * sizeof(cf32), cudaMemcpyHostToDevice, st.s), "H2D");
            check(lrc_fmdemod_run(g.ctx, (const float *)in.d, 1, x.size(), x.size(), d_state, (float *)out.d, x.size(), st.s),
                  "lrc_fmdemod_run");
            cuda_check(cudaMemcpyAsync(out.h, out.d, x.size() * sizeof(float), cudaMemcpyDeviceToHost, st.s), "D2H");
            st.sync();
            const float *p = (const float *)out.h;
            v.send(std::vector<float>(p, p + x.size()));
        }
    } catch (...) { cudaFree(d_state); in.release(g); out.release(g); throw; }
}

// ---- samplerate::resample(din, dout, ratio) -------------------------------------------------------------
inline void resample(Gpu &g, Receiver<std::vector<float>> din, Sender<std::vector<float>> dout, double ratio,
                     size_t max_chunk = 1 << 20)
{
    g.bind();
    lrc_resampler *rs = nullptr;
    check(lrc_resampler_create(g.ctx, ratio, 1, max_chunk, &rs), "lrc_resampler_create");   // src_new(1, 1) :61
    Stream st; Slot in, out;
    try {
        for (;;) {
            std::vector<float> vin = din.recv();
            const size_t lout = (size_t)(ratio * (double)vin.size() + 1.0) + 1;                  // :64
            in.reserve(g, vin.size() * 4 + 16); out.reserve(g, lout * 4);
            std::memcpy(in.h, vin.data(), vin.size() * 4);
            cuda_check(cudaMemcpyAsync(in.d, in.h, vin.size() * 4, cudaMemcpyHostToDevice, st.s), "H2D");
            size_t n_out = 0;
            // a non-zero status here is the reference's panic!(src_strerror(error)) :77-83
            check(lrc_resampler_process(rs, (const float *)in.d, vin.size(), vin.size(), (float *)out.d, lout, &n_out, st.s),
                  "lrc_resampler_process");
            cuda_check(cudaMemcpyAsync(out.h, out.d, n_out * 4, cudaMemcpyDeviceToHost, st.s), "D2H");
            st.sync();
            const float *p = (const float *)out.h;
            dout.send(std::vector<float>(p, p + n_out));                                          // set_len(output_frames_gen) :84
        }
    } catch (...) { lrc_resampler_destroy(rs); in.release(g); out.release(g); throw; }
}

// ---- FM broadcast receiver over MANY channels (BASELINE config 3), device-resident between stages ------
// rtlsdr u8 IQ chunks in, 48 kHz-style audio chunks out:  fused unpack + FIR/decimate (seam-exact stream state) ->
// quadrature discriminator (carried x[-1]) -> rational resampler (carried history), three launches per batch with
// the 1/decim-rate intermediates never leaving the device.  One chunk (chunk_bytes, even) is taken from every
// channel's port and packed channel-major into a pinned slot; two slots alternate like fir_decimate_multi: while
// slot A's batch is on the device the block is already packing slot B, and A's audio is scattered to the senders
// when the block comes back to A.  The reference would wire rtlsdr::data_to_samples -> dsputils::convolve ->
// (discriminator) -> samplerate::resample with one thread and one channel message per stage and chunk.
// The device side is lrc_fmrx: ONE kernel per batch for the BASELINE shape (64 taps / 10, ratio 1/5).
inline void fm_receiver_multi(Gpu &g, std::vector<Receiver<std::vector<uint8_t>>> u, std::vector<Sender<std::vector<float>>> v,
                              std::vector<float> taps, size_t decim, double ratio, size_t chunk_bytes)
{
    g.bind();
    const size_t n_ch = u.size();
    if (v.size() != n_ch || n_ch == 0) throw std::invalid_argument("fm_receiver_multi: port count mismatch");
    if (chunk_bytes == 0 || (chunk_bytes & 1)) throw std::invalid_argument("fm_receiver_multi: chunk_bytes must be even");
    const size_t chunk = chunk_bytes / 2;                                   // samples per channel and batch
    const size_t cap_bb = (taps.size() + chunk) / decim + 2;               // decimated samples a batch can yield
    const size_t cap_au = ((size_t)(ratio * (double)cap_bb + 1.0) + 1 + 3) / 4 * 4;
    lrc_fmrx *rx = nullptr;
    float *d_au = nullptr;
    check(lrc_fmrx_create(g.ctx, taps.data(), (int)taps.size(), (int)decim, ratio, n_ch, chunk, &rx), "lrc_fmrx_create");
    cuda_check(cudaMalloc((void **)&d_au, n_ch * cap_au * sizeof(float)), "cudaMalloc");
    Stream st;
    struct RingSlot { Slot in, out; cudaEvent_t done = nullptr; size_t n_out = 0; bool busy = false; } ring[2];
    for (auto &r : ring) {
        r.in.reserve(g, n_ch * chunk_bytes); r.out.reserve(g, n_ch * cap_au * sizeof(float));
        cuda_check(cudaEventCreateWithFlags(&r.done, cudaEventDisableTiming), "cudaEventCreate");
    }
    auto drain = [&](RingSlot &r) {
        if (!r.busy) return;
        cuda_check(cudaEventSynchronize(r.done), "cudaEventSynchronize");
        const float *p = (const float *)r.out.h;
        if (r.n_out)
            for (size_t c = 0; c < n_ch; ++c) v[c].send(std::vector<float>(p + c * cap_au, p + c * cap_au + r.n_out));
        r.busy = false;
    };
    auto cleanup = [&]() {
        lrc_fmrx_destroy(rx);
        cudaFree(d_au);
        for (auto &r : ring) { r.in.release(g); r.out.release(g); if (r.done) cudaEventDestroy(r.done); }
    };
    try {
        for (size_t it = 0;; ++it) {
            RingSlot &r = ring[it & 1];
            drain(r);                                              // slot reuse: its previous batch must be out
            for (size_t c = 0; c < n_ch; ++c) {
                std::vector<uint8_t> x = u[c].recv();
                if (x.size() != chunk_bytes) throw std::length_error("fm_receiver_multi: chunk length != chunk_bytes");
                std::memcpy((uint8_t *)r.in.h + c * chunk_bytes, x.data(), chunk_bytes);
            }
            cuda_check(cudaMemcpyAsync(r.in.d, r.in.h, n_ch * chunk_bytes, cudaMemcpyHostToDevice, st.s), "H2D");
            size_t n_au = 0;
            check(lrc_fmrx_push(rx, (const uint8_t *)r.in.d, chunk, chunk, d_au, cap_au, &n_au, st.s), "lrc_fmrx_push");
            if (n_au)
                cuda_check(cudaMemcpyAsync(r.out.h, d_au, n_ch * cap_au * sizeof(float), cudaMemcpyDeviceToHost, st.s), "D2H");
            r.n_out = n_au;
            cuda_check(cudaEventRecord(r.done, st.s), "cudaEventRecord");
            r.busy = true;
            drain(ring[(it + 1) & 1]);                             // hand out the batch submitted one step ago
        }
    } catch (...) {
        try { drain(ring[0]); drain(ring[1]); } catch (...) {}
        cleanup();
        throw;
    }
}

// ---- headline chain: cf32 chunks (whole frames' worth) -> rows of |X|^2 -----------------------------------
// Each message must hold a whole number of k_avg-frame rows plus the ntaps-decim tail; one row per output
// message.  The device work goes through the double-buffered host ring of lrc_chain_run_host.
inline void chain_psd(Gpu &g, Receiver<std::vector<cf32>> u, Sender<std::vector<float>> v, std::vector<float> taps,
                      size_t decim, size_t nfft, size_t k_avg)
{
    g.bind();
    lrc_chain *ch = nullptr;
    check(lrc_chain_create(g.ctx, taps.data(), (int)taps.size(), (int)decim, (int)nfft, LRC_WINDOW_HANN, &ch), "lrc_chain_create");
    try {
        for (;;) {
            std::vector<cf32> x = u.recv();
            const size_t rows = lrc_chain_frames(ch, x.size()) / k_avg;
            std::vector<float> out(rows * nfft);
            size_t nr = 0;
            check(lrc_chain_run_host(ch, (const float *)x.data(), x.size(), k_avg, out.data(), &nr), "lrc_chain_run_host");
            for (size_t r = 0; r < nr; ++r) v.send(std::vector<float>(out.begin() + r * nfft, out.begin() + (r + 1) * nfft));
        }
    } catch (...) { lrc_chain_destroy(ch); throw; }
}

// ---- OOK: captures in, decoded packets out -----------------------------------------------------------------
struct OokPacket { uint32_t stream, proto; std::vector<size_t> bits; };

// Every message is one batch of n_streams captures, stream-major, n_blocks*1024 bytes each (the bytes
// rtl_source_cmplx would have delivered 1024 at a time, bitfount.rs:16-34).  Packets come out ordered by
// (stream, proto, sequence) -- per stream exactly what shaper_optional(36) / shaper_optional(24) send.
inline void ook_decode(Gpu &g, Receiver<std::vector<uint8_t>> u, Sender<OokPacket> v, size_t n_streams, size_t n_blocks,
                       unsigned s_rate, size_t max_runs = 1 << 16, size_t max_packets = 256)
{
    g.bind();
    lrc_ook *ook = nullptr;
    check(lrc_ook_create(g.ctx, n_streams, n_blocks, s_rate, max_runs, max_packets, &ook), "lrc_ook_create");
    Stream st; Slot in;
    const size_t bytes = n_streams * n_blocks * 1024;
    std::vector<lrc_ook_packet> pk(n_streams * 2 * max_packets);
    try {
        for (;;) {
            std::vector<uint8_t> cap = u.recv();
            if (cap.size() != bytes) throw std::length_error("ook_decode: batch size != n_streams*n_blocks*1024");
            in.reserve(g, bytes);
            std::memcpy(in.h, cap.data(), bytes);
            cuda_check(cudaMemcpyAsync(in.d, in.h, bytes, cudaMemcpyHostToDevice, st.s), "H2D");
            check(lrc_ook_decode(ook, (const uint8_t *)in.d, n_blocks * 1024, st.s), "lrc_ook_decode");
            size_t n = 0;
            check(lrc_ook_fetch_packets(ook, pk.data(), pk.size(), &n), "lrc_ook_fetch_packets");
            for (size_t k = 0; k < n; ++k) {
                OokPacket p{pk[k].stream, pk[k].proto, {}};
                for (uint32_t i = 0; i < pk[k].nbits; ++i) p.bits.push_back(pk[k].bits[i]);
                v.send(std::move(p));
            }
        }
    } catch (...) { lrc_ook_destroy(ook); in.release(g); throw; }
}

// The streaming form, for a live receiver: every message holds the NEXT k blocks of each of the n_streams streams,
// stream-major (n_streams * k * 1024 bytes), k free to change from message to message.  The state of the reference's
// trigger .. shaper_optional blocks lives on the device between messages, so the packets sent after a message are exactly
// those the reference's per-block threads would have sent on all the bytes so far: a packet that crosses a message
// boundary is not lost.  A message longer than max_push_blocks per stream is pushed in pieces (the result does not depend
// on how the stream is cut).  max_carry_blocks = 0: the exact carry (the trigger's OOM guard + 1 blocks per stream).
inline void ook_decode_stream(Gpu &g, Receiver<std::vector<uint8_t>> u, Sender<OokPacket> v, size_t n_streams, unsigned s_rate,
                              size_t max_push_blocks = 1024, size_t max_carry_blocks = 0, size_t max_runs_per_push = 1 << 16,
                              size_t max_packets_per_fetch = 256)
{
    g.bind();
    lrc_ook_stream *ook = nullptr;
    check(lrc_ook_stream_create(g.ctx, n_streams, max_push_blocks, s_rate, max_carry_blocks, max_runs_per_push,
                                max_packets_per_fetch, &ook), "lrc_ook_stream_create");
    Stream st; Slot in;
    std::vector<lrc_ook_packet> pk(n_streams * 2 * max_packets_per_fetch);
    try {
        for (;;) {
            std::vector<uint8_t> msg = u.recv();
            if (msg.empty() || msg.size() % (n_streams * 1024) != 0)
                throw std::length_error("ook_decode_stream: message size is not n_streams * k * 1024 bytes");
            const size_t k = msg.size() / (n_streams * 1024);
            in.reserve(g, msg.size());
            std::memcpy(in.h, msg.data(), msg.size());
            cuda_check(cudaMemcpyAsync(in.d, in.h, msg.size(), cudaMemcpyHostToDevice, st.s), "H2D");
            for (size_t b = 0; b < k; b += max_push_blocks) {
                const size_t n = std::min(max_push_blocks, k - b);
                check(lrc_ook_stream_push(ook, (const uint8_t *)in.d + b * 1024, n, k * 1024, st.s), "lrc_ook_stream_push");
                size_t np = 0;
                check(lrc_ook_stream_fetch_packets(ook, pk.data(), pk.size(), &np), "lrc_ook_stream_fetch_packets");
                for (size_t q = 0; q < np; ++q) {
                    OokPacket p{pk[q].stream, pk[q].proto, {}};
                    for (uint32_t i = 0; i < pk[q].nbits; ++i) p.bits.push_back(pk[q].bits[i]);
                    v.send(std::move(p));
                }
            }
        }
    } catch (...) { lrc_ook_stream_destroy(ook); in.release(g); throw; }
}

// the packets of ook_decode back onto the reference's two ports: what shaper_optional(36) and shaper_optional(24) send
// towards binconv (ratpak.rs:105-119) -- the bit vector of every protocol-A packet on `a`, of every protocol-B packet on `b`
inline void split_protocols(Receiver<OokPacket> u, Sender<std::vector<size_t>> a, Sender<std::vector<size_t>> b)
{
    for (;;) {
        OokPacket p = u.recv();
        (p.proto == 0 ? a : b).send(std::move(p.bits));
    }
}

}  // namespace kpn_gpu
