//! Raw declarations of `include/libredio_cuda.h`.  Pointers prefixed `d_` are device pointers, `h_` host
//! pointers; every function returns a status (`LRC_OK == 0`), `lrc_last_error()` has the detail text.
#![allow(non_camel_case_types)]
use libc::{c_char, c_double, c_float, c_int, c_uint, c_void, size_t};

pub const LRC_OK: c_int = 0;
pub const LRC_ERR_INVALID: c_int = 1;
pub const LRC_ERR_CUDA: c_int = 2;
pub const LRC_ERR_UNSUPPORTED: c_int = 3;
pub const LRC_ERR_NOMEM: c_int = 4;
pub const LRC_ERR_CAPACITY: c_int = 5;
pub const LRC_ERR_ODD_LENGTH: c_int = 6;
pub const LRC_ERR_LENGTH: c_int = 7;
pub const LRC_WINDOW_NONE: c_int = 0;
pub const LRC_WINDOW_HANN: c_int = 1;

macro_rules! opaque { ($($n:ident),*) => { $( #[repr(C)] pub struct $n { _p: [u8; 0] } )* } }
opaque!(lrc_ctx, lrc_fir, lrc_fir_stream, lrc_fft, lrc_rfft, lrc_psd, lrc_chain, lrc_fastfir, lrc_resampler, lrc_fmrx, lrc_ook,
        lrc_ook_stream, lrc_gather);

#[repr(C)]
#[derive(Clone, Copy)]
pub struct lrc_ook_packet {
    pub stream: u32,
    pub proto: u32,
    pub seq: u32,
    pub nbits: u32,
    pub bits: [u8; 40],
}

extern "C" {
    pub fn lrc_version() -> c_int;
    pub fn lrc_strerror(status: c_int) -> *const c_char;
    pub fn lrc_last_error() -> *const c_char;
    pub fn lrc_ctx_create(device: c_int, ctx: *mut *mut lrc_ctx) -> c_int;
    pub fn lrc_ctx_destroy(ctx: *mut lrc_ctx) -> c_int;
    pub fn lrc_ctx_sync(ctx: *mut lrc_ctx) -> c_int;
    pub fn lrc_ctx_sm_count(ctx: *mut lrc_ctx, n_sm: *mut c_int) -> c_int;
    pub fn lrc_ctx_numa_node(ctx: *mut lrc_ctx, node: *mut c_int, n_nodes: *mut c_int) -> c_int;
    pub fn lrc_ctx_bind_thread(ctx: *mut lrc_ctx, n_cpus: *mut c_int) -> c_int;
    pub fn lrc_host_alloc(ctx: *mut lrc_ctx, bytes: size_t, h_ptr: *mut *mut c_void) -> c_int;
    pub fn lrc_host_free(ctx: *mut lrc_ctx, h_ptr: *mut c_void) -> c_int;
    // device memory, streams and asynchronous copies: what kpn-gpu builds its pinned double-buffered rings from
    pub fn lrc_dev_alloc(ctx: *mut lrc_ctx, bytes: size_t, d_ptr: *mut *mut c_void) -> c_int;
    pub fn lrc_dev_free(ctx: *mut lrc_ctx, d_ptr: *mut c_void) -> c_int;
    pub fn lrc_dev_memset(ctx: *mut lrc_ctx, d_ptr: *mut c_void, value: c_int, bytes: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_stream_create(ctx: *mut lrc_ctx, stream: *mut *mut c_void) -> c_int;
    pub fn lrc_stream_destroy(ctx: *mut lrc_ctx, stream: *mut c_void) -> c_int;
    pub fn lrc_stream_sync(ctx: *mut lrc_ctx, stream: *mut c_void) -> c_int;
    pub fn lrc_event_create(ctx: *mut lrc_ctx, event: *mut *mut c_void) -> c_int;
    pub fn lrc_event_destroy(ctx: *mut lrc_ctx, event: *mut c_void) -> c_int;
    pub fn lrc_event_record(ctx: *mut lrc_ctx, event: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn lrc_event_sync(ctx: *mut lrc_ctx, event: *mut c_void) -> c_int;
    pub fn lrc_copy_h2d_async(ctx: *mut lrc_ctx, d_dst: *mut c_void, h_src: *const c_void, bytes: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_copy_d2h_async(ctx: *mut lrc_ctx, h_dst: *mut c_void, d_src: *const c_void, bytes: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_copy_to_host(ctx: *mut lrc_ctx, h_dst: *mut c_void, d_src: *const c_void, bytes: size_t) -> c_int;

    pub fn lrc_unpack_u8_cf32(ctx: *mut lrc_ctx, d_iq: *const u8, n_bytes: size_t, d_out: *mut c_float, stream: *mut c_void) -> c_int;

    pub fn lrc_fir_create(ctx: *mut lrc_ctx, h_taps: *const c_float, ntaps: c_int, decim: c_int, fir: *mut *mut lrc_fir) -> c_int;
    pub fn lrc_fir_destroy(fir: *mut lrc_fir) -> c_int;
    pub fn lrc_fir_out_len(fir: *const lrc_fir, n_in: size_t) -> size_t;
    pub fn lrc_fir_run_cf32(fir: *mut lrc_fir, d_in: *const c_float, n_ch: size_t, n_in: size_t, in_stride: size_t,
                            d_out: *mut c_float, out_stride: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_fir_run_u8(fir: *mut lrc_fir, d_in: *const u8, n_ch: size_t, n_in: size_t, in_stride: size_t,
                          d_out: *mut c_float, out_stride: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_fir_stream_create(fir: *mut lrc_fir, n_ch: size_t, max_chunk: size_t, input_is_u8: c_int, st: *mut *mut lrc_fir_stream) -> c_int;
    pub fn lrc_fir_stream_destroy(st: *mut lrc_fir_stream) -> c_int;
    pub fn lrc_fir_stream_push(st: *mut lrc_fir_stream, d_chunk: *const c_void, n: size_t, chunk_stride: size_t,
                               d_out: *mut c_float, out_stride: size_t, n_out: *mut size_t, stream: *mut c_void) -> c_int;

    pub fn lrc_fft_create(ctx: *mut lrc_ctx, nfft: c_int, inverse: c_int, fft: *mut *mut lrc_fft) -> c_int;
    pub fn lrc_fft_destroy(fft: *mut lrc_fft) -> c_int;
    pub fn lrc_fft_run(fft: *mut lrc_fft, d_in: *const c_float, d_out: *mut c_float, batch: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_fft_run_host(fft: *mut lrc_fft, h_in: *const c_float, h_out: *mut c_float, n_samples: size_t) -> c_int;
    // kiss_fftr / kiss_fftri (libkissfft/tools/kiss_fftr.c:67-159)
    pub fn lrc_rfft_create(ctx: *mut lrc_ctx, nfft: c_int, inverse: c_int, rfft: *mut *mut lrc_rfft) -> c_int;
    pub fn lrc_rfft_destroy(rfft: *mut lrc_rfft) -> c_int;
    pub fn lrc_rfft_run(rfft: *mut lrc_rfft, d_in: *const c_float, d_out: *mut c_float, batch: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_rfft_run_host(rfft: *mut lrc_rfft, h_in: *const c_float, h_out: *mut c_float, batch: size_t) -> c_int;
    // tools/psdpng.c:120-185 spectrogram rows
    pub fn lrc_psdpng_rows(ctx: *mut lrc_ctx, d_pcm: *const i16, n_samples: size_t, nfft: c_int, navg: c_int, remove_dc: c_int,
                           stereo: c_int, d_rows: *mut c_float, n_rows: *mut size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_psd_create(ctx: *mut lrc_ctx, nfft: c_int, window: c_int, psd: *mut *mut lrc_psd) -> c_int;
    pub fn lrc_psd_set_window(psd: *mut lrc_psd, h_window: *const c_float) -> c_int;
    pub fn lrc_psd_destroy(psd: *mut lrc_psd) -> c_int;
    pub fn lrc_psd_run(psd: *mut lrc_psd, d_in: *const c_float, n_frames: size_t, k_avg: size_t, d_rows: *mut c_float, stream: *mut c_void) -> c_int;

    pub fn lrc_chain_create(ctx: *mut lrc_ctx, h_taps: *const c_float, ntaps: c_int, decim: c_int, nfft: c_int, window: c_int,
                            chain: *mut *mut lrc_chain) -> c_int;
    pub fn lrc_chain_destroy(chain: *mut lrc_chain) -> c_int;
    pub fn lrc_chain_frames(chain: *const lrc_chain, n_in: size_t) -> size_t;
    pub fn lrc_chain_kind(chain: *const lrc_chain) -> c_int;
    pub fn lrc_chain_run(chain: *mut lrc_chain, d_in: *const c_float, n_in: size_t, k_avg: size_t, d_rows: *mut c_float,
                         n_rows: *mut size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_chain_run_u8(chain: *mut lrc_chain, d_iq: *const u8, n_in: size_t, k_avg: size_t, d_rows: *mut c_float,
                            n_rows: *mut size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_chain_run_host(chain: *mut lrc_chain, h_in: *const c_float, n_in: size_t, k_avg: size_t, h_rows: *mut c_float,
                              n_rows: *mut size_t) -> c_int;
    pub fn lrc_chain_run_host_u8(chain: *mut lrc_chain, h_iq: *const u8, n_in: size_t, k_avg: size_t, h_rows: *mut c_float,
                                 n_rows: *mut size_t) -> c_int;

    pub fn lrc_fastfir_create(ctx: *mut lrc_ctx, h_taps_cpx: *const c_float, nh: size_t, nfft: size_t, ff: *mut *mut lrc_fastfir) -> c_int;
    pub fn lrc_fastfir_destroy(ff: *mut lrc_fastfir) -> c_int;
    pub fn lrc_fastfir_nfft(ff: *const lrc_fastfir) -> size_t;
    pub fn lrc_fastfir_out_len(ff: *const lrc_fastfir, n_in: size_t, flush: c_int) -> size_t;
    pub fn lrc_fastfir_run(ff: *mut lrc_fastfir, d_in: *const c_float, n_in: size_t, d_out: *mut c_float, flush: c_int,
                           n_out: *mut size_t, stream: *mut c_void) -> c_int;

    pub fn lrc_fmdemod_run(ctx: *mut lrc_ctx, d_in: *const c_float, n_ch: size_t, n: size_t, in_stride: size_t,
                           d_state: *mut c_float, d_out: *mut c_float, out_stride: size_t, stream: *mut c_void) -> c_int;

    pub fn lrc_resampler_create(ctx: *mut lrc_ctx, ratio: c_double, n_ch: size_t, max_chunk: size_t, rs: *mut *mut lrc_resampler) -> c_int;
    pub fn lrc_resampler_destroy(rs: *mut lrc_resampler) -> c_int;
    pub fn lrc_resampler_reset(rs: *mut lrc_resampler) -> c_int;
    pub fn lrc_resampler_get_taps(rs: *const lrc_resampler, h_taps: *mut c_double, cap: size_t, ntaps: *mut size_t,
                                  l: *mut c_int, m: *mut c_int) -> c_int;
    pub fn lrc_resampler_next_out_len(rs: *const lrc_resampler, n_in: size_t) -> size_t;
    pub fn lrc_resampler_process(rs: *mut lrc_resampler, d_in: *const c_float, n_in: size_t, in_stride: size_t,
                                 d_out: *mut c_float, out_stride: size_t, n_out: *mut size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_resampler_process_host(rs: *mut lrc_resampler, h_in: *const c_float, n_in: size_t, h_out: *mut c_float,
                                      out_cap: size_t, n_out: *mut size_t) -> c_int;

    // BASELINE config 3 as one streaming receiver: u8 IQ -> FIR/decimate -> discriminator -> resampler (one kernel per push
    // for 64 taps / 10, ratio 1/5)
    pub fn lrc_fmrx_create(ctx: *mut lrc_ctx, h_taps: *const c_float, ntaps: c_int, decim: c_int, ratio: c_double, n_ch: size_t,
                           max_chunk: size_t, rx: *mut *mut lrc_fmrx) -> c_int;
    pub fn lrc_fmrx_destroy(rx: *mut lrc_fmrx) -> c_int;
    pub fn lrc_fmrx_reset(rx: *mut lrc_fmrx) -> c_int;
    pub fn lrc_fmrx_is_fused(rx: *const lrc_fmrx) -> c_int;
    pub fn lrc_fmrx_next_out_len(rx: *const lrc_fmrx, n: size_t) -> size_t;
    pub fn lrc_fmrx_push(rx: *mut lrc_fmrx, d_iq: *const u8, n: size_t, chunk_stride: size_t, d_audio: *mut c_float,
                         out_stride: size_t, n_out: *mut size_t, stream: *mut c_void) -> c_int;

    pub fn lrc_ook_create(ctx: *mut lrc_ctx, n_streams: size_t, n_blocks: size_t, sample_rate: c_uint, max_runs: size_t,
                          max_packets: size_t, ook: *mut *mut lrc_ook) -> c_int;
    pub fn lrc_ook_destroy(ook: *mut lrc_ook) -> c_int;
    pub fn lrc_ook_decode(ook: *mut lrc_ook, d_iq: *const u8, stream_stride_bytes: size_t, stream: *mut c_void) -> c_int;
    pub fn lrc_ook_fetch_packets(ook: *mut lrc_ook, h_packets: *mut lrc_ook_packet, cap: size_t, n_packets: *mut size_t) -> c_int;
    pub fn lrc_ook_debug_ptrs(ook: *mut lrc_ook, d_block_sums: *mut *const c_float, d_run_counts: *mut *const u32,
                              d_runs: *mut *const u32, d_n_bits: *mut *const u32) -> c_int;
    pub fn lrc_ook_stream_create(ctx: *mut lrc_ctx, n_streams: size_t, max_push_blocks: size_t, sample_rate: c_uint,
                                 max_carry_blocks: size_t, max_runs_per_push: size_t, max_packets_per_fetch: size_t,
                                 st: *mut *mut lrc_ook_stream) -> c_int;
    pub fn lrc_ook_stream_destroy(st: *mut lrc_ook_stream) -> c_int;
    pub fn lrc_ook_stream_reset(st: *mut lrc_ook_stream) -> c_int;
    pub fn lrc_ook_stream_push(st: *mut lrc_ook_stream, d_iq: *const u8, n_blocks: size_t, stream_stride_bytes: size_t,
                               stream: *mut c_void) -> c_int;
    pub fn lrc_ook_stream_fetch_packets(st: *mut lrc_ook_stream, h_packets: *mut lrc_ook_packet, cap: size_t,
                                        n_packets: *mut size_t) -> c_int;
    pub fn lrc_ook_stream_debug_ptrs(st: *mut lrc_ook_stream, d_block_sums: *mut *const c_float, d_run_counts: *mut *const u32,
                                     d_runs: *mut *const u32, d_n_bits: *mut *const u32) -> c_int;
    pub fn lrc_eat(bits: *const u8, nbits: size_t, widths: *const size_t, n_widths: size_t, out: *mut size_t) -> c_int;
    pub fn lrc_ook_envelope_table(ctx: *mut lrc_ctx, d_table: *mut c_float, stream: *mut c_void) -> c_int;

    // output gather between GPUs (copy engines over NVLink): the `v.send(x)` of kpn.rs:27 when the producer blocks
    // are sharded over several devices
    pub fn lrc_gather_create(ctx: *mut lrc_ctx, rank: c_int, world: c_int, bytes_per_rank: size_t, slots: c_int,
                             g: *mut *mut lrc_gather) -> c_int;
    pub fn lrc_gather_create_host(ctx: *mut lrc_ctx, rank: c_int, world: c_int, bytes_per_rank: size_t, slots: c_int,
                                  shm_name: *const c_char, root: c_int, g: *mut *mut lrc_gather) -> c_int;
    pub fn lrc_gather_destroy(g: *mut lrc_gather) -> c_int;
    pub fn lrc_gather_wait_host(g: *mut lrc_gather, slot: c_int, timeout_ms: c_uint) -> c_int;
    pub fn lrc_gather_set_root(g: *mut lrc_gather, root: c_int) -> c_int;
    pub fn lrc_gather_handle_bytes() -> size_t;
    pub fn lrc_gather_export(g: *mut lrc_gather, h_handle: *mut c_void, cap: size_t) -> c_int;
    pub fn lrc_gather_connect(g: *mut lrc_gather, h_handles: *const c_void) -> c_int;
    pub fn lrc_gather_connect_local(g: *mut lrc_gather, all: *const *mut lrc_gather) -> c_int;
    pub fn lrc_gather_push(g: *mut lrc_gather, slot: c_int, d_src: *const c_void, stream: *mut c_void) -> c_int;
    pub fn lrc_gather_wait_sent(g: *mut lrc_gather, slot: c_int, stream: *mut c_void) -> c_int;
    pub fn lrc_gather_wait(g: *mut lrc_gather, slot: c_int, stream: *mut c_void) -> c_int;
    pub fn lrc_gather_buffer(g: *mut lrc_gather, slot: c_int, d_ptr: *mut *mut c_void, block_stride: *mut size_t) -> c_int;
}
