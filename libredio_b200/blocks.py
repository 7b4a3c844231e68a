"""Host-side mirror of the reference's block interfaces over the C ABI, for tests and bench.py.

One class per reference function; names and argument meaning follow the reference:

    unpack / data_to_samples   rtlsdr::data_to_samples          src/rtlsdr/src/rtlsdr.rs:160-162
    Fir (convolve + decimate)  dsputils::convolve               src/dsputils/src/dsputils.rs:30-32
    Fft (block_size, inv)      kissfft::fft                     src/kissfft/src/kissfft.rs:18-31
    Resampler (ratio)          samplerate::resample             src/samplerate/src/samplerate.rs:59-87
    Ook                        trigger/discretize/rle/dle/...   src/bitfount/src/bitfount.rs:36-96, src/ratpak.rs:60-111
    FastFir                    kiss_fastfir                     libkissfft/tools/kiss_fastfir.c:65-245

torch is used for device memory and streams only.  Errors follow the reference's convention: what would
panic there (odd unpack length, frame length != block_size, closed port) raises here.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import capi
from .capi import check


def _p(t) -> C.c_void_p:
    if t is None:
        return C.c_void_p(None)
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    return C.c_void_p(t.data_ptr())


def _stream() -> C.c_void_p:
    """torch's current stream as a cudaStream_t.  torch reports the legacy default stream as handle 0,
    which the C ABI reads as "use the context's own stream"; pass cudaStreamLegacy (0x1) instead so the
    launch is ordered with the torch ops around it."""
    h = torch.cuda.current_stream().cuda_stream
    return C.c_void_p(h if h else 1)


class Context:
    """One per GPU (one process per GPU under torch.distributed)."""

    def __init__(self, device: int = 0):
        self.lib = capi.load()
        if not torch.cuda.is_available():
            raise RuntimeError("libredio_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = device
        torch.cuda.set_device(device)
        self.h = C.c_void_p()
        check(self.lib.lrc_ctx_create(device, C.byref(self.h)), "lrc_ctx_create")
        n = C.c_int()
        check(self.lib.lrc_ctx_sm_count(self.h, C.byref(n)), "lrc_ctx_sm_count")
        self.sm_count = n.value
        self.tdev = torch.device("cuda", device)
        node, nodes = C.c_int(), C.c_int()
        check(self.lib.lrc_ctx_numa_node(self.h, C.byref(node), C.byref(nodes)), "lrc_ctx_numa_node")
        self.numa_node, self.numa_nodes = node.value, nodes.value
        self._pinned = []

    def sync(self):
        torch.cuda.synchronize(self.device)

    def close(self):
        if self.h:
            for p in self._pinned:
                self.lib.lrc_host_free(self.h, p)
            self._pinned = []
            self.lib.lrc_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def bind_thread(self) -> int:
        """pin the calling thread to the CPUs of the GPU's NUMA node; returns the CPUs bound to (0 = left alone)"""
        n = C.c_int()
        check(self.lib.lrc_ctx_bind_thread(self.h, C.byref(n)), "lrc_ctx_bind_thread")
        return n.value

    def pinned(self, shape, dtype):
        """pinned host tensor from lrc_host_alloc (placed on the GPU's NUMA node); lives until the context closes"""
        if isinstance(shape, int):
            shape = (shape,)
        n = int(np.prod(shape))
        es = torch.empty(0, dtype=dtype).element_size()
        p = C.c_void_p()
        check(self.lib.lrc_host_alloc(self.h, max(n * es, 1), C.byref(p)), "lrc_host_alloc")
        self._pinned.append(p)
        buf = (C.c_char * max(n * es, 1)).from_address(p.value)
        return torch.frombuffer(buf, dtype=dtype, count=n).reshape(shape)


# ---- (1) -------------------------------------------------------------------------------------------
def data_to_samples(ctx: Context, iq: torch.Tensor) -> torch.Tensor:
    """u8 IQ (device, 1-D, even length) -> complex64."""
    assert iq.dtype == torch.uint8 and iq.is_cuda and iq.is_contiguous()
    n = iq.numel()
    out = torch.empty(n // 2 + (n & 1), dtype=torch.complex64, device=iq.device)
    check(ctx.lib.lrc_unpack_u8_cf32(ctx.h, _p(iq), n, _p(out), _stream()), "lrc_unpack_u8_cf32")
    return out


# ---- (2) -------------------------------------------------------------------------------------------
class Fir:
    def __init__(self, ctx: Context, taps, decim: int = 1):
        self.ctx = ctx
        self.taps = np.ascontiguousarray(taps, dtype=np.float32)
        self.decim = int(decim)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_fir_create(ctx.h, _p(self.taps), self.taps.size, self.decim, C.byref(self.h)), "lrc_fir_create")

    def out_len(self, n_in: int) -> int:
        return int(self.ctx.lib.lrc_fir_out_len(self.h, n_in))

    def run(self, x: torch.Tensor) -> torch.Tensor:
        """x: complex64 [n] or [n_ch, n] -> [.., n_out]"""
        assert x.dtype == torch.complex64 and x.is_cuda and x.is_contiguous()
        x2 = x.reshape(-1, x.shape[-1])
        n_ch, n = x2.shape
        no = self.out_len(n)
        out = torch.empty((n_ch, no), dtype=torch.complex64, device=x.device)
        check(self.ctx.lib.lrc_fir_run_cf32(self.h, _p(x2), n_ch, n, n, _p(out), max(no, 1), _stream()), "lrc_fir_run_cf32")
        return out.reshape(*x.shape[:-1], no)

    def run_u8(self, iq: torch.Tensor) -> torch.Tensor:
        """iq: uint8 [2n] or [n_ch, 2n] -> complex64 [.., n_out] (fused unpack + FIR)"""
        assert iq.dtype == torch.uint8 and iq.is_cuda and iq.is_contiguous() and iq.shape[-1] % 2 == 0
        q2 = iq.reshape(-1, iq.shape[-1])
        n_ch, nb = q2.shape
        n = nb // 2
        no = self.out_len(n)
        out = torch.empty((n_ch, no), dtype=torch.complex64, device=iq.device)
        check(self.ctx.lib.lrc_fir_run_u8(self.h, _p(q2), n_ch, n, n, _p(out), max(no, 1), _stream()), "lrc_fir_run_u8")
        return out.reshape(*iq.shape[:-1], no)

    def close(self):
        if self.h:
            self.ctx.lib.lrc_fir_destroy(self.h)
            self.h = C.c_void_p()


class FirStream:
    """Seam-exact streaming FIR+decimate over n_ch channels."""

    def __init__(self, fir: Fir, n_ch: int, max_chunk: int, u8: bool = False):
        self.fir, self.n_ch, self.max_chunk, self.u8 = fir, n_ch, max_chunk, u8
        self.h = C.c_void_p()
        check(fir.ctx.lib.lrc_fir_stream_create(fir.h, n_ch, max_chunk, int(u8), C.byref(self.h)), "lrc_fir_stream_create")

    def push(self, chunk: torch.Tensor) -> torch.Tensor:
        assert chunk.is_cuda and chunk.is_contiguous()
        c2 = chunk.reshape(self.n_ch, -1)
        n = c2.shape[1] // 2 if self.u8 else c2.shape[1]
        cap = (self.fir.taps.size + n) // self.fir.decim + 2
        out = torch.empty((self.n_ch, cap), dtype=torch.complex64, device=chunk.device)
        no = C.c_size_t()
        check(self.fir.ctx.lib.lrc_fir_stream_push(self.h, _p(c2), n, n, _p(out), cap, C.byref(no), _stream()),
              "lrc_fir_stream_push")
        return out[:, : no.value]

    def close(self):
        if self.h:
            self.fir.ctx.lib.lrc_fir_stream_destroy(self.h)
            self.h = C.c_void_p()


# ---- (3) -------------------------------------------------------------------------------------------
class Fft:
    """kissfft::fft(pin, cout, block_size, inv): frames of exactly block_size samples, unscaled."""

    def __init__(self, ctx: Context, block_size: int, inv: int = 0):
        self.ctx, self.block_size, self.inv = ctx, int(block_size), int(inv)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_fft_create(ctx.h, self.block_size, self.inv, C.byref(self.h)), "lrc_fft_create")

    def run(self, x: torch.Tensor, inplace: bool = False) -> torch.Tensor:
        assert x.dtype == torch.complex64 and x.is_cuda and x.is_contiguous()
        if x.shape[-1] != self.block_size:
            # assert!(din.len() == block_size)  kissfft.rs:24
            raise capi.LrcError(capi.ERR_LENGTH, "Fft.run", f"frame length {x.shape[-1]} != block_size {self.block_size}")
        out = x if inplace else torch.empty_like(x)
        batch = x.numel() // self.block_size
        check(self.ctx.lib.lrc_fft_run(self.h, _p(x), _p(out), batch, _stream()), "lrc_fft_run")
        return out

    def run_host(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.complex64)
        out = np.empty_like(x)
        check(self.ctx.lib.lrc_fft_run_host(self.h, _p(x), _p(out), x.size), "lrc_fft_run_host")
        return out

    def close(self):
        if self.h:
            self.ctx.lib.lrc_fft_destroy(self.h)
            self.h = C.c_void_p()


class Rfft:
    """kiss_fftr / kiss_fftri (tools/kiss_fftr.c:67-159): nfft reals <-> nfft/2+1 bins, unscaled both ways."""

    def __init__(self, ctx: Context, nfft: int, inv: int = 0):
        self.ctx, self.nfft, self.inv = ctx, int(nfft), int(inv)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_rfft_create(ctx.h, self.nfft, self.inv, C.byref(self.h)), "lrc_rfft_create")

    def run(self, x: torch.Tensor) -> torch.Tensor:
        assert x.is_cuda and x.is_contiguous()
        nb = self.nfft // 2 + 1
        if self.inv:
            assert x.dtype == torch.complex64 and x.shape[-1] == nb
            out = torch.empty(x.shape[:-1] + (self.nfft,), dtype=torch.float32, device=x.device)
            batch = x.numel() // nb
        else:
            assert x.dtype == torch.float32 and x.shape[-1] == self.nfft
            out = torch.empty(x.shape[:-1] + (nb,), dtype=torch.complex64, device=x.device)
            batch = x.numel() // self.nfft
        check(self.ctx.lib.lrc_rfft_run(self.h, _p(x), _p(out), batch, _stream()), "lrc_rfft_run")
        return out

    def close(self):
        if self.h:
            self.ctx.lib.lrc_rfft_destroy(self.h)
            self.h = C.c_void_p()


class Psd:
    def __init__(self, ctx: Context, nfft: int, window: int = capi.WINDOW_HANN):
        self.ctx, self.nfft = ctx, int(nfft)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_psd_create(ctx.h, self.nfft, window, C.byref(self.h)), "lrc_psd_create")

    def set_window(self, w):
        w = np.ascontiguousarray(w, dtype=np.float32)
        assert w.size == self.nfft
        check(self.ctx.lib.lrc_psd_set_window(self.h, _p(w)), "lrc_psd_set_window")

    def run(self, x: torch.Tensor, k_avg: int) -> torch.Tensor:
        assert x.dtype == torch.complex64 and x.is_cuda and x.is_contiguous()
        n_frames = x.numel() // self.nfft
        rows = n_frames // k_avg
        out = torch.empty((rows, self.nfft), dtype=torch.float32, device=x.device)
        check(self.ctx.lib.lrc_psd_run(self.h, _p(x), n_frames, k_avg, _p(out), _stream()), "lrc_psd_run")
        return out

    def close(self):
        if self.h:
            self.ctx.lib.lrc_psd_destroy(self.h)
            self.h = C.c_void_p()


def psdpng_rows(ctx: Context, pcm: torch.Tensor, nfft: int = 1024, navg: int = 20, remove_dc: bool = False,
                stereo: bool = False) -> torch.Tensor:
    """tools/psdpng.c transform_signal: int16 PCM -> rows of 10 log10(avg |X|^2 + 1), nfft/2+1 bins each."""
    assert pcm.dtype == torch.int16 and pcm.is_cuda and pcm.is_contiguous()
    n_samples = pcm.numel() // (2 if stereo else 1)
    rows_max = (n_samples // nfft) // navg
    out = torch.empty((max(rows_max, 1), nfft // 2 + 1), dtype=torch.float32, device=pcm.device)
    n_rows = C.c_size_t(0)
    check(ctx.lib.lrc_psdpng_rows(ctx.h, _p(pcm), n_samples, nfft, navg, int(remove_dc), int(stereo), _p(out),
                                  C.byref(n_rows), _stream()), "lrc_psdpng_rows")
    return out[: n_rows.value]


class Chain:
    """cf32 -> FIR/decimate -> window -> FFT -> |X|^2 average, one fused kernel."""

    def __init__(self, ctx: Context, taps, decim: int, nfft: int, window: int = capi.WINDOW_HANN):
        self.ctx, self.nfft, self.decim = ctx, int(nfft), int(decim)
        self.taps = np.ascontiguousarray(taps, dtype=np.float32)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_chain_create(ctx.h, _p(self.taps), self.taps.size, self.decim, self.nfft, window,
                                       C.byref(self.h)), "lrc_chain_create")

    def frames(self, n_in: int) -> int:
        return int(self.ctx.lib.lrc_chain_frames(self.h, n_in))

    @property
    def kind(self) -> int:
        """0 = unfused kernels, 1 = fused BASELINE instance, 2 = fused generic instance (lrc_chain_kind)"""
        return int(self.ctx.lib.lrc_chain_kind(self.h))

    def run(self, x: torch.Tensor, k_avg: int, out: torch.Tensor | None = None) -> torch.Tensor:
        assert x.dtype == torch.complex64 and x.is_cuda and x.is_contiguous() and x.dim() == 1
        rows = self.frames(x.numel()) // k_avg
        if out is None:
            out = torch.empty((rows, self.nfft), dtype=torch.float32, device=x.device)
        nr = C.c_size_t()
        check(self.ctx.lib.lrc_chain_run(self.h, _p(x), x.numel(), k_avg, _p(out), C.byref(nr), _stream()), "lrc_chain_run")
        assert nr.value == rows
        return out

    def run_u8(self, iq: torch.Tensor, k_avg: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """iq: device uint8 [2 n] of interleaved I,Q (the rtlsdr wire format); the unpack happens inside the kernel"""
        assert iq.dtype == torch.uint8 and iq.is_cuda and iq.is_contiguous() and iq.dim() == 1 and iq.numel() % 2 == 0
        n = iq.numel() // 2
        rows = self.frames(n) // k_avg
        if out is None:
            out = torch.empty((rows, self.nfft), dtype=torch.float32, device=iq.device)
        nr = C.c_size_t()
        check(self.ctx.lib.lrc_chain_run_u8(self.h, _p(iq), n, k_avg, _p(out), C.byref(nr), _stream()), "lrc_chain_run_u8")
        assert nr.value == rows
        return out

    def run_host(self, x, k_avg: int, out=None):
        """x: pinned CPU complex64 tensor (or numpy array); returns rows as a CPU tensor/array of the same kind."""
        n = x.numel() if isinstance(x, torch.Tensor) else x.size
        rows = self.frames(n) // k_avg
        if out is None:
            out = (torch.empty((rows, self.nfft), dtype=torch.float32, pin_memory=True)
                   if isinstance(x, torch.Tensor) else np.empty((rows, self.nfft), dtype=np.float32))
        nr = C.c_size_t()
        check(self.ctx.lib.lrc_chain_run_host(self.h, _p(x), n, k_avg, _p(out), C.byref(nr)), "lrc_chain_run_host")
        return out

    def run_host_u8(self, iq, k_avg: int, out=None):
        """iq: pinned CPU uint8 tensor (or numpy array) of interleaved I,Q bytes -- the rtlsdr wire format;
        2 bytes per sample cross PCIe and data_to_samples runs on the device in front of the chain."""
        n = (iq.numel() if isinstance(iq, torch.Tensor) else iq.size) // 2
        rows = self.frames(n) // k_avg
        if out is None:
            out = (torch.empty((rows, self.nfft), dtype=torch.float32, pin_memory=True)
                   if isinstance(iq, torch.Tensor) else np.empty((rows, self.nfft), dtype=np.float32))
        nr = C.c_size_t()
        check(self.ctx.lib.lrc_chain_run_host_u8(self.h, _p(iq), n, k_avg, _p(out), C.byref(nr)), "lrc_chain_run_host_u8")
        return out

    def close(self):
        if self.h:
            self.ctx.lib.lrc_chain_destroy(self.h)
            self.h = C.c_void_p()


# ---- (4) -------------------------------------------------------------------------------------------
def fm_demod(ctx: Context, x: torch.Tensor, state: torch.Tensor | None = None) -> torch.Tensor:
    """d[n] = arg(x[n] conj(x[n-1])); x: complex64 [n] or [n_ch, n]; state: complex64 [n_ch] carried x[-1]
    (updated in place), None = stateless (x[-1] = 0)."""
    assert x.dtype == torch.complex64 and x.is_cuda and x.is_contiguous()
    x2 = x.reshape(-1, x.shape[-1])
    n_ch, n = x2.shape
    out = torch.empty((n_ch, n), dtype=torch.float32, device=x.device)
    if state is not None:
        assert state.dtype == torch.complex64 and state.numel() == n_ch and state.is_cuda
    check(ctx.lib.lrc_fmdemod_run(ctx.h, _p(x2), n_ch, n, n, _p(state), _p(out), max(n, 1), _stream()), "lrc_fmdemod_run")
    return out.reshape(x.shape)


class Resampler:
    """samplerate::resample(din, dout, ratio): streaming, state carried across chunks (samplerate.rs:59-87)."""

    def __init__(self, ctx: Context, ratio: float, n_ch: int = 1, max_chunk: int = 1 << 20):
        self.ctx, self.ratio, self.n_ch, self.max_chunk = ctx, float(ratio), n_ch, max_chunk
        self.h = C.c_void_p()
        check(ctx.lib.lrc_resampler_create(ctx.h, C.c_double(self.ratio), n_ch, max_chunk, C.byref(self.h)),
              "lrc_resampler_create")
        nt, L, M = C.c_size_t(), C.c_int(), C.c_int()
        check(ctx.lib.lrc_resampler_get_taps(self.h, None, 0, C.byref(nt), C.byref(L), C.byref(M)), "lrc_resampler_get_taps")
        self.L, self.M, self.ntaps = L.value, M.value, nt.value

    def taps(self) -> np.ndarray:
        h = np.empty(self.ntaps, dtype=np.float64)
        check(self.ctx.lib.lrc_resampler_get_taps(self.h, _p(h), h.size, None, None, None), "lrc_resampler_get_taps")
        return h

    def reset(self):
        check(self.ctx.lib.lrc_resampler_reset(self.h), "lrc_resampler_reset")

    def process(self, x: torch.Tensor) -> torch.Tensor:
        """x: float32 [n] or [n_ch, n] -> [.., n_out]; the reference sizes the output ratio*len + 1 (:64)."""
        assert x.dtype == torch.float32 and x.is_cuda and x.is_contiguous()
        x2 = x.reshape(self.n_ch, -1)
        n = x2.shape[1]
        cap = int(self.ratio * n + 1) + 1
        out = torch.empty((self.n_ch, cap), dtype=torch.float32, device=x.device)
        no = C.c_size_t()
        check(self.ctx.lib.lrc_resampler_process(self.h, _p(x2), n, n, _p(out), cap, C.byref(no), _stream()),
              "lrc_resampler_process")
        res = out[:, : no.value]
        return res.reshape(-1) if x.dim() == 1 else res

    def close(self):
        if self.h:
            self.ctx.lib.lrc_resampler_destroy(self.h)
            self.h = C.c_void_p()


class FmReceiver:
    """BASELINE config 3 as one streaming object: rtlsdr u8 IQ chunks [n_ch, 2 n] -> audio chunks [n_ch, m]
    (lrc_fmrx: unpack + FIR/decimate, discriminator, resampler; ONE kernel per push for the BASELINE shape 64 taps / 10,
    ratio 1/5, the three stand-alone stages otherwise) -- the Python twin of kpn_gpu::fm_receiver_multi.  Output is
    independent of how the stream is chunked."""

    def __init__(self, ctx: Context, taps, decim: int, ratio: float, n_ch: int, max_chunk: int):
        self.ctx, self.n_ch, self.max_chunk = ctx, n_ch, max_chunk
        self.taps = np.ascontiguousarray(taps, dtype=np.float32)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_fmrx_create(ctx.h, _p(self.taps), self.taps.size, int(decim), C.c_double(float(ratio)), n_ch,
                                      max_chunk, C.byref(self.h)), "lrc_fmrx_create")
        self.fused = bool(ctx.lib.lrc_fmrx_is_fused(self.h))

    def next_out_len(self, n: int) -> int:
        return int(self.ctx.lib.lrc_fmrx_next_out_len(self.h, n))

    def reset(self):
        check(self.ctx.lib.lrc_fmrx_reset(self.h), "lrc_fmrx_reset")

    def push(self, iq: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        assert iq.dtype == torch.uint8 and iq.is_cuda and iq.is_contiguous()
        q2 = iq.reshape(self.n_ch, -1)
        n = q2.shape[1] // 2
        want = self.next_out_len(n)
        if out is None:
            out = torch.empty((self.n_ch, max(want, 1)), dtype=torch.float32, device=iq.device)
        no = C.c_size_t()
        check(self.ctx.lib.lrc_fmrx_push(self.h, _p(q2), n, n, _p(out), out.shape[1], C.byref(no), _stream()), "lrc_fmrx_push")
        assert no.value == want
        return out[:, : no.value]

    def close(self):
        if self.h:
            self.ctx.lib.lrc_fmrx_destroy(self.h)
            self.h = C.c_void_p()


# ---- long FIR (config 5) ----------------------------------------------------------------------------
class FastFir:
    """kiss_fastfir: overlap-save convolution with the nh-1 transient removed (tools/kiss_fastfir.c)."""

    def __init__(self, ctx: Context, h, nfft: int = 0):
        self.ctx = ctx
        self.taps = np.ascontiguousarray(h, dtype=np.complex64)
        self.h = C.c_void_p()
        check(ctx.lib.lrc_fastfir_create(ctx.h, _p(self.taps), self.taps.size, nfft, C.byref(self.h)), "lrc_fastfir_create")
        self.nfft = int(ctx.lib.lrc_fastfir_nfft(self.h))
        self.ngood = self.nfft - self.taps.size + 1

    def out_len(self, n_in: int, flush: bool = False) -> int:
        return int(self.ctx.lib.lrc_fastfir_out_len(self.h, n_in, int(flush)))

    def run(self, x: torch.Tensor, flush: bool = False, out: torch.Tensor | None = None) -> torch.Tensor:
        assert x.dtype == torch.complex64 and x.is_cuda and x.is_contiguous() and x.dim() == 1
        no = self.out_len(x.numel(), flush)
        if out is None:
            out = torch.empty(max(no, 1), dtype=torch.complex64, device=x.device)
        n = C.c_size_t()
        check(self.ctx.lib.lrc_fastfir_run(self.h, _p(x), x.numel(), _p(out), int(flush), C.byref(n), _stream()),
              "lrc_fastfir_run")
        assert n.value == no
        return out[:no]

    def close(self):
        if self.h:
            self.ctx.lib.lrc_fastfir_destroy(self.h)
            self.h = C.c_void_p()


# ---- (5) OOK ------------------------------------------------------------------------------------------
class Ook:
    """The OOK chain of ratpak.rs:60-111 over n_streams finite u8-IQ captures of n_blocks*512 samples."""

    FIELDS_A1 = (4, 8, 4, 12, 8)      # binconv, ratpak.rs:115
    FIELDS_A2 = (4, 8, 2, 10, 12)     # binconv, ratpak.rs:119

    def __init__(self, ctx: Context, n_streams: int, n_blocks: int, sample_rate: int = 256000,
                 max_runs: int = 4096, max_packets: int = 64):
        self.ctx, self.n_streams, self.n_blocks = ctx, n_streams, n_blocks
        self.max_runs, self.max_packets = max_runs, max_packets
        self.h = C.c_void_p()
        check(ctx.lib.lrc_ook_create(ctx.h, n_streams, n_blocks, sample_rate, max_runs, max_packets, C.byref(self.h)),
              "lrc_ook_create")

    def decode(self, iq: torch.Tensor):
        """iq: uint8 [n_streams, n_blocks*1024] on the device.  Asynchronous."""
        assert iq.dtype == torch.uint8 and iq.is_cuda and iq.is_contiguous()
        assert iq.shape == (self.n_streams, self.n_blocks * 1024)
        check(self.ctx.lib.lrc_ook_decode(self.h, _p(iq), iq.shape[1], _stream()), "lrc_ook_decode")

    def packets(self):
        """-> list of (stream, proto, seq, bits uint8[nbits]) ordered by (stream, proto, seq)."""
        n = C.c_size_t()
        cap = self.n_streams * 2 * self.max_packets
        buf = (capi.OokPacket * max(cap, 1))()
        check(self.ctx.lib.lrc_ook_fetch_packets(self.h, buf, cap, C.byref(n)), "lrc_ook_fetch_packets")
        out = []
        for k in range(n.value):
            p = buf[k]
            out.append((p.stream, p.proto, p.seq, np.frombuffer(bytes(p.bits)[: p.nbits], dtype=np.uint8).copy()))
        return out

    def debug(self) -> dict:
        """Intermediate products copied to the host: block_sums [S, B] f32, n_runs [S], runs [S, max_runs]
        as (value << 31 | length), n_bits [S]."""
        ps = [C.c_void_p() for _ in range(4)]
        check(self.ctx.lib.lrc_ook_debug_ptrs(self.h, *[C.byref(p) for p in ps]), "lrc_ook_debug_ptrs")
        S, B, R = self.n_streams, self.n_blocks, self.max_runs
        out = {}
        for name, ptr, shape, dt in (("block_sums", ps[0], (S, B), np.float32), ("n_runs", ps[1], (S,), np.uint32),
                                     ("runs", ps[2], (S, R), np.uint32), ("n_bits", ps[3], (S,), np.uint32)):
            host = np.empty(shape, dtype=dt)
            check(self.ctx.lib.lrc_copy_to_host(self.ctx.h, _p(host), ptr, host.nbytes), "lrc_copy_to_host")
            out[name] = host
        return out

    @staticmethod
    def eat(bits, widths):
        lib = capi.load()
        b = np.ascontiguousarray(bits, dtype=np.uint8)
        w = np.ascontiguousarray(widths, dtype=np.uint64)
        out = np.empty(w.size, dtype=np.uint64)
        check(lib.lrc_eat(_p(b), b.size, _p(w), w.size, _p(out)), "lrc_eat")
        return [int(v) for v in out]

    def close(self):
        if self.h:
            self.ctx.lib.lrc_ook_destroy(self.h)
            self.h = C.c_void_p()


class OokStream:
    """The OOK chain of ratpak.rs:60-111 on n_streams endless streams, pushed a few 512-sample blocks at a time: the
    packets after any push are those the reference emits on everything pushed so far, whatever the push sizes.
    max_carry_blocks = 0 keeps the exact carry (the trigger's OOM guard + 1 blocks per stream)."""

    def __init__(self, ctx: Context, n_streams: int, max_push_blocks: int, sample_rate: int = 256000,
                 max_carry_blocks: int = 0, max_runs: int = 4096, max_packets: int = 64):
        self.ctx, self.n_streams, self.max_push_blocks = ctx, n_streams, max_push_blocks
        self.max_runs, self.max_packets = max_runs, max_packets
        self.last_push = 0
        self.h = C.c_void_p()
        check(ctx.lib.lrc_ook_stream_create(ctx.h, n_streams, max_push_blocks, sample_rate, max_carry_blocks, max_runs,
                                            max_packets, C.byref(self.h)), "lrc_ook_stream_create")

    def push(self, iq: torch.Tensor):
        """iq: uint8 [n_streams, k*1024] on the device, the next k blocks of every stream.  Asynchronous."""
        assert iq.dtype == torch.uint8 and iq.is_cuda and iq.dim() == 2 and iq.stride(1) == 1
        assert iq.shape[0] == self.n_streams and iq.shape[1] % 1024 == 0
        n = iq.shape[1] // 1024
        check(self.ctx.lib.lrc_ook_stream_push(self.h, _p(iq), n, iq.stride(0), _stream()), "lrc_ook_stream_push")
        self.last_push = n

    def packets(self):
        """-> the packets completed since the last call, as (stream, proto, seq, bits uint8[nbits]) ordered by
        (stream, proto, seq); seq counts from create / reset."""
        n = C.c_size_t()
        cap = self.n_streams * 2 * self.max_packets
        buf = (capi.OokPacket * max(cap, 1))()
        check(self.ctx.lib.lrc_ook_stream_fetch_packets(self.h, buf, cap, C.byref(n)), "lrc_ook_stream_fetch_packets")
        out = []
        for k in range(n.value):
            p = buf[k]
            out.append((p.stream, p.proto, p.seq, np.frombuffer(bytes(p.bits)[: p.nbits], dtype=np.uint8).copy()))
        return out

    def reset(self):
        check(self.ctx.lib.lrc_ook_stream_reset(self.h), "lrc_ook_stream_reset")
        self.last_push = 0

    def debug(self) -> dict:
        """The last push's intermediate products on the host: block_sums [S, k] f32, n_runs [S] (runs it completed),
        runs [S, max_runs] as (value << 31 | length), n_bits [S] (bits it emitted)."""
        ps = [C.c_void_p() for _ in range(4)]
        check(self.ctx.lib.lrc_ook_stream_debug_ptrs(self.h, *[C.byref(p) for p in ps]), "lrc_ook_stream_debug_ptrs")
        S, B, R = self.n_streams, self.last_push, self.max_runs
        out = {}
        for name, ptr, shape, dt in (("block_sums", ps[0], (S, B), np.float32), ("n_runs", ps[1], (S,), np.uint32),
                                     ("runs", ps[2], (S, R), np.uint32), ("n_bits", ps[3], (S,), np.uint32)):
            host = np.empty(shape, dtype=dt)
            check(self.ctx.lib.lrc_copy_to_host(self.ctx.h, _p(host), ptr, host.nbytes), "lrc_copy_to_host")
            out[name] = host
        return out

    def close(self):
        if self.h:
            self.ctx.lib.lrc_ook_stream_destroy(self.h)
            self.h = C.c_void_p()


def ook_envelope_table(ctx: Context) -> torch.Tensor:
    """|i2f(b0) + j i2f(b1)| for all 65536 byte pairs, computed by the device routine the OOK kernels use."""
    t = torch.empty(65536, dtype=torch.float32, device=ctx.tdev)
    check(ctx.lib.lrc_ook_envelope_table(ctx.h, _p(t), _stream()), "lrc_ook_envelope_table")
    return t.reshape(256, 256)


# ---- (e) output gather over NVLink ---------------------------------------------------------------
class Gather:
    """Copy-engine gather of equally sized per-rank output blocks (include/libredio_cuda.h "(e)"): the multi-GPU
    form of the reference's `v.send(x)` between blocks (src/kpn/src/kpn.rs:127-131).  One process per GPU:
    `Gather(ctx, rank, world, nbytes, slots).connect_distributed()`; several contexts in one process:
    `Gather.connect_local([g0, g1, ...])`."""

    def __init__(self, ctx: Context, rank: int, world: int, bytes_per_rank: int, slots: int = 2, host_shm: str | None = None,
                 root: int = 0):
        """host_shm = "/name": gather into page-locked POSIX shared memory of the node instead of a GPU (lrc_gather_create_host;
        rank `root` creates the segment, the others open it) -- for consumers that run on the CPU."""
        self.ctx, self.rank, self.world, self.bytes_per_rank, self.slots = ctx, rank, world, bytes_per_rank, slots
        self.is_host = host_shm is not None
        self.h = C.c_void_p()
        if self.is_host:
            check(ctx.lib.lrc_gather_create_host(ctx.h, rank, world, bytes_per_rank, slots, host_shm.encode(), root, C.byref(self.h)),
                  "lrc_gather_create_host")
        else:
            check(ctx.lib.lrc_gather_create(ctx.h, rank, world, bytes_per_rank, slots, C.byref(self.h)), "lrc_gather_create")

    def set_root(self, root: int):
        """root >= 0: only that rank receives (a gather); -1: every rank receives everything (the default)"""
        check(self.ctx.lib.lrc_gather_set_root(self.h, root), "lrc_gather_set_root")
        return self

    def export(self) -> bytes:
        n = self.ctx.lib.lrc_gather_handle_bytes()
        buf = C.create_string_buffer(n)
        check(self.ctx.lib.lrc_gather_export(self.h, buf, n), "lrc_gather_export")
        return buf.raw

    def connect(self, handles: list[bytes]):
        blob = b"".join(handles)
        check(self.ctx.lib.lrc_gather_connect(self.h, C.c_char_p(blob)), "lrc_gather_connect")

    def connect_distributed(self, group=None):
        """Exchange the IPC handles through torch.distributed (host objects) and map every peer."""
        import torch.distributed as dist
        if self.world == 1:
            return self
        handles = [None] * self.world
        dist.all_gather_object(handles, self.export(), group=group)
        self.connect(handles)
        dist.barrier(group=group)              # nobody pushes before everybody has mapped everybody
        return self

    @staticmethod
    def connect_local(gathers: list["Gather"]):
        arr = (C.c_void_p * len(gathers))(*[g.h for g in gathers])
        for g in gathers:
            check(g.ctx.lib.lrc_gather_connect_local(g.h, arr), "lrc_gather_connect_local")

    def push(self, slot: int, src: torch.Tensor):
        assert src.is_cuda and src.is_contiguous() and src.numel() * src.element_size() == self.bytes_per_rank
        check(self.ctx.lib.lrc_gather_push(self.h, slot, _p(src), _stream()), "lrc_gather_push")

    def wait_sent(self, slot: int):
        check(self.ctx.lib.lrc_gather_wait_sent(self.h, slot, _stream()), "lrc_gather_wait_sent")

    def wait(self, slot: int):
        check(self.ctx.lib.lrc_gather_wait(self.h, slot, _stream()), "lrc_gather_wait")

    def wait_host(self, slot: int, timeout_ms: int = 10000):
        """host gather: block this CPU thread until every rank's latest push into the slot has arrived"""
        check(self.ctx.lib.lrc_gather_wait_host(self.h, slot, timeout_ms), "lrc_gather_wait_host")

    def buffer(self, slot: int, dtype=torch.float32) -> torch.Tensor:
        """The slot's receive buffer as a [world, elems_per_rank] tensor view (no copy)."""
        ptr, stride = C.c_void_p(), C.c_size_t()
        check(self.ctx.lib.lrc_gather_buffer(self.h, slot, C.byref(ptr), C.byref(stride)), "lrc_gather_buffer")
        es = torch.empty(0, dtype=dtype).element_size()
        assert stride.value % es == 0 and self.bytes_per_rank % es == 0
        if self.is_host:
            # host gather: the segment as a CPU tensor [world, elems_per_rank] (a view of the shared memory, no copy)
            npdt = np.dtype(torch.empty(0, dtype=dtype).numpy().dtype)
            raw = (C.c_uint8 * (self.world * stride.value)).from_address(ptr.value)
            arr = np.frombuffer(raw, dtype=npdt).reshape(self.world, stride.value // es)
            self._keep = raw
            return torch.from_numpy(arr)[:, : self.bytes_per_rank // es]
        iface = {"shape": (self.world, stride.value // es), "typestr": np.dtype(torch.empty(0, dtype=dtype).numpy().dtype).str,
                 "data": (ptr.value, False), "version": 3}
        holder = type("_Buf", (), {"__cuda_array_interface__": iface})()
        t = torch.as_tensor(holder, device=self.ctx.tdev)
        self._keep = holder
        return t[:, : self.bytes_per_rank // es]

    def close(self):
        if self.h:
            self.ctx.lib.lrc_gather_destroy(self.h)
            self.h = C.c_void_p()
