"""GPU parity at every kernel the FFT, PSD, overlap-save, FIR and resampler plans can dispatch to.

Each plan picks its kernel from the size, the input alignment, the batch and the filter shape.  The other test files
cover the shapes the benchmark runs; this one walks the dispatch tables, compares every case with a plain f64
reference of the same operation, and shows with torch.profiler that the case reached the kernel it names.

kernel (file)                                   -> test
fft_tma_kernel<9|11, fwd|inv> (k_fft.cu)        -> test_fft_every_launch_branch_vs_f64 (512 / 2048, 16-byte aligned, batch >= 64)
fft_batch_kernel<L, fwd|inv>, every L but 10    -> test_fft_every_launch_branch_vs_f64 (incl. 512 / 2048 at batch < 64 or 8-byte offset)
fft1024_warp_kernel                             -> test_fft_every_launch_branch_vs_f64 (1024)
psd_tma_kernel<9|11>                            -> test_psd_rows_per_row_vs_f64, test_psd_tma_ring_crosses_items_and_rows
psd_kernel<L> (incl. <9|10|11> at 8-byte offset)-> test_psd_rows_per_row_vs_f64
psd1024_warp_kernel                             -> test_psd_rows_per_row_vs_f64 (1024, aligned)
lrc_psd_set_window                              -> test_psd_rows_per_row_vs_f64 (window "random")
fastfir_kernel<1..12> (k_fastfir.cu)            -> test_fastfir_every_instance_vs_f64_convolution
fastfir16k_kernel, nh = 1 (k_fastfir16k.cu)     -> test_fastfir_16k_path_one_tap
fir_generic_kernel<true> (k_fir.cu)             -> test_fir_u8_generic_kernel_vs_oracle
lrc_fir_stream_push: skip path, generic kernel,
  u8 on a tile shape, fir_generic_kernel<false>
  grid stride                                   -> test_fir_stream_dispatch_is_seam_exact_and_matches_oracle
resample_kernel<4> (k_fm_resample.cu)           -> test_resampler_general_ratio_streams_bit_exact, test_resampler_general_ratio_wraps_the_grid
chain run_host on a kind-2 plan                 -> test_chain_kind2_host_ring_matches_device_path
chain WINDOW_NONE, kinds 1 and 2                -> test_chain_window_none_vs_f64

Tolerances are the repository's: max |err| <= 1e-4 x RMS of the reference (per frame, per row or per channel as
named), >= 100 dB SNR for the FFT and the resampler, bit equality where two paths run the same arithmetic.
"""
import re

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import oracle
from oracle import defined_f64 as D
from libredio_b200 import capi, synth

pytestmark = pytest.mark.gpu

TOL = 1e-4          # x RMS of the reference output
MIN_SNR_DB = 100.0


def rms(a, axis=None):
    return np.sqrt(np.mean(np.abs(np.asarray(a, dtype=np.complex128)) ** 2, axis=axis))


def dev(a, ctx):
    return torch.from_numpy(np.ascontiguousarray(a)).to(ctx.tdev)


def assert_close_rms(got, ref, tol=TOL, what=""):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if ref.size == 0:
        return
    err = float(np.max(np.abs(got.astype(np.complex128) - ref.astype(np.complex128))))
    assert err <= tol * rms(ref), f"{what}: max|err| {err:.3e} > {tol} x rms {rms(ref):.3e}"


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def launched(fn):
    """Run fn under torch.profiler (CUDA activities) and return (fn's result, names of the CUDA kernels it launched)."""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.key for e in prof.key_averages()}


def assert_ran(names, *kernels):
    """kernels: base name and first template argument, e.g. "fft_tma_kernel<9" or "psd1024_warp_kernel"."""
    for k in kernels:
        tail = "" if k.endswith("<") else (r"[,>]" if "<" in k else r"\b")
        pat = re.compile(r"(?:^|[\s:])" + re.escape(k) + tail)
        assert any(pat.search(n) for n in names), f"{k} did not run; kernels launched: {sorted(names)}"


def cnoise(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


# ---- FFT: every size, both directions, every launch branch ------------------------------------------------------
def _fft_groups(n):
    """transforms per CTA of fft_batch_kernel / fft_tma_kernel (CtaFFT: 16 points per thread, 128-thread CTAs at least)"""
    t = max(1, n // 16)
    return max(1, 128 // t)


@pytest.mark.parametrize("inv", [0, 1])
@pytest.mark.parametrize("n", [1 << k for k in range(1, 14)])
def test_fft_every_launch_branch_vs_f64(ctx, n, inv):
    """batch 1, 63, 64 (the TMA threshold), 65 (a last CTA with idle groups) and a batch sized from the SM count; input
    16-byte aligned and at an 8-byte offset (a [1:] view); out of place and in place.  512 and 2048 points take the
    TMA ring only when the input is 16-byte aligned and batch >= 64; the big batch there gives every transform group
    at least six frames (resident groups <= 3 CTAs per SM by shared memory), so its 3-stage ring wraps twice."""
    from libredio_b200 import blocks
    log2n = n.bit_length() - 1
    tma = n in (512, 2048)
    big = ctx.sm_count * 3 * _fft_groups(n) * 6 + 5 if tma else (1 << 20) // n + 3
    f = blocks.Fft(ctx, n, inv)
    rng = np.random.default_rng(1000 * n + inv)
    expect = set()

    def run_all():
        for batch in (1, 63, 64, 65, big):
            x = cnoise(rng, (batch, n))
            xr = x.astype(np.complex128)
            ref = np.fft.ifft(xr, axis=-1) * n if inv else np.fft.fft(xr, axis=-1)
            for off in (0, 1):
                buf = torch.empty(batch * n + 1, dtype=torch.complex64, device=ctx.tdev)
                d = buf[off: off + batch * n].view(batch, n)
                assert (d.data_ptr() % 16 == 0) == (off == 0)
                d.copy_(dev(x, ctx))
                got = f.run(d).cpu().numpy()
                f.run(d, inplace=True)
                assert bits_equal(d.cpu().numpy(), got), (batch, off, "in place differs from out of place")
                err = np.max(np.abs(got - ref), axis=-1)
                assert np.all(err <= TOL * rms(ref, axis=-1)), (batch, off, float(np.max(err / rms(ref, axis=-1))))
                p_err = np.sum(np.abs(got - ref) ** 2, axis=-1)
                snr = 10 * np.log10(np.sum(np.abs(ref) ** 2, axis=-1) / np.maximum(p_err, 1e-300))
                assert np.min(snr) >= MIN_SNR_DB, (batch, off, float(np.min(snr)))
                if n == 1024:
                    expect.add("fft1024_warp_kernel")
                elif tma and off == 0 and batch >= 64:
                    expect.add(f"fft_tma_kernel<{log2n}")
                else:
                    expect.add(f"fft_batch_kernel<{log2n}")

    _, names = launched(run_all)
    assert_ran(names, *sorted(expect))
    if tma:
        assert {f"fft_tma_kernel<{log2n}", f"fft_batch_kernel<{log2n}"} <= expect
    f.close()


# ---- PSD: window + FFT + |X|^2 rows --------------------------------------------------------------------------------
def _psd_kernels(nfft, aligned):
    l2 = nfft.bit_length() - 1
    if aligned and nfft == 1024:
        return {"psd1024_warp_kernel", "psd_reduce_kernel"}
    if aligned and nfft in (512, 2048):
        return {f"psd_tma_kernel<{l2}", "psd_reduce_kernel"}
    return {f"psd_kernel<{l2}", "psd_reduce_kernel"}


def _row_scaled_frames(rng, nfft, k, rows, tail):
    """rows*k + tail frames of complex noise; every row's frames scaled by the row's own factor, so a frame counted
    into the wrong row or item moves that row's power"""
    x = cnoise(rng, (rows * k + tail, nfft))
    scale = np.concatenate([np.repeat(0.25 + 0.6 * np.arange(rows), k), np.full(tail, 7.0)]).astype(np.float32)
    return (x * scale[:, None]).reshape(-1)


def _assert_rows(got, ref, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    for r in range(ref.shape[0]):
        err = float(np.max(np.abs(got[r] - ref[r])))
        tol = TOL * float(np.sqrt(np.mean(ref[r] ** 2)))
        assert err <= tol, f"{what} row {r}: max|err| {err:.3e} > {tol:.3e}"


def _psd_case(ctx, p, x, nfft, k, win, off):
    buf = torch.empty(x.size + 1, dtype=torch.complex64, device=ctx.tdev)
    d = buf[off: off + x.size]
    assert (d.data_ptr() % 16 == 0) == (off == 0)
    d.copy_(dev(x, ctx))
    got = p.run(d, k).cpu().numpy()
    _assert_rows(got, D.psd_rows(x, nfft, k, win), f"nfft {nfft} k {k} offset {off}")


@pytest.mark.parametrize("window", ["none", "hann", "random"])
@pytest.mark.parametrize("nfft", [256, 512, 1024, 2048, 4096, 8192])
def test_psd_rows_per_row_vs_f64(ctx, nfft, window):
    """k_avg 1, 15, 16, 17, 40, 64: items of up to 16 frames, several items per row, a ragged last item and a dropped
    tail; input 16-byte aligned (TMA / warp kernels at 512..2048) and at an 8-byte offset (psd_kernel)."""
    from libredio_b200 import blocks
    rng = np.random.default_rng(nfft + len(window))
    p = blocks.Psd(ctx, nfft, capi.WINDOW_HANN if window == "hann" else capi.WINDOW_NONE)
    if window == "none":
        win = np.ones(nfft, np.float32)
    elif window == "hann":
        win = D.hann_periodic(nfft)
    else:
        win = rng.uniform(0.2, 1.8, nfft).astype(np.float32)
        p.set_window(win)
    expect = set()

    def run_all():
        for k in (1, 15, 16, 17, 40, 64):
            x = _row_scaled_frames(rng, nfft, k, 3, min(k - 1, 5))
            for off in (0, 1):
                _psd_case(ctx, p, x, nfft, k, win, off)
                expect.update(_psd_kernels(nfft, off == 0))

    _, names = launched(run_all)
    assert_ran(names, *sorted(expect))
    p.close()


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("nfft", [512, 2048])
def test_psd_tma_ring_crosses_items_and_rows(ctx, nfft, k):
    """twice as many work items as transform groups can be resident (3 CTAs per SM by shared memory), so each group's
    3-stage ring runs on from one item and one row into the next"""
    from libredio_b200 import blocks
    groups = ctx.sm_count * 3 * _fft_groups(nfft)
    rows = 2 * groups + 1                               # k < 16: one item per row
    rng = np.random.default_rng(nfft * 10 + k)
    x = cnoise(rng, (rows * k, nfft)) * (0.5 + (np.arange(rows * k) // k % 7)).astype(np.float32)[:, None]
    x = x.reshape(-1)
    p = blocks.Psd(ctx, nfft, capi.WINDOW_HANN)
    _, names = launched(lambda: _psd_case(ctx, p, x, nfft, k, D.hann_periodic(nfft), 0))
    assert_ran(names, f"psd_tma_kernel<{nfft.bit_length() - 1}")
    p.close()


# ---- overlap-save ---------------------------------------------------------------------------------------------------
def conv_valid_f64(x, h):
    """y[k] = sum_j h[j] x[k + nh - 1 - j], the outputs kiss_fastfir keeps, in f64 (by FFT when the direct sum is large)"""
    x = np.asarray(x, np.complex128)
    h = np.asarray(h, np.complex128)
    if x.size < h.size:
        return np.empty(0, np.complex128)
    if x.size * h.size <= 20_000_000:
        return np.convolve(x, h, mode="valid")
    from scipy.signal import oaconvolve
    return oaconvolve(x, h, mode="valid")


def _fastfir_cases():
    out = []
    for l2 in range(1, 13):
        nfft = 1 << l2
        for nh in sorted({1, min(nfft // 2, 1024), min(nfft, 1024)}):
            out.append((nfft, nh))
    return out


@pytest.mark.parametrize("nfft,nh", _fastfir_cases())
def test_fastfir_every_instance_vs_f64_convolution(ctx, nfft, nh):
    """inputs with no full block (flush only), exactly nfft, nfft + 3 ngood - 1, and enough blocks that the
    n_sm x occupancy grid strides round (occupancy bounded by 32 CTAs or 2048 threads per SM); flush and no flush"""
    from libredio_b200 import blocks
    rng = np.random.default_rng(nfft * 7 + nh)
    h = cnoise(rng, nh) / np.float32(np.sqrt(nh))
    ff = blocks.FastFir(ctx, h, nfft)
    assert ff.nfft == nfft and ff.ngood == nfft - nh + 1
    ngood = ff.ngood
    occ_bound = min(32, 2048 // max(1, nfft // 16))
    blocks_long = ctx.sm_count * occ_bound + 3
    lengths = [nfft - 1, nfft, nfft + 3 * ngood - 1, (blocks_long - 1) * ngood + nfft + ngood // 2]

    def run_all():
        for n in lengths:
            x = cnoise(rng, n)
            ref = conv_valid_f64(x, h)
            xd = dev(x, ctx)
            for flush in (False, True):
                got = ff.run(xd, flush).cpu().numpy()
                if flush:
                    n_out = max(n - nh + 1, 0)
                else:
                    n_out = ((n - nfft) // ngood + 1) * ngood if n >= nfft else 0
                want = ref[:n_out]
                assert_close_rms(got, want, what=f"n {n} flush {flush} vs f64")
                assert_close_rms(got, oracle.fastfir(h, x, nfft, flush), what=f"n {n} flush {flush} vs oracle")

    _, names = launched(run_all)
    assert_ran(names, f"fastfir_kernel<{nfft.bit_length() - 1}")
    ff.close()


@pytest.mark.parametrize("nfft", [8192, 16384])
def test_fastfir_16k_path_one_tap(ctx, nfft):
    """nh = 1 at nfft >= 8192 computes in 16384-point blocks with ngood16 = 16384: no overlap between blocks"""
    from libredio_b200 import blocks
    rng = np.random.default_rng(nfft)
    h = cnoise(rng, 1)
    ff = blocks.FastFir(ctx, h, nfft)

    def run_all():
        for n in (nfft - 1, nfft, nfft + 3 * nfft - 1, 5 * 16384 + 7):
            x = cnoise(rng, n)
            for flush in (False, True):
                got = ff.run(dev(x, ctx), flush).cpu().numpy()
                want = conv_valid_f64(x, h)[: ff.out_len(n, flush)]
                assert_close_rms(got, want, what=f"n {n} flush {flush} vs f64")
                assert_close_rms(got, oracle.fastfir(h, x, nfft, flush), what=f"n {n} flush {flush} vs oracle")

    _, names = launched(run_all)
    assert_ran(names, "fastfir16k_kernel")
    ff.close()


# ---- FIR + decimate ---------------------------------------------------------------------------------------------------
def _taps(ntaps, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal(ntaps) / np.sqrt(ntaps)).astype(np.float32)


@pytest.mark.parametrize("ntaps,decim", [(1, 1), (3, 7), (4, 10), (5, 3), (33, 4), (64, 5), (129, 16)])
def test_fir_u8_generic_kernel_vs_oracle(ctx, ntaps, decim):
    """u8 input of every shape but 64/10 runs fir_generic_kernel<true>, tile shapes (33/4, 64/5) included"""
    from libredio_b200 import blocks
    taps = _taps(ntaps, ntaps * 100 + decim)
    n_ch, n = 3, 20_003
    iq = np.stack([synth.iq_tone_noise_u8(n, seed=40 + c) for c in range(n_ch)])
    fir = blocks.Fir(ctx, taps, decim)
    got, names = launched(lambda: fir.run_u8(dev(iq, ctx)).cpu().numpy())
    assert_ran(names, "fir_generic_kernel<true")
    for c in range(n_ch):
        assert_close_rms(got[c], oracle.fir_decimate(oracle.data_to_samples(iq[c]), taps, decim), what=f"channel {c}")
    fir.close()


# (ntaps, decim, u8, n_ch, kernel the pushes run)
STREAM_CASES = [
    (3, 7, False, 3, "fir_generic_kernel<false"),      # decim > ntaps: skip path, generic kernel
    (3, 7, True, 3, "fir_generic_kernel<true"),
    (2, 16, False, 3, "fir_gentile_kernel<"),           # decim > ntaps on a tile shape
    (2, 16, True, 3, "fir_generic_kernel<true"),
    (129, 3, False, 3, "fir_generic_kernel<false"),    # no tile instance
    (129, 3, True, 3, "fir_generic_kernel<true"),
    (64, 8, True, 3, "fir_generic_kernel<true"),        # u8 on a tile shape
]


def _stream_check(ctx, ntaps, decim, u8, n_ch, chunks, kernel):
    from libredio_b200 import blocks
    taps = _taps(ntaps, ntaps * 10 + decim)
    n = sum(chunks)
    if u8:
        x = np.stack([synth.iq_tone_noise_u8(n, seed=60 + c) for c in range(n_ch)])
    else:
        x = np.stack([synth.cf32_noise_tones(n, seed=60 + c) for c in range(n_ch)])
    fir = blocks.Fir(ctx, taps, decim)
    whole = (fir.run_u8(dev(x, ctx)) if u8 else fir.run(dev(x, ctx))).cpu().numpy()
    st = blocks.FirStream(fir, n_ch, max(chunks), u8=u8)

    def push_all():
        outs, pos = [], 0
        for c in chunks:
            w, p = (2 * c, 2 * pos) if u8 else (c, pos)
            outs.append(st.push(dev(x[:, p:p + w], ctx)).cpu().numpy())
            pos += c
        return np.concatenate(outs, axis=1)

    got, names = launched(push_all)
    assert_ran(names, kernel)
    assert bits_equal(got, whole), "chunked output differs from one call over the whole input"
    for c in range(n_ch):
        xc = oracle.data_to_samples(x[c]) if u8 else x[c]
        assert_close_rms(got[c], oracle.fir_decimate(xc, taps, decim), what=f"channel {c}")
    st.close(); fir.close()


@pytest.mark.parametrize("ntaps,decim,u8,n_ch,kernel", STREAM_CASES)
def test_fir_stream_dispatch_is_seam_exact_and_matches_oracle(ctx, ntaps, decim, u8, n_ch, kernel):
    """chunks shorter than decim, chunks of 1, and chunks that end inside the samples a window skips"""
    chunks = [1, 2, 6, 1, 1, 13, 100, 5, 1000, 3, 1, 2000, 17, 4001]
    _stream_check(ctx, ntaps, decim, u8, n_ch, chunks, kernel)


def test_fir_stream_generic_kernel_wraps_the_grid(ctx):
    """a push with n_ch x n_out above the generic kernel's n_sm x 8 CTAs x 256 threads"""
    n_ch, decim = 8, 3
    chunk = (ctx.sm_count * 8 * 256 * 3 // 2) * decim // n_ch
    _stream_check(ctx, 129, decim, False, n_ch, [5, 1, chunk, 77], "fir_generic_kernel<false")


# ---- resampler, general L/M -------------------------------------------------------------------------------------------
def _rs_input(n_ch, n, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    return np.stack([(np.sin(2 * np.pi * (0.004 + 0.003 * c) * t) + 0.3 * np.sin(2 * np.pi * 0.031 * t + c)
                      + 0.1 * rng.standard_normal(n)).astype(np.float32) for c in range(n_ch)])


def _rs_check(ctx, ratio, n_ch, chunks):
    from libredio_b200 import blocks
    x = _rs_input(n_ch, sum(chunks), int(ratio * 1000) + n_ch)
    rs = blocks.Resampler(ctx, ratio, n_ch, max(chunks))
    assert rs.L > 1 or rs.M == 1 or rs.M > 6, "this ratio has a decimator kernel"

    def stream():
        parts, pos = [], 0
        for c in chunks:
            parts.append(rs.process(dev(x[:, pos:pos + c], ctx)).cpu().numpy())
            pos += c
        return np.concatenate(parts, axis=1)

    got, names = launched(stream)
    assert_ran(names, "resample_kernel<4")
    one = blocks.Resampler(ctx, ratio, n_ch, x.shape[1])
    whole = one.process(dev(x, ctx)).cpu().numpy()
    assert bits_equal(got, whole), "chunked output differs from one call over the whole input"
    for c in range(n_ch):
        ref = D.resample(x[c], ratio)
        assert got[c].shape == ref.shape
        assert D.snr_db(ref, got[c]) >= MIN_SNR_DB, f"channel {c}"
    rs.close(); one.close()


@pytest.mark.parametrize("n_ch", [1, 5])
@pytest.mark.parametrize("ratio", [2.0, 48000 / 44100, 3 / 7, 1.0, 1 / 7])
def test_resampler_general_ratio_streams_bit_exact(ctx, ratio, n_ch):
    """L > 1, or L = 1 with M = 1 or M > 6: one thread per output.  Pushes shorter than the carried history (tpp - 1)
    make the next window reach back through two carries."""
    L, M = D.resampler_ratio(ratio)
    tpp = -(-(2 * 32 * max(L, M) + 1) // L)
    chunks = [1, 3, tpp - 2, 1, 500, 7, tpp - 1, 2000, tpp, 1, 3001]
    _rs_check(ctx, ratio, n_ch, chunks)


def test_resampler_general_ratio_wraps_the_grid(ctx):
    """n_ch x n_out above the n_sm x 16 CTAs x 256 threads of resample_kernel in one push"""
    ratio, n_ch = 48000 / 44100, 5
    n = int(ctx.sm_count * 16 * 256 * 1.25 / n_ch / ratio)
    _rs_check(ctx, ratio, n_ch, [5, n, 1])


# ---- fused chain -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("frames,k", [(37, 1), (900, 300), (1000, 450)])
def test_chain_kind2_host_ring_matches_device_path(ctx, frames, k):
    """the pinned host ring over the generic fused instance: rows of whole segments and rows sliced across segments
    (k_avg above the ring's 400 frames per segment)"""
    from libredio_b200 import blocks
    taps = synth.lpf_taps(64, 0.04)
    ntaps, decim, nfft = 64, 8, 1024
    n = (frames - 1) * nfft * decim + (nfft - 1) * decim + ntaps
    xh = torch.from_numpy(synth.cf32_noise_tones(n, seed=frames)).pin_memory()
    ch = blocks.Chain(ctx, taps, decim, nfft)
    assert ch.kind == 2
    a = ch.run(xh.to(ctx.tdev), k).cpu()
    b, names = launched(lambda: ch.run_host(xh, k))
    assert_ran(names, "chain_gen_kernel<64")
    assert a.shape == b.shape == (frames // k, nfft)
    assert (a - b).abs().max().item() <= 1e-5 * a.pow(2).mean().sqrt().item()
    ch.close()


@pytest.mark.parametrize("decim,kind,kernel", [(10, 1, "chain_kernel<64"), (8, 2, "chain_gen_kernel<64")])
def test_chain_window_none_vs_f64(ctx, decim, kind, kernel):
    from libredio_b200 import blocks
    taps = synth.lpf_taps(64, 0.04)
    nfft, frames, k = 1024, 70, 7
    n = (frames - 1) * nfft * decim + (nfft - 1) * decim + 64
    x = synth.cf32_noise_tones(n, seed=decim)
    ch = blocks.Chain(ctx, taps, decim, nfft, capi.WINDOW_NONE)
    assert ch.kind == kind
    got, names = launched(lambda: ch.run(dev(x, ctx), k).cpu().numpy())
    assert_ran(names, kernel)
    ref = D.psd_rows(oracle.fir_decimate(x, taps, decim), nfft, k, np.ones(nfft))
    _assert_rows(got, ref, f"decim {decim}")
    ch.close()
