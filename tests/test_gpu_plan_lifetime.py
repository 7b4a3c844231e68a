"""GPU: plan lifetimes through the C ABI.

Every plan type goes through create -> run -> destroy several times on one context; destroy(NULL) is a no-op; and a
create that fails after part of the plan exists returns its documented status, leaves the out-pointer null and leaves
the context usable for the next create and run.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from libredio_b200 import blocks, capi, synth

pytestmark = pytest.mark.gpu

TAPS64 = synth.lpf_taps(64, 0.04).astype(np.float32)


@pytest.fixture(scope="module")
def ctx():
    c = blocks.Context(0)
    yield c
    c.close()


def ok(status, what):
    capi.check(status, what)


def dev(a):
    """numpy array -> device tensor, complete before the library's own stream reads it"""
    t = torch.from_numpy(np.ascontiguousarray(a)).to("cuda")
    torch.cuda.synchronize()
    return t


def p(t):
    return C.c_void_p(t.data_ptr())


def h(a):
    return a.ctypes.data_as(C.c_void_p)


def cf32(n_ch, n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n_ch, n)) + 1j * rng.standard_normal((n_ch, n))).astype(np.complex64)


def u8(n_bytes, seed):
    return np.random.default_rng(seed).integers(0, 256, n_bytes, dtype=np.uint8)


def finish(lib, ctx):
    ok(lib.lrc_ctx_sync(ctx.h), "lrc_ctx_sync")
    torch.cuda.synchronize()


# ---- one create -> run -> destroy per plan type ------------------------------------------------------------------------
def cycle_fir(lib, ctx):
    f = C.c_void_p()
    ok(lib.lrc_fir_create(ctx.h, h(TAPS64), 64, 10, C.byref(f)), "lrc_fir_create")
    x = dev(cf32(1, 20000, 1))
    n_out = lib.lrc_fir_out_len(f, 20000)
    y = torch.empty(2 * n_out, dtype=torch.float32, device="cuda")
    ok(lib.lrc_fir_run_cf32(f, p(x), 1, 20000, 20000, p(y), n_out, None), "lrc_fir_run_cf32")
    finish(lib, ctx)
    assert torch.isfinite(y).all()
    ok(lib.lrc_fir_destroy(f), "lrc_fir_destroy")


def cycle_fir_stream(lib, ctx):
    f, st = C.c_void_p(), C.c_void_p()
    ok(lib.lrc_fir_create(ctx.h, h(TAPS64), 64, 10, C.byref(f)), "lrc_fir_create")
    ok(lib.lrc_fir_stream_create(f, 2, 1000, 0, C.byref(st)), "lrc_fir_stream_create")
    y = torch.empty((2, 2 * 200), dtype=torch.float32, device="cuda")
    n_out = C.c_size_t()
    for k in range(3):
        x = dev(cf32(2, 1000, 2 + k))
        ok(lib.lrc_fir_stream_push(st, p(x), 1000, 1000, p(y), 200, C.byref(n_out), None), "lrc_fir_stream_push")
        assert n_out.value > 0
    finish(lib, ctx)
    ok(lib.lrc_fir_stream_destroy(st), "lrc_fir_stream_destroy")
    ok(lib.lrc_fir_destroy(f), "lrc_fir_destroy")


def cycle_fft(lib, ctx):
    f = C.c_void_p()
    ok(lib.lrc_fft_create(ctx.h, 1024, 0, C.byref(f)), "lrc_fft_create")
    x = cf32(4, 1024, 3)
    y = np.empty_like(x)
    ok(lib.lrc_fft_run_host(f, h(x), h(y), x.size), "lrc_fft_run_host")
    np.testing.assert_allclose(y, np.fft.fft(x, axis=1), rtol=0, atol=1e-3 * np.abs(y).max())
    ok(lib.lrc_fft_destroy(f), "lrc_fft_destroy")


def cycle_rfft(lib, ctx):
    f = C.c_void_p()
    ok(lib.lrc_rfft_create(ctx.h, 512, 0, C.byref(f)), "lrc_rfft_create")
    x = np.random.default_rng(4).standard_normal((3, 512)).astype(np.float32)
    y = np.empty((3, 257), dtype=np.complex64)
    ok(lib.lrc_rfft_run_host(f, h(x), h(y), 3), "lrc_rfft_run_host")
    np.testing.assert_allclose(y, np.fft.rfft(x, axis=1), rtol=0, atol=1e-3 * np.abs(y).max())
    ok(lib.lrc_rfft_destroy(f), "lrc_rfft_destroy")


def cycle_psd(lib, ctx):
    f = C.c_void_p()
    ok(lib.lrc_psd_create(ctx.h, 1024, capi.WINDOW_HANN, C.byref(f)), "lrc_psd_create")
    x = dev(cf32(8, 1024, 5))
    rows = torch.empty((2, 1024), dtype=torch.float32, device="cuda")
    ok(lib.lrc_psd_run(f, p(x), 8, 4, p(rows), None), "lrc_psd_run")
    finish(lib, ctx)
    assert torch.isfinite(rows).all() and (rows > 0).any()
    ok(lib.lrc_psd_destroy(f), "lrc_psd_destroy")


def run_chain(lib, ctx, ntaps, decim, nfft):
    taps = synth.lpf_taps(ntaps, 0.04).astype(np.float32)
    c = C.c_void_p()
    ok(lib.lrc_chain_create(ctx.h, h(taps), ntaps, decim, nfft, capi.WINDOW_HANN, C.byref(c)), "lrc_chain_create")
    n_in = 8 * nfft * decim + ntaps
    x = cf32(1, n_in, 6)
    rows = np.empty((2, nfft), dtype=np.float32)
    n_rows = C.c_size_t()
    ok(lib.lrc_chain_run_host(c, h(x), n_in, 4, h(rows), C.byref(n_rows)), "lrc_chain_run_host")
    assert n_rows.value == 2 and np.isfinite(rows).all()
    iq = u8(2 * n_in, 7)
    ok(lib.lrc_chain_run_host_u8(c, h(iq), n_in, 4, h(rows), C.byref(n_rows)), "lrc_chain_run_host_u8")
    d_iq, d_rows = dev(iq), torch.empty((2, nfft), dtype=torch.float32, device="cuda")
    ok(lib.lrc_chain_run_u8(c, p(d_iq), n_in, 4, p(d_rows), C.byref(n_rows), None), "lrc_chain_run_u8")
    finish(lib, ctx)
    assert n_rows.value == 2 and torch.isfinite(d_rows).all()
    ok(lib.lrc_chain_destroy(c), "lrc_chain_destroy")


def cycle_chain(lib, ctx):
    run_chain(lib, ctx, 64, 10, 1024)          # the fused instance


def cycle_chain_unfused(lib, ctx):
    run_chain(lib, ctx, 33, 3, 256)            # FIR into a scratch signal, then the PSD kernel


def cycle_resampler(lib, ctx):
    r = C.c_void_p()
    ok(lib.lrc_resampler_create(ctx.h, 0.2, 2, 5000, C.byref(r)), "lrc_resampler_create")
    x = np.random.default_rng(8).standard_normal((2, 5000)).astype(np.float32)
    y = np.empty((2, 1002), dtype=np.float32)
    n_out = C.c_size_t()
    ok(lib.lrc_resampler_process_host(r, h(x), 5000, h(y), 1002, C.byref(n_out)), "lrc_resampler_process_host")
    assert 990 <= n_out.value <= 1001 and np.isfinite(y[:, :n_out.value]).all()
    ok(lib.lrc_resampler_destroy(r), "lrc_resampler_destroy")


def run_fmrx(lib, ctx, ntaps, decim, ratio):
    taps = synth.lpf_taps(ntaps, 0.04).astype(np.float32)
    rx = C.c_void_p()
    ok(lib.lrc_fmrx_create(ctx.h, h(taps), ntaps, decim, ratio, 2, 8000, C.byref(rx)), "lrc_fmrx_create")
    out = torch.empty((2, 400), dtype=torch.float32, device="cuda")
    n_out = C.c_size_t()
    for k in range(3):
        want = lib.lrc_fmrx_next_out_len(rx, 8000)
        iq = dev(u8(2 * 2 * 8000, 9 + k).reshape(2, -1))
        ok(lib.lrc_fmrx_push(rx, p(iq), 8000, 8000, p(out), 400, C.byref(n_out), None), "lrc_fmrx_push")
        assert n_out.value == want
    finish(lib, ctx)
    ok(lib.lrc_fmrx_destroy(rx), "lrc_fmrx_destroy")


def cycle_fmrx(lib, ctx):
    run_fmrx(lib, ctx, 64, 10, 0.2)            # the fused instance


def cycle_fmrx_composed(lib, ctx):
    run_fmrx(lib, ctx, 32, 8, 0.25)            # FIR stream, demodulator and resampler plans


def fastfir_taps():
    rng = np.random.default_rng(10)
    return ((rng.standard_normal(50) + 1j * rng.standard_normal(50)) / 8).astype(np.complex64)


def cycle_fastfir(lib, ctx):
    ff = C.c_void_p()
    hh = fastfir_taps()
    ok(lib.lrc_fastfir_create(ctx.h, h(hh), 50, 0, C.byref(ff)), "lrc_fastfir_create")
    x = dev(cf32(1, 5000, 11))
    y = torch.empty(2 * lib.lrc_fastfir_out_len(ff, 5000, 1), dtype=torch.float32, device="cuda")
    n_out = C.c_size_t()
    ok(lib.lrc_fastfir_run(ff, p(x), 5000, p(y), 1, C.byref(n_out), None), "lrc_fastfir_run")
    finish(lib, ctx)
    assert 2 * n_out.value == y.numel() and torch.isfinite(y).all()
    ok(lib.lrc_fastfir_destroy(ff), "lrc_fastfir_destroy")


def cycle_fastfir_stream(lib, ctx):
    ff, st = C.c_void_p(), C.c_void_p()
    hh = fastfir_taps()
    ok(lib.lrc_fastfir_create(ctx.h, h(hh), 50, 0, C.byref(ff)), "lrc_fastfir_create")
    ok(lib.lrc_fastfir_stream_create(ff, 2, C.byref(st)), "lrc_fastfir_stream_create")
    y = torch.empty((2, 2 * 4000), dtype=torch.float32, device="cuda")
    n_out = C.c_size_t()
    for k, flush in enumerate((0, 0, 1)):
        want = lib.lrc_fastfir_stream_next_out_len(st, 1500, flush)
        x = dev(cf32(2, 1500, 12 + k))
        ok(lib.lrc_fastfir_stream_push(st, p(x), 1500, 1500, p(y), 4000, flush, C.byref(n_out), None),
           "lrc_fastfir_stream_push")
        assert n_out.value == want
    finish(lib, ctx)
    ok(lib.lrc_fastfir_stream_destroy(st), "lrc_fastfir_stream_destroy")
    ok(lib.lrc_fastfir_destroy(ff), "lrc_fastfir_destroy")


OOK_STREAMS, OOK_BLOCKS, OOK_RATE = 2, 800, 256000


def ook_input():
    """[stream][block][1024] bytes, two packets per stream"""
    return dev(np.stack([synth.ook_capture_u8(OOK_BLOCKS, seed=14 + s, n_packets=2)[0] for s in range(OOK_STREAMS)]))


def cycle_ook(lib, ctx):
    o = C.c_void_p()
    ok(lib.lrc_ook_create(ctx.h, OOK_STREAMS, OOK_BLOCKS, OOK_RATE, 1 << 16, 256, C.byref(o)), "lrc_ook_create")
    ok(lib.lrc_ook_decode(o, p(ook_input()), OOK_BLOCKS * 1024, None), "lrc_ook_decode")
    pk = (capi.OokPacket * 256)()
    n = C.c_size_t()
    ok(lib.lrc_ook_fetch_packets(o, pk, 256, C.byref(n)), "lrc_ook_fetch_packets")
    assert n.value > 0
    ok(lib.lrc_ook_destroy(o), "lrc_ook_destroy")


def cycle_ook_stream(lib, ctx):
    st = C.c_void_p()
    half = OOK_BLOCKS // 2
    ok(lib.lrc_ook_stream_create(ctx.h, OOK_STREAMS, half, OOK_RATE, 0, 1 << 16, 256, C.byref(st)), "lrc_ook_stream_create")
    iq = ook_input()
    pk = (capi.OokPacket * 256)()
    n = C.c_size_t()
    total = 0
    for k in range(2):
        ok(lib.lrc_ook_stream_push(st, C.c_void_p(iq.data_ptr() + k * half * 1024), half, OOK_BLOCKS * 1024, None),
           "lrc_ook_stream_push")
        ok(lib.lrc_ook_stream_fetch_packets(st, pk, 256, C.byref(n)), "lrc_ook_stream_fetch_packets")
        total += n.value
    assert total > 0
    ok(lib.lrc_ook_stream_destroy(st), "lrc_ook_stream_destroy")


CYCLES = {name[len("cycle_"):]: fn for name, fn in globals().items() if name.startswith("cycle_")}


@pytest.mark.parametrize("plan", sorted(CYCLES))
def test_create_run_destroy_repeats(ctx, plan):
    for _ in range(3):
        CYCLES[plan](ctx.lib, ctx)


@pytest.mark.parametrize("plan", ["fir", "fir_stream", "fft", "rfft", "psd", "chain", "resampler", "fmrx", "fastfir",
                                  "fastfir_stream", "ook", "ook_stream"])
def test_destroy_null_is_ok(ctx, plan):
    assert getattr(ctx.lib, f"lrc_{plan}_destroy")(None) == capi.OK


# ---- creates that fail after part of the plan exists --------------------------------------------------------------------
HUGE = 1 << 38          # bytes: well beyond the 180 GB of HBM


def fail_fmrx_ratio(lib, ctx, out):
    # the FIR plan exists when the resampler finds that 1/4099 is not L/M with L, M <= 4096
    return lib.lrc_fmrx_create(ctx.h, h(TAPS64), 64, 10, 1.0 / 4099, 2, 4096, C.byref(out)), capi.ERR_UNSUPPORTED


def fail_chain_nan_tap(lib, ctx, out):
    taps = TAPS64.copy()
    taps[17] = np.nan
    return lib.lrc_chain_create(ctx.h, h(taps), 64, 10, 1024, capi.WINDOW_HANN, C.byref(out)), capi.ERR_INVALID


def fail_ook_stream_carry(lib, ctx, out):
    # the chain's buffers exist when the carry of 2^28 blocks (256 GiB) does not fit
    return (lib.lrc_ook_stream_create(ctx.h, 1, OOK_BLOCKS, OOK_RATE, HUGE // 1024, 0, 0, C.byref(out)), capi.ERR_NOMEM)


def fail_fir_stream_size(lib, ctx, out):
    f = C.c_void_p()
    ok(lib.lrc_fir_create(ctx.h, h(TAPS64), 64, 10, C.byref(f)), "lrc_fir_create")
    try:
        return lib.lrc_fir_stream_create(f, 1, HUGE // 8, 0, C.byref(out)), capi.ERR_CUDA
    finally:
        ok(lib.lrc_fir_destroy(f), "lrc_fir_destroy")


def fail_fastfir_stream_size(lib, ctx, out):
    ff = C.c_void_p()
    hh = fastfir_taps()
    ok(lib.lrc_fastfir_create(ctx.h, h(hh), 50, 0, C.byref(ff)), "lrc_fastfir_create")
    try:
        return lib.lrc_fastfir_stream_create(ff, HUGE // (1024 * 8), C.byref(out)), capi.ERR_CUDA
    finally:
        ok(lib.lrc_fastfir_destroy(ff), "lrc_fastfir_destroy")


FAILS = {name[len("fail_"):]: fn for name, fn in globals().items() if name.startswith("fail_")}


# device memory a failed create may leave unaccounted for: allocator granularity and other work on the device, far below
# what the half-built plans hold (the OOK stream case has allocated its chain's 21 GiB when the carry fails)
FREE_SLACK = 1 << 30


@pytest.mark.parametrize("case", sorted(FAILS))
def test_failed_create_leaves_nothing_behind(ctx, case):
    out = C.c_void_p()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    status, want = FAILS[case](ctx.lib, ctx, out)
    assert status == want, ctx.lib.lrc_last_error().decode()
    assert out.value is None
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info()[0] >= free0 - FREE_SLACK
    cycle_fir(ctx.lib, ctx)
    cycle_chain(ctx.lib, ctx)
