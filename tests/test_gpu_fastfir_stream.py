"""GPU: streaming overlap-save over many channels (lrc_fastfir_stream_*, blocks.FastFirStream, kpn_gpu::fast_fir_multi).

The contract pinned here: for every channel and every way of cutting the input into pushes, the outputs of the pushes
concatenated, with flush on the last push, equal lrc_fastfir_run(whole input, flush=1) bit for bit, and after any push
without flush the outputs so far are a bitwise prefix of it.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle
from libredio_b200 import blocks, capi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (nh, nfft): plans on fastfir_kernel<LOG2N> (nh <= 1024 and nfft < 8192) and on fastfir16k_kernel
PLANS = [(1, 0), (50, 128), (300, 0), (1024, 0), (100, 8192), (4096, 0), (8192, 16384)]


def compute_block(ff):
    nh = ff.taps.size
    nc = 16384 if (nh > 1024 or ff.nfft >= 8192) else ff.nfft
    return nc, nc - nh + 1


def taps(nh, seed):
    rng = np.random.default_rng(seed)
    return ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / np.sqrt(nh)).astype(np.complex64)


def signal(n_ch, n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n_ch, n)) + 1j * rng.standard_normal((n_ch, n))).astype(np.complex64)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def oneshot(ctx, ff, x):
    """lrc_fastfir_run(x, flush=1) per channel row"""
    return [ff.run(torch.from_numpy(np.ascontiguousarray(r)).to(ctx.tdev), True).cpu().numpy() for r in x]


def stream(ctx, fs, x, cuts, refs=None):
    """push x[:, a:b] for consecutive cuts, flush on the last; with refs, check the bitwise prefix after every push"""
    got = [[] for _ in range(x.shape[0])]
    done = 0
    for k, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        flush = k == len(cuts) - 2
        want = fs.next_out_len(b - a, flush)
        y = fs.push(torch.from_numpy(np.ascontiguousarray(x[:, a:b])).to(ctx.tdev), flush).cpu().numpy()
        assert y.shape == (x.shape[0], want)
        done += want
        for c in range(x.shape[0]):
            got[c].append(y[c])
            if refs is not None:
                assert done <= refs[c].size
                assert np.array_equal(bits(np.concatenate(got[c])), bits(refs[c][:done])), (k, c)
    return [np.concatenate(g) for g in got]


def random_cuts(rng, n, nc, good):
    sizes = []
    while sum(sizes) < n:
        sizes.append(int(rng.choice([0, 1, int(rng.integers(2, good)), good, nc, int(rng.integers(1, 2 * nc))])))
    cuts = np.minimum(np.cumsum([0] + sizes), n)
    return [int(v) for v in cuts] + [n]


@pytest.mark.parametrize("n_ch", [1, 3, 64])
@pytest.mark.parametrize("nh,nfft", PLANS)
def test_stream_equals_oneshot_bitwise_whatever_the_cuts(ctx, nh, nfft, n_ch):
    ff = blocks.FastFir(ctx, taps(nh, nh), nfft)
    nc, good = compute_block(ff)
    n = 4 * nc + 777
    x = signal(n_ch, n, nh + n_ch)
    refs = oneshot(ctx, ff, x)
    fs = blocks.FastFirStream(ff, n_ch)
    rng = np.random.default_rng(nh * 7 + n_ch)
    for cuts in (random_cuts(rng, n, nc, good), random_cuts(rng, n, nc, good), [0, n]):
        fs.reset()
        got = stream(ctx, fs, x, cuts, refs)
        for c in range(n_ch):
            assert np.array_equal(bits(got[c]), bits(refs[c]))
    fs.close(); ff.close()


def test_every_two_push_split_of_a_short_stream(ctx):
    ff = blocks.FastFir(ctx, taps(50, 1), 128)
    n = 400
    x = signal(1, n, 2)
    refs = oneshot(ctx, ff, x)
    fs = blocks.FastFirStream(ff, 1)
    for s in range(n + 1):
        got = stream(ctx, fs, x, [0, s, n], refs)
        assert np.array_equal(bits(got[0]), bits(refs[0])), s
    fs.close(); ff.close()


def rms(a):
    return float(np.sqrt(np.mean(np.abs(np.asarray(a, dtype=np.complex128)) ** 2)))


@pytest.mark.parametrize("nh,nfft", [(300, 0), (100, 8192), (4096, 0)])
def test_accuracy_against_the_restated_kiss_fastfir_and_f64_convolution_at_seams(ctx, nh, nfft):
    ff = blocks.FastFir(ctx, taps(nh, 11), nfft)
    nc, good = compute_block(ff)
    n = 3 * nc + 1000
    x = signal(1, n, 12)
    fs = blocks.FastFirStream(ff, 1)
    cuts = [0, 1000, nc + 17, 2 * nc + 5, n]
    y = stream(ctx, fs, x, cuts)[0]
    ref = oracle.fastfir(ff.taps, x[0], nfft, True)
    assert y.shape == ref.shape
    assert np.max(np.abs(y - ref)) <= 1e-4 * rms(ref)
    hr = ff.taps[::-1].astype(np.complex128)
    seams = [c - nh + 1 for c in cuts[1:-1]] + [b * good for b in range(1, y.size // good)]
    for s0 in seams:
        s0 = max(0, min(s0 - 16, y.size - 32))
        seg = x[0, s0: s0 + 32 + nh - 1].astype(np.complex128)
        win = np.array([np.dot(seg[k:k + nh], hr) for k in range(32)])
        assert np.max(np.abs(y[s0:s0 + 32] - win)) <= 1e-4 * rms(win)
    fs.close(); ff.close()


def test_channels_are_independent(ctx):
    ff = blocks.FastFir(ctx, taps(1024, 3), 0)
    nc, good = compute_block(ff)
    n = 3 * nc + 99
    x = signal(64, n, 4)
    cuts = random_cuts(np.random.default_rng(5), n, nc, good)
    fs = blocks.FastFirStream(ff, 64)
    many = stream(ctx, fs, x, cuts)
    one = blocks.FastFirStream(ff, 1)
    for c in (0, 17, 63):
        one.reset()
        assert np.array_equal(bits(stream(ctx, one, x[c:c + 1], cuts)[0]), bits(many[c]))
    one.close(); fs.close(); ff.close()


@pytest.mark.parametrize("nh,nfft", [(300, 0), (4096, 0)])
def test_strides_larger_than_the_push(ctx, nh, nfft):
    lib = ctx.lib
    ff = blocks.FastFir(ctx, taps(nh, 8), nfft)
    nc, good = compute_block(ff)
    n_ch, n = 5, 2 * nc + 300
    x = signal(n_ch, n, 9)
    refs = oneshot(ctx, ff, x)
    fs = blocks.FastFirStream(ff, n_ch)
    got = [[] for _ in range(n_ch)]
    for a, b, flush in ((0, nc + 3, 0), (nc + 3, n, 1)):
        m = b - a
        cs, os_ = m + 37, fs.next_out_len(m, bool(flush)) + 51
        buf = torch.zeros((n_ch, cs), dtype=torch.complex64, device=ctx.tdev)
        buf[:, :m] = torch.from_numpy(x[:, a:b]).to(ctx.tdev)
        out = torch.full((n_ch, os_), 7.0 + 7.0j, dtype=torch.complex64, device=ctx.tdev)
        no = C.c_size_t()
        capi.check(lib.lrc_fastfir_stream_push(fs.h, C.c_void_p(buf.data_ptr()), m, cs, C.c_void_p(out.data_ptr()), os_,
                                               flush, C.byref(no), blocks._stream()), "push")
        o = out.cpu().numpy()
        assert np.all(o[:, no.value:] == 7.0 + 7.0j)              # nothing written past n_out in a row
        for c in range(n_ch):
            got[c].append(o[c, :no.value])
    for c in range(n_ch):
        assert np.array_equal(bits(np.concatenate(got[c])), bits(refs[c]))
    fs.close(); ff.close()


@pytest.mark.parametrize("nh,nfft", [(300, 0), (4096, 0)])
def test_reset_and_flush_return_to_the_initial_state(ctx, nh, nfft):
    ff = blocks.FastFir(ctx, taps(nh, 21), nfft)
    nc, good = compute_block(ff)
    n = 2 * nc + 500
    x = signal(2, n, 22)
    refs = oneshot(ctx, ff, x)
    fs = blocks.FastFirStream(ff, 2)
    fs.push(torch.from_numpy(signal(2, nc + 123, 23)).to(ctx.tdev))   # some history, then reset
    fs.reset()
    got = stream(ctx, fs, x, [0, 333, nc + 1, n], refs)
    got2 = stream(ctx, fs, x, [0, n // 2, n], refs)                     # right after a flushing push
    for c in range(2):
        assert np.array_equal(bits(got[c]), bits(refs[c])) and np.array_equal(bits(got2[c]), bits(refs[c]))
    # a flush with fewer than nh samples held emits nothing
    for held in (0, 1, nh - 1):
        if held:
            assert fs.push(torch.from_numpy(signal(2, held, 24)).to(ctx.tdev)).shape == (2, 0)
        assert fs.next_out_len(0, True) == 0
        assert fs.push(torch.zeros((2, 0), dtype=torch.complex64, device=ctx.tdev), True).shape == (2, 0)
    # ... and with held samples past whole blocks, only what the one-shot keeps
    m = nc + good                                           # two blocks, then nh - 1 samples: no flush outputs
    assert fs.next_out_len(m, True) == fs.next_out_len(m, False) == 2 * good
    fs.close(); ff.close()


def test_errors(ctx):
    lib = ctx.lib
    ff = blocks.FastFir(ctx, taps(300, 31), 0)
    st = C.c_void_p()
    assert lib.lrc_fastfir_stream_create(ff.h, 0, C.byref(st)) == capi.ERR_INVALID
    assert lib.lrc_fastfir_stream_create(None, 2, C.byref(st)) == capi.ERR_INVALID
    fs = blocks.FastFirStream(ff, 2)
    n = 3000
    x = torch.zeros((2, n + 1), dtype=torch.complex64, device=ctx.tdev)
    out = torch.empty((2, 4096), dtype=torch.complex64, device=ctx.tdev)
    no = C.c_size_t()
    s = blocks._stream()
    xp, op = x.data_ptr(), out.data_ptr()
    push = lambda *a: lib.lrc_fastfir_stream_push(*a)
    assert push(None, C.c_void_p(xp), n, n, C.c_void_p(op), 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    assert push(fs.h, None, n, n, C.c_void_p(op), 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    assert push(fs.h, C.c_void_p(xp), n, n, None, 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    assert push(fs.h, C.c_void_p(xp), n, n, C.c_void_p(op), 4096, 0, None, s) == capi.ERR_INVALID
    assert push(fs.h, C.c_void_p(xp + 4), n, n, C.c_void_p(op), 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    assert push(fs.h, C.c_void_p(xp), n, n, C.c_void_p(op + 4), 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    assert push(fs.h, C.c_void_p(xp), n, n - 1, C.c_void_p(op), 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    assert push(fs.h, C.c_void_p(xp), n, n, C.c_void_p(xp + 8 * 100), 4096, 0, C.byref(no), s) == capi.ERR_INVALID
    want = fs.next_out_len(n, False)
    assert want > 0
    assert push(fs.h, C.c_void_p(xp), n, n, C.c_void_p(op), want - 1, 0, C.byref(no), s) == capi.ERR_CAPACITY
    # a refused push consumed nothing: the stream still equals a fresh one
    xs = signal(2, 5000, 32)
    refs = oneshot(ctx, ff, xs)
    got = stream(ctx, fs, xs, [0, 2500, 5000], refs)
    assert all(np.array_equal(bits(got[c]), bits(refs[c])) for c in range(2))
    fs.close(); ff.close()


def test_config5_shape_8_channels_of_2_24_random_pushes(ctx):
    """config 5's taps (4096, rng(6)/64), 8 channels x 2^24 samples on the device, pushes of about 2^20"""
    nh, n, n_ch = 4096, 1 << 24, 8
    rng = np.random.default_rng(6)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64).astype(np.complex64)
    ff = blocks.FastFir(ctx, h, 0)
    g = torch.Generator(device=ctx.tdev).manual_seed(7)
    x = torch.view_as_complex(torch.randn(n_ch, n, 2, device=ctx.tdev, generator=g))
    fs = blocks.FastFirStream(ff, n_ch)
    cuts = [0]
    while cuts[-1] < n:
        cuts.append(min(n, cuts[-1] + int(rng.integers(1 << 19, 3 << 19))))
    outs = []
    for k, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        outs.append(fs.push(x[:, a:b].contiguous(), k == len(cuts) - 2))
    y = torch.cat(outs, dim=1)
    for c in range(n_ch):
        ref = ff.run(x[c].contiguous(), True)
        assert y.shape[1] == ref.numel() == n - nh + 1
        assert torch.equal(torch.view_as_real(y[c]).view(torch.int32), torch.view_as_real(ref).view(torch.int32)), c
    fs.close(); ff.close()


def test_kpn_fast_fir_multi_block_in_a_threaded_graph():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "kpn"), "test_gpu_fastfir_stream"])
    out = subprocess.run([os.path.join(ROOT, "kpn", "test_gpu_fastfir_stream")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "kpn fastfir stream OK" in out.stdout, out.stdout + out.stderr
