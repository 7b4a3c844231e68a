"""CPU suite, part 1: the oracle against the reference's own golden vectors, known-answer tests and the
fixtures generated from the vendored kissfft (tests/golden/make_golden.py).  No GPU, no product code."""
import os

import numpy as np
import pytest

import oracle
from oracle import defined_f64 as D


# ---- (1) i2f / data_to_samples: rtlsdr.rs:159-162 ----------------------------------------------------
def test_i2f_hand_computed_micro_cases():
    assert oracle.i2f(0) == np.float32(-1.0)
    assert oracle.i2f(127) == np.float32(0.0)
    assert oracle.i2f(254) == np.float32(1.0)
    assert oracle.i2f(255) == np.float32(1.007874)
    assert oracle.i2f(128) == np.float32(np.float32(128) / np.float32(127)) - np.float32(1)


def test_data_to_samples_all_bytes_against_numpy_f32_ops():
    b = np.arange(256, dtype=np.uint8).repeat(2)
    got = oracle.data_to_samples(b)
    ref = b.astype(np.float32) / np.float32(127.0) - np.float32(1.0)      # one f32 div, one f32 sub
    assert np.array_equal(got.view(np.float32), ref)
    with pytest.raises(IndexError):
        oracle.data_to_samples(np.zeros(3, np.uint8))


# ---- (2) convolve: dsputils.rs:30-32 --------------------------------------------------------------------
def test_convolve_is_valid_mode_correlation_left_fold():
    u = np.array([1, 2, 3, 4, 5], np.float32)
    v = np.array([10, 1], np.float32)
    assert oracle.convolve(u, v).tolist() == [12.0, 23.0, 34.0, 45.0]      # taps NOT reversed
    assert oracle.convolve(u[:1], v).size == 0
    # left fold from 0 in f32: (((0 + a) + b) + c), visible with cancellation
    u = np.array([1e8, 1.0, -1e8], np.float32)
    v = np.ones(3, np.float32)
    assert oracle.convolve(u, v)[0] == np.float32(np.float32(np.float32(0 + 1e8) + 1) - 1e8) == 0.0


def test_fir_decimate_definition():
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(1000) + 1j * rng.standard_normal(1000)).astype(np.complex64)
    taps = rng.standard_normal(64).astype(np.float32)
    for d in (1, 3, 10, 64, 100):
        z = oracle.fir_decimate(x, taps, d)
        assert z.size == (1000 - 64) // d + 1
        assert np.array_equal(z.view(np.float32), oracle.fir_decimate(x, taps, d, full=True).view(np.float32))
        assert np.array_equal(z.real, oracle.convolve(x.real.copy(), taps)[::d])
        assert np.array_equal(z.imag, oracle.convolve(x.imag.copy(), taps)[::d])
        ref = np.correlate(x.astype(np.complex128), taps.astype(np.float64), "valid")[::d]
        assert np.max(np.abs(z - ref)) < 1e-4 * np.sqrt(np.mean(np.abs(ref) ** 2))


def test_window_bug_of_reference_is_reproduced_and_corrected_designer_is_finite():
    w = oracle.window(64, faithful=True)                 # dsputils.rs:49 swapped arguments
    assert w.size == 65 and not np.isfinite(w[1])
    assert not np.all(np.isfinite(oracle.lpf(64, 0.04, faithful=True)))
    good = oracle.lpf(64, 0.04, faithful=False)
    assert np.all(np.isfinite(good)) and abs(good.sum() - 1.0) < 0.05
    from libredio_b200 import synth
    assert np.max(np.abs(synth.lpf_taps(64, 0.04) - good)) < 1e-6


def test_hpf_bsf_bpf_designers_restated_and_corrected():
    """dsputils.rs:74-94.  Faithful restatement: NaN like lpf (the window bug, :49).  Corrected window: finite, the
    product's host designers (libredio_b200/synth.py) equal the oracle's, and the formulas are kept as written --
    the 1.0 of hpf at index m/2 - 1 (:77), bsf = lpf(fc1) + hpf(fc2) (:82-88), bpf = -bsf (:91-94)."""
    from libredio_b200 import synth
    m = 64
    for fn, args in ((oracle.hpf, (0.1,)), (oracle.bsf, (0.05, 0.2)), (oracle.bpf, (0.05, 0.2))):
        assert np.isnan(fn(m, *args, faithful=True)).any()
        assert np.isfinite(fn(m, *args)).all()
    lp, hp = oracle.lpf(m, 0.1), oracle.hpf(m, 0.1)
    want = -lp
    want[m // 2 - 1] = np.float32(want[m // 2 - 1] + np.float32(1.0))
    assert np.array_equal(hp.view(np.uint32), want.view(np.uint32))
    bs, bp = oracle.bsf(m, 0.05, 0.2), oracle.bpf(m, 0.05, 0.2)
    assert np.array_equal(bs.view(np.uint32), (oracle.lpf(m, 0.05) + oracle.hpf(m, 0.2)).view(np.uint32))
    assert np.array_equal(bp.view(np.uint32), (-bs).view(np.uint32))
    assert np.max(np.abs(synth.hpf_taps(m, 0.1) - hp)) < 1e-6
    assert np.max(np.abs(synth.bsf_taps(m, 0.05, 0.2) - bs)) < 1e-6
    assert np.max(np.abs(synth.bpf_taps(m, 0.05, 0.2) - bp)) < 1e-6

    def gain(h, f):
        n = np.arange(h.size)
        return abs(np.sum(h.astype(np.float64) * np.exp(-2j * np.pi * f * n)))
    assert gain(hp, 0.0) < 2e-3 and abs(gain(hp, 0.3) - 1.0) < 2e-3            # a high-pass
    assert abs(gain(bs, 0.0) - 1.0) < 5e-3 and abs(gain(bs, 0.35) - 1.0) < 5e-3 and gain(bs, 0.1) < 0.7


# ---- (3) FFT vs the reference's outputs -----------------------------------------------------------------
def test_restated_fft_vs_golden_fixtures_from_vendored_kissfft(golden):
    import tests.golden.make_golden as mg
    for n in golden["fft_sizes"]:
        n = int(n)
        x = mg.fft_input(n)
        for inv, key in ((False, f"fwd_{n}"), (True, f"inv_{n}")):
            got = oracle.fft(x, inv)
            ref = golden[key]
            if n & (n - 1) == 0:     # radix-4/2 path restated operation by operation: bit-identical
                assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (n, inv)
            else:                    # radix 3/5 use the generic O(p^2) sum: last-bit differences only
                assert np.max(np.abs(got - ref)) < 2e-6 * np.sqrt(np.mean(np.abs(ref) ** 2)), (n, inv)


def test_restated_fft_vs_mixed_radix_and_real_fixtures(golden):
    """radix 3/5/generic sizes and the kiss_fftr pair: fixtures from the vendored build vs the restatement
    and vs f64 numpy (SNR thresholds of the reference's self tests, mk_test.py:30)."""
    import tests.golden.make_golden as mg
    for n in golden["mixed_sizes"]:
        n = int(n)
        x = mg.fft_input(n)
        for inv, key in ((False, f"fwd_{n}"), (True, f"inv_{n}")):
            ref = golden[key]
            assert np.max(np.abs(oracle.fft(x, inv) - ref)) < 2e-5 * np.sqrt(np.mean(np.abs(ref) ** 2)), (n, inv)
            exact = np.fft.ifft(x.astype(np.complex128)) * n if inv else np.fft.fft(x.astype(np.complex128))
            assert D.snr_db(exact, ref) >= 100.0, (n, inv)
    for n in golden["rfft_sizes"]:
        n = int(n)
        t = mg.rfft_input(n)
        assert D.snr_db(np.fft.rfft(t.astype(np.float64)), golden[f"rfft_{n}"]) >= 100.0
        assert D.snr_db(n * t.astype(np.float64), golden[f"irfft_{n}"]) >= 100.0
        if oracle.have_ref():
            assert np.array_equal(oracle.ref_fftr(t).view(np.uint32), golden[f"rfft_{n}"].view(np.uint32))


def test_psdpng_rows_restatement_vs_fixture_and_f64(golden):
    """psdpng.c:120-185 restated around the vendored kiss_fftr == committed fixture; and close to an f64 model."""
    import tests.golden.make_golden as mg
    for stereo in (False, True):
        for dc in (False, True):
            pcm = mg.psdpng_input(stereo)
            ref = golden[f"psdpng_{int(stereo)}{int(dc)}"]
            if oracle.have_ref():
                assert np.array_equal(oracle.psdpng_rows(pcm, 256, 3, dc, stereo).view(np.uint32), ref.view(np.uint32))
            x = pcm.astype(np.float64)
            x = x.reshape(-1, 2).sum(axis=1) if stereo else x
            fr = x[: 6 * 256].reshape(6, 256)
            if dc:
                fr = fr - fr.mean(axis=1, keepdims=True)
            p = (np.abs(np.fft.rfft(fr, axis=1)) ** 2).reshape(2, 3, 129).mean(axis=1)
            # after -a the DC bin is rounding noise of the mean removal: compare above a 0 dB floor (the +1 of :173)
            model = 10 * np.log10(p + 1)
            assert np.max(np.abs(model - ref)) < 1e-3 * np.sqrt(np.mean(model ** 2))


def test_only_golden_vector_of_the_reference_tree(golden):
    """test/fft.py:95-98, tolerance 1e-5 (:104)"""
    F = oracle.fft(golden["fftpy_tvec"].astype(np.complex64))
    assert np.max(np.abs(F - golden["fftpy_Ftvec"])) < 1e-5


@pytest.mark.parametrize("n", [8, 36, 240, 1024, 1800])
def test_fft_self_test_thresholds_of_reference(n):
    """test_vs_dft.c / mk_test.py:30: SNR vs an exact DFT >= 100 dB for float"""
    rng = np.random.default_rng(n)
    x = (rng.integers(-32768, 32768, n) + 1j * rng.integers(-32768, 32768, n)).astype(np.complex64)
    assert D.snr_db(np.fft.fft(x.astype(np.complex128)), oracle.fft(x)) >= 100.0
    assert D.snr_db(np.fft.ifft(x.astype(np.complex128)) * n, oracle.fft(x, True)) >= 100.0


def test_restated_fft_and_fastfir_bit_exact_vs_vendored_build(golden):
    """Bit for bit against the vendored kissfft: its stored outputs (tests/golden) always -- radix 4/2 and the generic odd-prime
    butterfly (7; 11 and 13 inside 1001), kiss_fastfir with and without flush -- and the live build too where oracle/_ref exists."""
    import tests.golden.make_golden as mg
    for n in (2, 64, 1024, 8192, 7, 97, 1001, 7919):
        x = mg.fft_input(n)
        for inv, key in ((False, f"fwd_{n}"), (True, f"inv_{n}")):
            assert np.array_equal(oracle.fft(x, inv).view(np.uint32), golden[key].view(np.uint32)), (n, inv)
    h, x = mg.fastfir_case()
    for flush, key in ((False, "fastfir_noflush"), (True, "fastfir_flush")):
        assert np.array_equal(oracle.fastfir(h, x, 0, flush).view(np.uint32), golden[key].view(np.uint32)), flush
    if not oracle.have_ref():
        return
    rng = np.random.default_rng(1)
    for n in (2, 64, 1024, 8192, 7, 11):
        x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        for inv in (False, True):
            assert np.array_equal(oracle.fft(x, inv).view(np.uint32), oracle.ref_kissfft(x, inv).view(np.uint32))
    h = (rng.standard_normal(77) + 1j * rng.standard_normal(77)).astype(np.complex64)
    x = (rng.standard_normal(5000) + 1j * rng.standard_normal(5000)).astype(np.complex64)
    for flush in (False, True):
        assert np.array_equal(oracle.fastfir(h, x, 0, flush).view(np.uint32), oracle.ref_fastfir(h, x, 0, flush).view(np.uint32))
    assert np.max(np.abs(oracle.ref_fftr(np.arange(8, dtype=np.float32)) - np.fft.rfft(np.arange(8)))) < 1e-5


def test_fastfir_vs_golden_and_definition(golden):
    import tests.golden.make_golden as mg
    h, x = mg.fastfir_case()
    for flush, key in ((False, "fastfir_noflush"), (True, "fastfir_flush")):
        got = oracle.fastfir(h, x, 0, flush)
        assert np.array_equal(got.view(np.uint32), golden[key].view(np.uint32))
    full = np.convolve(x.astype(np.complex128), h.astype(np.complex128))[h.size - 1:]
    got = oracle.fastfir(h, x, 0, True)
    assert got.size == x.size - h.size + 1                       # flush recovers every valid output
    assert np.max(np.abs(got - full[: got.size])) < 1e-4 * np.sqrt(np.mean(np.abs(full) ** 2))
    assert oracle.fastfir(h, x[:500], 0, False).size == 0        # less than one block (nfft = 1024)


# ---- (5) OOK chain ------------------------------------------------------------------------------------------
def f32(x):
    return np.float32(x)


def test_trigger_state_machine_hand_traced():
    """bitfount.rs:46-81 traced by hand in numpy f32 on constant blocks"""
    env = np.full(512, 0.01, np.float32)
    s = f32(0)
    for v in env:
        s = f32(s + v)
    quiet = np.zeros(20 * 1024, np.uint8) + 127                   # envelope exactly 0 -> s = 0 every block
    r = oracle.ook_decode(quiet)
    assert r["n_bursts"] == 0 and np.all(r["block_sums"] == 0) and r["bits"].size == 0
    # threshold evolution for a constant block sum s: thr0 = s; each block thr += s/1000; thr -= thr*0.002
    thr = s
    for _ in range(5):
        thr = f32(thr + f32(s / f32(1000)))
        thr = f32(thr - f32(thr * f32(0.002)))
    assert thr < s and not (s > f32(thr * f32(4)))                 # a constant floor never fires


def test_first_burst_has_leading_zero_and_49_blocks():
    rng = np.random.default_rng(3)
    n_blocks = 200
    iq = np.clip(np.rint(127 + rng.standard_normal(n_blocks * 1024)), 0, 255).astype(np.uint8)
    iq[100 * 1024:101 * 1024] = 255                                # one loud block fires the trigger
    r = oracle.ook_decode(iq)
    assert r["n_bursts"] == 1
    # counter 50 (the firing block) .. 2 are collected = 49 blocks, plus the 0.0 of vec!(0.0) (bitfount.rs:43)
    assert r["bits"].size == 49 * 512 + 1
    assert r["bits"][0] == 0 and r["bits"][1:513].all() and not r["bits"][513:].any()
    # rle: (0,1) then (1,512) are emitted; the trailing zero run is never flushed (kpn.rs:17-29)
    assert r["run_val"].tolist() == [0, 1] and r["run_len"].tolist() == [1, 512]


def test_discretize_and_norm_definition():
    b = oracle.discretize(np.array([0.0, 1.0, 0.5, 0.50001, 2.0], np.float32))
    assert b.tolist() == [0, 0, 0, 0, 1]                           # x > max/2, strict
    assert oracle.norm(3.0, 4.0) == 5.0
    t = oracle.norm_table()
    assert t.shape == (256, 256) and t[127, 127] == 0 and np.array_equal(t, t.T)


def test_b2d_and_eat_micro_cases():
    assert oracle.b2d([1, 0, 1]) == 5 and oracle.b2d([]) == 0 and oracle.b2d([1] * 12) == 4095
    bits = [0, 1, 0, 1] + [1, 0, 0, 0, 0, 1, 1, 1] + [0, 1, 1, 0] + [0] * 11 + [1] + [1] * 8
    assert oracle.eat(bits, [4, 8, 4, 12, 8]) == [5, 135, 6, 1, 255]
    assert oracle.eat(bits, [4, 8, 2, 10, 12]) == [5, 135, 1, 512, 511]


def test_ook_chain_decodes_constructed_packets():
    from libredio_b200 import synth
    for seed in range(6):
        iq, sent = synth.ook_capture_u8(800, seed=seed, n_packets=3)
        r = oracle.ook_decode(iq)
        assert [tuple(p) for p in r["a_packets"]] == [tuple(b) for pr, b in sent if pr == 0]
        assert [tuple(p) for p in r["b_packets"]] == [tuple(b) for pr, b in sent if pr == 1]


# ---- north-star-defined stages ---------------------------------------------------------------------------------
def _same(a: dict, b: dict):
    assert a["n_bursts"] == b["n_bursts"]
    for k in ("block_sums", "bits", "run_val", "run_len", "a_packets", "b_packets"):
        x, y = a[k], b[k]
        assert x.shape == y.shape, k
        if x.dtype == np.float32:
            x, y = x.view(np.uint32), y.view(np.uint32)
        assert np.array_equal(x, y), k


@pytest.mark.parametrize("seed,n_blocks,n_packets", [(4, 420, 2), (7, 300, 1), (11, 520, 3), (23, 64, 0)])
def test_ook_chain_two_independent_restatements_agree_bit_for_bit(seed, n_blocks, n_packets):
    """The reference has no test or vector for the OOK chain, so the C restatement (the GPU's oracle) is checked
    against a second restatement written independently from the same Rust as a network of generator blocks
    (oracle/restated_py.py): block sums, bursts, bit stream, every run and the packets must be identical."""
    from oracle import restated_py as P
    from libredio_b200 import synth                     # synthetic input generator only (numpy, no device code)
    iq, sent = synth.ook_capture_u8(n_blocks, seed=seed, n_packets=n_packets)
    a, b = oracle.ook_decode(iq), P.ook_decode(iq)
    _same(a, b)
    if n_packets:       # rle never flushes its last run, so the final packet may stay inside the chain (kpn.rs:17-29)
        assert len(sent) - 1 <= a["a_packets"].shape[0] + a["b_packets"].shape[0] <= len(sent)


@pytest.mark.parametrize("loud,before", [(72, False), (73, True), (200, True)])
def test_ook_chain_restatements_agree_on_the_oom_guard_path(loud, before):
    """bitfount.rs:52-54 with the guard shrunk to 120 blocks in both restatements (the reference's 50 000 blocks would need 100 s
    of capture): abandoned pieces, the remainder sent with a leading 0.0, and -- loud + 48 collected blocks == the guard -- the
    reset buffer [0.0] sent on its own as a single 0 bit."""
    from oracle import restated_py as P
    from libredio_b200 import synth
    iq = synth.ook_guard_capture_u8(loud, seed=loud, before=before, after=True)
    oracle.set_trigger_guard_blocks(120)
    try:
        a, b = oracle.ook_decode(iq), P.ook_decode(iq)
    finally:
        oracle.set_trigger_guard_blocks(0)
    _same(a, b)
    if loud != 200:
        assert a["bits"].size == (2 if before else 1) * (51 * 512 + 1), "the lone 0 bit is there (the other +1: vec!(0.0) of the first burst)"
    full = oracle.ook_decode(iq)                             # the reference's constant: a capture this short never reaches it,
    if loud != 200:                                          # the stretch is sent whole instead of its reset buffer
        assert full["bits"].size == a["bits"].size - 1 + (loud + 48) * 512 + (0 if before else 1)      # + its own vec!(0.0)


def test_ook_chain_restatements_agree_on_unstructured_input():
    """not packets: amplitude steps and noise bursts that drive the threshold arithmetic (bitfount.rs:57-70) through
    re-triggers, a burst still open at the end of the capture and runs spanning burst boundaries"""
    from oracle import restated_py as P
    rng = np.random.default_rng(99)
    n_blocks = 520
    n = n_blocks * 512
    amp = np.zeros(n)
    pos = 50 * 512
    k = 0
    while pos < n - 3000:
        ln = int(rng.integers(40, 20_000))
        amp[pos:pos + ln] = rng.uniform(0.05, 0.9)
        # short gaps keep a burst open (re-trigger, bitfount.rs:68-70); every third gap is long enough (> 50 blocks)
        # for the counter to run out so that the burst is sent
        k += 1
        pos += ln + (int(rng.integers(100, 9000)) if k % 3 else int(rng.integers(56, 70)) * 512)
    amp[-20_000:] = 0.8                                        # open burst at the end: never sent (bitfount.rs:78-81)
    ph = rng.uniform(0, 2 * np.pi, n)
    i = 127 + 127 * amp * np.cos(ph) + 1.5 * rng.standard_normal(n)
    q = 127 + 127 * amp * np.sin(ph) + 1.5 * rng.standard_normal(n)
    iq = np.empty(2 * n)
    iq[0::2], iq[1::2] = i, q
    iq = np.clip(np.rint(iq), 0, 255).astype(np.uint8)
    a, b = oracle.ook_decode(iq), P.ook_decode(iq)
    assert a["n_bursts"] >= 2 and a["run_len"].size > 5
    _same(a, b)


def test_unpack_and_convolve_two_independent_restatements_agree_bit_for_bit():
    """rtlsdr.rs:159-162 and dsputils.rs:30-32 have no test in the reference either: C restatement == Python restatement"""
    from oracle import restated_py as P
    rng = np.random.default_rng(17)
    data = rng.integers(0, 256, 4096, dtype=np.uint8)
    a = oracle.data_to_samples(data)
    b = np.array([complex(float(re), float(im)) for re, im in P.data_to_samples(data)], dtype=np.complex64)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    with pytest.raises(IndexError):
        P.data_to_samples(data[:7])                                # odd length: the reference panics (rtlsdr.rs:161)
    u = (rng.standard_normal(700) * 3).astype(np.float32)
    for m in (1, 2, 64, 699, 700):
        v = rng.standard_normal(m).astype(np.float32)
        c = oracle.convolve(u, v)
        p = np.array(P.convolve(u, v), dtype=np.float32)
        assert c.shape == p.shape == (700 - m + 1,)
        assert np.array_equal(c.view(np.uint32), p.view(np.uint32))
    assert P.convolve(u[:3], u[:5]) == [] and oracle.convolve(u[:3], u[:5]).size == 0


def test_python_restatement_micro_cases():
    from oracle import restated_py as P
    assert [float(P.i2f(b)) for b in (0, 127, 254)] == [-1.0, 0.0, 1.0]
    assert P.i2f(255).view(np.uint32) == oracle.i2f(255).view(np.uint32)
    assert P.b2d([1, 0, 1]) == 5 and P.eat([1, 0, 1, 1, 1, 1], [3, 3]) == [5, 7]
    assert list(P.rle(iter([1, 1, 0, 0, 0, 1]))) == [(1, 2), (0, 3)]           # the last run is never flushed
    assert list(P.shaper_optional(iter([1, 0, None, 1, None, 1, 1, None]), 2)) == [[1, 0], [1, 1]]
    # matcher A consumes the next run only after a matching pulse (ratpak.rs:91)
    d = [(1, np.float32(3e-4)), (0, np.float32(2e-3)), (0, np.float32(2e-3)), (1, np.float32(3e-4)), (0, np.float32(4e-3)),
         (1, np.float32(3e-4)), (0, np.float32(3e-3))]
    assert list(P.matcher_a(iter(d))) == [0, None, 1, None]


@pytest.mark.parametrize("ratio", [0.2, 0.5, 2.0, 48000 / 44100, 3 / 7])
def test_resampler_definition_is_plain_polyphase_and_in_sinc_medium_class(ratio):
    """libsamplerate is absent (parity unpinned, DESIGN.md section 2), so the f64 definition is checked two ways:
    (1) it IS the textbook rational polyphase filter -- identical to scipy.signal.upfirdn with the same prototype;
    (2) the prototype sits in the class of the converter the reference asks for (SRC_SINC_MEDIUM_QUALITY,
    samplerate.rs:61: ~121 dB SNR, ~90 % bandwidth): >= 120 dB rejection from 1.1x the slower Nyquist on, -6 dB at
    0.9x, < 0.01 dB ripple over the lower 80 %."""
    import scipy.signal as ss
    L, M = D.resampler_ratio(ratio)
    h = D.resampler_taps(L, M)
    x = np.random.default_rng(5).standard_normal(5000)
    y = D.resample(x, ratio)
    u = ss.upfirdn(h, x, up=L, down=M)[: y.size]
    assert np.max(np.abs(y - u)) < 1e-12
    nfft = 1 << 22 if h.size > (1 << 12) else 1 << 20
    H = np.abs(np.fft.rfft(h, nfft)) / L
    f = np.arange(H.size) / nfft                        # cycles per sample at the L-times-upsampled rate
    fc = 0.5 / max(L, M)                                # Nyquist of the slower of the two rates
    assert 20 * np.log10(H[f >= 1.1 * fc].max()) <= -120.0
    pb = H[f <= 0.8 * fc]
    assert 20 * np.log10(pb.max() / pb.min()) < 0.01
    assert abs(20 * np.log10(H[np.searchsorted(f, 0.9 * fc)]) + 6.02) < 0.1


def _load_model(name):
    import importlib.util
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "models", name + ".py")
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_packed_resampler_index_model_matches_the_definition_on_many_shapes():
    """tools/models/resample_dec2_model.py follows the host and device index arithmetic of the packed two-tile
    decimator line by line (virtual row, s0, tile pairing, the three fill paths, windows, store predicates, carry
    update); swept here over kernel configurations, channel counts and chunkings the GPU tests do not reach -- odd tile
    counts, a pair spanning two channels, outputs that are an exact multiple of a tile, one-sample chunks."""
    m = _load_model("resample_dec2_model")
    rng = np.random.default_rng(0)
    seen = {"full": 0, "fast": 0, "generic": 0}
    for M, R, NT in [(5, 6, 64), (5, 6, 128), (2, 7, 128), (3, 6, 128), (6, 5, 128)]:
        h = D.resampler_taps(1, M)
        tile = R * NT * M
        for n_ch, chunks in [(1, [5000]), (3, [1, 4, 5, 990, 11_000]), (2, [1200 * M + 7, 3]), (5, [2 * tile]),
                             (4, [2 * tile + 1, tile - 1]), (1, [6 * tile])]:
            mod = m.Dec2Model(M, R, NT, n_ch, h)
            x = rng.standard_normal((n_ch, sum(chunks)))
            outs, pos = [], 0
            for c in chunks:
                outs.append(mod.process(x[:, pos:pos + c]))
                pos += c
            got = np.concatenate(outs, axis=1)
            for c in range(n_ch):
                ref = D.resample(x[c], 1.0 / M, taps=h)
                assert got[c].shape == ref.shape
                assert np.max(np.abs(got[c] - ref)) < 1e-10
            for k in seen:
                seen[k] += mod.paths[k]
    assert all(v > 0 for v in seen.values()), seen            # every fill path was taken


def test_fastfir16k_design_model_is_an_exact_overlap_save():
    """tools/models/fastfir16k_model.py mirrors, index for index, the data flow of the nfft = 16384 kernel (k_fastfir16k.cu)
    (16 x 1024 split, lane-slab rows of pitch 34, column pairs per P1 thread, warp-level 32 x 32 sub-transforms through
    the row buffer, H stored as Hq[k1][i][lane][c]); it must reproduce the direct convolution to f64 accuracy."""
    m = _load_model("fastfir16k_model")
    rng = np.random.default_rng(3)
    nh = 4096
    h = (rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64
    x = rng.standard_normal(m.N + 12289) + 1j * rng.standard_normal(m.N + 12289)
    y = m.fastfir(h, x)
    assert y.size == 2 * 12289
    ref = np.convolve(x, h)[nh - 1: nh - 1 + y.size]
    assert np.max(np.abs(y - ref)) <= 1e-12 * np.sqrt(np.mean(np.abs(ref) ** 2))


def test_round2_index_models_exhaustive():
    """the integer arithmetic the round-2 kernels rely on (tools/models/index_models.py restates it index for index)"""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "models"))
    import index_models as im
    # folded envelope table: every sorted pair has its own slot inside the table, whatever the order of the two bytes
    seen = {}
    for hi in range(256):
        for lo in range(hi + 1):
            idx = im.ook_fold_index(hi << 8 | lo)
            assert im.OOK_FOLD_MIN <= idx <= im.OOK_FOLD_MAX and idx not in seen
            seen[idx] = (hi, lo)
    assert len(seen) == 256 * 257 // 2
    rng = np.random.default_rng(0)
    for w in rng.integers(0, 1 << 32, 20000, dtype=np.uint64).tolist() + [0, 0xFFFFFFFF, 0x00FF00FF, 0xFF00FF00, 0x7F7F7F7F]:
        b = [(w >> (8 * i)) & 255 for i in range(4)]
        k0, k1 = im.sorted_key_pair(w)
        assert k0 == max(b[0], b[1]) << 8 | min(b[0], b[1]) and k1 == max(b[2], b[3]) << 8 | min(b[2], b[3])
    # rows of both tables start 8 banks apart (4-byte / 2-byte entries: 264 entries per row)
    assert im.ook_fold_index(200 << 8) - im.ook_fold_index(199 << 8) == 264
    slots = {im.ook_rank_slot(raw) for raw in range(65536)}
    assert len(slots) == 65536 and max(slots) < 256 * 264
    # padded-chunk tile: windows never straddle a pad inside a 16-byte pair load, thread windows start an odd number of
    # 16-byte units apart, and every sample a (zero-padded) tap can reach is either copied or lies behind the copied extent
    for ntaps_max in (64, 128):
        for decim, r in ((4, 8), (5, 8), (8, 7), (10, 7), (16, 4)):
            step, win, winl, padb, pitch = im.gen_tile(ntaps_max, decim, r)
            offs = im.gen_tile_offsets(ntaps_max, decim, r)
            assert pitch % 16 == 0 and (pitch // 16) % 2 == 1
            assert all(o % 8 == 0 for o in offs) and all(offs[j + 1] == offs[j] + 8 for j in range(0, winl, 2))
            assert all(offs[j] % 16 == 0 for j in range(0, winl, 2))
            for t in (0, 1, 5):                                  # window of thread t = the same samples seen from chunk t
                for j in range(winl):
                    i = t * step + j                             # tile sample index
                    assert t * pitch + offs[j] == (i // step) * pitch + (i % step) * 8
            for n in (512, 1024):
                for ntaps in (1, 2, 17, 63, ntaps_max - 1, ntaps_max):
                    tile_in = (n - 1) * decim + ntaps
                    covered = np.zeros(tile_in, bool)
                    for c, s0, ns, hand in im.chunk_plan(tile_in, step):
                        assert ns % 2 == 0 and (s0 * 8) % 16 == 0
                        covered[s0:s0 + ns] = True
                        if hand is not None:
                            assert s0 <= hand < s0 + step and not covered[hand]
                            covered[hand] = True
                    assert covered.all()


def test_trigger_bookkeeping_from_masks_equals_the_blockwise_statements():
    """ook_trigger_kernel, round 2: the walker leaves collect / send bit masks per tile of 32 blocks; the keeper steps from send to
    send (buffer length by popc) and the helpers expand the tags (burst index at the start of the tile + sends before the block).
    tools/models/index_models.py restates both that and bitfount.rs:52-54,73-81 taken block by block: same tags, same burst
    events, same state -- with the reference's guard, a shrunk one (the block-by-block tiles near it) and a tiny burst capacity."""
    import sys
    import random
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "models"))
    import index_models as im
    random.seed(1)

    def masks(n_tiles, p_fire, long_run):
        tiles, trig = [], 0
        for t in range(n_tiles):
            cm = sm = 0
            nb = 32 if t < n_tiles - 1 else random.randint(1, 32)
            for u in range(nb):
                trig -= 1
                if random.random() < (0.9 if long_run else p_fire):
                    trig = 50 if long_run else random.choice([50, 50, 3, 2])
                cm |= (trig > 1) << u
                sm |= (trig == 0) << u
            tiles.append((cm, sm, nb))
        return tiles

    n_events = 0
    for it in range(300):
        tiles = masks(random.randint(1, 20), random.choice([0.01, 0.05, 0.3]), it % 7 == 0)
        for guard in (1000 * 50 * 512, 120 * 512, 40 * 512):
            for cap in (1000, 3):
                a, b = im.keeper_blockwise(tiles, guard, cap), im.keeper_send_to_send(tiles, guard, cap)
                assert a == b
                n_events += len(a[1])
    assert n_events > 1000


def test_split_slicer_model_equals_the_flattened_bit_stream():
    """ook_slice_kernel / ook_scan_kernel / ook_scatter_kernel place every collected block in the bit stream and in the transition
    list from per-block summaries and prefix sums, 32 blocks per step.  That is restated in tools/models/index_models.py and
    compared with the plainest statement there is: flatten the sent bursts (leading 0.0 bit, lone [0.0] bursts of the OOM guard,
    abandoned bursts contributing nothing) and record where the value changes (kpn.rs:17-29)."""
    import sys
    import random
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "models"))
    import index_models as im
    random.seed(3)

    def stream(n_blocks, p_lone, noisy):
        blocks, flags, burst, k, first = [], [], 0, 0, True
        while k < n_blocks:
            for _ in range(min(random.randint(0, 40), n_blocks - k)):
                blocks.append((-1, None)); k += 1
            if k >= n_blocks:
                break
            while random.random() < p_lone:                      # abandoned (0) or lone [0.0] (3) bursts in front of this one
                flags.append(random.choice([0, 3])); burst += 1
            flags.append(1 | (2 if (first or random.random() < 0.3) else 0)); first = False
            for i in range(min(random.randint(1, 70), n_blocks - k)):
                if i and random.random() < 0.1:                  # a hole: the block at counter 1 is not collected
                    blocks.append((-1, None)); k += 1
                    continue
                m = random.random()
                if m < 0.5:
                    bits = [0] * 512
                elif m < 0.6:
                    bits = [1] * 512
                elif noisy:
                    bits = [random.getrandbits(1) for _ in range(512)]
                else:
                    bits, v = [], random.getrandbits(1)
                    while len(bits) < 512:
                        bits += [v] * random.randint(1, 200); v ^= 1
                    bits = bits[:512]
                blocks.append((burst, bits)); k += 1
            burst += 1
        while random.random() < p_lone:
            flags.append(random.choice([0, 3])); burst += 1
        return blocks, flags, burst

    def flattened(blocks, flags, n_bursts):
        flat = []
        for j in range(n_bursts):
            if not flags[j] & 1:
                continue
            if flags[j] & 2:
                flat.append(0)
            for t, b in blocks:
                if t == j:
                    flat += b
        return [i for i in range(1, len(flat)) if flat[i] != flat[i - 1]], len(flat)

    n_tr = 0
    for it in range(120):
        blocks, flags, nb = stream(random.randint(1, 300), random.choice([0, 0.2, 0.5]), it % 3 == 0)
        want = flattened(blocks, flags, nb)
        assert im.rle_split(blocks, flags, nb) == want
        n_tr += len(want[0])
    assert n_tr > 100_000


def test_defined_stages_sanity():
    w = D.hann_periodic(1024)
    assert w[0] == 0 and w[512] == 1 and abs(w.sum() - 512) < 1e-3
    x = np.exp(2j * np.pi * 0.05 * np.arange(100))
    d = D.fm_discriminator(x)
    assert d[0] == 0 and np.allclose(d[1:], 2 * np.pi * 0.05)
    rng = np.random.default_rng(0)
    z = rng.standard_normal(4096) + 1j * rng.standard_normal(4096)
    rows = D.psd_rows(z, 1024, 2, None)
    assert rows.shape == (2, 1024) and np.isclose(rows.sum(), 1024 * np.sum(np.abs(z) ** 2) / 2)   # Parseval
    assert D.resampler_ratio(0.2) == (1, 5) and D.resampler_ratio(48000 / 44100) == (160, 147)
    with pytest.raises(ValueError):
        D.resampler_ratio(np.pi)
    h = D.resampler_taps(1, 5)
    assert h.size == 321 and abs(h.sum() - 1) < 1e-12
    y = D.resample(np.ones(4000), 0.2)
    assert y.size == 800 and np.allclose(y[200:], 1.0, atol=1e-6)    # unity DC gain once the filter is full
    assert D.resample(np.ones(1000), 2.0).size == 2000
