"""GPU parity, part 3: the bit-exact OOK chain (north_star subsystem 5) and the overlap-save long FIR.

OOK: every intermediate that the reference computes in f32 (envelope, block sums) must be BIT-identical to
the CPU restatement, and so must the run lengths and decoded packet bits.
"""
import os

import numpy as np
import pytest
import torch

import oracle
from libredio_b200 import capi, synth

pytestmark = pytest.mark.gpu


def dev(a, ctx):
    return torch.from_numpy(np.ascontiguousarray(a)).to(ctx.tdev)


# ---- OOK -------------------------------------------------------------------------------------------------
def test_envelope_exhaustive_65536_pairs_bit_exact(ctx):
    """inputs come from u8, so there are only 65536 distinct (re, im) pairs: CPU == GPU is checked exhaustively"""
    from libredio_b200 import blocks
    got = blocks.ook_envelope_table(ctx).cpu().numpy()
    ref = oracle.norm_table()
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert got[127, 127] == 0.0 and got[254, 127] == 1.0
    # spot-check the table builder against the scalar C function
    for b0, b1 in ((0, 0), (255, 255), (3, 200), (128, 126)):
        assert ref[b0, b1] == oracle.norm(oracle.i2f(b0), oracle.i2f(b1))


def noisy_burst_capture(seed, n_blocks=400):
    """quiet floor with two stretches of full-scale random bytes: the envelope crosses max/2 thousands of times"""
    rng = np.random.default_rng(seed)
    iq = np.clip(np.rint(127 + 1.0 * rng.standard_normal(n_blocks * 1024)), 0, 255).astype(np.uint8)
    for start, length in ((100, 30), (250, 5)):
        iq[start * 1024:(start + length) * 1024] = rng.integers(0, 256, length * 1024, dtype=np.uint8)
    return iq


def run_ook(ctx, caps, max_runs=4096):
    from libredio_b200 import blocks
    iq = np.stack(caps)
    n_streams, nbytes = iq.shape
    ook = blocks.Ook(ctx, n_streams, nbytes // 1024, 256000, max_runs, 64)
    ook.decode(dev(iq, ctx))
    pk = ook.packets()
    dbg = ook.debug()
    ook.close()
    return pk, dbg


def check_against_oracle(caps, pk, dbg):
    for s, iq in enumerate(caps):
        r = oracle.ook_decode(iq)
        # f32 block sums: bit-identical (sequential order + exact envelope)
        assert np.array_equal(dbg["block_sums"][s].view(np.uint32), r["block_sums"].view(np.uint32)), f"stream {s} sums"
        assert dbg["n_bits"][s] == r["bits"].size, f"stream {s} bit count"
        nr = int(dbg["n_runs"][s])
        assert nr == r["run_val"].size, f"stream {s} run count"
        runs = dbg["runs"][s][:nr]
        assert np.array_equal(runs >> 31, r["run_val"]) and np.array_equal(runs & 0x7FFFFFFF, r["run_len"])
        a = [p[3] for p in pk if p[0] == s and p[1] == 0]
        b = [p[3] for p in pk if p[0] == s and p[1] == 1]
        assert len(a) == len(r["a_packets"]) and len(b) == len(r["b_packets"])
        for x, y in zip(a, r["a_packets"]):
            assert np.array_equal(x, y)
        for x, y in zip(b, r["b_packets"]):
            assert np.array_equal(x, y)


def test_ook_decodes_known_packets_bit_exact(ctx):
    caps, sent = [], []
    for s in range(16):
        iq, snt = synth.ook_capture_u8(800, seed=4 + s, n_packets=3)
        caps.append(iq); sent.append(snt)
    pk, dbg = run_ook(ctx, caps)
    check_against_oracle(caps, pk, dbg)
    # and the decoded bits are the bits the generator sent (known by construction)
    for s in range(16):
        for proto in (0, 1):
            got = [p[3] for p in pk if p[0] == s and p[1] == proto]
            want = [b for pr, b in sent[s] if pr == proto]
            assert len(got) == len(want)
            for g, w in zip(got, want):
                assert np.array_equal(g, w)
    assert sum(len(x) for x in sent) == len(pk) > 16


@pytest.mark.parametrize("case", ["noise_only", "loud_noise", "ragged_blocks", "all_zero", "saturated", "burst_at_end",
                                  "long_gapped_burst_at_end", "gapped_bursts_sent"])
def test_ook_edge_cases_match_oracle(ctx, case):
    rng = np.random.default_rng(hash(case) % 1000)
    if case == "noise_only":
        caps = [np.clip(np.rint(127 + 1.5 * rng.standard_normal(300 * 1024)), 0, 255).astype(np.uint8) for _ in range(3)]
    elif case == "loud_noise":      # thousands of short runs, nothing decodable
        caps = [noisy_burst_capture(70 + s) for s in range(3)]
    elif case == "ragged_blocks":   # n_blocks not a multiple of the 32-block warp group
        caps = [synth.ook_capture_u8(401, seed=80 + s, n_packets=1)[0] for s in range(5)]
    elif case == "all_zero":
        caps = [np.zeros(64 * 1024, np.uint8), np.full(64 * 1024, 127, np.uint8)]
    elif case == "saturated":
        caps = [np.full(200 * 1024, 255, np.uint8), rng.integers(0, 256, 200 * 1024, dtype=np.uint8)]
    elif case in ("long_gapped_burst_at_end", "gapped_bursts_sent"):
        # one loud block every 50: the counter reaches 1 (that block is NOT collected) and the next block re-fires, so the burst
        # goes on with single-block holes in it (bitfount.rs:68-75).  Open at the end of the capture: 250+ blocks to un-tag,
        # with holes; or followed by silence: the same bursts are sent and sliced.
        def quiet(n):
            return np.clip(np.rint(127 + 1.5 * rng.standard_normal(n * 1024)), 0, 255).astype(np.uint8)
        def loud(n):
            return np.clip(np.rint(127 + 60 * rng.standard_normal(n * 1024)), 0, 255).astype(np.uint8)
        caps = []
        for s in range(3):
            parts = [quiet(100 + s)]
            for _ in range(5 + s):
                parts += [loud(1), quiet(49)]
            parts += [loud(1), quiet(20 if case == "long_gapped_burst_at_end" else 120)]
            caps.append(np.concatenate(parts))
        n = min(c.size for c in caps) // 1024 * 1024
        caps = [c[:n] for c in caps]
        r0 = oracle.ook_decode(caps[0])                       # the construction does what it says: nothing sent / one holed burst
        assert (r0["bits"].size == 0) if case == "long_gapped_burst_at_end" else (r0["n_bursts"] == 1 and r0["bits"].size == 294 * 512 + 1)
    else:                           # a burst still open when the capture ends is never sent (bitfount.rs:78-81)
        iq, _ = synth.ook_capture_u8(500, seed=90, n_packets=1)
        iq = iq.copy(); iq[-40 * 1024:] = np.clip(np.rint(127 + 90 * rng.standard_normal(40 * 1024)), 0, 255).astype(np.uint8)
        caps = [iq]
    pk, dbg = run_ook(ctx, caps, max_runs=1 << 18)
    check_against_oracle(caps, pk, dbg)


def test_ook_oom_guard_path_matches_oracle_with_the_guard_shrunk_on_both_sides(ctx, monkeypatch):
    """bitfount.rs:52-54: a buffer longer than 1000*50*512 samples is thrown away and collection restarts from [0.0].  The real
    constant needs 100 s of capture per stream, so the test shrinks it to 120 blocks in the oracle AND in the plan (test hooks on
    both sides) and drives every way through the guard: a long loud stretch cut into abandoned pieces whose remainder is sent with
    a leading 0.0; the guard firing exactly on the block where the counter stands at 1, after which the reference sends the
    lone [0.0] -- one 0 bit, first, between and after ordinary bursts; several firings in one stretch."""
    guard = 120
    cases = [(L, bf, af) for L in (60, 71, 72, 73, 74, 200, 400) for bf in (True, False) for af in (True, False)]
    caps = [synth.ook_guard_capture_u8(L, seed=1000 + i, before=bf, after=af) for i, (L, bf, af) in enumerate(cases)]
    n = max(c.size for c in caps)
    rng = np.random.default_rng(5)
    caps = [np.concatenate([c, np.clip(np.rint(127 + 1.5 * rng.standard_normal(n - c.size)), 0, 255).astype(np.uint8)]) for c in caps]
    monkeypatch.setenv("LRC_OOK_TEST_GUARD_BLOCKS", str(guard))
    oracle.set_trigger_guard_blocks(guard)
    try:
        # the construction reaches the corner: the whole output of these two captures is the lone 0 bit / two 51-block bursts + 2
        lone = oracle.ook_decode(caps[cases.index((72, False, False))])
        assert lone["n_bursts"] == 1 and lone["bits"].size == 1
        mid = oracle.ook_decode(caps[cases.index((73, True, True))])
        assert mid["n_bursts"] == 3 and mid["bits"].size == 2 * 51 * 512 + 2
        pk, dbg = run_ook(ctx, caps, max_runs=1 << 15)
        check_against_oracle(caps, pk, dbg)
    finally:
        oracle.set_trigger_guard_blocks(0)
    # and with the reference's constant the same captures never reach the guard: both sides agree there too
    monkeypatch.delenv("LRC_OOK_TEST_GUARD_BLOCKS")
    pk, dbg = run_ook(ctx, caps[:6], max_runs=1 << 18)
    check_against_oracle(caps[:6], pk, dbg)


def test_ook_quiet_block_boundary_block_maximum_equal_to_half_the_burst_maximum(ctx):
    """The slicer does not read a collected block whose maximum does not exceed the burst's max/2 (k_ook.cu, quiet blocks): such a
    block is 512 zeros because `x > max/2` (bitfount.rs:91) is false for x <= max/2 -- INCLUDING equality.  Byte pairs whose envelope
    is exactly half of another pair's exist (2229 of the distinct values): (78, 115) is 0.3972283, (29, 103) twice that.  A burst
    whose maximum is the latter gets one block that peaks exactly at max/2 (all zeros, not read) and one that peaks at the next
    envelope value above it (one 1 bit: must be read); everything against the oracle."""
    env = lambda b0, b1: oracle.norm(oracle.i2f(b0), oracle.i2f(b1))
    top, mid = (29, 103), (78, 115)
    assert np.float32(env(*top)) / np.float32(2) == np.float32(env(*mid))
    # the smallest envelope above max/2, by brute force over the byte pairs
    above = min(((env(a, b), a, b) for a in range(0, 256, 1) for b in (103, 115, 127, 140) if env(a, b) > env(*mid)))
    rng = np.random.default_rng(12)
    n_blocks = 260

    def floor_block():
        return np.clip(np.rint(127 + 1.2 * rng.standard_normal(1024)), 0, 255).astype(np.uint8)

    blocks = [floor_block() for _ in range(n_blocks)]
    loud = floor_block()
    loud[0:600:2], loud[1:600:2] = 200, 60                       # fires the trigger; envelope below the top pair's
    loud[700], loud[701] = top                                   # the burst's maximum
    assert max(env(200, 60), env(*mid)) < env(*top)
    blocks[100] = loud
    at_half = floor_block(); at_half[300], at_half[301] = mid; at_half[640], at_half[641] = mid[::-1]
    blocks[103] = at_half                                        # block maximum == max/2: quiet by equality
    just_above = floor_block(); just_above[500], just_above[501] = above[1], above[2]
    blocks[105] = just_above                                     # block maximum just above max/2: one sample is a 1
    cap = np.concatenate(blocks)
    r = oracle.ook_decode(cap)
    assert r["n_bursts"] == 1 and r["bits"].size == 1 + 49 * 512
    ones = np.flatnonzero(r["bits"])
    assert 1 + 5 * 512 + 250 in ones and not np.any((ones > 1 + 3 * 512) & (ones <= 1 + 4 * 512))   # block 105 has its 1, block 103 none
    pk, dbg = run_ook(ctx, [cap, cap[::-1].copy(), cap], max_runs=1 << 12)
    check_against_oracle([cap, cap[::-1].copy(), cap], pk, dbg)


@pytest.mark.parametrize("n_blocks", [1, 5, 31, 32, 33, 65])
def test_ook_captures_shorter_than_a_warp_group(ctx, n_blocks):
    """the block-sum kernel's TMA box is 32 blocks tall: captures with fewer blocks (and a ragged second group) rely on the
    out-of-bounds rows being zero-filled and never stored; every stage must still equal the oracle"""
    rng = np.random.default_rng(n_blocks)
    caps = [np.clip(np.rint(127 + (2 + 40 * (s % 2)) * rng.standard_normal(n_blocks * 1024)), 0, 255).astype(np.uint8) for s in range(3)]
    pk, dbg = run_ook(ctx, caps, max_runs=1 << 17)
    check_against_oracle(caps, pk, dbg)


def test_ook_run_capacity_overflow_is_reported(ctx):
    caps = [noisy_burst_capture(70)]
    assert oracle.ook_decode(caps[0])["run_val"].size > 64
    with pytest.raises(capi.LrcError) as e:
        run_ook(ctx, caps, max_runs=64)
    assert e.value.status == capi.ERR_CAPACITY


def test_eat_and_b2d_micro_cases():
    """kpn.rs:111-124 on the two field layouts of ratpak.rs:115,119 (host helper, no GPU work)"""
    from libredio_b200 import blocks
    assert blocks.Ook.eat([1, 0, 1], [3]) == [5] == [oracle.b2d([1, 0, 1])]
    rng = np.random.default_rng(1)
    bits = rng.integers(0, 2, 36).astype(np.uint8)
    for w in (blocks.Ook.FIELDS_A1, blocks.Ook.FIELDS_A2):
        assert blocks.Ook.eat(bits, w) == oracle.eat(bits, w)
    with pytest.raises(capi.LrcError):
        blocks.Ook.eat(bits[:24], blocks.Ook.FIELDS_A1)


def test_ook_many_streams_sharded_equals_whole(ctx):
    """config 4 shards streams across GPUs with no exchange: decoding a subset of the streams must give the
    same packets as decoding them inside the full batch."""
    caps = [synth.ook_capture_u8(450, seed=200 + s, n_packets=2)[0] for s in range(24)]
    whole, _ = run_ook(ctx, caps)
    for lo, hi in ((0, 12), (12, 24)):
        part, _ = run_ook(ctx, caps[lo:hi])
        want = [(p[0] - lo, p[1], p[2], p[3].tobytes()) for p in whole if lo <= p[0] < hi]
        assert [(p[0], p[1], p[2], p[3].tobytes()) for p in part] == want


# ---- overlap-save long FIR ---------------------------------------------------------------------------------
def rms(a):
    return float(np.sqrt(np.mean(np.abs(np.asarray(a, dtype=np.complex128)) ** 2)))


def test_fastfir_vs_reference_golden(ctx, golden):
    """outputs of the vendored tools/kiss_fastfir.c on the fixture of tests/golden/make_golden.py"""
    from libredio_b200 import blocks
    import tests.golden.make_golden as mg
    h, x = mg.fastfir_case()
    ff = blocks.FastFir(ctx, h, 0)
    assert ff.nfft == 1024                                   # auto size: next pow2 >= 2*300, floor 1024
    for flush, key in ((False, "fastfir_noflush"), (True, "fastfir_flush")):
        got = ff.run(dev(x, ctx), flush).cpu().numpy()
        ref = golden[key]
        assert got.shape == ref.shape
        assert np.max(np.abs(got - ref)) <= 1e-4 * rms(ref)
    ff.close()


@pytest.mark.parametrize("nh,n,nfft", [(1, 3000, 0), (50, 10_000, 128), (300, 6000, 0), (1024, 40_000, 0),
                                       (4096, 70_000, 0), (4096, 8192, 0), (4096, 8191, 0), (17, 16, 64)])
def test_fastfir_vs_oracle_and_direct_convolution(ctx, nh, n, nfft):
    from libredio_b200 import blocks
    rng = np.random.default_rng(nh + n)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / np.sqrt(nh)).astype(np.complex64)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    ff = blocks.FastFir(ctx, h, nfft)
    for flush in (False, True):
        got = ff.run(dev(x, ctx), flush).cpu().numpy()
        ref = oracle.fastfir(h, x, nfft, flush)
        assert got.shape == ref.shape == (ff.out_len(n, flush),)
        if ref.size:
            assert np.max(np.abs(got - ref)) <= 1e-4 * rms(ref)
            # true convolution with the transient removed: y[k] = sum_j h[j] x[k + nh - 1 - j]
            full = np.convolve(x.astype(np.complex128), h.astype(np.complex128))[nh - 1:]
            assert np.max(np.abs(got - full[: got.size])) <= 1e-4 * rms(full)
    ff.close()


def test_fastfir_config5_shape_spot_windows(ctx):
    """config 5 at a size the CPU cannot filter whole: 4096 taps, 2^24 samples generated on the device;
    check random output windows (incl. block seams) against an f64 direct convolution."""
    from libredio_b200 import blocks
    nh, n = 4096, 1 << 24
    rng = np.random.default_rng(6)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64).astype(np.complex64)
    g = torch.Generator(device=ctx.tdev).manual_seed(5)
    x = torch.view_as_complex(torch.randn(n, 2, device=ctx.tdev, generator=g))
    ff = blocks.FastFir(ctx, h, 0)
    assert ff.nfft == 8192 and ff.ngood == 4097
    y = ff.run(x)
    assert y.numel() == ff.out_len(n) == ((n - 8192) // 4097 + 1) * 4097
    hr = h[::-1].astype(np.complex128)
    starts = [0, 4097 - 8, 4097 * 100 - 3, y.numel() - 64] + [int(v) for v in rng.integers(0, y.numel() - 64, 8)]
    for s0 in starts:
        seg = x[s0: s0 + 64 + nh - 1].cpu().numpy().astype(np.complex128)
        ref = np.array([np.dot(seg[k:k + nh], hr) for k in range(64)])
        got = y[s0:s0 + 64].cpu().numpy()
        assert np.max(np.abs(got - ref)) <= 1e-4 * rms(ref)
    ff.close()


# ---- nfft = 16384 blocks (k_fastfir16k.cu) --------------------------------------------------------------------
@pytest.mark.parametrize("nh,n", [(4096, 16384), (4096, 16384 + 12289 * 3 + 100), (4096, 20_000), (1000, 70_000),
                                  (4096, 1 << 22), (8192, 50_000), (5000, 16383)])
def test_fastfir_nfft_16384_vs_oracle(ctx, nh, n):
    """explicit 16384-point blocks: against the restated kiss_fastfir at the same block size (itself pinned to the
    vendored build by the golden fixture) and against the f64 convolution on windows incl. block seams"""
    from libredio_b200 import blocks
    rng = np.random.default_rng(nh + n)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / np.sqrt(nh)).astype(np.complex64)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    ff = blocks.FastFir(ctx, h, 16384)
    assert ff.nfft == 16384 and ff.ngood == 16384 - nh + 1
    for flush in (False, True):
        got = ff.run(dev(x, ctx), flush).cpu().numpy()
        assert got.shape == (ff.out_len(n, flush),)
        if n <= 100_000:
            ref = oracle.fastfir(h, x, 16384, flush)
            assert got.shape == ref.shape
            if ref.size:
                assert np.max(np.abs(got - ref)) <= 1e-4 * rms(ref)
        # true convolution with the transient removed, on windows (incl. block seams)
        hr = h[::-1].astype(np.complex128)
        for s0 in [0, ff.ngood - 8, got.size - 64] + [int(v) for v in rng.integers(0, max(1, got.size - 64), 6)]:
            if s0 < 0 or s0 + 64 > got.size:
                continue
            seg = x[s0: s0 + 64 + nh - 1].astype(np.complex128)
            ref = np.array([np.dot(seg[k:k + nh], hr) for k in range(64)])
            assert np.max(np.abs(got[s0:s0 + 64] - ref)) <= 1e-4 * rms(ref)
    ff.close()


@pytest.mark.parametrize("nh,n", [(4096, 70_000), (4096, 8192), (4096, 8191), (4096, 8192 + 4097 * 5 - 1), (2049, 30_000),
                                  (1025, 9000), (3000, 100_001), (6000, 60_000), (8192, 16384), (8192, 16383)])
def test_fastfir_automatic_size_keeps_kiss_fastfir_output_length_whatever_the_compute_block(ctx, nh, n):
    """nfft = 0: the OUTPUT LENGTH is the one kiss_fastfir's own block size gives (kiss_fastfir.c:81-93, :199-204 -- a call
    without flush stops at the reference's last full block) although the arithmetic runs in 16384-point blocks for
    nh > 1024; values against the restated kiss_fastfir at the reference's size"""
    from libredio_b200 import blocks
    rng = np.random.default_rng(7 * nh + n)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / np.sqrt(nh)).astype(np.complex64)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    ff = blocks.FastFir(ctx, h, 0)
    ref_nfft = max(1024, 2 << max(1, (nh - 1).bit_length()))     # kiss_fastfir.c:81-93
    assert ff.nfft == ref_nfft
    for flush in (False, True):
        got = ff.run(dev(x, ctx), flush).cpu().numpy()
        ref = oracle.fastfir(h, x, 0, flush)
        assert got.shape == ref.shape == (ff.out_len(n, flush),)
        if ref.size:
            assert np.max(np.abs(got - ref)) <= 1e-4 * rms(ref)
    ff.close()


def test_fastfir_explicit_8192_blocks_agree_with_the_automatic_plan(ctx):
    """the two compute paths (8192-point kernel on request, 16384-point blocks by default) give the same stream"""
    from libredio_b200 import blocks
    rng = np.random.default_rng(11)
    nh, n = 4096, 1 << 21
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64).astype(np.complex64)
    g = torch.Generator(device=ctx.tdev).manual_seed(3)
    x = torch.view_as_complex(torch.randn(n, 2, device=ctx.tdev, generator=g))
    a, b = blocks.FastFir(ctx, h, 0), blocks.FastFir(ctx, h, 8192)
    assert a.nfft == b.nfft == 8192
    for flush in (False, True):
        ya, yb = a.run(x, flush), b.run(x, flush)
        assert ya.shape == yb.shape
        assert (ya - yb).abs().max().item() <= 1e-5 * yb.abs().pow(2).mean().sqrt().item()
    a.close(); b.close()


def test_fastfir_sizes_beyond_16384_are_refused(ctx):
    from libredio_b200 import blocks
    with pytest.raises(capi.LrcError) as e:
        blocks.FastFir(ctx, np.ones(8193, dtype=np.complex64), 0)          # kiss_fastfir would pick 32768
    assert e.value.status == capi.ERR_UNSUPPORTED
    with pytest.raises(capi.LrcError) as e:
        blocks.FastFir(ctx, np.ones(100, dtype=np.complex64), 32768)
    assert e.value.status == capi.ERR_UNSUPPORTED
