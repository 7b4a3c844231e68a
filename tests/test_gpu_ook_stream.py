"""GPU: the streaming OOK plan (lrc_ook_stream).  The reference chain is causal, so after pushes 0..k the packets emitted
so far must equal the oracle's decode of the concatenation of those pushes -- same bursts left open, same run unflushed,
same pulse pair pending -- and every push's block sums and completed runs must be the oracle's for that stretch.  Checked
at every seam of seeded random splits, of every two-push split of a short capture and of one-block pushes."""
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle
from libredio_b200 import capi, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev(a, ctx):
    return torch.from_numpy(np.ascontiguousarray(a)).to(ctx.tdev)


def random_splits(n_blocks, seed, lo=1, hi=97):
    rng = np.random.default_rng(seed)
    out, done = [], 0
    while done < n_blocks:
        k = min(int(rng.integers(lo, hi + 1)), n_blocks - done)
        out.append(k)
        done += k
    return out


def quiet(rng, n):
    return np.clip(np.rint(127 + 1.5 * rng.standard_normal(n * 1024)), 0, 255).astype(np.uint8)


def loud(rng, n, sd=60):
    return np.clip(np.rint(127 + sd * rng.standard_normal(n * 1024)), 0, 255).astype(np.uint8)


def by_stream_proto(pk, n_streams):
    out = {(s, p): [] for s in range(n_streams) for p in (0, 1)}
    for s, p, seq, bits in pk:
        out[(s, p)].append((seq, bits.tobytes()))
    return out


def oracle_packets(r):
    return {0: [p.tobytes() for p in r["a_packets"]], 1: [p.tobytes() for p in r["b_packets"]]}


def stream_and_check(ctx, caps, splits, max_carry=0, max_runs=1 << 16, check_each=True, ook=None):
    """push `caps` (equal-length u8 captures, one per stream) in pieces of `splits` blocks; after every push compare the
    push's block sums, the runs completed so far and the packets emitted so far with the oracle on the prefix
    (check_each=False: the packets after the last push only).  Returns the packets, ordered by (stream, proto, seq)."""
    from libredio_b200 import blocks
    iq = np.stack(caps)
    S, nbytes = iq.shape
    n_blocks = nbytes // 1024
    assert sum(splits) == n_blocks
    own = ook is None
    if own:
        ook = blocks.OokStream(ctx, S, max(splits), 256000, max_carry, max_runs, 256)
    d_iq = dev(iq, ctx)
    full = [oracle.ook_decode(c) for c in caps]
    runs = [[] for _ in range(S)]
    pk_all = []
    done = 0
    for k in splits:
        ook.push(d_iq[:, done * 1024:(done + k) * 1024])
        pk = ook.packets()
        pk_all += pk
        done += k
        if not check_each and done < n_blocks:
            continue
        dbg = ook.debug()
        got = by_stream_proto(pk_all, S)
        for s in range(S):
            r = oracle.ook_decode(caps[s][: done * 1024]) if done < n_blocks else full[s]
            want = oracle_packets(r)
            for p in (0, 1):
                assert [b for _, b in got[(s, p)]] == want[p], f"stream {s} proto {p}: packets after block {done}"
                assert [q for q, _ in got[(s, p)]] == list(range(len(want[p]))), "sequence numbers"
            if not check_each:                  # the runs of the pushes in between were not collected
                continue
            assert np.array_equal(dbg["block_sums"][s].view(np.uint32), full[s]["block_sums"][done - k:done].view(np.uint32)), \
                f"stream {s}: block sums of the push ending at {done}"
            nr = int(dbg["n_runs"][s])
            runs[s] += dbg["runs"][s][:nr].tolist()
            rr = np.array(runs[s], dtype=np.uint32)
            assert rr.size == r["run_val"].size, f"stream {s}: {rr.size} runs after block {done}, oracle {r['run_val'].size}"
            assert np.array_equal(rr >> 31, r["run_val"]) and np.array_equal(rr & 0x7FFFFFFF, r["run_len"]), \
                f"stream {s}: runs after block {done}"
    if own:
        ook.close()
    return sorted(pk_all, key=lambda p: (p[0], p[1], p[2]))


def batch_packets(ctx, caps):
    from libredio_b200 import blocks
    iq = np.stack(caps)
    ook = blocks.Ook(ctx, iq.shape[0], iq.shape[1] // 1024, 256000, 1 << 16, 256)
    ook.decode(dev(iq, ctx))
    pk = ook.packets()
    ook.close()
    return pk


def same_packets(a, b):
    return [(p[0], p[1], p[2], p[3].tobytes()) for p in a] == [(p[0], p[1], p[2], p[3].tobytes()) for p in b]


def test_seeded_random_push_sizes(ctx):
    caps, sent = [], []
    for s in range(16):
        iq, snt = synth.ook_capture_u8(800, seed=4 + s, n_packets=3)
        caps.append(iq); sent.append(snt)
    pk = stream_and_check(ctx, caps, random_splits(800, seed=1))
    assert same_packets(pk, batch_packets(ctx, caps))
    for s in range(16):
        for proto in (0, 1):
            got = [p[3] for p in pk if p[0] == s and p[1] == proto]
            want = [b for pr, b in sent[s] if pr == proto]
            assert len(got) == len(want) and all(np.array_equal(g, w) for g, w in zip(got, want))
    assert len(pk) > 16


def test_every_seam_position(ctx):
    """a capture with one packet burst, split into two pushes at every k in 1..N-1, and as N one-block pushes: seams on the
    firing block, inside the pulses, on the 49th trailing block, on the send block and on the block after it"""
    from libredio_b200 import blocks
    seed = next(sd for sd in range(300, 400) if len(oracle.ook_decode(synth.ook_capture_u8(300, seed=sd, n_packets=1)[0])["a_packets"])
                + len(oracle.ook_decode(synth.ook_capture_u8(300, seed=sd, n_packets=1)[0])["b_packets"]) == 1)
    cap = synth.ook_capture_u8(300, seed=seed, n_packets=1)[0]
    caps = [cap, np.roll(cap, 37 * 1024)]
    n = 300
    ook = blocks.OokStream(ctx, 2, n - 1, 256000, 0, 1 << 16, 256)
    want = batch_packets(ctx, caps)
    for k in range(1, n):
        pk = stream_and_check(ctx, caps, [k, n - k], ook=ook)
        assert same_packets(pk, want), f"split at {k}"
        ook.reset()
    ook.close()
    assert same_packets(stream_and_check(ctx, caps, [1] * n), want)


@pytest.mark.parametrize("case", ["loud_noise", "gapped_bursts", "saturated", "all_zero", "burst_at_end"])
def test_edge_cases_pushed_in_pieces(ctx, case):
    rng = np.random.default_rng(sum(map(ord, case)))
    if case == "loud_noise":          # thousands of short runs across the seams
        caps = []
        for _ in range(3):
            c = quiet(rng, 400)
            c[100 * 1024:130 * 1024] = rng.integers(0, 256, 30 * 1024, dtype=np.uint8)
            c[250 * 1024:255 * 1024] = rng.integers(0, 256, 5 * 1024, dtype=np.uint8)
            caps.append(c)
    elif case == "gapped_bursts":     # one loud block every 50: the counter reaches 1 and the next block re-fires
        caps = []
        for s in range(3):
            parts = [quiet(rng, 100 + s)]
            for _ in range(5 + s):
                parts += [loud(rng, 1), quiet(rng, 49)]
            parts += [loud(rng, 1), quiet(rng, 120)]
            caps.append(np.concatenate(parts))
        n = min(c.size for c in caps)
        caps = [c[:n] for c in caps]
    elif case == "saturated":
        caps = [np.full(200 * 1024, 255, np.uint8), rng.integers(0, 256, 200 * 1024, dtype=np.uint8)]
    elif case == "all_zero":          # the threshold stays 0
        caps = [np.zeros(64 * 1024, np.uint8), np.full(64 * 1024, 127, np.uint8)]
    else:                             # a burst still open when the stream so far ends
        iq, _ = synth.ook_capture_u8(500, seed=90, n_packets=1)
        iq = iq.copy(); iq[-40 * 1024:] = np.clip(np.rint(127 + 90 * rng.standard_normal(40 * 1024)), 0, 255).astype(np.uint8)
        caps = [iq]
    n = caps[0].size // 1024
    for seed in (2, 3):
        stream_and_check(ctx, caps, random_splits(n, seed, 1, 41), max_runs=1 << 18)
    if case == "gapped_bursts":       # and a seam on every block: the counter reaches 1 exactly at a seam
        stream_and_check(ctx, caps, [1] * n, max_runs=1 << 18)


def test_oom_guard_across_seams(ctx, monkeypatch):
    """bitfount.rs:52-54 with the guard shrunk to 120 blocks on both sides; one-block pushes put a seam on the block where the
    guard fires and on the lone-[0.0] corner (the guard firing with the counter at 1, the next block sending [0.0])"""
    guard = 120
    cases = [(72, False, False), (73, True, True), (71, True, False), (200, False, True), (400, True, True)]
    caps = [synth.ook_guard_capture_u8(L, seed=1000 + i, before=bf, after=af) for i, (L, bf, af) in enumerate(cases)]
    n = max(c.size for c in caps)
    rng = np.random.default_rng(5)
    caps = [np.concatenate([c, quiet(rng, (n - c.size) // 1024)]) for c in caps]
    monkeypatch.setenv("LRC_OOK_TEST_GUARD_BLOCKS", str(guard))
    oracle.set_trigger_guard_blocks(guard)
    try:
        lone = oracle.ook_decode(caps[0])
        assert lone["n_bursts"] == 1 and lone["bits"].size == 1
        nb = n // 1024
        stream_and_check(ctx, caps, [1] * nb, max_runs=1 << 15)
        stream_and_check(ctx, caps, random_splits(nb, 7, 1, 60), max_runs=1 << 15)
        # the exact carry of a plan created under the hook is guard + 1 blocks: no overflow however the input is split
        stream_and_check(ctx, caps, random_splits(nb, 8, 100, 200), max_runs=1 << 15)
    finally:
        oracle.set_trigger_guard_blocks(0)


def test_quiet_block_rule_against_the_final_maximum(ctx):
    """discretize compares with the FINAL maximum of a burst (bitfount.rs:90-91).  A block whose maximum equals the final max/2
    ((78, 115) against (29, 103)) and one just above it are collected in pushes before the one that brings the burst's
    maximum; the first slices to zeros, the second has its 1 bit -- decided against the final maximum, not a running one."""
    env = lambda b0, b1: oracle.norm(oracle.i2f(b0), oracle.i2f(b1))
    top, mid = (29, 103), (78, 115)
    assert np.float32(env(*top)) / np.float32(2) == np.float32(env(*mid))
    above = min(((env(a, b), a, b) for a in range(0, 256) for b in (103, 115, 127, 140) if env(a, b) > env(*mid)))
    rng = np.random.default_rng(12)

    def floor_block():
        return np.clip(np.rint(127 + 1.2 * rng.standard_normal(1024)), 0, 255).astype(np.uint8)

    blks = [floor_block() for _ in range(260)]
    fire = floor_block(); fire[0:600:2], fire[1:600:2] = 200, 60      # fires the trigger below the final maximum
    blks[100] = fire
    at_half = floor_block(); at_half[300], at_half[301] = mid
    blks[103] = at_half                                                # == final max/2, above the running max/2 at the time
    just_above = floor_block(); just_above[500], just_above[501] = above[1], above[2]
    blks[105] = just_above
    peak = floor_block(); peak[700], peak[701] = top
    blks[110] = peak                                                   # the burst's maximum arrives last
    cap = np.concatenate(blks)
    r = oracle.ook_decode(cap)
    assert r["n_bursts"] == 1
    ones = np.flatnonzero(r["bits"])
    assert 1 + 5 * 512 + 250 in ones and not np.any((ones > 1 + 3 * 512) & (ones <= 1 + 4 * 512))
    for splits in ([104, 156], [101, 3, 2, 4, 150], [1] * 260, random_splits(260, 9, 1, 13)):
        stream_and_check(ctx, [cap, cap[::-1].copy()], splits, max_runs=1 << 12)


def test_carry_overflow_is_reported_and_reset_starts_over(ctx):
    from libredio_b200 import blocks
    rng = np.random.default_rng(3)
    cap, _ = synth.ook_capture_u8(400, seed=5, n_packets=2)
    caps = [quiet(rng, 400), cap]
    ook = blocks.OokStream(ctx, 2, 400, 256000, 20, 1 << 16, 256)
    d_iq = dev(np.stack(caps), ctx)
    with pytest.raises(capi.LrcError) as e:
        for b in range(0, 400, 10):
            ook.push(d_iq[:, b * 1024:(b + 10) * 1024])
            ook.packets()
    assert e.value.status == capi.ERR_CAPACITY and "stream 1" in str(e.value) and "max_carry_blocks" in str(e.value)
    with pytest.raises(capi.LrcError) as e2:                      # loud until reset
        ook.push(d_iq[:, :1024])
    assert e2.value.status == capi.ERR_CAPACITY
    ook.reset()
    # whole bursts inside one push need no carry: the capture in one push decodes as the oracle from scratch
    pk = stream_and_check(ctx, caps, [400], ook=ook)
    assert same_packets(pk, batch_packets(ctx, caps)) and len(pk) >= 1
    ook.close()


def test_streams_stay_independent(ctx):
    """config 4 shards streams over GPUs: streaming a subset gives the packets it gets inside the full set"""
    caps = [synth.ook_capture_u8(450, seed=200 + s, n_packets=2)[0] for s in range(24)]
    splits = random_splits(450, 11, 5, 80)
    whole = stream_and_check(ctx, caps, splits, check_each=False)
    for lo, hi in ((0, 12), (12, 24), (5, 6)):
        part = stream_and_check(ctx, caps[lo:hi], splits, check_each=False)
        want = [(p[0] - lo, p[1], p[2], p[3].tobytes()) for p in whole if lo <= p[0] < hi]
        assert [(p[0], p[1], p[2], p[3].tobytes()) for p in part] == want


def test_kpn_app_ook_stream_from_an_iq_capture_file(tmp_path):
    """iq_file_source_u8 -> batch(37) -> kpn_gpu::ook_decode_stream -> split_protocols -> fork -> binconv x 2 / applicator: the
    field lines equal those of the whole file (37 does not divide a burst's length: packets cross message boundaries)"""
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "kpn"), "test_gpu_apps"])
    n_blocks = 600
    iq, sent = synth.ook_capture_u8(n_blocks, seed=77, n_packets=3)
    ref = oracle.ook_decode(iq)

    def eat(bits, widths):                                        # kpn.rs:111-124
        out, i = [], 0
        for w in widths:
            out.append(int("".join(str(int(b)) for b in bits[i:i + w]), 2))
            i += w
        return out
    a_ref, b_ref = [list(p) for p in ref["a_packets"]], [list(p) for p in ref["b_packets"]]
    assert len(a_ref) >= 1 and len(b_ref) >= 1
    assert len(a_ref) + len(b_ref) == len(sent)
    lines = []
    for tag, widths in {"A": (4, 8, 4, 12, 8), "C": (4, 8, 2, 10, 12)}.items():
        lines += [tag + " " + " ".join(str(v) for v in eat(p, widths)) for p in a_ref]
    lines += ["B " + " ".join(str(int(v)) for v in p) + " 0" for p in b_ref]
    cap = tmp_path / "capture.iq"
    iq.tofile(cap)
    exp = tmp_path / "expected.txt"
    exp.write_text("\n".join(lines) + "\n")
    exe = os.path.join(ROOT, "kpn", "test_gpu_apps")
    out = subprocess.run([exe, "ook_stream", str(cap), "37", str(exp)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "kpn app ook_stream OK" in out.stdout, out.stdout + out.stderr
