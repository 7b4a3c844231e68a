"""CPU: a model of the streaming OOK plan's seam hand-over (k_ook.cu, lrc_ook_stream), pushed block range by block range.

Each push starts from explicit per-stream state only -- the trigger's threshold and counter, the buffer length, whether the
buffer starts with the 0.0 of vec!(0.0), the open burst's collected blocks (the carry) and their running maximum, the open
run of rle, each matcher's pending pulse and partial packet -- and leaves the same state for the next push.  After every push
the runs it has completed and the packets it has emitted must equal the oracle's decode of the concatenation of the pushes so
far (the reference chain is causal).  The carry may drop the bytes of a block whose maximum does not exceed half the running
maximum (it slices to 512 zeros against any later, larger maximum); the model checks that rule too."""
import numpy as np
import pytest

import oracle
from oracle.restated_py import _in
from libredio_b200 import synth

F = np.float32
TABLE = None


def envelope_blocks(iq):
    global TABLE
    if TABLE is None:
        TABLE = oracle.norm_table()
    e = TABLE[iq[0::2], iq[1::2]]
    return e.reshape(-1, 512)


class Matcher:
    """ratpak.rs:88-97 looper body + shaper_optional (kpn.rs:266-275), one run at a time"""

    def __init__(self, proto):
        self.proto, self.want = proto, (36 if proto == 0 else 24)
        self.pending, self.d, self.acc = False, F(0), []

    def first_ok(self, v, d):
        if self.proto == 0:
            return v == 1 and _in(d, 2e-4, 6e-4)
        return v == 1 and (_in(d, 125e-6, 250e-6) or _in(d, 500e-6, 650e-6))

    def second(self, v, e):
        if v != 0:
            return None
        if self.proto == 0:
            return 0 if _in(e, 1.5e-3, 2.5e-3) else 1 if _in(e, 3.5e-3, 4.5e-3) else None
        ok = _in(e, 125e-6, 250e-6) or _in(e, 500e-6, 650e-6)
        return (1 if self.d > e else 0) if ok else None

    def feed(self, v, d, out):
        if self.pending:
            self.pending = False
            y = self.second(v, d)
        elif self.first_ok(v, d):
            self.pending, self.d = True, d
            return
        else:
            y = None
        if y is not None:
            self.acc.append(y)
        else:
            if len(self.acc) == self.want:
                out.append(bytes(self.acc))
            self.acc = []


class SeamModel:
    def __init__(self, guard_blocks=50000, quiet_drop=False, s_rate=256000):
        self.guard = guard_blocks * 512
        self.quiet_drop, self.s_rate = quiet_drop, F(s_rate)
        self.threshold, self.trig, self.buf_len, self.lead0 = F(0), 0, 1, True       # bitfount.rs:41-44
        self.carry, self.run_max = [], F(0)       # open burst: collected blocks (None = dropped quiet block), running max
        self.run_val, self.run_len = 0, 0         # the open run of rle
        self.matchers = [Matcher(0), Matcher(1)]
        self.max_carry = 0

    def push(self, env):
        """env: [k, 512] f32 envelopes of the push's blocks -> (runs completed, packets emitted per proto)"""
        sent = []                                 # (lead0, blocks, maximum) of every burst sent in this push
        for blk in env:
            self.trig -= 1
            s = F(np.cumsum(blk, dtype=np.float32)[-1])
            if self.buf_len > self.guard:         # :52-54
                self.carry, self.run_max, self.buf_len, self.lead0 = [], F(0), 1, True
            if self.threshold == F(0):
                self.threshold = s
            if self.trig < 0:
                self.threshold = F(self.threshold + F(s / F(1000)))
                self.threshold = F(self.threshold - F(self.threshold * F(0.002)))
            if s > F(self.threshold * F(4)):
                self.trig = 50
            if self.trig > 1:                     # :73-75
                bm = F(blk.max())
                drop = self.quiet_drop and bm <= F(self.run_max / F(2))
                self.carry.append(None if drop else blk)
                self.run_max = max(self.run_max, bm)
                self.buf_len += 512
            if self.trig == 0:                    # :78-81
                sent.append((self.lead0, self.carry, self.run_max))
                self.carry, self.run_max, self.buf_len, self.lead0 = [], F(0), 0, False
        self.trig = max(self.trig, -1)            # every counter below 0 walks the same way
        self.max_carry = max(self.max_carry, len(self.carry))
        bits = []
        for lead0, blocks, mx in sent:            # discretize :87-96 against the burst's final maximum
            half = F(mx / F(2))
            if lead0:
                bits.append(0)
            for b in blocks:
                bits += [0] * 512 if b is None else (b > half).astype(np.uint8).tolist()
        runs = []                                 # rle across the seam: the open run continues
        for x in bits:
            if self.run_len and x != self.run_val:
                runs.append((self.run_val, self.run_len))
                self.run_len = 0
            self.run_val = x
            self.run_len += 1
        pk = ([], [])
        for v, n in runs:                         # dle + both matchers (fork kpn.rs:182)
            d = F(F(n) / self.s_rate)
            for m in self.matchers:
                m.feed(v, d, pk[m.proto])
        return runs, pk


def splits_of(n, seed, lo, hi):
    rng = np.random.default_rng(seed)
    out, done = [], 0
    while done < n:
        k = min(int(rng.integers(lo, hi + 1)), n - done)
        out.append(k)
        done += k
    return out


def check_on_prefixes(cap, splits, guard_blocks=50000, quiet_drop=False):
    env = envelope_blocks(cap)
    model = SeamModel(guard_blocks, quiet_drop)
    runs, pk, done = [], ([], []), 0
    for k in splits:
        r, p = model.push(env[done:done + k])
        runs += r
        pk[0].extend(p[0]); pk[1].extend(p[1])
        done += k
        ref = oracle.ook_decode(cap[: done * 1024])
        assert [v for v, _ in runs] == ref["run_val"].tolist() and [n for _, n in runs] == ref["run_len"].tolist(), \
            f"runs after block {done}"
        assert pk[0] == [bytes(p) for p in ref["a_packets"]] and pk[1] == [bytes(p) for p in ref["b_packets"]], \
            f"packets after block {done}"
    return model, pk


@pytest.mark.parametrize("quiet_drop", [False, True])
def test_seam_model_equals_the_oracle_on_every_prefix(quiet_drop):
    for s in range(3):
        cap, sent = synth.ook_capture_u8(500, seed=40 + s, n_packets=3)
        model, pk = check_on_prefixes(cap, splits_of(500, s, 1, 97), quiet_drop=quiet_drop)
        assert sum(len(x) for x in pk) == len(sent) >= 1
        assert model.max_carry <= 50001


def test_seam_model_one_block_pushes_and_the_quiet_boundary():
    """every seam position; and a block whose maximum equals the burst's final max/2 collected before the maximum arrives"""
    cap, _ = synth.ook_capture_u8(300, seed=303, n_packets=1)
    check_on_prefixes(cap, [1] * 300, quiet_drop=True)
    env = lambda b0, b1: oracle.norm(oracle.i2f(b0), oracle.i2f(b1))
    top, mid = (29, 103), (78, 115)
    rng = np.random.default_rng(12)
    blks = [np.clip(np.rint(127 + 1.2 * rng.standard_normal(1024)), 0, 255).astype(np.uint8) for _ in range(200)]
    blks[100][0:600:2], blks[100][1:600:2] = 200, 60
    blks[103][300], blks[103][301] = mid
    blks[110][700], blks[110][701] = top
    assert env(200, 60) < env(*top)
    cap = np.concatenate(blks)
    for qd in (False, True):
        check_on_prefixes(cap, [1] * 200, quiet_drop=qd)


def test_seam_model_oom_guard_path():
    """bitfount.rs:52-54 with the guard shrunk to 120 blocks on both sides: abandoned pieces, the lone [0.0], seams anywhere;
    the carry never holds more than guard + 1 blocks"""
    guard = 120
    oracle.set_trigger_guard_blocks(guard)
    try:
        for i, (L, bf, af) in enumerate([(72, False, False), (73, True, True), (200, False, True), (400, True, False)]):
            cap = synth.ook_guard_capture_u8(L, seed=1000 + i, before=bf, after=af)
            n = cap.size // 1024
            for splits in ([1] * n, splits_of(n, i, 1, 150)):
                model, _ = check_on_prefixes(cap, splits, guard_blocks=guard, quiet_drop=bool(i % 2))
                assert model.max_carry <= guard + 1
    finally:
        oracle.set_trigger_guard_blocks(0)
