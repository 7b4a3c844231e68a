"""Streaming OOK decode (lrc_ook_stream) against the one-shot decode of the same capture, config 4's shape.

    python tools/ook_stream_bench.py [--streams 4096] [--blocks 500] [--pushes 500,100,50,10,1] [--reps 3] [--out DIR]
    python tools/ook_stream_bench.py --profile --out DIR      # per-kernel split with torch.profiler (a separate run)

The capture is bench.py's config-4 input (16 synthetic streams with packets, repeated to --streams).  Each repetition
times, in turn, the one-shot lrc_ook_decode of the whole capture and, for every push size P, the same capture streamed as
blocks/P pushes of P blocks per stream (reset outside the timed window), with CUDA events around the device work.  The
streamed packets are checked against the one-shot packets.  Prints one JSON object: ms per push, Msamples/s, the ratio of
time per sample to the one-shot decode, the carry memory, and the GPU name and power limit."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:                      # the numbers stand without it, but say why it is missing
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--blocks", type=int, default=500)
    ap.add_argument("--pushes", default="500,100,50,10,1")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-carry", type=int, default=512, help="carry blocks per stream (0 = the exact guard + 1)")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200); nothing is measured on the CPU")
    from libredio_b200 import blocks, synth
    ctx = blocks.Context(0)
    S, B = a.streams, a.blocks
    caps = [synth.ook_capture_u8(B, seed=4 + s, n_packets=2)[0] for s in range(16)]
    iq = torch.from_numpy(np.stack(caps)).to(ctx.tdev)[torch.arange(S, device=ctx.tdev) % 16].contiguous()
    pushes = [int(p) for p in a.pushes.split(",")]
    one = blocks.Ook(ctx, S, B, 256000, 4096, 64)
    plans = {P: blocks.OokStream(ctx, S, P, 256000, a.max_carry, 4096, 64) for P in pushes}
    key = lambda pk: [(p[0], p[1], p[2], p[3].tobytes()) for p in pk]

    def run_one():
        one.decode(iq)

    def run_stream(P):
        for b in range(0, B, P):
            plans[P].push(iq[:, b * 1024:min(b + P, B) * 1024])

    # warm-up and parity: every streamed pass gives the one-shot packets
    run_one()
    ref = key(one.packets())
    for P in pushes:
        run_stream(P)
        assert key(plans[P].packets()) == ref, f"push size {P}: packets differ from the one-shot decode"
        plans[P].reset()

    if a.profile:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_one()
            torch.cuda.synchronize()
            for P in pushes:
                if P >= 10:
                    run_stream(P)
                    torch.cuda.synchronize()
                    plans[P].reset()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=30)
        print(table)
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            open(os.path.join(a.out, "ook_stream_profile.txt"), "w").write(table)
        return

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    t_one, t_push = [], {P: [] for P in pushes}
    for _ in range(a.reps):                     # alternated: one-shot, then every push size, then again
        t_one.append(timed(run_one))
        for P in pushes:
            t_push[P].append(timed(lambda: run_stream(P)) / ((B + P - 1) // P))
            plans[P].packets()
            plans[P].reset()
    ms_one = float(np.median(t_one))
    res = {"workload": f"{S} streams x {B} blocks of 512 u8 IQ samples (bench.py config 4 input)", **gpu_info(),
           "one_shot": {"ms": ms_one, "msamples_per_s": S * B * 512 / (ms_one * 1e-3) / 1e6},
           "carry_bytes_allocated": S * ((a.max_carry + 31) // 32 * 32) * 1024, "max_carry_blocks": a.max_carry, "pushes": {}}
    for P in pushes:
        ms = float(np.median(t_push[P]))
        res["pushes"][str(P)] = {"ms_per_push": ms, "ms_per_push_best": float(np.min(t_push[P])),
                                 "msamples_per_s": S * P * 512 / (ms * 1e-3) / 1e6,
                                 "time_per_sample_vs_one_shot": (ms / P) / (ms_one / B)}
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "ook_stream_bench.json"), "w").write(json.dumps(res, indent=1))
    for p in plans.values():
        p.close()
    one.close()
    ctx.close()


if __name__ == "__main__":
    main()
