"""Streaming overlap-save (lrc_fastfir_stream) against the one-shot lrc_fastfir_run, config 5's filter.

    python tools/fastfir_stream_bench.py [--reps 3] [--out DIR]

Taps are config 5's (4096, rng(6)/64); the input is generated on the device.  Two workloads, each repetition timing the
arms in turn in one process with CUDA events around the device work of a whole pass:
  - 1 channel x 2^30 samples: one lrc_fastfir_run, and the same stream pushed in 2^16 .. 2^24-sample pushes;
  - 64 channels x 2^24 samples: 64 lrc_fastfir_run calls, and the 64 channels pushed together in 2^14 .. 2^20 samples
    per channel (the rate is also compared with the one-shot of one channel of 2^30).
Pushes read the input in place (chunk_stride = the channel's row) and write into one output buffer, so a pass has no
copies besides the carry update.  Every streamed pass (flushed on its last push) is checked bit for bit against the
one-shot.  Prints one JSON object: ms per push, Gsamples/s, time per sample over the one-shot's, and the GPU name and
power limit."""
from __future__ import annotations

import argparse
import ctypes as C
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
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log2n", type=int, default=30, help="samples of the one-channel stream (2^N)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200); nothing is measured on the CPU")
    from libredio_b200 import blocks
    from libredio_b200.capi import check
    ctx = blocks.Context(0)
    lib = ctx.lib
    nh = 4096
    rng = np.random.default_rng(6)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64).astype(np.complex64)
    ff = blocks.FastFir(ctx, h, 0)
    s = blocks._stream()
    ES = 8
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(fn):
        e0, e1 = ev(), ev()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    def oneshot(x, out):
        no = C.c_size_t()
        check(lib.lrc_fastfir_run(ff.h, C.c_void_p(x.data_ptr()), x.numel(), C.c_void_p(out.data_ptr()), 1, C.byref(no), s),
              "lrc_fastfir_run")
        return no.value

    def streamed(st, x, n_ch, n, push, out, out_stride):
        """x: [n_ch, n] rows (any row stride); out: [n_ch, out_stride]; returns the pushes made"""
        done, k = 0, 0
        no = C.c_size_t()
        for p0 in range(0, n, push):
            m = min(push, n - p0)
            check(lib.lrc_fastfir_stream_push(st, C.c_void_p(x.data_ptr() + p0 * ES), m, x.stride(0),
                                              C.c_void_p(out.data_ptr() + done * ES), out_stride, int(p0 + m == n),
                                              C.byref(no), s), "lrc_fastfir_stream_push")
            done += no.value
            k += 1
        assert done == n - nh + 1
        return k

    g = torch.Generator(device=ctx.tdev).manual_seed(5)
    res = {"workload": "config-5 taps (4096, rng(6)/64), cf32 generated on the device", **gpu_info()}

    # ---- 1 channel x 2^N ---------------------------------------------------------------------------------------
    n1 = 1 << a.log2n
    x1 = torch.view_as_complex(torch.randn(n1, 2, device=ctx.tdev, generator=g))
    tot = n1 - nh + 1
    ref = torch.empty(tot, dtype=torch.complex64, device=ctx.tdev)
    got = torch.empty(tot, dtype=torch.complex64, device=ctx.tdev)
    st1 = C.c_void_p()
    check(lib.lrc_fastfir_stream_create(ff.h, 1, C.byref(st1)), "lrc_fastfir_stream_create")
    pushes1 = [p for p in (1 << 16, 1 << 18, 1 << 20, 1 << 22, 1 << 24) if p <= n1]
    same = lambda u, v: torch.equal(torch.view_as_real(u).view(torch.int32), torch.view_as_real(v).view(torch.int32))
    oneshot(x1, ref)
    for p in pushes1:                                        # warm-up and parity
        streamed(st1, x1.view(1, -1), 1, n1, p, got.view(1, -1), tot)
        assert same(got, ref), f"1 channel, push {p}: differs from the one-shot"
    t1 = {"oneshot": []} | {p: [] for p in pushes1}
    for _ in range(a.reps):
        t1["oneshot"].append(timed(lambda: oneshot(x1, ref)))
        for p in pushes1:
            t1[p].append(timed(lambda: streamed(st1, x1.view(1, -1), 1, n1, p, got.view(1, -1), tot)))
    ms1 = float(np.median(t1["oneshot"]))
    res["one_channel"] = {"samples": n1, "oneshot_ms": ms1, "oneshot_gsps": n1 / ms1 / 1e6, "pushes": {}}
    for p in pushes1:
        ms = float(np.median(t1[p]))
        k = -(-n1 // p)
        res["one_channel"]["pushes"][str(p)] = {"pushes": k, "ms_per_push": ms / k, "gsps": n1 / ms / 1e6,
                                                "time_per_sample_vs_oneshot": ms / ms1}
    lib.lrc_fastfir_stream_destroy(st1)
    del x1, ref, got
    torch.cuda.empty_cache()

    # ---- 64 channels x 2^24 --------------------------------------------------------------------------------------
    n_ch, n = 64, 1 << 24
    xm = torch.view_as_complex(torch.randn(n_ch, n, 2, device=ctx.tdev, generator=g))
    tot = n - nh + 1
    refm = torch.empty(n_ch, tot, dtype=torch.complex64, device=ctx.tdev)
    gotm = torch.empty(n_ch, tot, dtype=torch.complex64, device=ctx.tdev)
    stm = C.c_void_p()
    check(lib.lrc_fastfir_stream_create(ff.h, n_ch, C.byref(stm)), "lrc_fastfir_stream_create")
    pushesm = (1 << 14, 1 << 16, 1 << 18, 1 << 20)

    def oneshot_all():
        for c in range(n_ch):
            oneshot(xm[c], refm[c])

    oneshot_all()
    for p in pushesm:
        streamed(stm, xm, n_ch, n, p, gotm, tot)
        assert same(gotm, refm), f"64 channels, push {p}: differs from the one-shot"
    tm = {"oneshot": []} | {p: [] for p in pushesm}
    for _ in range(a.reps):
        tm["oneshot"].append(timed(oneshot_all))
        for p in pushesm:
            tm[p].append(timed(lambda: streamed(stm, xm, n_ch, n, p, gotm, tot)))
    msm = float(np.median(tm["oneshot"]))
    res["64_channels"] = {"samples_per_channel": n, "oneshot_64_calls_ms": msm, "oneshot_64_calls_gsps": n_ch * n / msm / 1e6,
                          "pushes": {}}
    for p in pushesm:
        ms = float(np.median(tm[p]))
        k = -(-n // p)
        res["64_channels"]["pushes"][str(p)] = {
            "pushes": k, "ms_per_push": ms / k, "gsps": n_ch * n / ms / 1e6,
            "time_per_sample_vs_64_oneshot_calls": ms / msm,
            "time_per_sample_vs_one_channel_oneshot": (ms / (n_ch * n)) / (ms1 / n1)}
    res["parity"] = "every streamed pass bitwise equal to the one-shot"
    lib.lrc_fastfir_stream_destroy(stm)
    ff.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "fastfir_stream_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
