#!/usr/bin/env python
"""Per-kernel roofline table for every BASELINE.json config (device-resident inputs, CUDA events, inputs
>> L2).  Not the headline bench (that is bench.py); this feeds DESIGN.md / profiles/ and tells which kernel
to tune next.  Usage: python tools/bench_kernels.py [--quick] > gpurun_out/kernels.jsonl"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from libredio_b200 import blocks, synth, capi  # noqa: E402

PEAK = 6551.4
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ts = [ev[i].elapsed_time(ev[i + 1]) for i in range(iters)]
    return float(np.median(ts)), float(np.min(ts))




def cpu_rate(fn, samples_per_call, seconds=2.0):
    """Reference CPU path timed beside the GPU number (SURVEY 8d): `fn` (an oracle/ call; ctypes releases the
    GIL) on every host core for ~`seconds`; returns {"cpu_Msamples/s", "cpu_cores", "cpu_kind"}."""
    import time
    from concurrent.futures import ThreadPoolExecutor
    cores = os.cpu_count() or 1
    t0 = time.perf_counter(); fn(); per = time.perf_counter() - t0
    calls = max(1, int(seconds / max(per, 1e-6)))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:
        list(ex.map(lambda _: [fn() for _ in range(calls)], range(cores)))
    dt = time.perf_counter() - t0
    return {"cpu_Msamples/s": cores * calls * samples_per_call / dt / 1e6, "cpu_cores": cores}


def report(name, samples, alg_bytes, ms, extra=None):
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    line = {"kernel": name, "Msamples/s": samples / (ms * 1e-3) / 1e6, "ms": ms, "GB/s": gbs, "frac_hbm": gbs / PEAK,
            "alg_bytes": alg_bytes}
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--only", default="")
    ap.add_argument("--cpu", action="store_true", help="time the reference's CPU path (oracle/) beside each config")
    ap.add_argument("--ook-streams", type=int, default=0, help="streams of the OOK config (default 4096; 512 = one GPU's shard of eight)")
    a = ap.parse_args()
    if a.cpu:
        import oracle
    q = 4 if a.quick else 1
    ctx = blocks.Context(0)
    dev = ctx.tdev
    g = torch.Generator(device=dev).manual_seed(0)
    taps = synth.lpf_taps(64, 0.04)
    want = lambda k: (not a.only) or (k in a.only.split(","))

    if want("unpack"):
        n = (1 << 30) // q
        iq = torch.randint(0, 256, (n,), dtype=torch.uint8, device=dev, generator=g)
        out = torch.empty(n // 2, dtype=torch.complex64, device=dev)
        import ctypes as C
        def f():
            capi.check(ctx.lib.lrc_unpack_u8_cf32(ctx.h, C.c_void_p(iq.data_ptr()), n, C.c_void_p(out.data_ptr()), blocks._stream()), "unpack")
        ms, _ = timeit(f)
        extra = None
        if a.cpu:
            hb = np.random.default_rng(0).integers(0, 256, 1 << 22, dtype=np.uint8)
            extra = cpu_rate(lambda: oracle.data_to_samples(hb), hb.size // 2)
            extra["cpu_what"] = "restated rtlsdr::data_to_samples (rtlsdr.rs:159-162), strict f32 C"
        report("unpack u8->cf32 (K1)", n // 2, n + n * 4, ms, extra)
        del iq, out

    if want("fir"):
        # config 1/3 shape: 1024 channels x 2.4 Msps x 0.1 s
        n_ch, n = 1024 // q, 240_000
        x = torch.view_as_complex(torch.randn(n_ch, n, 2, device=dev, generator=g))
        fir = blocks.Fir(ctx, taps, 10)
        ms, _ = timeit(lambda: fir.run(x))
        extra = {"n_ch": n_ch}
        if a.cpu:
            hx = synth.cf32_noise_tones(240_000, seed=1)
            extra.update(cpu_rate(lambda: oracle.fir_decimate(hx, taps, 10), hx.size))
            extra["cpu_what"] = "restated dsputils::convolve (dsputils.rs:30-32) on kept outputs only, strict f32 C"
            full = cpu_rate(lambda: oracle.fir_decimate(hx[:60_000], taps, 10, full=True), 60_000, 1.0)
            extra["cpu_Msamples/s_faithful_all_outputs"] = full["cpu_Msamples/s"]
        report("FIR64/10 cf32 (K2 tile)", n_ch * n, n_ch * n * 8.8, ms, extra)
        iq = torch.randint(0, 256, (n_ch, 2 * n), dtype=torch.uint8, device=dev, generator=g)
        ms, _ = timeit(lambda: fir.run_u8(iq))
        report("unpack+FIR64/10 u8 fused (K1+K2)", n_ch * n, n_ch * n * 2.8, ms,
               {"flop_per_sample": 25.6, "TFLOP/s": n_ch * n * 25.6 / (ms * 1e-3) / 1e12})
        del x, iq
        fir.close()

    if want("fft"):
        n = (1 << 26) // q * 4
        x = torch.view_as_complex(torch.randn(n, 2, device=dev, generator=g))
        f = blocks.Fft(ctx, 1024, 0)
        y = torch.empty_like(x)
        xv = x.view(-1, 1024)
        import ctypes as C
        def run():
            capi.check(ctx.lib.lrc_fft_run(f.h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), n // 1024, blocks._stream()), "fft")
        ms, _ = timeit(run)
        extra = None
        if a.cpu and oracle.have_ref():
            hx = synth.cf32_noise_tones(1024 * 256, seed=2).reshape(256, 1024)
            extra = cpu_rate(lambda: oracle.kissfft_batch_cpu(hx), hx.size)
            extra["cpu_what"] = "vendored kiss_fft.c, reference build flags (libkissfft/Makefile:4, no -O)"
            extra["cpu_Msamples/s_O3"] = cpu_rate(lambda: oracle.kissfft_batch_cpu(hx, opt=True), hx.size, 1.0)["cpu_Msamples/s"]
        report("FFT1024 batched out-of-place (K3)", n, n * 16, ms, extra)
        p = blocks.Psd(ctx, 1024)
        ms, _ = timeit(lambda: p.run(x, 64))
        report("Hann+FFT1024+|X|^2 avg K=64 (config 2, K3 fused)", n, n * 8, ms,
               {"flop_per_sample": 55, "TFLOP/s": n * 55 / (ms * 1e-3) / 1e12})
        del x, y
        f.close(); p.close()

    if want("fm"):
        n_ch, n = 1024 // q, 240_000
        x = torch.view_as_complex(torch.randn(n_ch, n, 2, device=dev, generator=g))
        ms, _ = timeit(lambda: blocks.fm_demod(ctx, x))
        report("FM discriminator (K5)", n_ch * n, n_ch * n * 12, ms)
        d = torch.randn(n_ch, n, device=dev, generator=g)
        rs = blocks.Resampler(ctx, 0.2, n_ch, n)
        ms, _ = timeit(lambda: rs.process(d))
        report("resample 240k->48k, 321 taps (K6)", n_ch * n, n_ch * n * 4.8, ms,
               {"flop_per_sample": 2 * 321 / 5, "TFLOP/s": n_ch * n * 2 * 321 / 5 / (ms * 1e-3) / 1e12})
        del x, d
        rs.close()

    if want("fmchain"):
        # config 3: 1024 channels of rtlsdr u8 IQ at 2.4 Msps -> unpack+FIR64/10 -> discriminator -> resample 1/5 -> 48 kHz
        # audio.  (a) the fused receiver, ONE kernel per push (lrc_fmrx); (b) the three stand-alone stages, 3 launches
        # (+ the carry update) with the 240 kHz intermediates in HBM
        n_ch, n = 1024 // q, 240_000
        iq = torch.randint(0, 256, (n_ch, 2 * n), dtype=torch.uint8, device=dev, generator=g)
        n_bb = (n - 64) // 10 + 1
        rx = blocks.FmReceiver(ctx, taps, 10, 0.2, n_ch, n)
        n_audio = rx.next_out_len(n)
        out = torch.empty((n_ch, n_audio), dtype=torch.float32, device=dev)
        def fused():
            rx.reset()
            return rx.push(iq, out)
        ms, _ = timeit(fused)
        alg = n_ch * (n * 2 + n_audio * 4)                       # u8 IQ in, f32 audio out
        flop = 25.6 + 12.84
        report("config 3 fused receiver u8 IQ -> FIR64/10 -> FM -> 1/5 resample (one kernel)", n_ch * n, alg, ms,
               {"n_ch": n_ch, "audio_samples_per_ch": int(n_audio), "fused": rx.fused,
                "flop_per_sample": flop, "TFLOP/s": n_ch * n * flop / (ms * 1e-3) / 1e12})
        rx.close()
        fir = blocks.Fir(ctx, taps, 10)
        rs = blocks.Resampler(ctx, 0.2, n_ch, n_bb)
        def pipe():
            rs.reset()
            return rs.process(blocks.fm_demod(ctx, fir.run_u8(iq)))
        ms, _ = timeit(pipe)
        moved = n_ch * (n * 2 + n_bb * 8 * 2 + n_bb * 4 * 2 + n_audio * 4)
        report("config 3 three-stage pipeline (K1+K2, K5, K6)", n_ch * n, alg, ms,
               {"n_ch": n_ch, "bytes_moved_incl_intermediates": moved,
                "flop_per_sample": flop, "TFLOP/s": n_ch * n * flop / (ms * 1e-3) / 1e12})
        del iq
        fir.close(); rs.close()

    if want("fastfir"):
        n = (1 << 28) // q
        x = torch.view_as_complex(torch.randn(n, 2, device=dev, generator=g))
        rng = np.random.default_rng(6)
        h = ((rng.standard_normal(4096) + 1j * rng.standard_normal(4096)) / 64).astype(np.complex64)
        flop = (2 * 5 * 16384 * 14 + 6 * 16384) / 12289.0
        ff = blocks.FastFir(ctx, h, 0)
        out = torch.empty(ff.out_len(n) + 1, dtype=torch.complex64, device=dev)
        ms, _ = timeit(lambda: ff.run(x, out=out), iters=5)
        extra = {"flop_per_sample_nominal": flop, "TFLOP/s_nominal": n * flop / (ms * 1e-3) / 1e12}
        if a.cpu and oracle.have_ref():
            hx = synth.cf32_noise_tones(1 << 20, seed=5)
            extra.update(cpu_rate(lambda: oracle.ref_fastfir(h, hx), hx.size))
            extra["cpu_what"] = "vendored tools/kiss_fastfir.c (-O3, tools/Makefile:43), 2^20-sample buffers"
        report("overlap-save FIR 4096 taps, 16384-point blocks (config 5, K4)", n, n * 16, ms, extra)
        del out, x
        ff.close()

    if want("firg"):
        # stand-alone FIR for shapes without a dedicated instance: the padded-chunk tile kernel vs the one-thread-per-output kernel
        for ntaps, decim in [(64, 4), (128, 4), (64, 5), (64, 8), (128, 8), (128, 10), (64, 16), (128, 16)]:
            tp = synth.lpf_taps(ntaps, 0.4 / decim)
            n_ch, n = 256 // q, 1_000_000
            x = torch.view_as_complex(torch.randn(n_ch, n, 2, device=dev, generator=g))
            fir = blocks.Fir(ctx, tp, decim)
            ms, _ = timeit(lambda: fir.run(x))
            os.environ["LRC_FIR_NO_GENTILE"] = "1"
            ms_old, _ = timeit(lambda: fir.run(x), iters=3, warm=1)
            os.environ.pop("LRC_FIR_NO_GENTILE")
            no = (n - ntaps) // decim + 1
            report(f"FIR{ntaps}/{decim} cf32 (tile, generic shapes)", n_ch * n, n_ch * (n * 8.0 + no * 8.0), ms,
                   {"n_ch": n_ch, "flop_per_sample": 4.0 * ntaps / decim, "TFLOP/s": n_ch * n * 4.0 * ntaps / decim / (ms * 1e-3) / 1e12,
                    "one_thread_per_output_ms": ms_old, "speedup": ms_old / ms})
            fir.close()
            del x

    if want("chaing"):
        # generic fused chain instances (chain_generic.cuh) beside the unfused FIR -> HBM -> PSD path, ~2.7 GB of cf32 each
        os_env = os.environ
        for ntaps, decim, nfft in [(64, 10, 1024), (64, 4, 1024), (128, 4, 1024), (64, 5, 1024), (64, 8, 1024), (128, 8, 2048),
                                   (128, 10, 1024), (64, 10, 2048), (64, 10, 512), (64, 16, 1024), (64, 16, 512), (64, 4, 512), (64, 16, 2048), (64, 5, 2048)]:
            tp = synth.lpf_taps(ntaps, 0.4 / decim)
            k = 64
            frames = max(k, ((1 << 25) // q // (nfft * decim)) // k * k * 10)
            n = (frames - 1) * nfft * decim + (nfft - 1) * decim + ntaps
            x = torch.view_as_complex(torch.randn(n, 2, device=dev, generator=g))
            res = {}
            for label, env in (("fused", None), ("unfused", "1")):
                os_env["LRC_CHAIN_NO_GENERIC" if env else "LRC_CHAIN_GENERIC_ALL"] = "1"
                ch = blocks.Chain(ctx, tp, decim, nfft)
                os_env.pop("LRC_CHAIN_NO_GENERIC", None); os_env.pop("LRC_CHAIN_GENERIC_ALL", None)
                if label == "unfused" and (ntaps, decim, nfft) == (64, 10, 1024):
                    ch.close(); continue
                out = torch.empty((frames // k, nfft), dtype=torch.float32, device=dev)
                ms, _ = timeit(lambda: ch.run(x, k, out))
                res[label] = (ms, ch.kind)
                ch.close()
            ms, kind = res["fused"]
            extra = {"kind": kind, "flop_per_sample": 2.0 * 2 * ntaps / decim + 55.0 / decim}
            extra["TFLOP/s"] = n * extra["flop_per_sample"] / (ms * 1e-3) / 1e12
            if "unfused" in res:
                extra["unfused_ms"] = res["unfused"][0]
                extra["speedup_vs_unfused"] = res["unfused"][0] / ms
            report(f"chain {ntaps}/{decim}/{nfft} fused (kind {kind})", n, n * 8.0 + frames // k * nfft * 4, ms, extra)
            del x

    if want("ook"):
        n_streams, n_blocks = (a.ook_streams or 4096 // q), 500
        caps = [synth.ook_capture_u8(n_blocks, seed=4 + s, n_packets=2)[0] for s in range(32)]
        iq = torch.from_numpy(np.stack(caps)).to(dev).repeat(n_streams // 32, 1).contiguous()
        ook = blocks.Ook(ctx, n_streams, n_blocks, 256000, 4096, 64)
        ms, _ = timeit(lambda: ook.decode(iq), iters=5)
        ns = n_streams * n_blocks * 512
        extra = {"packets": len(ook.packets())}
        if a.cpu:
            extra.update(cpu_rate(lambda: oracle.ook_decode(caps[0]), n_blocks * 512))
            extra["cpu_what"] = "restated ratpak.rs:60-111 chain (envelope..shaper_optional), strict f32 C, one stream per core"
        report(f"OOK chain, {n_streams} streams (config 4, K7)", ns, ns * 2, ms, extra)
        ook.close()
    ctx.close()


if __name__ == "__main__":
    main()
