#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

metric : Msamples/s of cf32 through the FIR-decimate + FFT chain (64-tap low-pass /10 -> 1024-pt Hann FFT ->
         |X|^2 averaged over K=64 frames), absolute and as a fraction of the HBM roofline.
step   : one pass of the fused chain kernel over one batch of synthetic cf32 samples resident in HBM:
         65536 frames = 2^26 decimated samples into the FFT (configs[1]) = 671 088 694 input samples (5.4 GB),
         much larger than the 126 MB L2, so no L2 flush is needed between steps.
N > 1  : one process per GPU (torchrun); each rank owns an independent stream of the same size (weak
         scaling, channels sharded across GPUs); the only exchange is the gather of the 4 MB of output rows
         per rank over NVLink, inside the timed region: lrc_gather (copy-engine P2P pushes, no SMs) by
         default, NCCL all-gather with --gather nccl or when CUDA IPC is unavailable.
e2e    : the same step through the host-buffer entry point lrc_chain_run_host (pinned host input, chunked
         H2D overlapped with the kernel through the double-buffered device ring, rows copied back).
extra  : the other BASELINE.json configs measured in the same run (device-resident inputs >> L2, CUDA events, max over
         ranks): config 1 from u8 IQ, config 2 (PSD), config 3 (1024-channel FM receiver, one fused kernel), config 4
         (4096 OOK streams, sharded across the ranks) and config 5 (4096 taps over 2^30 samples, chunk-sharded across
         the ranks; outputs left sharded and gathered to rank 0), each with its roofline fraction.  --no-extra skips it.
--impl reference : the reference's own CPU path (oracle/: strict-f32 restatement of dsputils::convolve +
         the vendored kissfft built with the reference's flags), all host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the bench runs from a built tree that may be read-only: it leaves no caches in it

NTAPS, DECIM, NFFT, K_AVG = 64, 10, 1024, 64
FRAMES = 65536                      # 2^26 decimated samples / 1024
BYTES_PER_SAMPLE = 8.0              # SURVEY 8d: compulsory traffic = first read of cf32 (+ 4/(10*K) B of rows)
METRIC = "Msamples/s cf32 through FIR-decimate+FFT chain"
UNIT = "Msamples/s"


def n_input(frames: int) -> int:
    return frames * NFFT * DECIM + NTAPS - DECIM


def workload_name(frames: int) -> str:
    return (f"cf32 {n_input(frames)} samples -> FIR{NTAPS}/{DECIM} -> {frames} frames x {NFFT}-pt Hann FFT "
            f"(2^{int(np.log2(frames * NFFT))} samples into the FFT) -> |X|^2 avg K={K_AVG}")


def chain_source_sha() -> str:
    """sha256 over the sources the fused chain kernel is compiled from (what roofline.traffic is tied to)"""
    import hashlib
    h = hashlib.sha256()
    for f in ("k_chain.cu", "fir_core.cuh", "fft_core.cuh", "common.cuh"):
        with open(os.path.join(ROOT, "libredio_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def config_dict(frames: int, world: int) -> dict:
    """what the number was measured on; the SAME dict in both arms (the CPU arm times a bounded sample of it, described
    under cpu_baseline.sample)"""
    return {"workload": workload_name(frames), "ntaps": NTAPS, "decim": DECIM, "nfft": NFFT, "k_avg": K_AVG,
            "window": "hann", "frames": frames, "l2": "input 5.4 GB per step >> 126 MB L2, no flush needed",
            "sharding": f"{world} independent streams, one per GPU; gather of output rows only"}


FP32_PEAK_TFLOPS = 73.7      # packed FFMA2 micro-benchmark on a B200 (tools/ubench/f32x2.cu, profiles/r1_s8_f32x2_ubench.txt)


# ------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and clock-event reasons sampled through NVML every ~2 ms from a thread (nvidia-smi -lms cannot
    deliver a sample inside a region that lasts tens of milliseconds); nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, uuid: str | None = None):
        self.index, self.uuid = index, uuid
        self.sm, self.mx, self.pw, self.reasons = [], [], [], set()
        self.stop_flag = threading.Event()
        self.th = None
        self.how = None
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                for cand in (uuid, "GPU-" + uuid):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand if isinstance(cand, bytes) else cand.encode())
                        break
                    except Exception:
                        h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nv, self.h = pynvml, h
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.how = "nvml"
        except Exception:
            self.nv = None

    def _poll_nvml(self):
        nv, h = self.nv, self.h
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake_slowdown"}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mx.append(self.max_sm)
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                try:
                    self.pw.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
            except Exception:
                break
            time.sleep(0.002)

    def _poll_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.proc.stdout:
            p = [s.strip() for s in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                self.sm.append(float(p[1])); self.mx.append(float(p[2])); self.pw.append(float(p[3]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    self.reasons.add(nm)

    def start(self):
        if self.nv is not None:
            self.th = threading.Thread(target=self._poll_nvml, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi -lms 20"
            self.th = threading.Thread(target=self._poll_smi, daemon=True)
            self.th.start()
        except Exception:
            self.how = None

    def n(self) -> int:
        return len(self.sm)

    def stop(self) -> dict:
        if self.how is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"], "samples": 0}
        self.stop_flag.set()
        if self.nv is None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.th:
            self.th.join(timeout=2)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None,
                "power_w_max": max(self.pw) if self.pw else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "how": self.how}


# ------------------------------------------------------------------------------------------------------
# CPU reference arm / baseline
# ------------------------------------------------------------------------------------------------------
def cpu_model() -> str:
    """host CPU model string (SURVEY 8d: the CPU baseline states core count and model of the box it ran on)"""
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_chain_rate(seconds_target: float, threads: int, frames_per_call: int = 64, full: bool = False):
    """Time the CPU chain (oracle FIR restatement + vendored kissfft at the reference's build flags) on a
    bounded sample with `threads` host threads.  Returns (Msamples/s, description, kind, frames, secs)."""
    import oracle
    from libredio_b200 import synth
    from concurrent.futures import ThreadPoolExecutor
    taps = synth.lpf_taps(NTAPS, 0.04)
    win = synth.hann_periodic(NFFT)
    x = synth.cf32_noise_tones(n_input(frames_per_call), seed=2)
    use_ref = oracle.have_ref()

    def one(_):
        psd, nfr = oracle.chain_psd_cpu(x, taps, DECIM, NFFT, win, use_ref=use_ref, opt=False, full=full)
        return nfr

    t0 = time.perf_counter()
    one(0)
    per_call = time.perf_counter() - t0
    calls = max(threads, int(seconds_target / max(per_call, 1e-6)) * threads)
    calls = (calls + threads - 1) // threads * threads
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        frames = sum(ex.map(one, range(calls)))
    dt = time.perf_counter() - t0
    msps = frames * NFFT * DECIM / dt / 1e6
    kind = "port"
    desc = (f"{frames} frames ({frames * NFFT * DECIM} input samples) of the same workload, {threads} threads: "
            f"strict-f32 C restatement of dsputils::convolve "
            + ("(every lag computed as in dsputils.rs:30-32, then every 10th kept) + " if full
               else "(decimating: only kept outputs are computed) + ")
            + ("vendored kiss_fft.c built with the reference's flags (libkissfft/Makefile:4, no -O)" if use_ref
               else "restated kissfft (oracle/_ref not present)") + " + Hann + |X|^2 accumulation")
    return msps, desc, kind, frames, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    vals = []
    for _ in range(args.warmup):
        cpu_chain_rate(0.5, cores)
    per_step = max(2.0, min(20.0, 90.0 / max(args.steps, 1)))
    t_all = 0.0
    frames_all = 0
    desc = kind = ""
    for _ in range(args.steps):
        msps, desc, kind, frames, dt = cpu_chain_rate(per_step, cores)
        vals.append(msps); t_all += dt; frames_all += frames
    value = frames_all * NFFT * DECIM / t_all / 1e6
    f_msps, f_desc, _, _, _ = cpu_chain_rate(1.0, cores, full=True)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.frames, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "cpu_model": cpu_model(), "kind": kind, "sample": desc,
                         "as_written_all_lags": {"value": f_msps, "unit": UNIT, "sample": f_desc,
                                                 "note": "informational: the reference has no decimating FIR; `value` is the "
                                                         "stronger CPU baseline that skips the 9 of 10 dropped outputs"}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)



# ------------------------------------------------------------------------------------------------------
# the other BASELINE configs, in the same run (device-resident inputs, CUDA events, max over ranks)
# ------------------------------------------------------------------------------------------------------
def _timed(fn, iters, warm, world, dev, inner=4):
    """median / best milliseconds per call of fn(): `iters` measurements of `inner` back-to-back calls between two CUDA
    events on the current stream (launch latency amortised as in a stream of chunks), after `warm` calls; with several
    ranks every measurement starts behind a barrier and counts as the slowest rank's time"""
    import torch
    import torch.distributed as dist
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(inner):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / inner], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ts.append(float(t.item()))
    return float(np.median(ts)), float(np.min(ts))


def run_extras(ctx, world, rank, peak_hbm, quick=False):
    """configs 1 (u8), 2, 3, 4, 5 of BASELINE.json.  Configs 1-3 are per-rank replicas of the full-size workload (weak
    scaling, like the headline); configs 4 and 5 are ONE job of BASELINE size split across the ranks (strong scaling):
    streams for config 4, 16384-point overlap-save blocks for config 5 (every rank reads its own nh-1 halo from its
    slice of the source, no exchange), timed with the outputs left sharded and with the outputs gathered to rank 0."""
    import torch
    import torch.distributed as dist
    from libredio_b200 import blocks, synth, capi, shard
    dev = ctx.tdev
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    taps = synth.lpf_taps(NTAPS, 0.04)
    q = 8 if quick else 1
    out = {}

    def entry(name, samples_total, ms, best, bound, alg_bytes_total, flop_per_sample=None, **kw):
        e = {"value": samples_total / (ms * 1e-3) / 1e6, "unit": UNIT, "ms": ms, "ms_best": best, "n_gpus": world}
        gbs = alg_bytes_total / (ms * 1e-3) / 1e9
        roof = {"bound": bound, "hbm_gbs_algorithmic": gbs, "hbm_frac": gbs / (peak_hbm * world)}
        if flop_per_sample is not None:
            tf = samples_total * flop_per_sample / (ms * 1e-3) / 1e12
            roof.update({"tflops_nominal": tf, "fp32_frac": tf / (FP32_PEAK_TFLOPS * world), "flop_per_sample_nominal": flop_per_sample,
                         "fp32_peak_tflops": FP32_PEAK_TFLOPS})
        roof["frac"] = roof["fp32_frac"] if bound == "fp32" else roof["hbm_frac"]
        e["roofline"] = roof
        e.update(kw)
        out[name] = e

    # ---- config 1 from the wire format: 1024 channels x 240 k samples of u8 IQ -> fused unpack + FIR64/10 ------------
    n_ch, n = 1024 // q, 240_000
    iq = torch.randint(0, 256, (n_ch, 2 * n), dtype=torch.uint8, device=dev, generator=g)
    fir = blocks.Fir(ctx, taps, DECIM)
    ms, best = _timed(lambda: fir.run_u8(iq), 6, 3, world, dev)
    entry("config1_u8_fir64_decim10", world * n_ch * n, ms, best, "fp32", world * n_ch * n * 2.8, 25.6,
          workload=f"{n_ch} channels x {n} samples of rtlsdr u8 IQ per GPU -> unpack + FIR64/10 (one kernel), cf32 out",
          scaling="weak")
    fir.close()
    # ---- the headline chain fed the wire format (device-resident u8 IQ): unpack inside the kernel's tile load ------------
    fr8 = 16384 // q
    n8 = n_input(fr8)
    iq8 = torch.randint(0, 256, (2 * n8,), dtype=torch.uint8, device=dev, generator=g)
    ch8 = blocks.Chain(ctx, taps, DECIM, NFFT, capi.WINDOW_HANN)
    rows8 = torch.empty((fr8 // K_AVG, NFFT), dtype=torch.float32, device=dev)
    ms, best = _timed(lambda: ch8.run_u8(iq8, K_AVG, rows8), 6, 3, world, dev)
    entry("headline_chain_from_u8", world * n8, ms, best, "fp32", world * (n8 * 2.0 + rows8.numel() * 4), 31.6 + 20.0,
          workload=f"{n8} samples of u8 IQ per GPU -> i2f in the tile (bit-exact) -> FIR64/10 -> {fr8} x 1024-pt Hann FFT -> |X|^2 "
                   f"avg K={K_AVG}; one kernel, 2 B/sample from HBM", scaling="weak")
    ch8.close()
    del iq8, rows8
    # ---- config 3: the same input through the whole FM receiver, one fused kernel -------------------------------------
    rx = blocks.FmReceiver(ctx, taps, DECIM, 0.2, n_ch, n)
    n_audio = rx.next_out_len(n)
    audio = torch.empty((n_ch, max(n_audio, 1)), dtype=torch.float32, device=dev)

    def fm():
        rx.reset()
        rx.push(iq, audio)
    ms, best = _timed(fm, 6, 3, world, dev)
    entry("config3_fm_receiver_1024ch", world * n_ch * n, ms, best, "fp32", world * n_ch * (n * 2 + n_audio * 4), 25.6 + 12.84,
          workload=f"{n_ch} channels x {n} samples of u8 IQ per GPU -> FIR64/10 -> discriminator -> 1/5 resampler -> "
                   f"{n_audio} audio samples per channel; one kernel per push (fused={rx.fused})",
          scaling="weak", parity_note="resampler parity UNPINNED (libsamplerate absent): held to the builder's own f64 definition")
    rx.close()
    del iq, audio
    # ---- config 2: Hann + FFT1024 + |X|^2 averaged over K = 64, 2^26 samples --------------------------------------------
    n2 = (1 << 26) // q
    x = torch.view_as_complex(torch.randn(n2, 2, device=dev, generator=g))
    psd = blocks.Psd(ctx, NFFT, capi.WINDOW_HANN)
    ms, best = _timed(lambda: psd.run(x, K_AVG), 6, 3, world, dev)
    entry("config2_psd_1024_hann_k64", world * n2, ms, best, "hbm", world * (n2 * 8 + n2 // K_AVG * 4), 55.0,
          workload=f"2^{int(np.log2(n2))} cf32 samples per GPU -> Hann -> FFT1024 -> |X|^2 averaged over K=64", scaling="weak")
    psd.close()
    del x
    # ---- config 4: 4096 OOK streams, sharded across the ranks ---------------------------------------------------------
    n_streams, n_blocks = 4096 // q, 500
    lo, hi = shard.split_units(n_streams, rank, world)
    caps = [synth.ook_capture_u8(n_blocks, seed=4 + s, n_packets=2)[0] for s in range(16)]
    iq = torch.from_numpy(np.stack(caps)).to(dev)[torch.arange(lo, hi, device=dev) % 16].contiguous()
    ook = blocks.Ook(ctx, hi - lo, n_blocks, 256000, 4096, 64)
    ms, best = _timed(lambda: ook.decode(iq), 4, 2, world, dev, inner=3)
    ns = n_streams * n_blocks * 512
    n_pk = torch.tensor([len(ook.packets())], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(n_pk)
    entry("config4_ook_4096_streams", ns, ms, best, "hbm", ns * 2.0,
          workload=f"{n_streams} streams x {n_blocks} blocks of 512 u8 IQ samples, {n_streams // world} streams per GPU, "
                   "envelope -> trigger -> slicer -> rle -> matchers -> packets (bit-exact chain; blocks that cannot hold a 1 bit are sliced unread)",
          scaling="strong", packets_decoded=int(n_pk.item()))
    ook.close()
    del iq
    # ---- config 5: 4096 taps over 2^30 samples, 16384-point blocks sharded across the ranks -------------------------------
    nh, n5, nfft = 4096, (1 << 30) // q, 16384
    rng = np.random.default_rng(6)
    h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64).astype(np.complex64)
    sh = shard.fastfir_shard(n5, nh, nfft, rank, world)
    xs = torch.empty(max(sh.in_len, 1), dtype=torch.complex64, device=dev)
    for a0 in range(0, sh.in_len, 1 << 27):                      # generated in pieces: randn's temporaries stay small
        a1 = min(sh.in_len, a0 + (1 << 27))
        xs[a0:a1] = torch.view_as_complex(torch.randn(a1 - a0, 2, device=dev, generator=g))
    ff = blocks.FastFir(ctx, h, nfft)
    ys = torch.empty(sh.out_len + 1, dtype=torch.complex64, device=dev)
    ms, best = _timed(lambda: ff.run(xs[: sh.in_len], out=ys), 4, 2, world, dev, inner=2)
    n_out_all = shard.fastfir_shard(n5, nh, nfft, world - 1, world)
    n_out_all = n_out_all.out_start + n_out_all.out_len          # outputs of the whole job
    flop16 = (2 * 5 * nfft * 14 + 6 * nfft) / float(nfft - nh + 1)
    entry("config5_fastfir_4096taps_2pow30", n_out_all, ms, best, "fp32", n_out_all * 16.0, flop16,
          workload=f"4096 complex taps over a 2^{int(np.log2(n5))}-sample cf32 stream, overlap-save in 16384-point blocks "
                   f"(12289 outputs kept per block), {world} contiguous block ranges, outputs left sharded",
          scaling="strong")
    if world > 1:
        # the same with every shard's output gathered on rank 0 (SURVEY 7.7: the gather, not the filter, bounds this form)
        width = max(shard.fastfir_shard(n5, nh, nfft, r, world).out_len for r in range(world)) + 1
        ysend = ys if ys.numel() == width else torch.cat([ys, ys.new_zeros(width - ys.numel())])
        glist = [torch.empty(width, dtype=torch.complex64, device=dev) for _ in range(world)] if rank == 0 else None

        def filt_and_gather():
            ff.run(xs[: sh.in_len], out=ysend[: sh.out_len + 1])
            dist.gather(torch.view_as_real(ysend), [torch.view_as_real(t) for t in glist] if rank == 0 else None, dst=0)
        ms_g, best_g = _timed(filt_and_gather, 3, 1, world, dev, inner=1)
        out["config5_fastfir_4096taps_2pow30"]["gathered_to_rank0"] = {
            "value": n_out_all / (ms_g * 1e-3) / 1e6, "unit": UNIT, "ms": ms_g, "ms_best": best_g,
            "gather": f"dist.gather (NCCL) of {width * 8 / 2**30:.2f} GiB per rank into rank 0"}
        del glist, ysend
    ff.close()
    del xs, ys
    torch.cuda.empty_cache()
    return out


def dump_rows(out_dir, rows, world, rank):
    """DIR/psd_rows.npy: the f32 PSD rows of the last timed step, every rank's rows in rank order (4 MB per rank)"""
    import torch
    import torch.distributed as dist
    if world > 1:
        full = torch.empty((world * rows.shape[0], rows.shape[1]), dtype=rows.dtype, device=rows.device)
        dist.all_gather_into_tensor(full, rows)
        rows = full
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "psd_rows.npy"), rows.cpu().numpy())


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from libredio_b200 import blocks, synth, capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = blocks.Context(local)
    dev = ctx.tdev
    frames = args.frames
    n_in = n_input(frames)
    taps = synth.lpf_taps(NTAPS, 0.04)
    chain = blocks.Chain(ctx, taps, DECIM, NFFT, capi.WINDOW_HANN)

    # synthetic input, generated on the device for the HBM-resident leg: noise + 3 tones, seeded per rank
    g = torch.Generator(device=dev).manual_seed(2 + rank)
    x = torch.view_as_complex(torch.randn(n_in, 2, device=dev, generator=g))
    CH = 1 << 24
    for f, a in ((0.011, 2.0), (-0.0273, 1.0), (0.0402, 0.5)):
        for s in range(0, n_in, CH):
            e = min(n_in, s + CH)
            ph = (2 * np.pi * f) * torch.arange(s, e, device=dev, dtype=torch.float64)
            x[s:e] += torch.polar(torch.full((e - s,), a, device=dev, dtype=torch.float32), (ph % (2 * np.pi)).float())
    rows = frames // K_AVG
    # two output slots: the NVLink gather of step i (NCCL's stream) overlaps the kernel of step i+1
    outs = [torch.empty((rows, NFFT), dtype=torch.float32, device=dev) for _ in range(2)]
    pending = [None, None]
    # the only exchange: every rank's output rows go to every peer.  Default: lrc_gather (copy engines over NVLink,
    # zero SMs, overlaps the next step's persistent kernel); fallback / --gather nccl: NCCL all-gather, whose kernel
    # cannot start while the chain kernel fills every SM and therefore serialises with it.
    gather, gather_kind, gath, gather_all, gather_rot, gather_host, gather_p2p = None, "none (1 GPU)", None, None, None, None, None
    if world > 1:
        ok = torch.zeros(1, device=dev)
        if args.gather == "ce":
            # the host gather (diagnostic line, or the gather itself with --gather-to host) is set up on its own: a node without
            # usable POSIX shared memory must not cost the run its NVLink gather.  Every collective below is reached by all ranks.
            shm = [f"/lrc_bench_{os.getpid()}_{os.environ.get('MASTER_PORT', '0')}" if rank == 0 else None]
            dist.broadcast_object_list(shm, src=0)
            hok = torch.zeros(1, device=dev)
            try:
                gather_host = blocks.Gather(ctx, rank, world, rows * NFFT * 4, slots=2, host_shm=shm[0], root=0)
                hok += 1
            except Exception as e:
                print(f"bench.py rank {rank}: host gather unavailable ({e})", file=sys.stderr)
                gather_host = None
            dist.all_reduce(hok)
            if int(hok.item()) != world:
                if gather_host is not None:
                    gather_host.close()
                gather_host = None
                if args.gather_to == "host":
                    args.gather_to = "root"
            try:
                gather_p2p = blocks.Gather(ctx, rank, world, rows * NFFT * 4, slots=2).connect_distributed()
                gather = gather_host if args.gather_to == "host" else gather_p2p
                if args.gather_to == "root":
                    gather.set_root(0)
                elif args.gather_to == "rotate":
                    gather.set_root(-2)
                # diagnostics only: the same loop with the other two placements of the receiver
                gather_all = blocks.Gather(ctx, rank, world, rows * NFFT * 4, slots=2).connect_distributed()
                gather_rot = blocks.Gather(ctx, rank, world, rows * NFFT * 4, slots=2).connect_distributed().set_root(-2)
                ok += 1
            except Exception as e:                         # e.g. CUDA IPC not permitted in this container
                print(f"bench.py rank {rank}: lrc_gather unavailable ({e}); using the NCCL all-gather", file=sys.stderr)
                gather = None
        dist.all_reduce(ok)                                # all ranks must agree on the mechanism BEFORE anyone waits on a peer
        if int(ok.item()) != world:
            if gather is not None:
                gather.close()
            for gx in (gather_all, gather_rot, gather_host, gather_p2p):
                if gx is not None and gx is not gather:
                    gx.close()
            gather = gather_all = gather_rot = gather_host = gather_p2p = None
        # bounded-time probe before the timed loop depends on it (every rank created and connected its Gather): one push +
        # arrival wait per slot on a side stream, polled from the host.  A peer whose flag write never arrives would
        # otherwise hang the bench inside a device-side wait; the probing stream can never drain in that case, so the
        # process cannot fall back: it fails fast with a message instead (rerun with --gather nccl).
        if gather is not None:
            side = torch.cuda.Stream(device=dev)
            with torch.cuda.stream(side):
                for b in range(2):
                    gather.push(b, outs[b])
                    gather.wait(b)
                pev = torch.cuda.Event()
                pev.record()
            t0, probe_stuck = time.perf_counter(), False
            while not pev.query():
                if time.perf_counter() - t0 > args.gather_probe_s:
                    probe_stuck = True
                    break
                time.sleep(0.005)
            if probe_stuck:
                print(f"bench.py rank {rank}: lrc_gather probe did not complete in {args.gather_probe_s:.0f} s "
                      "(a peer's arrival flag never came); rerun with --gather nccl", file=sys.stderr, flush=True)
                os._exit(3)
        if gather is None:
            gath = [torch.empty((world * rows, NFFT), dtype=torch.float32, device=dev) for _ in range(2)]
            gather_kind = "NCCL all_gather_into_tensor of output rows (async, 2 slots)"
        else:
            gather_kind = ("lrc_gather to HOST memory: every rank copies its output rows D2H over its own PCIe link into one page-locked "
                           "shared-memory segment of the node, rank 0 (where the consumer block runs on the CPU) orders on the flags"
                           if args.gather_to == "host" else
                           "lrc_gather, root 0: copy-engine P2P push of every rank's output rows into rank 0's slot (CUDA IPC, 2 slots)"
                           if args.gather_to == "root" else
                           "lrc_gather, rotating receiver: step n's rows of every rank land on rank (n - 1 + slot) % world"
                           if args.gather_to == "rotate" else
                           "lrc_gather, all ranks: copy-engine P2P push of output rows into every peer's slot (CUDA IPC, 2 slots)")

    def step(i):
        b = i & 1
        if gather is not None:
            gather.wait_sent(b)                            # slot reuse: the previous push must have read outs[b]
        elif pending[b] is not None:
            pending[b].wait()                              # slot reuse: its previous gather must be done
            pending[b] = None
        chain.run(x, K_AVG, outs[b])
        if gather is not None:
            gather.push(b, outs[b])
        elif world > 1:
            pending[b] = dist.all_gather_into_tensor(gath[b], outs[b], async_op=True)

    def drain():
        for b in range(2):
            if gather is not None:
                gather.wait(b)                             # every peer's rows for this slot have ARRIVED here
            elif pending[b] is not None:
                pending[b].wait()
                pending[b] = None

    for i in range(max(args.warmup, 3)):
        step(i)
    drain()
    torch.cuda.synchronize()

    try:
        uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local, uuid) if rank == 0 else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.start()
    def timed_loop(with_gather: bool, gather=gather):
        """EXACTLY `steps` steps between two events (per-step kernel events inside); the last gathers are drained inside"""
        def drain():
            for b in range(2):
                if gather is not None:
                    gather.wait(b)                             # every peer's rows for this slot have ARRIVED here
                elif pending[b] is not None:
                    pending[b].wait()
                    pending[b] = None
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        ev0.record()
        for i in range(args.steps):
            b = i & 1
            if with_gather:
                if gather is not None:
                    gather.wait_sent(b)
                elif pending[b] is not None:
                    pending[b].wait()
                    pending[b] = None
            kev[i][0].record()
            chain.run(x, K_AVG, outs[b])
            kev[i][1].record()
            if with_gather:
                if gather is not None:
                    gather.push(b, outs[b])
                elif world > 1:
                    pending[b] = dist.all_gather_into_tensor(gath[b], outs[b], async_op=True)
                if i == args.steps - 1:
                    drain()                                    # the last gathers are inside the timed region
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1), float(np.mean([a.elapsed_time(b) for a, b in kev]))

    total_ms, kern_ms = timed_loop(True)
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_rows(args.dump_outputs, outs[(args.steps - 1) & 1], world, rank)
    if world > 1:
        dist.barrier()
    if gather is not None:
        # the gathered rows must be what an NCCL all-gather of the same outputs gives (every step computes the same
        # rows from the same resident input, so both slots hold the final result of every rank)
        torch.cuda.synchronize()
        for b in range(2):
            want = torch.empty((world * rows, NFFT), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(want, outs[b])
            if args.gather_to == "host":
                if rank == 0:
                    gather.wait(b)
                    torch.cuda.synchronize()
                    if not torch.equal(gather.buffer(b).reshape(world * rows, NFFT), want.cpu()):
                        raise SystemExit(f"bench.py rank {rank}: host gather slot {b} differs from the NCCL all-gather")
                continue
            got = gather.buffer(b).reshape(world * rows, NFFT)
            w_ = max(args.warmup, 3)
            last_push = 1 + (w_ + 1 - b) // 2 + (args.steps + 1 - b) // 2     # pushes of slot b so far: probe, warm-up, timed
            mine = (args.gather_to == "all" or (args.gather_to == "root" and rank == 0) or
                    (args.gather_to == "rotate" and rank == (last_push - 1 + b) % world))
            if mine and not torch.equal(got, want):
                raise SystemExit(f"bench.py rank {rank}: lrc_gather slot {b} differs from the NCCL all-gather")
    # ---- where a multi-GPU step's time goes (VERDICT r1: 0.93 at 8 GPUs unexplained): every rank's own kernel time, the
    # same timed loop again WITHOUT the gather (no pushes, no arrival waits; max over ranks), and rank 0 alone
    diag = None
    if world > 1:
        kall = torch.zeros(world, device=dev, dtype=torch.float64)
        kall[rank] = kern_ms
        dist.all_reduce(kall)
        dist.barrier()
        torch.cuda.synchronize()
        ng_ms, ng_kern = timed_loop(False)
        tn = torch.tensor([ng_ms, ng_kern], device=dev, dtype=torch.float64)
        dist.all_reduce(tn, op=dist.ReduceOp.MAX)
        ta = tr = None
        if gather_all is not None:                             # the same loop with the rows pushed to EVERY rank ...
            dist.barrier()
            torch.cuda.synchronize()
            ag_ms, ag_kern = timed_loop(True, gather_all)
            ta = torch.tensor([ag_ms, ag_kern], device=dev, dtype=torch.float64)
            dist.all_reduce(ta, op=dist.ReduceOp.MAX)
            dist.barrier()                                     # ... and with the receiver rotating from step to step
            torch.cuda.synchronize()
            rg_ms, rg_kern = timed_loop(True, gather_rot)
            tr = torch.tensor([rg_ms, rg_kern], device=dev, dtype=torch.float64)
            dist.all_reduce(tr, op=dist.ReduceOp.MAX)
        th = None
        if gather_host is not None:                            # ... and with the rows gathered into the node's HOST memory
            dist.barrier()
            torch.cuda.synchronize()
            hg_ms, hg_kern = timed_loop(True, gather_host)
            th = torch.tensor([hg_ms, hg_kern], device=dev, dtype=torch.float64)
            dist.all_reduce(th, op=dist.ReduceOp.MAX)
        # one rank alone (the others idle): is the kernel itself slower when its peers run (power, NVLink inbound writes)?
        solo = torch.zeros(2, device=dev, dtype=torch.float64)
        dist.barrier()
        if rank == 0:
            a_ms, a_kern = timed_loop(False)
            solo[0], solo[1] = a_ms / args.steps, a_kern
        dist.barrier()
        dist.all_reduce(solo)
        # Isolation of the receiver's slow-down: rank 0 runs the kernel-only loop while its peers run NO kernel that touches HBM --
        # a spin kernel paces them to one push of their (stale) rows per step time, into rank 0's slot.  Same inbound bytes per
        # step as the real loop, no peer compute, no peer power draw to speak of: what is left is the inbound traffic itself.
        # Second pass: only ONE peer pushes (1/7 of the bytes).
        iso = [None, None]
        if gather is not None and args.gather_to == "root":
            try:
                clk_hz = torch.cuda.clock_rate() * 1e6 if hasattr(torch.cuda, "clock_rate") else 1.6e9    # MHz -> Hz
            except Exception:
                clk_hz = 1.6e9
            spin = int(0.78e-3 * clk_hz)                           # torch.cuda._sleep counts SM cycles
            for pi, pushers in enumerate((range(1, world), (1,))):
                dist.barrier()
                torch.cuda.synchronize()
                res = torch.zeros(1, device=dev, dtype=torch.float64)
                if rank == 0:
                    _, k_iso = timed_loop(False)
                    res[0] = k_iso
                elif rank in pushers:
                    for i in range(args.steps + 6):                # a little longer than rank 0's loop
                        b = i & 1
                        gather.wait_sent(b)
                        torch.cuda._sleep(spin)
                        gather.push(b, outs[b])
                    torch.cuda.synchronize()
                dist.barrier()
                dist.all_reduce(res)
                iso[pi] = float(res[0].item())
            if rank == 0:                                           # leave the slots consistent: nothing reads them after this
                torch.cuda.synchronize()
        # the loops above ran one after the other on GPUs held at their power cap: later loops run a little slower whatever they do
        # (the clocks sag as the run goes on).  The main loop once more, last, shows how much of a difference is just that.
        dist.barrier()
        torch.cuda.synchronize()
        rp_ms, rp_kern = timed_loop(True)
        trp = torch.tensor([rp_ms, rp_kern], device=dev, dtype=torch.float64)
        dist.all_reduce(trp, op=dist.ReduceOp.MAX)
        diag = {"ms_per_step_main_loop_again_after_the_diagnostics": float(trp[0].item()) / args.steps,
                "kernel_ms_main_loop_again_after_the_diagnostics": float(trp[1].item()),
                "ms_per_step_host_gather_max_over_ranks": (float(th[0].item()) / args.steps) if th is not None else None,
                "kernel_ms_host_gather_max_over_ranks": float(th[1].item()) if th is not None else None,
                "kernel_ms_rank0_while_idle_peers_only_push": iso[0],
                "kernel_ms_rank0_while_ONE_idle_peer_pushes": iso[1],
                "kernel_ms_per_rank": [float(v) for v in kall.tolist()],
                "ms_per_step_without_gather_max_over_ranks": float(tn[0].item()) / args.steps,
                "kernel_ms_without_gather_max_over_ranks": float(tn[1].item()),
                "ms_per_step_all_gather_max_over_ranks": (float(ta[0].item()) / args.steps) if ta is not None else None,
                "kernel_ms_all_gather_max_over_ranks": float(ta[1].item()) if ta is not None else None,
                "ms_per_step_rotating_receiver_max_over_ranks": (float(tr[0].item()) / args.steps) if tr is not None else None,
                "kernel_ms_rotating_receiver_max_over_ranks": float(tr[1].item()) if tr is not None else None,
                "ms_per_step_rank0_alone_peers_idle": float(solo[0].item()),
                "kernel_ms_rank0_alone_peers_idle": float(solo[1].item()),
                "note": "ORDER MATTERS: these loops run one after the other and the later ones are slower whatever they do (power-capped "
                        "clocks sag during the run: compare main_loop_again with the bench line's ms_per_step); A/B claims come from "
                        "separate bench.py runs with the mode under test as the main loop (profiles/r2_z_gather_ab_n8.txt).  "
                        "kernel_ms_per_rank: only the RECEIVER of the gather runs a slower kernel (inbound P2P writes into an "
                        "HBM-saturated GPU); ms_per_step - ms_per_step_without_gather = what the gather costs in all; the all-gather and "
                        "rotating-receiver lines are the same loop with the receiver placed differently; without_gather - rank0_alone "
                        "= what running next to busy peers costs"}
    clocks = None
    if sampler:
        # NVML refreshes its clock reading only every few tens of ms: when the timed region was too short
        # to be seen, keep the same steps running (untimed) under the sampler until it has a few readings.
        window = "timed region"
        if sampler.n() < 8 or total_ms < 300.0:
            t_end = time.perf_counter() + 0.6
            i = 0
            while time.perf_counter() < t_end:
                chain.run(x, K_AVG, outs[i & 1]); i += 1
                if i % 16 == 0:
                    torch.cuda.synchronize()
            torch.cuda.synchronize()
            window = f"timed region ({total_ms:.0f} ms) + 0.6 s of the same step repeated untimed right after it"
        clocks = sampler.stop()
        clocks["window"] = window
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * n_in / (ms_per_step * 1e-3) / 1e6

    # ---- e2e through the host-buffer entry point (rank-local pinned input) ---------------------------
    e2e_steps = max(1, min(args.steps, 3))
    e2e_frames = min(frames, args.e2e_frames)
    n_e = n_input(e2e_frames)
    bound_cpus = ctx.bind_thread()                         # this rank's thread on the GPU's NUMA node (no-op on one node)
    xh = ctx.pinned(n_e, torch.complex64)                  # lrc_host_alloc: pinned, on the GPU's NUMA node
    xh.copy_(x[:n_e])
    rows_h = ctx.pinned((e2e_frames // K_AVG, NFFT), torch.float32)
    chain.run_host(xh, K_AVG, rows_h)                      # warm-up (allocates the ring)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        chain.run_host(xh, K_AVG, rows_h)                  # synchronous: returns when rows are on the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * n_e * e2e_steps / float(te.item()) / 1e6
    # the same chain fed in the reference's own wire format (rtlsdr u8 I,Q, rtlsdr.rs:160-162: 2 bytes per sample over
    # PCIe, data_to_samples on the device): first-class beside the cf32 figure, with its own copies declared
    iqh = ctx.pinned(2 * n_e, torch.uint8)
    iqh.copy_((x[:n_e].view(torch.float32).reshape(-1).clamp(-1, 1) * 127 + 127).round().to(torch.uint8))
    chain.run_host_u8(iqh, K_AVG, rows_h)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        chain.run_host_u8(iqh, K_AVG, rows_h)
    torch.cuda.synchronize()
    tu = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tu, op=dist.ReduceOp.MAX)
    e2e_u8_value = world * n_e * e2e_steps / float(tu.item()) / 1e6
    # what bounds e2e: bare pinned-host -> device copies of the same buffer, ALL ranks copying at the same time (the host
    # side -- DRAM and PCIe root complexes -- is shared by the GPUs of a box), max over ranks
    xd = torch.empty(n_e, dtype=torch.complex64, device=dev)
    xd.copy_(xh, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(3):
        xd.copy_(xh, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    tc = torch.tensor([c0.elapsed_time(c1) * 1e-3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    h2d_gbs = 3 * n_e * 8 / float(tc.item()) / 1e9        # per GPU, with every GPU of the job copying
    del xd

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback (B200_PROFILING.md 6.65 TB/s)"
    # ---- the other BASELINE configs (every rank takes part: configs 4 and 5 are sharded across the ranks) ----------------
    extra = None
    if not args.no_extra:
        del x, xh
        torch.cuda.empty_cache()
        extra = run_extras(ctx, world, rank, peak, quick=args.quick_extra)
    if rank == 0:
        alg_bytes = n_in * BYTES_PER_SAMPLE + rows * NFFT * 4
        achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
        # DRAM bytes per launch from the committed ncu capture -- only while the capture still describes THIS kernel: the
        # file records the sha256 of the kernel's sources at capture time (tools/chain_traffic.py writes it)
        traffic, traffic_note = None, "no ncu capture committed for this kernel source"
        tp = os.path.join(ROOT, "profiles", "chain_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if tj.get("kernel_source_sha256") == chain_source_sha():
                    traffic = tj.get("dram_bytes_per_launch")
                    traffic_note = f"ncu dram__bytes_read+write of one launch, {tj.get('capture', 'profiles/')}"
                else:
                    traffic_note = "profiles/chain_traffic.json was captured for an older kernel source: not reported"
            except Exception:
                traffic = None
        cpu = None
        if world == 1 and not args.no_cpu:
            msps, desc, kind, _, _ = cpu_chain_rate(args.cpu_seconds, os.cpu_count() or 1)
            cpu = {"value": msps, "unit": UNIT, "cores": os.cpu_count() or 1, "cpu_model": cpu_model(), "kind": kind,
                   "sample": desc}
            f_msps, f_desc, _, _, _ = cpu_chain_rate(0.4, os.cpu_count() or 1, full=True)
            cpu["as_written_all_lags"] = {"value": f_msps, "unit": UNIT, "sample": f_desc,
                                          "note": "informational: the reference has no decimating FIR; `value` is the "
                                                  "stronger CPU baseline that skips the 9 of 10 dropped outputs"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(frames, world),
            "run": {"gather": gather_kind, "numa": {"gpu_node": ctx.numa_node, "host_nodes": ctx.numa_nodes,
                                                    "rank_thread_bound_to_cpus": bound_cpus,
                                                    "pinned_buffers": "lrc_host_alloc (preferred node = the GPU's)"}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                         "kernel": "chain_kernel<64,10,10,7> (+ psd_reduce)",
                         "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": alg_bytes},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n_e * 8,
                    "d2h_bytes_per_step": (e2e_frames // K_AVG) * NFFT * 4,
                    "workload": workload_name(e2e_frames) + f" ({e2e_steps} steps through lrc_chain_run_host; a smaller batch than "
                                "the device-resident step: the rate is PCIe-bound and does not depend on it)",
                    "bound": "pcie h2d", "h2d_copy_gbs_per_gpu_all_ranks_copying": h2d_gbs,
                    "frac_of_h2d_copy": (e2e_value / world) * 8e6 / (h2d_gbs * 1e9)},
            "e2e_u8": {"value": e2e_u8_value, "unit": UNIT, "h2d_bytes_per_step": n_e * 2,
                       "d2h_bytes_per_step": (e2e_frames // K_AVG) * NFFT * 4,
                       "frac_of_h2d_copy": (e2e_u8_value / world) * 2e6 / (h2d_gbs * 1e9),
                       "note": "the same chain and step through lrc_chain_run_host_u8: host buffers hold the reference's own wire "
                               "format, rtlsdr u8 I,Q (rtlsdr.rs:160-162); data_to_samples runs on the device"},
            "gpu_launches": 2 * args.steps,
            "clocks": clocks,
        }
        if diag:
            line["scaling_diagnostics"] = diag
        if extra:
            line["extra"] = extra
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
    if gather is not None:
        gather.close()
    for gx in (gather_all, gather_rot, gather_host, gather_p2p):
        if gx is not None and gx is not gather:
            gx.close()
    chain.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES, help="frames per step (default: BASELINE config)")
    ap.add_argument("--e2e-frames", type=int, default=16384, dest="e2e_frames",
                    help="frames per e2e step through host buffers (1.3 GB pinned by default)")
    ap.add_argument("--cpu-seconds", type=float, default=1.5, dest="cpu_seconds",
                    help="per-thread seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true", dest="no_cpu")
    ap.add_argument("--no-extra", action="store_true", dest="no_extra", help="skip the per-config extra block")
    ap.add_argument("--quick-extra", action="store_true", dest="quick_extra", help="extra block at 1/8 size (smoke runs)")
    ap.add_argument("--gather-probe-s", type=float, default=30.0, dest="gather_probe_s",
                    help="N > 1: seconds the lrc_gather connectivity probe may take before falling back to NCCL")
    ap.add_argument("--gather-to", default="host", choices=["host", "root", "all", "rotate"], dest="gather_to",
                    help="N > 1: who receives the output rows: the node's host memory (default: the consumer of PSD rows is a CPU "
                         "block in the reference -- vidsink / psdpng -- and rows pushed into a computing GPU cost its kernel 4.7 %%), "
                         "rank 0's GPU (a gather over NVLink), every rank (all-gather), or a receiver that rotates from step to step")
    ap.add_argument("--gather", default="ce", choices=["ce", "nccl"],
                    help="N > 1: output gather by lrc_gather (copy engines over NVLink, default) or NCCL all-gather")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", dest="dump_outputs",
                    help="write the PSD rows of the last timed step to DIR/psd_rows.npy (f32; the input is seeded, so two "
                         "builds run with the same arguments can be compared row for row)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the rows of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
