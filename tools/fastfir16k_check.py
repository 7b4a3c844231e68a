#!/usr/bin/env python
"""One-process check + timing of the 16384-point overlap-save kernel: windows of the output (incl. block seams and
the flush block) against an f64 direct convolution, then the throughput of the two plans on the same input:
nfft = 0 (kiss_fastfir's output length, computed in 16384-point blocks) and explicit 16384."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from libredio_b200 import blocks  # noqa: E402

ctx = blocks.Context(0)
rng = np.random.default_rng(6)
nh = 4096
h = ((rng.standard_normal(nh) + 1j * rng.standard_normal(nh)) / 64).astype(np.complex64)
hr = h[::-1].astype(np.complex128)
g = torch.Generator(device=ctx.tdev).manual_seed(5)
res = {}
for nfft in (0, 16384):
    ff = blocks.FastFir(ctx, h, nfft)
    worst = 0.0
    for n, flush in ((16384, False), (70_001, True), (1 << 22, False)):
        x = torch.view_as_complex(torch.randn(n, 2, device=ctx.tdev, generator=g))
        y = ff.run(x, flush)
        assert y.numel() == ff.out_len(n, flush), (nfft, n, y.numel(), ff.out_len(n, flush))
        starts = [0, ff.ngood - 8, y.numel() - 64] + [int(v) for v in rng.integers(0, max(1, y.numel() - 64), 6)]
        for s0 in starts:
            if s0 < 0 or s0 + 64 > y.numel():
                continue
            seg = x[s0: s0 + 64 + nh - 1].cpu().numpy().astype(np.complex128)
            ref = np.array([np.dot(seg[k:k + nh], hr) for k in range(64)])
            got = y[s0:s0 + 64].cpu().numpy()
            worst = max(worst, float(np.max(np.abs(got - ref)) / np.sqrt(np.mean(np.abs(ref) ** 2))))
    n = 1 << 27
    x = torch.view_as_complex(torch.randn(n, 2, device=ctx.tdev, generator=g))
    out = torch.empty(ff.out_len(n) + 1, dtype=torch.complex64, device=ctx.tdev)
    for _ in range(2):
        ff.run(x, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        ff.run(x, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    res[str(nfft)] = {"max_err_over_rms": worst, "ms": ms, "Msamples/s": n / (ms * 1e-3) / 1e6}
    ff.close()
    del x, out
print(json.dumps(res), flush=True)
assert all(v["max_err_over_rms"] <= 1e-4 for v in res.values()), res
