"""CPU suite, part 2: the C-ABI library loads and exports every symbol include/*.h declares, fails loudly
without a GPU, and the host-side sharding logic works at world_size 2 (gloo)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "libredio_cuda.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(lrc_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from libredio_b200 import capi
    lib = capi.load()                                  # raises if the .so is missing or a symbol is absent
    syms = header_symbols()
    assert len(syms) >= 45
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/libredio_cuda.h but not exported"
    assert sorted(capi.SIGNATURES) == syms, "capi.SIGNATURES out of sync with the header"
    assert lib.lrc_version() == 100


def test_rust_sys_crate_declares_every_header_symbol():
    """rust/libredio-cuda-sys is shipped as source only (no rustc in this image): keep its extern block in step with the
    header so the reference-side binding a maintainer would build (INTEGRATION.md) is complete."""
    txt = open(os.path.join(ROOT, "rust", "libredio-cuda-sys", "src", "lib.rs")).read()
    declared = set(re.findall(r"\bpub fn (lrc_[a-z0-9_]+)\s*\(", txt))
    missing = [s for s in header_symbols() if s not in declared]
    assert not missing, f"missing from the Rust -sys crate: {missing}"
    stale = sorted(declared - set(header_symbols()))
    assert not stale, f"declared in Rust but not in the header: {stale}"


def test_status_strings_and_host_helper():
    from libredio_b200 import capi
    lib = capi.load()
    for code in range(8):
        assert lib.lrc_strerror(code)
    assert b"no CPU fallback" in lib.lrc_strerror(capi.ERR_CUDA)
    # kpn::eat is pure host code in the library
    bits = np.array([1, 0, 1, 1, 1, 1], np.uint8)
    w = np.array([3, 3], np.uint64)
    out = np.zeros(2, np.uint64)
    assert lib.lrc_eat(C.c_void_p(bits.ctypes.data), 6, C.c_void_p(w.ctypes.data), 2, C.c_void_p(out.ctypes.data)) == 0
    assert out.tolist() == [5, 7]


def test_no_gpu_means_loud_failure_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("this box has a GPU")
    from libredio_b200 import capi, blocks
    lib = capi.load()
    h = C.c_void_p()
    assert lib.lrc_ctx_create(0, C.byref(h)) == capi.ERR_CUDA
    assert lib.lrc_last_error()
    with pytest.raises(RuntimeError):
        blocks.Context(0)


def test_product_package_never_imports_the_oracle():
    """only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/"""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "libredio_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "liboracle" not in txt, f
    for d in ("kpn", "rust", "include"):
        p = os.path.join(ROOT, d)
        if os.path.isdir(p):
            for dirpath, _, files in os.walk(p):
                for f in files:
                    txt = open(os.path.join(dirpath, f), errors="ignore").read()
                    assert "liboracle" not in txt and "restated.h" not in txt, f


def test_library_reads_only_the_documented_environment_switches():
    """Every stage compiles one kernel per shape; an environment variable may size a grid, select the reference a test
    compares against, or be a test hook, but not pick a second kernel form.  The list is DESIGN.md's "Tuning knobs"."""
    documented = {
        # grid multipliers
        "LRC_UNPACK_CAP", "LRC_FM_CAP", "LRC_FIR_GRID", "LRC_FIRU8_GRID", "LRC_FFT_GRID", "LRC_PSD_GRID", "LRC_RS_GRID",
        "LRC_CHAIN_GRID",
        # reference switches that tests compare against
        "LRC_RS_VARIANT", "LRC_CHAIN_NO_GENERIC", "LRC_CHAIN_GENERIC_ALL", "LRC_FIR_NO_GENTILE",
        # test hook
        "LRC_OOK_TEST_GUARD_BLOCKS",
        # device of the kissfft / libsamplerate ABI shims
        "LIBREDIO_DEVICE",
    }
    csrc = os.path.join(ROOT, "libredio_b200", "csrc")
    found = set()
    for f in os.listdir(csrc):
        found |= set(re.findall(r'"((?:LRC|LIBREDIO)_[A-Z0-9_]+)"', open(os.path.join(csrc, f)).read()))
    assert found == documented, f"undocumented: {sorted(found - documented)}, no longer read: {sorted(documented - found)}"


def test_split_units_covers_everything():
    from libredio_b200 import shard
    for n in (0, 1, 7, 8, 4096, 4099):
        for world in (1, 2, 3, 8):
            spans = [shard.split_units(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_chain_and_fastfir_shards_tile_the_stream():
    from libredio_b200 import shard
    n_in = 64 * 10240 + 54 + 5
    for world in (1, 2, 4, 8):
        sh = [shard.chain_shard(n_in, 64, 10, 1024, 8, r, world) for r in range(world)]
        assert sh[0].row_lo == 0 and sh[-1].row_hi == 8
        for a in sh:
            assert a.in_start == a.row_lo * 8 * 10240
            assert a.in_start + a.in_len <= n_in
    n_in, nh, nfft = 1 << 20, 4096, 8192
    for world in (1, 2, 4, 8):
        sh = [shard.fastfir_shard(n_in, nh, nfft, r, world) for r in range(world)]
        assert sh[0].out_start == 0
        assert sum(s.out_len for s in sh) == ((n_in - nfft) // 4097 + 1) * 4097
        for a, b in zip(sh, sh[1:]):
            assert a.out_start + a.out_len == b.out_start
            assert b.in_start == b.block_lo * 4097                      # own halo, no exchange
        assert all(s.in_start + s.in_len <= n_in for s in sh)


_WORKER = r'''
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
import oracle
from oracle import defined_f64 as D
from libredio_b200 import shard, synth
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
taps = synth.lpf_taps(64, 0.04)
frames, k = 16, 4
x = synth.cf32_noise_tones(frames * 10240 + 54, seed=2)
whole = D.psd_rows(oracle.fir_decimate(x, taps, 10), 1024, k, D.hann_periodic(1024))
sh = shard.chain_shard(x.size, 64, 10, 1024, k, rank, world)
mine = x[sh.in_start: sh.in_start + sh.in_len]                 # own halo, nothing exchanged
loc = D.psd_rows(oracle.fir_decimate(mine, taps, 10), 1024, k, D.hann_periodic(1024))
assert loc.shape[0] == sh.row_hi - sh.row_lo
rows_max = -(-(frames // k) // world)
g = shard.gather_rows(shard.pad_rows(torch.from_numpy(loc), rows_max), world).numpy()
got = np.concatenate([g[r * rows_max: r * rows_max + (shard.split_units(frames // k, r, world)[1] - shard.split_units(frames // k, r, world)[0])] for r in range(world)])
assert got.shape == whole.shape and np.allclose(got, whole, rtol=1e-12, atol=0), "sharded rows differ"
# config 5: overlap-save blocks sharded, outputs concatenate to the unsharded result bit for bit
rng = np.random.default_rng(5)
h = (rng.standard_normal(100) + 1j * rng.standard_normal(100)).astype(np.complex64)
sig = (rng.standard_normal(20000) + 1j * rng.standard_normal(20000)).astype(np.complex64)
full = oracle.fastfir(h, sig, 1024, False)
fs = shard.fastfir_shard(sig.size, 100, 1024, rank, world)
part = oracle.fastfir(h, sig[fs.in_start: fs.in_start + fs.in_len], 1024, False)
assert part.size == fs.out_len and np.array_equal(part.view(np.uint32), full[fs.out_start: fs.out_start + fs.out_len].view(np.uint32))
t = torch.tensor([float(part.size)]); dist.all_reduce(t)
assert int(t.item()) == full.size
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_world_size_2_gloo_sharded_chain_and_gather(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29617", WORLD_SIZE="2", OMP_NUM_THREADS="1")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o}"
        assert f"rank {r} ok" in o


def test_rust_kpn_gpu_mirrors_every_cpp_gpu_block_name_and_argument_order():
    """north_star: 'Host code stays in Rust'.  rust/kpn-gpu cannot be compiled here (no rustc), so it is kept in step with
    the compiled and GPU-tested C++ mirror kpn/gpu_blocks.hpp by text: every block of namespace kpn_gpu has a `pub fn` of the
    same name whose parameters are the same, in the same order (ports first, then parameters: kpn.rs:127-131); C++ parameters
    that have a default value are tuning knobs the Rust side fixes."""
    hpp = open(os.path.join(ROOT, "kpn", "gpu_blocks.hpp")).read()
    rs = open(os.path.join(ROOT, "rust", "kpn-gpu", "src", "lib.rs")).read()
    hpp = re.sub(r"//[^\n]*", "", hpp)
    cpp = {}
    for m in re.finditer(r"inline\s+void\s+(\w+)\s*\(([^)]*)\)", hpp):
        name, params = m.group(1), m.group(2)
        names = []
        depth, cur = 0, ""
        for ch in params + ",":                                  # split on top-level commas (templates contain commas)
            if ch in "<(":
                depth += 1
            elif ch in ">)":
                depth -= 1
            if ch == "," and depth == 0:
                if cur.strip():
                    names.append(cur.strip())
                cur = ""
            else:
                cur += ch
        keep = [re.sub(r"\s*=.*", "", p).split()[-1].lstrip("&*") for p in names if "=" not in p]
        cpp[name] = keep
    blocks = {k: v for k, v in cpp.items() if k not in ("check", "cuda_check")}
    assert {"data_to_samples", "fft", "fir_decimate", "fir_decimate_multi", "fm_demod", "resample", "fm_receiver_multi",
            "chain_psd", "ook_decode", "split_protocols"} <= set(blocks)
    rust = {m.group(1): [p.split(":")[0].strip() for p in m.group(2).split(",") if p.strip()]
            for m in re.finditer(r"pub fn (\w+)\s*\(([^)]*)\)", rs)}
    alias = {"g": "gpu"}
    for name, params in blocks.items():
        assert name in rust, f"kpn_gpu::{name} has no Rust counterpart in rust/kpn-gpu/src/lib.rs"
        want = [alias.get(p, p) for p in params]
        assert rust[name] == want, f"{name}: Rust parameters {rust[name]} != C++ {want}"
    # and it binds only symbols the -sys crate declares
    sys_txt = open(os.path.join(ROOT, "rust", "libredio-cuda-sys", "src", "lib.rs")).read()
    declared = set(re.findall(r"\bpub fn (lrc_[a-z0-9_]+)\s*\(", sys_txt))
    used = set(re.findall(r"sys::(lrc_[a-z0-9_]+)\s*\(", rs)) | set(re.findall(r", sys::(lrc_[a-z0-9_]+_destroy)\)", rs))
    assert used and used <= declared, sorted(used - declared)
