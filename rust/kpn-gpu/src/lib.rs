//! GPU blocks with the block signature of LibRedio's `kpn` crate
//! (`pub fn name(u: Receiver<In>, v: Sender<Out>, params…)`, src/kpn/src/kpn.rs:127-131).
//! Each spawns on its own thread exactly like the blocks of src/ratpak.rs:60-185; a closed port or a
//! non-zero status of the GPU library panics the block, which drops its ports and tears the graph down --
//! the reference's own convention (`.unwrap()` everywhere, `panic!(src_strerror(..))` samplerate.rs:77-83).
//!
//! SOURCE ONLY in this repository (no Rust toolchain in the build image); the compiled and tested host
//! layer is the C++ mirror kpn/gpu_blocks.hpp, and tests/test_cpu_abi_host.py keeps the two in step block by
//! block (same names, same argument order).  The crate needs no CUDA bindings of its own: pinned host memory,
//! device memory, streams and asynchronous copies all come from the C ABI (`lrc_host_alloc`, `lrc_dev_alloc`,
//! `lrc_stream_*`, `lrc_event_*`, `lrc_copy_*_async`).
//!
//! | reference block / function                      | here                                   |
//! |-------------------------------------------------|----------------------------------------|
//! | `rtlsdr::data_to_samples` rtlsdr.rs:160-162      | [`data_to_samples`]                    |
//! | `dsputils::convolve` (+ /D) dsputils.rs:30-32    | [`fir_decimate`], [`fir_decimate_multi`] (channel ring) |
//! | `kiss_fastfir` (streaming) kiss_fastfir.c:228-245 | [`fast_fir_multi`] (channel ring)      |
//! | `kissfft::fft` kissfft.rs:18-31                  | [`fft`]                                |
//! | `samplerate::resample` samplerate.rs:59-87       | [`resample`]                           |
//! | (north-star) discriminator                      | [`fm_demod`]                           |
//! | (north-star) FIR -> FFT -> \|X\|^2 chain           | [`chain_psd`]                          |
//! | (north-star) config-3 receiver, N channels      | [`fm_receiver_multi`] (one kernel per batch) |
//! | `trigger` .. `shaper_optional` ratpak.rs:60-111  | [`ook_decode`], [`ook_decode_stream`], [`split_protocols`] |
//! | `kpn::eat` kpn.rs:116-124                        | [`eat`]                                |
use libredio_cuda_sys as sys;
use num_complex::Complex;
use std::ffi::CStr;
use std::os::raw::c_void;
use std::ptr;
use std::sync::mpsc::{Receiver, Sender};

type Cf32 = Complex<f32>;

fn check(rc: i32, what: &str) {
    if rc != sys::LRC_OK {
        let detail = unsafe { CStr::from_ptr(sys::lrc_last_error()) }.to_string_lossy().into_owned();
        panic!("{}: {}", what, detail);
    }
}

/// One context per GPU; share it between the blocks of a graph (every block owns its plans and their state).
pub struct Gpu(pub *mut sys::lrc_ctx);
unsafe impl Send for Gpu {}
unsafe impl Sync for Gpu {}
impl Gpu {
    pub fn new(device: i32) -> Gpu {
        let mut ctx = ptr::null_mut();
        check(unsafe { sys::lrc_ctx_create(device, &mut ctx) }, "lrc_ctx_create");
        Gpu(ctx)
    }
    /// pin the calling block thread to the CPUs of the GPU's NUMA node (no-op on a single-node host)
    pub fn bind_thread(&self) {
        let mut n = 0;
        check(unsafe { sys::lrc_ctx_bind_thread(self.0, &mut n) }, "lrc_ctx_bind_thread");
    }
}
impl Drop for Gpu {
    fn drop(&mut self) { unsafe { sys::lrc_ctx_destroy(self.0); } }
}

/// Pinned host + device buffer pair: one half of a ring slot (kpn/gpu_blocks.hpp `Slot`).
struct Slot { ctx: *mut sys::lrc_ctx, h: *mut c_void, d: *mut c_void, bytes: usize }
impl Slot {
    fn new(g: &Gpu) -> Slot { Slot { ctx: g.0, h: ptr::null_mut(), d: ptr::null_mut(), bytes: 0 } }
    fn reserve(&mut self, n: usize) {
        if n <= self.bytes { return; }
        self.release();
        check(unsafe { sys::lrc_host_alloc(self.ctx, n, &mut self.h) }, "lrc_host_alloc");
        check(unsafe { sys::lrc_dev_alloc(self.ctx, n, &mut self.d) }, "lrc_dev_alloc");
        self.bytes = n;
    }
    fn release(&mut self) {
        unsafe {
            if !self.h.is_null() { sys::lrc_host_free(self.ctx, self.h); }
            if !self.d.is_null() { sys::lrc_dev_free(self.ctx, self.d); }
        }
        self.h = ptr::null_mut(); self.d = ptr::null_mut(); self.bytes = 0;
    }
    fn put<T: Copy>(&mut self, offset_elems: usize, src: &[T]) {
        unsafe { ptr::copy_nonoverlapping(src.as_ptr(), (self.h as *mut T).add(offset_elems), src.len()); }
    }
    fn take<T: Copy + Default>(&self, offset_elems: usize, n: usize) -> Vec<T> {
        let mut out = vec![T::default(); n];
        unsafe { ptr::copy_nonoverlapping((self.h as *const T).add(offset_elems), out.as_mut_ptr(), n); }
        out
    }
    fn h2d(&self, bytes: usize, st: &Stream) {
        check(unsafe { sys::lrc_copy_h2d_async(self.ctx, self.d, self.h, bytes, st.0) }, "lrc_copy_h2d_async");
    }
    fn d2h(&self, bytes: usize, st: &Stream) {
        check(unsafe { sys::lrc_copy_d2h_async(self.ctx, self.h, self.d, bytes, st.0) }, "lrc_copy_d2h_async");
    }
}
impl Drop for Slot { fn drop(&mut self) { self.release(); } }

/// A CUDA stream owned by a block (kpn/gpu_blocks.hpp `Stream`).
struct Stream(*mut c_void, *mut sys::lrc_ctx);
impl Stream {
    fn new(g: &Gpu) -> Stream {
        let mut s = ptr::null_mut();
        check(unsafe { sys::lrc_stream_create(g.0, &mut s) }, "lrc_stream_create");
        Stream(s, g.0)
    }
    fn sync(&self) { check(unsafe { sys::lrc_stream_sync(self.1, self.0) }, "lrc_stream_sync"); }
}
impl Drop for Stream { fn drop(&mut self) { unsafe { sys::lrc_stream_destroy(self.1, self.0); } } }

// plan handles freed when the block dies (a panic unwinds through these)
macro_rules! plan_guard {
    ($name:ident, $ty:ty, $destroy:path) => {
        struct $name(*mut $ty);
        impl Drop for $name { fn drop(&mut self) { unsafe { $destroy(self.0); } } }
    };
}
plan_guard!(FirPlan, sys::lrc_fir, sys::lrc_fir_destroy);
plan_guard!(FirStreamPlan, sys::lrc_fir_stream, sys::lrc_fir_stream_destroy);
plan_guard!(FastFirPlan, sys::lrc_fastfir, sys::lrc_fastfir_destroy);
plan_guard!(FastFirStreamPlan, sys::lrc_fastfir_stream, sys::lrc_fastfir_stream_destroy);
plan_guard!(FftPlan, sys::lrc_fft, sys::lrc_fft_destroy);
plan_guard!(ResamplerPlan, sys::lrc_resampler, sys::lrc_resampler_destroy);
plan_guard!(ChainPlan, sys::lrc_chain, sys::lrc_chain_destroy);
plan_guard!(FmRxPlan, sys::lrc_fmrx, sys::lrc_fmrx_destroy);
plan_guard!(OokPlan, sys::lrc_ook, sys::lrc_ook_destroy);
plan_guard!(OokStreamPlan, sys::lrc_ook_stream, sys::lrc_ook_stream_destroy);

/// Drop-in for `rtlsdr::data_to_samples` as a block (src/rtlsdr/src/rtlsdr.rs:160-162; wired in bitfount.rs:24-28):
/// bytes pairwise to `Complex<f32>`, bit-exact `i2f`.  An odd length panics like the reference's `i[1]`.
pub fn data_to_samples(gpu: &Gpu, u: Receiver<Vec<u8>>, v: Sender<Vec<Cf32>>) {
    let st = Stream::new(gpu);
    let (mut inp, mut out) = (Slot::new(gpu), Slot::new(gpu));
    loop {
        let data = u.recv().unwrap();
        inp.reserve(data.len() + 16); out.reserve(data.len() * 4 + 16);
        inp.put(0, &data);
        inp.h2d(data.len(), &st);
        check(unsafe { sys::lrc_unpack_u8_cf32(gpu.0, inp.d as *const u8, data.len(), out.d as *mut f32, st.0) }, "lrc_unpack_u8_cf32");
        out.d2h(data.len() * 4, &st);
        st.sync();
        v.send(out.take::<Cf32>(0, data.len() / 2)).unwrap();
    }
}

/// Drop-in for `kissfft::fft(pin, cout, block_size, inv)` (src/kissfft/src/kissfft.rs:18-31).
/// Every frame already queued on `pin` (up to 4096) goes to the device in one launch.
pub fn fft(gpu: &Gpu, pin: Receiver<Vec<Cf32>>, cout: Sender<Vec<Cf32>>, block_size: u32, inv: u32) {
    let mut plan = ptr::null_mut();
    check(unsafe { sys::lrc_fft_create(gpu.0, block_size as i32, inv as i32, &mut plan) }, "lrc_fft_create");   // kiss_fft_alloc once, :19
    let plan = FftPlan(plan);
    let st = Stream::new(gpu);
    let mut buf = Slot::new(gpu);
    let n = block_size as usize;
    loop {
        let mut frames = vec![pin.recv().unwrap()];
        while frames.len() < 4096 { match pin.try_recv() { Ok(f) => frames.push(f), Err(_) => break } }
        buf.reserve(frames.len() * n * 8);
        for (k, f) in frames.iter().enumerate() {
            assert!(f.len() == n);                                       // kissfft.rs:24
            buf.put(k * n, f);
        }
        buf.h2d(frames.len() * n * 8, &st);
        check(unsafe { sys::lrc_fft_run(plan.0, buf.d as *const f32, buf.d as *mut f32, frames.len(), st.0) }, "lrc_fft_run");
        buf.d2h(frames.len() * n * 8, &st);
        st.sync();
        for k in 0..frames.len() { cout.send(buf.take::<Cf32>(k * n, n)).unwrap(); }
    }
}

/// `dsputils::convolve` (src/dsputils/src/dsputils.rs:30-32) on the re/im planes followed by decimation, ONE channel,
/// seam-exact across messages: the concatenated outputs equal one call over the concatenated input.
pub fn fir_decimate(gpu: &Gpu, u: Receiver<Vec<Cf32>>, v: Sender<Vec<Cf32>>, taps: &[f32], decim: usize) {
    let max_chunk = 1usize << 20;
    let mut fir = ptr::null_mut();
    check(unsafe { sys::lrc_fir_create(gpu.0, taps.as_ptr(), taps.len() as i32, decim as i32, &mut fir) }, "lrc_fir_create");
    let fir = FirPlan(fir);
    let mut fs = ptr::null_mut();
    check(unsafe { sys::lrc_fir_stream_create(fir.0, 1, max_chunk, 0, &mut fs) }, "lrc_fir_stream_create");
    let fs = FirStreamPlan(fs);
    let st = Stream::new(gpu);
    let (mut inp, mut out) = (Slot::new(gpu), Slot::new(gpu));
    loop {
        let x = u.recv().unwrap();
        assert!(x.len() <= max_chunk, "fir_decimate: chunk longer than max_chunk");
        let cap = (taps.len() + x.len()) / decim + 2;
        inp.reserve(x.len() * 8 + 16); out.reserve(cap * 8);
        inp.put(0, &x);
        inp.h2d(x.len() * 8, &st);
        let mut n_out = 0usize;
        check(unsafe { sys::lrc_fir_stream_push(fs.0, inp.d, x.len(), x.len(), out.d as *mut f32, cap, &mut n_out, st.0) },
              "lrc_fir_stream_push");
        out.d2h(n_out * 8, &st);
        st.sync();
        v.send(out.take::<Cf32>(0, n_out)).unwrap();
    }
}

/// Completion marker of one ring slot's batch (kpn/gpu_blocks.hpp: `cudaEvent_t done`).
struct Event(*mut c_void, *mut sys::lrc_ctx);
impl Event {
    fn new(g: &Gpu) -> Event {
        let mut e = ptr::null_mut();
        check(unsafe { sys::lrc_event_create(g.0, &mut e) }, "lrc_event_create");
        Event(e, g.0)
    }
    fn record(&self, st: &Stream) { check(unsafe { sys::lrc_event_record(self.1, self.0, st.0) }, "lrc_event_record"); }
    fn sync(&self) { check(unsafe { sys::lrc_event_sync(self.1, self.0) }, "lrc_event_sync"); }
}
impl Drop for Event { fn drop(&mut self) { unsafe { sys::lrc_event_destroy(self.1, self.0); } } }

/// One slot of a channel ring: pinned + device input, pinned + device output, the event that marks its batch as out, the
/// count of the batch in flight (kpn/gpu_blocks.hpp `RingSlot`).  All slots of a ring submit on the block's ONE stream, so
/// the launches reach the plan's carried state in order.
struct RingSlot { inp: Slot, out: Slot, done: Event, n_out: usize, busy: bool }

/// FIR + decimate over MANY channels: the channel ring.  One chunk (`chunk_len` samples) is taken from every channel's
/// port, packed channel-major into a pinned slot, and the whole batch goes through ONE kernel launch
/// (`lrc_fir_stream_push`, per-channel carried state on the device).  Two slots alternate: while slot A's batch is on the
/// device the block is already packing slot B from the ports, and A's outputs are scattered to the senders when the block
/// comes back to A.
pub fn fir_decimate_multi(gpu: &Gpu, u: Vec<Receiver<Vec<Cf32>>>, v: Vec<Sender<Vec<Cf32>>>, taps: &[f32], decim: usize, chunk_len: usize) {
    let n_ch = u.len();
    assert!(v.len() == n_ch && n_ch > 0, "fir_decimate_multi: port count mismatch");
    let mut fir = ptr::null_mut();
    check(unsafe { sys::lrc_fir_create(gpu.0, taps.as_ptr(), taps.len() as i32, decim as i32, &mut fir) }, "lrc_fir_create");
    let fir = FirPlan(fir);
    let mut fs = ptr::null_mut();
    check(unsafe { sys::lrc_fir_stream_create(fir.0, n_ch, chunk_len, 0, &mut fs) }, "lrc_fir_stream_create");
    let fs = FirStreamPlan(fs);
    let cap = (taps.len() + chunk_len) / decim + 2;
    let st = Stream::new(gpu);
    let mut ring: Vec<RingSlot> = (0..2).map(|_| RingSlot { inp: Slot::new(gpu), out: Slot::new(gpu), done: Event::new(gpu), n_out: 0, busy: false }).collect();
    for r in ring.iter_mut() { r.inp.reserve(n_ch * chunk_len * 8); r.out.reserve(n_ch * cap * 8); }
    let drain = |r: &mut RingSlot| {
        if !r.busy { return; }
        r.done.sync();
        for c in 0..n_ch { v[c].send(r.out.take::<Cf32>(c * cap, r.n_out)).unwrap(); }
        r.busy = false;
    };
    let mut it = 0usize;
    loop {
        let (a, b) = ring.split_at_mut(1);
        let (r, other) = if it & 1 == 0 { (&mut a[0], &mut b[0]) } else { (&mut b[0], &mut a[0]) };
        drain(r);                                                        // slot reuse: its previous batch must be out
        for c in 0..n_ch {
            let x = u[c].recv().unwrap();
            assert!(x.len() == chunk_len, "fir_decimate_multi: chunk length != chunk_len");
            r.inp.put(c * chunk_len, &x);
        }
        r.inp.h2d(n_ch * chunk_len * 8, &st);
        check(unsafe { sys::lrc_fir_stream_push(fs.0, r.inp.d, chunk_len, chunk_len, r.out.d as *mut f32, cap, &mut r.n_out, st.0) },
              "lrc_fir_stream_push");
        r.out.d2h(n_ch * cap * 8, &st);
        r.done.record(&st);
        r.busy = true;
        drain(other);                                                    // hand out the batch submitted one step ago
        it += 1;
    }
}

/// Long FIR by overlap-save over MANY channels (`kiss_fastfir` with a carried offset, tools/kiss_fastfir.c:228-245): the
/// channel ring of [`fir_decimate_multi`] over `lrc_fastfir_stream_push`, one chunk (`chunk_len` samples) per channel per
/// batch, one push per batch.  Outputs come as whole compute blocks complete (a batch that completes none sends nothing);
/// per channel they are a prefix of `lrc_fastfir_run` over the channel's whole input.  Never flushes: ports never end.
pub fn fast_fir_multi(gpu: &Gpu, u: Vec<Receiver<Vec<Cf32>>>, v: Vec<Sender<Vec<Cf32>>>, h: &[Cf32], nfft: usize, chunk_len: usize) {
    let n_ch = u.len();
    assert!(v.len() == n_ch && n_ch > 0, "fast_fir_multi: port count mismatch");
    let mut ff = ptr::null_mut();
    check(unsafe { sys::lrc_fastfir_create(gpu.0, h.as_ptr() as *const f32, h.len(), nfft, &mut ff) }, "lrc_fastfir_create");
    let ff = FastFirPlan(ff);
    let mut fs = ptr::null_mut();
    check(unsafe { sys::lrc_fastfir_stream_create(ff.0, n_ch, &mut fs) }, "lrc_fastfir_stream_create");
    let fs = FastFirStreamPlan(fs);
    let cap = chunk_len + 16384;                                         // the history is shorter than one compute block
    let st = Stream::new(gpu);
    let mut ring: Vec<RingSlot> = (0..2).map(|_| RingSlot { inp: Slot::new(gpu), out: Slot::new(gpu), done: Event::new(gpu), n_out: 0, busy: false }).collect();
    for r in ring.iter_mut() { r.inp.reserve(n_ch * chunk_len * 8); r.out.reserve(n_ch * cap * 8); }
    let drain = |r: &mut RingSlot| {
        if !r.busy { return; }
        r.done.sync();
        if r.n_out > 0 { for c in 0..n_ch { v[c].send(r.out.take::<Cf32>(c * cap, r.n_out)).unwrap(); } }
        r.busy = false;
    };
    let mut it = 0usize;
    loop {
        let (a, b) = ring.split_at_mut(1);
        let (r, other) = if it & 1 == 0 { (&mut a[0], &mut b[0]) } else { (&mut b[0], &mut a[0]) };
        drain(r);                                                        // slot reuse: its previous batch must be out
        for c in 0..n_ch {
            let x = u[c].recv().unwrap();
            assert!(x.len() == chunk_len, "fast_fir_multi: chunk length != chunk_len");
            r.inp.put(c * chunk_len, &x);
        }
        r.inp.h2d(n_ch * chunk_len * 8, &st);
        check(unsafe { sys::lrc_fastfir_stream_push(fs.0, r.inp.d as *const f32, chunk_len, chunk_len, r.out.d as *mut f32, cap, 0,
                                                    &mut r.n_out, st.0) }, "lrc_fastfir_stream_push");
        r.out.d2h(n_ch * cap * 8, &st);
        r.done.record(&st);
        r.busy = true;
        drain(other);                                                    // hand out the batch submitted one step ago
        it += 1;
    }
}

/// Drop-in for `samplerate::resample(din, dout, ratio)` (src/samplerate/src/samplerate.rs:59-87).
pub fn resample(gpu: &Gpu, din: Receiver<Vec<f32>>, dout: Sender<Vec<f32>>, ratio: f64) {
    let mut rs = ptr::null_mut();
    check(unsafe { sys::lrc_resampler_create(gpu.0, ratio, 1, 1 << 22, &mut rs) }, "lrc_resampler_create");   // src_new(1, 1) :61
    let rs = ResamplerPlan(rs);
    loop {
        let vin = din.recv().unwrap();
        let lout = ((ratio * vin.len() as f64) + 1f64) as usize + 1;      // samplerate.rs:64
        let mut vout = vec![0f32; lout];
        let mut n_out = 0usize;
        // a non-zero status here is the reference's panic!(src_strerror(error)) :77-83
        check(unsafe { sys::lrc_resampler_process_host(rs.0, vin.as_ptr(), vin.len(), vout.as_mut_ptr(), lout, &mut n_out) },
              "lrc_resampler_process_host");
        vout.truncate(n_out);                                             // set_len(output_frames_gen) :84
        dout.send(vout).unwrap();
    }
}

/// Quadrature FM discriminator (north-star stage): `d[n] = arg(x[n] conj(x[n-1]))`, `x[-1]` carried across messages
/// (0 at stream start).
pub fn fm_demod(gpu: &Gpu, u: Receiver<Vec<Cf32>>, v: Sender<Vec<f32>>) {
    let st = Stream::new(gpu);
    let (mut inp, mut out) = (Slot::new(gpu), Slot::new(gpu));
    let mut d_state: *mut c_void = ptr::null_mut();
    check(unsafe { sys::lrc_dev_alloc(gpu.0, 8, &mut d_state) }, "lrc_dev_alloc");
    check(unsafe { sys::lrc_dev_memset(gpu.0, d_state, 0, 8, st.0) }, "lrc_dev_memset");       // x[-1] = 0 at stream start
    struct DevBuf(*mut sys::lrc_ctx, *mut c_void);
    impl Drop for DevBuf { fn drop(&mut self) { unsafe { sys::lrc_dev_free(self.0, self.1); } } }
    let state = DevBuf(gpu.0, d_state);
    loop {
        let x = u.recv().unwrap();
        inp.reserve(x.len() * 8 + 16); out.reserve(x.len() * 4 + 16);
        inp.put(0, &x);
        inp.h2d(x.len() * 8, &st);
        check(unsafe { sys::lrc_fmdemod_run(gpu.0, inp.d as *const f32, 1, x.len(), x.len(), state.1 as *mut f32, out.d as *mut f32, x.len(), st.0) },
              "lrc_fmdemod_run");
        out.d2h(x.len() * 4, &st);
        st.sync();
        v.send(out.take::<f32>(0, x.len())).unwrap();
    }
}

/// The headline chain as one block: cf32 chunks holding whole rows of `k_avg` frames (+ the ntaps-decim tail)
/// in, one `Vec<f32>` of `nfft` averaged |X|^2 values per row out.  The device work goes through the double-buffered host
/// ring of `lrc_chain_run_host`.
pub fn chain_psd(gpu: &Gpu, u: Receiver<Vec<Cf32>>, v: Sender<Vec<f32>>, taps: &[f32], decim: usize, nfft: usize, k_avg: usize) {
    let mut ch = ptr::null_mut();
    check(unsafe { sys::lrc_chain_create(gpu.0, taps.as_ptr(), taps.len() as i32, decim as i32, nfft as i32, sys::LRC_WINDOW_HANN, &mut ch) },
          "lrc_chain_create");
    let ch = ChainPlan(ch);
    loop {
        let x = u.recv().unwrap();
        let rows = unsafe { sys::lrc_chain_frames(ch.0, x.len()) } / k_avg;
        let mut out = vec![0f32; rows * nfft];
        let mut nr = 0usize;
        check(unsafe { sys::lrc_chain_run_host(ch.0, x.as_ptr() as *const f32, x.len(), k_avg, out.as_mut_ptr(), &mut nr) },
              "lrc_chain_run_host");
        for r in 0..nr { v.send(out[r * nfft..(r + 1) * nfft].to_vec()).unwrap(); }
    }
}

/// FM broadcast receiver over MANY channels (BASELINE config 3): rtlsdr u8 IQ chunks in, audio chunks out, through
/// `lrc_fmrx` -- ONE kernel per batch for the BASELINE shape (64 taps / 10, ratio 1/5), stream state of all stages carried
/// on the device.  One chunk (`chunk_bytes`, even) is taken from every channel's port and packed channel-major into a pinned
/// slot; two slots alternate like `fir_decimate_multi`.  The reference would wire rtlsdr::data_to_samples ->
/// dsputils::convolve -> (discriminator) -> samplerate::resample with one thread and one channel message per stage and chunk.
pub fn fm_receiver_multi(gpu: &Gpu, u: Vec<Receiver<Vec<u8>>>, v: Vec<Sender<Vec<f32>>>, taps: &[f32], decim: usize, ratio: f64, chunk_bytes: usize) {
    let n_ch = u.len();
    assert!(v.len() == n_ch && n_ch > 0, "fm_receiver_multi: port count mismatch");
    assert!(chunk_bytes > 0 && chunk_bytes % 2 == 0, "fm_receiver_multi: chunk_bytes must be even");
    let chunk = chunk_bytes / 2;                                          // samples per channel and batch
    let cap_bb = (taps.len() + chunk) / decim + 2;
    let cap_au = (((ratio * cap_bb as f64 + 1.0) as usize) + 1 + 3) / 4 * 4;
    let mut rx = ptr::null_mut();
    check(unsafe { sys::lrc_fmrx_create(gpu.0, taps.as_ptr(), taps.len() as i32, decim as i32, ratio, n_ch, chunk, &mut rx) }, "lrc_fmrx_create");
    let rx = FmRxPlan(rx);
    let st = Stream::new(gpu);
    let mut ring: Vec<RingSlot> = (0..2).map(|_| RingSlot { inp: Slot::new(gpu), out: Slot::new(gpu), done: Event::new(gpu), n_out: 0, busy: false }).collect();
    for r in ring.iter_mut() { r.inp.reserve(n_ch * chunk_bytes); r.out.reserve(n_ch * cap_au * 4); }
    let drain = |r: &mut RingSlot| {
        if !r.busy { return; }
        r.done.sync();
        if r.n_out > 0 { for c in 0..n_ch { v[c].send(r.out.take::<f32>(c * cap_au, r.n_out)).unwrap(); } }
        r.busy = false;
    };
    let mut it = 0usize;
    loop {
        let (a, b) = ring.split_at_mut(1);
        let (r, other) = if it & 1 == 0 { (&mut a[0], &mut b[0]) } else { (&mut b[0], &mut a[0]) };
        drain(r);
        for c in 0..n_ch {
            let x = u[c].recv().unwrap();
            assert!(x.len() == chunk_bytes, "fm_receiver_multi: chunk length != chunk_bytes");
            r.inp.put(c * chunk_bytes, &x);
        }
        r.inp.h2d(n_ch * chunk_bytes, &st);
        check(unsafe { sys::lrc_fmrx_push(rx.0, r.inp.d as *const u8, chunk, chunk, r.out.d as *mut f32, cap_au, &mut r.n_out, st.0) },
              "lrc_fmrx_push");
        if r.n_out > 0 { r.out.d2h(n_ch * cap_au * 4, &st); }
        r.done.record(&st);
        r.busy = true;
        drain(other);
        it += 1;
    }
}

/// One decoded packet of the OOK chain: which stream, which protocol (0 = A, 36 bits; 1 = B, 24 bits), the bits.
pub struct OokPacket { pub stream: u32, pub proto: u32, pub bits: Vec<usize> }

/// The chain of src/ratpak.rs:60-111 (data_to_samples -> |x| -> bitfount::trigger -> discretize -> rle -> dle -> the two
/// matchers -> shaper_optional 36 / 24) over `n_streams` captures at once, bit-exact.  Every message is one batch of
/// `n_streams` captures, stream-major, `n_blocks * 1024` bytes each (the bytes `rtl_source_cmplx` would have delivered 1024
/// at a time, bitfount.rs:16-34).  Packets come out ordered by (stream, proto, sequence).
pub fn ook_decode(gpu: &Gpu, u: Receiver<Vec<u8>>, v: Sender<OokPacket>, n_streams: usize, n_blocks: usize, s_rate: u32) {
    let (max_runs, max_packets) = (1usize << 16, 256usize);
    let mut ook = ptr::null_mut();
    check(unsafe { sys::lrc_ook_create(gpu.0, n_streams, n_blocks, s_rate, max_runs, max_packets, &mut ook) }, "lrc_ook_create");
    let ook = OokPlan(ook);
    let st = Stream::new(gpu);
    let mut inp = Slot::new(gpu);
    let bytes = n_streams * n_blocks * 1024;
    let mut pk = vec![sys::lrc_ook_packet { stream: 0, proto: 0, seq: 0, nbits: 0, bits: [0u8; 40] }; n_streams * 2 * max_packets];
    loop {
        let cap = u.recv().unwrap();
        assert!(cap.len() == bytes, "ook_decode: batch size != n_streams*n_blocks*1024");
        inp.reserve(bytes);
        inp.put(0, &cap);
        inp.h2d(bytes, &st);
        check(unsafe { sys::lrc_ook_decode(ook.0, inp.d as *const u8, n_blocks * 1024, st.0) }, "lrc_ook_decode");
        let mut n = 0usize;
        check(unsafe { sys::lrc_ook_fetch_packets(ook.0, pk.as_mut_ptr(), pk.len(), &mut n) }, "lrc_ook_fetch_packets");
        for p in &pk[..n] {
            let bits = p.bits[..p.nbits as usize].iter().map(|&b| b as usize).collect();
            v.send(OokPacket { stream: p.stream, proto: p.proto, bits }).unwrap();
        }
    }
}

/// The streaming form of [`ook_decode`], for a live receiver: every message holds the NEXT `k` blocks of each of the
/// `n_streams` streams, stream-major (`n_streams * k * 1024` bytes), `k` free to change from message to message.  The state
/// of the reference's `trigger` .. `shaper_optional` blocks stays on the device between messages, so the packets sent after
/// a message are exactly those the reference sends on all the bytes so far.  The carry is the exact one (the trigger's OOM
/// guard + 1 blocks per stream).
pub fn ook_decode_stream(gpu: &Gpu, u: Receiver<Vec<u8>>, v: Sender<OokPacket>, n_streams: usize, s_rate: u32) {
    let (max_push, max_carry, max_runs, max_packets) = (1024usize, 0usize, 1usize << 16, 256usize);
    let mut ook = ptr::null_mut();
    check(unsafe { sys::lrc_ook_stream_create(gpu.0, n_streams, max_push, s_rate, max_carry, max_runs, max_packets, &mut ook) },
          "lrc_ook_stream_create");
    let ook = OokStreamPlan(ook);
    let st = Stream::new(gpu);
    let mut inp = Slot::new(gpu);
    let mut pk = vec![sys::lrc_ook_packet { stream: 0, proto: 0, seq: 0, nbits: 0, bits: [0u8; 40] }; n_streams * 2 * max_packets];
    loop {
        let msg = u.recv().unwrap();
        assert!(!msg.is_empty() && msg.len() % (n_streams * 1024) == 0, "ook_decode_stream: message is not n_streams * k * 1024 bytes");
        let k = msg.len() / (n_streams * 1024);
        inp.reserve(msg.len());
        inp.put(0, &msg);
        inp.h2d(msg.len(), &st);
        let mut b = 0usize;
        while b < k {
            let n = max_push.min(k - b);
            check(unsafe { sys::lrc_ook_stream_push(ook.0, (inp.d as *const u8).add(b * 1024), n, k * 1024, st.0) },
                  "lrc_ook_stream_push");
            let mut np = 0usize;
            check(unsafe { sys::lrc_ook_stream_fetch_packets(ook.0, pk.as_mut_ptr(), pk.len(), &mut np) },
                  "lrc_ook_stream_fetch_packets");
            for p in &pk[..np] {
                let bits = p.bits[..p.nbits as usize].iter().map(|&b| b as usize).collect();
                v.send(OokPacket { stream: p.stream, proto: p.proto, bits }).unwrap();
            }
            b += n;
        }
    }
}

/// The packets of [`ook_decode`] back onto the reference's two ports: what `shaper_optional(36)` and `shaper_optional(24)`
/// send towards `binconv` (ratpak.rs:105-119).
pub fn split_protocols(u: Receiver<OokPacket>, a: Sender<Vec<usize>>, b: Sender<Vec<usize>>) {
    loop {
        let p = u.recv().unwrap();
        if p.proto == 0 { a.send(p.bits).unwrap(); } else { b.send(p.bits).unwrap(); }
    }
}

/// `kpn::eat` (src/kpn/src/kpn.rs:116-124) served by the library's host helper.
pub fn eat(x: &[usize], is: &[usize]) -> Vec<usize> {
    let bits: Vec<u8> = x.iter().map(|&b| b as u8).collect();
    let mut out = vec![0usize; is.len()];
    check(unsafe { sys::lrc_eat(bits.as_ptr(), bits.len(), is.as_ptr(), is.len(), out.as_mut_ptr()) }, "lrc_eat");
    out
}
