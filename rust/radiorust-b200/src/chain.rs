//! Safe wrapper of `rr_chain`: a list of stages (one per reference block) that runs `n_streams` independent
//! streams in lock step on one B200.  The block types in [`crate::blocks`] are Tokio task loops around one of these.
use crate::pool::{PinnedChunk, PinnedChunkBuf};
use crate::{check, sys, Context, Error, GpuFloat};

use num::Complex;

use std::ffi::CStr;
use std::marker::PhantomData;
use std::os::raw::c_void;

/// Frequency response closure of `Filter` (src/blocks/filters.rs:128-131): evaluated on the host at (re)design time
pub type FreqResp = Box<dyn Fn(isize, f64) -> Complex<f64> + Send + Sync>;

/// Window function of `Filter` / `Fourier` (src/windowing.rs)
pub enum Window {
    /// `Kaiser::with_beta(beta)` (windowing.rs:24-51); `Filter::new` uses `Kaiser::with_null_at_bin(2.0)` = beta sqrt(3)
    Kaiser(f64),
    /// `Rectangular` (windowing.rs:14-20)
    Rectangular,
    /// any `radiorust::windowing::Window` (its `relative_value_at` is called on the host at design time)
    Custom(Box<dyn radiorust::windowing::Window + Send + Sync>),
}

impl Window {
    /// `Kaiser::with_null_at_bin(n)`: beta = sqrt(n^2 - 1) (math.rs:37-39)
    pub fn kaiser_with_null_at_bin(n: f64) -> Self {
        Window::Kaiser(unsafe { sys::rr_kaiser_null_at_bin_to_beta(n) })
    }
}

/// One stage = one reference block with its constructor arguments
pub enum Stage {
    /// `FreqShifter::with_precision_and_shift` (transform.rs:297)
    FreqShifter { precision: f64, shift: f64 },
    /// `Filter::with_window` (filters.rs:145-152)
    Filter { freq_resp: FreqResp, window: Window },
    /// `Downsampler::with_quality` (resampling.rs:45-50)
    Downsampler { output_chunk_len: usize, output_rate: f64, bandwidth: f64, quality: f64 },
    /// `Upsampler::with_quality` (resampling.rs:180-185)
    Upsampler { output_chunk_len: usize, output_rate: f64, bandwidth: f64, quality: f64 },
    /// `FmDemod::new` (modulation.rs:97)
    FmDemod { deviation: f64 },
    /// `FmMod::new` (modulation.rs:27)
    FmMod { deviation: f64 },
    /// `GainControl::new` (transform.rs:43)
    GainControl { gain: f64 },
    /// `Fourier::with_window` / `with_window_center_dc` (analysis.rs:38-59)
    Fourier { window: Window, center_dc: bool },
    /// `Rechunker::new` (chunks.rs:57)
    Rechunker { output_chunk_len: usize },
    /// `Overlapper::new` (chunks.rs:194)
    Overlapper { chunk_count: usize },
}

unsafe extern "C" fn freq_resp_trampoline(user: *mut c_void, bin: i64, freq_hz: f64, out_re: *mut f64, out_im: *mut f64) {
    let f = &*(user as *const FreqResp);
    let v = f(bin as isize, freq_hz);
    *out_re = v.re;
    *out_im = v.im;
}
unsafe extern "C" fn window_trampoline(user: *mut c_void, x: f64) -> f64 {
    let w = &*(user as *const Box<dyn radiorust::windowing::Window + Send + Sync>);
    w.relative_value_at(x)
}

/// Host closures a chain's stages point to; they must outlive the `rr_chain`
enum Callback {
    Resp(Box<FreqResp>),
    Win(Box<Box<dyn radiorust::windowing::Window + Send + Sync>>),
}

fn window_fields(window: Window, keep: &mut Vec<Callback>) -> (i32, f64, sys::rr_window_fn, *mut c_void) {
    match window {
        Window::Kaiser(beta) => (sys::RR_WINDOW_KAISER, beta, None, std::ptr::null_mut()),
        Window::Rectangular => (sys::RR_WINDOW_RECTANGULAR, 0.0, None, std::ptr::null_mut()),
        Window::Custom(w) => {
            let boxed = Box::new(w);
            let user = &*boxed as *const Box<dyn radiorust::windowing::Window + Send + Sync> as *mut c_void;
            keep.push(Callback::Win(boxed));
            (sys::RR_WINDOW_CUSTOM, 0.0, Some(window_trampoline), user)
        }
    }
}

fn resp_fields(f: FreqResp, keep: &mut Vec<Callback>) -> (sys::rr_freq_resp_fn, *mut c_void) {
    let boxed = Box::new(f);
    let user = &*boxed as *const FreqResp as *mut c_void;
    keep.push(Callback::Resp(boxed));
    (Some(freq_resp_trampoline), user)
}

/// What one push produced
#[derive(Clone, Copy, Debug, PartialEq)]
pub struct Pushed {
    /// samples per stream written to the output buffer
    pub count: usize,
    /// their sample rate
    pub sample_rate: f64,
}

/// `rr_chain`.  `Send` but not `Sync`: one task owns a chain (every entry point selects the CUDA device itself, so
/// the owning Tokio task may migrate between worker threads).
pub struct Chain<Flt: GpuFloat> {
    raw: *mut sys::rr_chain,
    ctx: Context,
    n_streams: usize,
    callbacks: Vec<Callback>,
    _flt: PhantomData<Flt>,
}
unsafe impl<Flt: GpuFloat> Send for Chain<Flt> {}

impl<Flt: GpuFloat> Drop for Chain<Flt> {
    fn drop(&mut self) {
        unsafe {
            sys::rr_chain_destroy(self.raw); // waits for the chain's streams
        }
        // `callbacks` drop after this body: the library no longer calls them
    }
}

impl<Flt: GpuFloat> Chain<Flt> {
    /// Build a chain of `stages` for `n_streams` streams.  Argument errors that make the reference constructors
    /// panic (resampling.rs:51-56) come back as `RR_ERR_INVALID`.
    pub fn new(ctx: &Context, stages: Vec<Stage>, n_streams: usize) -> Result<Self, Error> {
        let mut callbacks = Vec::new();
        let mut descs: Vec<sys::rr_stage_desc> = Vec::with_capacity(stages.len());
        for st in stages {
            let mut d: sys::rr_stage_desc = unsafe { std::mem::zeroed() };
            match st {
                Stage::FreqShifter { precision, shift } => {
                    d.kind = sys::RR_STAGE_FREQSHIFT;
                    d.precision = precision;
                    d.shift = shift;
                }
                Stage::Filter { freq_resp, window } => {
                    d.kind = sys::RR_STAGE_FILTER;
                    let (f, fu) = resp_fields(freq_resp, &mut callbacks);
                    d.freq_resp = f;
                    d.freq_resp_user = fu;
                    let (k, beta, w, wu) = window_fields(window, &mut callbacks);
                    d.window_kind = k;
                    d.window_beta = beta;
                    d.window_fn = w;
                    d.window_user = wu;
                }
                Stage::Downsampler { output_chunk_len, output_rate, bandwidth, quality } => {
                    d.kind = sys::RR_STAGE_DOWNSAMPLE;
                    d.output_chunk_len = output_chunk_len as u64;
                    d.output_rate = output_rate;
                    d.bandwidth = bandwidth;
                    d.quality = quality;
                }
                Stage::Upsampler { output_chunk_len, output_rate, bandwidth, quality } => {
                    d.kind = sys::RR_STAGE_UPSAMPLE;
                    d.output_chunk_len = output_chunk_len as u64;
                    d.output_rate = output_rate;
                    d.bandwidth = bandwidth;
                    d.quality = quality;
                }
                Stage::FmDemod { deviation } => {
                    d.kind = sys::RR_STAGE_FMDEMOD;
                    d.deviation = deviation;
                }
                Stage::FmMod { deviation } => {
                    d.kind = sys::RR_STAGE_FMMOD;
                    d.deviation = deviation;
                }
                Stage::GainControl { gain } => {
                    d.kind = sys::RR_STAGE_GAIN;
                    d.gain = gain;
                }
                Stage::Fourier { window, center_dc } => {
                    d.kind = sys::RR_STAGE_FOURIER;
                    let (k, beta, w, wu) = window_fields(window, &mut callbacks);
                    d.window_kind = k;
                    d.window_beta = beta;
                    d.window_fn = w;
                    d.window_user = wu;
                    d.center_dc = center_dc as i32;
                }
                Stage::Rechunker { output_chunk_len } => {
                    d.kind = sys::RR_STAGE_RECHUNK;
                    d.output_chunk_len = output_chunk_len as u64;
                }
                Stage::Overlapper { chunk_count } => {
                    d.kind = sys::RR_STAGE_OVERLAP;
                    d.chunk_count = chunk_count as i32;
                }
            }
            descs.push(d);
        }
        Self::create(ctx, descs, callbacks, n_streams)
    }

    fn create(ctx: &Context, descs: Vec<sys::rr_stage_desc>, callbacks: Vec<Callback>, n_streams: usize) -> Result<Self, Error> {
        let desc = sys::rr_chain_desc {
            dtype: Flt::DTYPE,
            n_streams: n_streams as i32,
            n_stages: descs.len() as i32,
            reserved: 0,
            stages: descs.as_ptr(),
        };
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::rr_chain_create(ctx.raw(), &desc, &mut raw) })?;
        Ok(Chain { raw, ctx: ctx.clone(), n_streams, callbacks, _flt: PhantomData })
    }

    /// Streams processed per push
    pub fn n_streams(&self) -> usize {
        self.n_streams
    }
    /// The device context
    pub fn context(&self) -> &Context {
        &self.ctx
    }

    // ---- live parameters (tokio watch channels in the reference) ----------------------------------------------
    /// `FreqShifter::set_shift` (transform.rs:384-386) for one stream, or for all with `stream = None`
    pub fn set_shift(&mut self, stage: usize, stream: Option<usize>, shift_hz: f64) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_set_shift(self.raw, stage as i32, stream.map_or(-1, |s| s as i32), shift_hz) })
    }
    /// One shift per stream (a channelizer's tuning table)
    pub fn set_shifts(&mut self, stage: usize, shifts_hz: &[f64]) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_set_shifts(self.raw, stage as i32, shifts_hz.as_ptr(), shifts_hz.len() as i32) })
    }
    /// `FreqShifter::shift` (transform.rs:380-382)
    pub fn shift(&self, stage: usize, stream: usize) -> Result<f64, Error> {
        let mut v = 0.0;
        check(unsafe { sys::rr_chain_get_shift(self.raw, stage as i32, stream as i32, &mut v) })?;
        Ok(v)
    }
    /// `Filter::update` (window `None`, filters.rs:279-286) / `Filter::update_with_window` (filters.rs:288-297)
    pub fn update_filter(&mut self, stage: usize, freq_resp: FreqResp, window: Option<Window>) -> Result<(), Error> {
        let (f, fu) = resp_fields(freq_resp, &mut self.callbacks);
        match window {
            None => check(unsafe { sys::rr_chain_update_filter(self.raw, stage as i32, f, fu, 0, 0.0, None, std::ptr::null_mut(), 1) }),
            Some(w) => {
                let (k, beta, wf, wu) = window_fields(w, &mut self.callbacks);
                check(unsafe { sys::rr_chain_update_filter(self.raw, stage as i32, f, fu, k, beta, wf, wu, 0) })
            }
        }
        // (replaced closures stay alive until the chain is dropped: a few boxes per retune)
    }
    /// `FmDemod::set_deviation` (modulation.rs:154-157) / `FmMod::set_deviation` (modulation.rs:76-79)
    pub fn set_deviation(&mut self, stage: usize, deviation: f64) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_set_deviation(self.raw, stage as i32, deviation) })
    }
    /// `GainControl::set` (transform.rs:89-91)
    pub fn set_gain(&mut self, stage: usize, gain: f64) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_set_gain(self.raw, stage as i32, gain) })
    }
    /// `Rechunker::set_output_chunk_len` (chunks.rs:171-175)
    pub fn set_output_chunk_len(&mut self, stage: usize, output_chunk_len: usize) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_set_output_chunk_len(self.raw, stage as i32, output_chunk_len) })
    }

    /// One in-band `Signal::Event`.  Returns how many `SamplesLost` events the chain's Rechunker / Overlapper stages
    /// generated because of it (chunks.rs:84-91, 226-233): the block task sends that many downstream first.
    pub fn event(&mut self, is_interrupt: bool) -> Result<u64, Error> {
        let before = unsafe { sys::rr_chain_samples_lost_count(self.raw) };
        check(unsafe { sys::rr_chain_event(self.raw, is_interrupt as i32) })?;
        Ok(unsafe { sys::rr_chain_samples_lost_count(self.raw) } - before)
    }
    /// Total `SamplesLost` events generated so far
    pub fn samples_lost_count(&self) -> u64 {
        unsafe { sys::rr_chain_samples_lost_count(self.raw) }
    }

    // ---- data path ---------------------------------------------------------------------------------------------
    /// Upper bound of output samples per stream for a push of `n_chunks` chunks of `chunk_len` samples
    pub fn max_output(&self, sample_rate: f64, chunk_len: usize, n_chunks: usize) -> usize {
        unsafe { sys::rr_chain_max_output(self.raw, sample_rate, chunk_len, n_chunks) }
    }

    /// `n_chunks` `Signal::Samples` messages per stream from host memory; `input` holds stream `s` at
    /// `s * in_stride`, `output` receives stream `s` at `s * out_stride`.  Asynchronous when both are pinned: call
    /// [`Chain::sync`] before reading `output` or modifying `input`.
    pub fn push(
        &mut self,
        sample_rate: f64,
        chunk_len: usize,
        n_chunks: usize,
        input: &[Complex<Flt>],
        in_stride: usize,
        output: &mut [Complex<Flt>],
        out_stride: usize,
    ) -> Result<Pushed, Error> {
        assert!(input.len() >= (self.n_streams - 1) * in_stride + chunk_len * n_chunks, "input slice too short");
        let out_capacity = if self.n_streams > 1 { out_stride.min(output.len() - (self.n_streams - 1) * out_stride) } else { output.len() };
        let (mut count, mut rate) = (0usize, 0f64);
        check(unsafe {
            sys::rr_chain_push(
                self.raw, sample_rate, chunk_len, n_chunks, input.as_ptr() as *const c_void, in_stride,
                output.as_mut_ptr() as *mut c_void, out_capacity, out_stride, &mut count, &mut rate,
            )
        })?;
        Ok(Pushed { count, sample_rate: rate })
    }

    /// One chunk of one stream straight from / into pinned pool buffers (no staging copy on the host); waits for the
    /// result and sets `output`'s length.
    pub fn push_pinned(&mut self, sample_rate: f64, input: &PinnedChunk<Complex<Flt>>, output: &mut PinnedChunkBuf<Complex<Flt>>) -> Result<Pushed, Error> {
        assert_eq!(self.n_streams, 1, "push_pinned is the single-stream form");
        let cap = output.capacity();
        let (mut count, mut rate) = (0usize, 0f64);
        check(unsafe {
            sys::rr_chain_push(
                self.raw, sample_rate, input.len(), 1, input.as_ptr() as *const c_void, input.len(),
                output.as_mut_ptr() as *mut c_void, cap, cap, &mut count, &mut rate,
            )
        })?;
        self.sync()?;
        unsafe { output.set_len(count) };
        Ok(Pushed { count, sample_rate: rate })
    }

    /// The same with device pointers (no PCIe traffic): lets two chains hand device buffers to each other
    ///
    /// # Safety
    /// `dev_in` / `dev_out` must be device allocations of the chain's device holding `n_streams` rows of
    /// `in_stride` / `out_stride` complex samples.
    pub unsafe fn push_device(
        &mut self,
        sample_rate: f64,
        chunk_len: usize,
        n_chunks: usize,
        dev_in: *const c_void,
        in_stride: usize,
        dev_out: *mut c_void,
        out_capacity: usize,
        out_stride: usize,
    ) -> Result<Pushed, Error> {
        let (mut count, mut rate) = (0usize, 0f64);
        check(sys::rr_chain_push_device(self.raw, sample_rate, chunk_len, n_chunks, dev_in, in_stride, dev_out, out_capacity, out_stride, &mut count, &mut rate))?;
        Ok(Pushed { count, sample_rate: rate })
    }

    /// A channelizer's push: every stream reads the same `chunk_len * n_chunks` samples of `input` (one wideband
    /// row, copied to the device once), each with its own shift and state; `output` receives stream `s` at
    /// `s * out_stride`.  Asynchronous when both are pinned: call [`Chain::sync`] before reading `output` or
    /// modifying `input`.
    pub fn push_shared(
        &mut self,
        sample_rate: f64,
        chunk_len: usize,
        n_chunks: usize,
        input: &[Complex<Flt>],
        output: &mut [Complex<Flt>],
        out_stride: usize,
    ) -> Result<Pushed, Error> {
        assert!(input.len() >= chunk_len * n_chunks, "input slice too short");
        let out_capacity = if self.n_streams > 1 { out_stride.min(output.len() - (self.n_streams - 1) * out_stride) } else { output.len() };
        let (mut count, mut rate) = (0usize, 0f64);
        check(unsafe {
            sys::rr_chain_push_shared(
                self.raw, sample_rate, chunk_len, n_chunks, input.as_ptr() as *const c_void, output.as_mut_ptr() as *mut c_void,
                out_capacity, out_stride, &mut count, &mut rate,
            )
        })?;
        Ok(Pushed { count, sample_rate: rate })
    }

    /// The same with device pointers: every stream reads the row at `dev_in` in place
    ///
    /// # Safety
    /// `dev_in` must be a device allocation of the chain's device holding `chunk_len * n_chunks` complex samples,
    /// `dev_out` one holding `n_streams` rows of `out_stride` complex samples.
    pub unsafe fn push_shared_device(
        &mut self,
        sample_rate: f64,
        chunk_len: usize,
        n_chunks: usize,
        dev_in: *const c_void,
        dev_out: *mut c_void,
        out_capacity: usize,
        out_stride: usize,
    ) -> Result<Pushed, Error> {
        let (mut count, mut rate) = (0usize, 0f64);
        check(sys::rr_chain_push_shared_device(self.raw, sample_rate, chunk_len, n_chunks, dev_in, dev_out, out_capacity, out_stride, &mut count, &mut rate))?;
        Ok(Pushed { count, sample_rate: rate })
    }

    /// Wait for everything enqueued by earlier pushes
    pub fn sync(&mut self) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_sync(self.raw) })
    }
    /// Force the stateful overlap-save path (`false`) or allow the fused polyphase kernels (`true`, default)
    pub fn set_fast_path(&mut self, enable: bool) -> Result<(), Error> {
        check(unsafe { sys::rr_chain_set_fast_path(self.raw, enable as i32) })
    }
    /// Name of the execution plan chosen at the last push (diagnostics)
    pub fn plan(&self) -> String {
        unsafe { CStr::from_ptr(sys::rr_chain_plan(self.raw)).to_string_lossy().into_owned() }
    }
}
