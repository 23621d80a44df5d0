//! vox_box_b200 — vox_box's trait/function surface on top of libvoxbox_b200 (C ABI, sm_100a CUDA).
//!
//! NOT COMPILED IN THE BUILD IMAGE (no cargo/rustc there): source only, see README.md.
//!
//! The module layout, trait names, method names and signatures are the reference crate's
//! (andrewcsmith/vox_box.rs `src/{periodic,spectrum,polynomial,waves,error,lib}.rs`), so a caller switches with
//! `use vox_box_b200 as vox_box;`:
//!
//!  * `periodic`   — `Autocorrelate<T>` for `[T]` and `VecDeque<T>`, `Pitch`, `PitchExtractor`, `Pitched<S, T>`,
//!                   `LagType` / `Hanning`, `interpolate_sinc`, `Interpolation`, `improve_extremum`;
//!  * `spectrum`   — `LPC<T>`, `LPCSolver`, `Resonance`, `ToResonance<T>`, `EstimateFormants<T>`,
//!                   `FormantExtractor`, `MFCC<T>`, `hz_to_mel`, `mel_to_hz`, `dct`, `dct_mut`;
//!  * `polynomial` — `Polynomial<'a, T>` for `[Complex<T>]`;
//!  * `waves`      — `RMS`, `Amplitude`, `MaxAmplitude`, `Normalize`, `Filter`;
//!  * `error`      — `VoxBoxError`, `VoxBoxResult`;
//!  * crate root   — `find_formants`, `find_formants_{real,complex}_work_size`, `MAX_RESONANCES`,
//!                   `{MALE,FEMALE}_FORMANT_ESTIMATES`.
//!
//! Every trait method is ONE frame = a batch of one through the C ABI, on a thread-local device context
//! (`with_context`).  `T` / `S` are `f32` or `f64` (the sealed `Elem` trait); f64 slices go to the device as
//! `VBX_F64` samples, so a frame the caller windowed in f64 is analysed exactly as the reference does.
//! Methods whose reference signature has no `Result` panic on a device failure (the reference panics on bad sizes
//! in the same places); there is no CPU fallback.  Real workloads should not call frame by frame: `batch::Batch`
//! (device-resident utterances, one call = all frames) and `batch::Multi` (all GPUs of the box, host-side gather)
//! are the intended drivers.
//!
//! `ffi` is the `extern "C"` block: one declaration per entry point of include/voxbox_b200.h.
#![allow(non_camel_case_types)]
#![allow(clippy::too_many_arguments)]

extern crate num_complex;

use std::cell::RefCell;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr;

pub use num_complex::Complex;

pub mod ffi {
    use super::*;

    #[repr(C)]
    pub struct vbx_ctx {
        _private: [u8; 0],
    }
    #[repr(C)]
    pub struct vbx_multi {
        _private: [u8; 0],
    }

    /// struct vbx_frames (include/voxbox_b200.h)
    #[repr(C)]
    #[derive(Clone, Copy)]
    pub struct vbx_frames {
        pub base: *const c_void,
        pub n_frames: i64,
        pub frame_stride: i64,
        pub frames_per_segment: i64,
        pub segment_stride: i64,
        pub frame_len: i32,
        pub dtype: i32,
        pub window: i32,
        /// samples between consecutive samples of a frame: 0 / 1 contiguous, C for C interleaved channels (the C header's
        /// `union { reserved; sample_step; }`)
        pub sample_step: i32,
    }

    pub const VBX_OK: c_int = 0;
    pub const VBX_ERR_LPC: c_int = 1;
    pub const VBX_ERR_PITCH: c_int = 2;
    pub const VBX_ERR_POLYNOMIAL: c_int = 3;
    pub const VBX_ERR_WORKSPACE: c_int = 4;
    pub const VBX_ERR_CUDA: c_int = 5;
    pub const VBX_ERR_BADARG: c_int = 6;
    pub const VBX_ERR_NOMEM: c_int = 7;
    pub const VBX_F32: i32 = 0;
    pub const VBX_F64: i32 = 1;
    pub const VBX_I16: i32 = 2;
    /// G.711 mu-law / A-law bytes, decoded to int16 PCM as the kernels load them (frame views only)
    pub const VBX_MULAW8: i32 = 3;
    pub const VBX_ALAW8: i32 = 4;
    pub const VBX_WINDOW_NONE: i32 = 0;
    pub const VBX_WINDOW_HANN_SYMMETRIC: i32 = 1;
    pub const VBX_WINDOW_HANN_PERIODIC: i32 = 2;
    pub const VBX_WINDOW_HANN_LAG: i32 = 3;
    pub const VBX_LPC_BURG: i32 = 0;
    pub const VBX_LPC_AUTOCORR: i32 = 1;

    #[link(name = "voxbox_b200")]
    extern "C" {
        pub fn vbx_ctx_create(device: c_int, out: *mut *mut vbx_ctx) -> c_int;
        pub fn vbx_ctx_destroy(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_sync(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_ctx_stream(ctx: *mut vbx_ctx) -> *mut c_void;
        pub fn vbx_last_error(ctx: *mut vbx_ctx) -> *const c_char;
        pub fn vbx_status_str(status: c_int) -> *const c_char;
        pub fn vbx_version() -> c_int;
        pub fn vbx_device_sm_count(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_kernel_launches(ctx: *mut vbx_ctx) -> i64;
        pub fn vbx_malloc(ctx: *mut vbx_ctx, bytes: usize, dev_out: *mut *mut c_void) -> c_int;
        pub fn vbx_free(ctx: *mut vbx_ctx, dev: *mut c_void) -> c_int;
        pub fn vbx_malloc_host(ctx: *mut vbx_ctx, bytes: usize, host_out: *mut *mut c_void) -> c_int;
        pub fn vbx_free_host(ctx: *mut vbx_ctx, host: *mut c_void) -> c_int;
        pub fn vbx_memcpy_h2d(ctx: *mut vbx_ctx, dev: *mut c_void, host: *const c_void, bytes: usize) -> c_int;
        pub fn vbx_memcpy_d2h(ctx: *mut vbx_ctx, host: *mut c_void, dev: *const c_void, bytes: usize) -> c_int;
        pub fn vbx_memcpy_d2d(ctx: *mut vbx_ctx, dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
        pub fn vbx_memset(ctx: *mut vbx_ctx, dev: *mut c_void, value: c_int, bytes: usize) -> c_int;
        pub fn vbx_timer_start(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_timer_stop_ms(ctx: *mut vbx_ctx, ms_out: *mut f32) -> c_int;
        pub fn vbx_profile_begin(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_profile_end(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_profile_count(ctx: *mut vbx_ctx) -> c_int;
        pub fn vbx_profile_entry(ctx: *mut vbx_ctx, index: c_int, name_out: *mut c_char, name_len: c_int, ms_total: *mut f64,
                                 launches: *mut i64) -> c_int;
        pub fn vbx_profile_counters(ctx: *mut vbx_ctx, out: *mut u64, n: i32) -> c_int;
        pub fn vbx_measure_peaks(ctx: *mut vbx_ctx, fp32_tflops: *mut f64, fp64_tflops: *mut f64) -> c_int;
        pub fn vbx_window_table_host(window: c_int, n: i32, out: *mut f64) -> c_int;

        pub fn vbx_autocorrelate(ctx: *mut vbx_ctx, frames: *const vbx_frames, n_lags: i32, r_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_autocorrelate_host(ctx: *mut vbx_ctx, frames: *const vbx_frames, n_lags: i32, r_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_autocorrelate_ring(ctx: *mut vbx_ctx, rings: *const c_void, dtype: i32, n_rings: i64, capacity: i64,
                                      heads: *const i64, n: i32, n_lags: i32, r_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_lpc_levinson(ctx: *mut vbx_ctx, r: *const c_void, r_dtype: i32, n_frames: i64, r_stride: i32, p: i32,
                                ac_out: *mut c_void, kc_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_lpc(ctx: *mut vbx_ctx, frames: *const vbx_frames, p: i32, r_out: *mut c_void, ac_out: *mut c_void,
                       kc_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_lpc_host(ctx: *mut vbx_ctx, frames: *const vbx_frames, p: i32, r_out: *mut c_void, ac_out: *mut c_void,
                            kc_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_lpc_burg(ctx: *mut vbx_ctx, frames: *const vbx_frames, p: i32, coeffs_out: *mut c_void, status_out: *mut u8,
                            out_dtype: i32) -> c_int;
        pub fn vbx_find_roots(ctx: *mut vbx_ctx, coeffs: *const c_void, dtype: i32, n_polys: i64, len: i32, roots_out: *mut c_void,
                              status_out: *mut u8) -> c_int;
        pub fn vbx_find_roots_work_size(len: i64) -> i64;
        pub fn vbx_laguerre(ctx: *mut vbx_ctx, coeffs: *const c_void, dtype: i32, n_polys: i64, len: i32, start_re: f64,
                            start_im: f64, z_out: *mut c_void) -> c_int;
        pub fn vbx_div_polynomial(ctx: *mut vbx_ctx, coeffs_inout: *mut c_void, dtype: i32, n_polys: i64, len: i32,
                                  other: *const c_void, other_per_poly: i32, rem_out: *mut c_void, status_out: *mut u8) -> c_int;
        pub fn vbx_roots_to_resonances(ctx: *mut vbx_ctx, roots: *const c_void, dtype: i32, n_frames: i64, n_roots: i32,
                                       sample_rate: f64, strict_im: i32, res_out: *mut c_void, res_slots: i32,
                                       nres_out: *mut i32, out_dtype: i32) -> c_int;
        pub fn vbx_lpc_to_resonances(ctx: *mut vbx_ctx, lpc: *const c_void, lpc_dtype: i32, n_frames: i64, lpc_stride: i32, p: i32,
                                     lpc_has_leading_one: i32, sample_rate: f64, strict_im: i32, status_in: *const u8,
                                     res_out: *mut c_void, res_slots: i32, nres_out: *mut i32, roots_out: *mut c_void,
                                     status_out: *mut u8, out_dtype: i32, precision: i32) -> c_int;
        pub fn vbx_estimate_formants(ctx: *mut vbx_ctx, resonances: *const c_void, res_dtype: i32, res_slots: i32,
                                     n_resonances: i32, n_segments: i64, frames_per_segment: i64, status_in: *const u8,
                                     est_inout: *mut c_void, n_estimates: i32, tracks_out: *mut c_void, dtype: i32) -> c_int;
        pub fn vbx_find_formants_real_work_size(buf_len: i64, n_coeffs: i64) -> i64;
        pub fn vbx_find_formants_complex_work_size(n_coeffs: i64) -> i64;
        pub fn vbx_find_formants(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, n_coeffs: i32, lpc_method: i32,
                                 est_inout: *mut c_void, n_formants: i32, tracks_out: *mut c_void, resonances_out: *mut c_void,
                                 nres_out: *mut i32, status_out: *mut u8, dtype: i32) -> c_int;
        pub fn vbx_find_formants_host(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, n_coeffs: i32,
                                      lpc_method: i32, est_inout: *mut c_void, n_formants: i32, tracks_out: *mut c_void,
                                      resonances_out: *mut c_void, nres_out: *mut i32, status_out: *mut u8, dtype: i32) -> c_int;
        pub fn vbx_find_formants_resampled(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, resample_ratio: f64,
                                           n_coeffs: i32, est_inout: *mut c_void, n_formants: i32, tracks_out: *mut c_void,
                                           resonances_out: *mut c_void, nres_out: *mut i32, status_out: *mut u8, dtype: i32) -> c_int;
        pub fn vbx_find_formants_buffered(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, resample_ratio: f64,
                                          resampled_buf_len: i64, n_coeffs: i32, est_inout: *mut c_void, n_formants: i32,
                                          tracks_out: *mut c_void, resonances_out: *mut c_void, nres_out: *mut i32,
                                          status_out: *mut u8, dtype: i32) -> c_int;
        pub fn vbx_pitch(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, threshold: f64, min_hz: f64, max_hz: f64,
                         max_candidates: i32, cand_out: *mut c_void, n_cand_out: *mut i32, status_out: *mut u8, out_dtype: i32) -> c_int;
        pub fn vbx_pitch_host(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, threshold: f64, min_hz: f64,
                              max_hz: f64, max_candidates: i32, cand_out: *mut c_void, n_cand_out: *mut i32, status_out: *mut u8,
                              out_dtype: i32) -> c_int;
        pub fn vbx_pitch_lag_function(ctx: *mut vbx_ctx, frames: *const vbx_frames, lag_out: *mut f64) -> c_int;
        pub fn vbx_frame_peaks(ctx: *mut vbx_ctx, frames: *const vbx_frames, local_out: *mut f64, global_out: *mut f64) -> c_int;
        pub fn vbx_pitch_with_peaks(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, threshold: f64,
                                    silence_threshold: f64, local_peaks: *const f64, global_peaks: *const f64, min_hz: f64,
                                    max_hz: f64, max_candidates: i32, cand_out: *mut c_void, n_cand_out: *mut i32,
                                    status_out: *mut u8, out_dtype: i32) -> c_int;
        pub fn vbx_pitch_with_peaks_host(ctx: *mut vbx_ctx, frames: *const vbx_frames, sample_rate: f64, threshold: f64,
                                         silence_threshold: f64, local_peaks: *const f64, global_peaks: *const f64, min_hz: f64,
                                         max_hz: f64, max_candidates: i32, cand_out: *mut c_void, n_cand_out: *mut i32,
                                         status_out: *mut u8, out_dtype: i32) -> c_int;
        pub fn vbx_pitch_extract(ctx: *mut vbx_ctx, cand: *const c_void, dtype: i32, n_frames: i64, max_candidates: i32,
                                 out: *mut c_void) -> c_int;
        pub fn vbx_pitch_viterbi(ctx: *mut vbx_ctx, cand: *const c_void, dtype: i32, n_cand: *const i32, n_segments: i64,
                                 frames_per_segment: i64, max_candidates: i32, voiced_unvoiced_cost: f64, octave_jump_cost: f64,
                                 octave_cost: f64, ceiling_hz: f64, path_out: *mut c_void, index_out: *mut i32) -> c_int;
        pub fn vbx_interpolate_sinc(ctx: *mut vbx_ctx, y: *const f64, n_series: i64, y_len: i64, offset: i64, nx: i64,
                                    x: *const f64, n_points: i64, max_depth: i64, out: *mut f64) -> c_int;
        pub fn vbx_improve_extremum(ctx: *mut vbx_ctx, y: *const f64, n_series: i64, y_len: i64, offset: i64, nx: i64,
                                    ixmid: *const f64, n_points: i64, interpolation: i32, sinc_depth: i64, is_max: i32,
                                    xmid_out: *mut f64, ymid_out: *mut f64) -> c_int;
        pub fn vbx_mfcc(ctx: *mut vbx_ctx, frames: *const vbx_frames, num_coeffs: i32, n_keep: i32, freq_lo: f64, freq_hi: f64,
                        sample_rate: f64, out: *mut c_void, energies_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_mfcc_host(ctx: *mut vbx_ctx, frames: *const vbx_frames, num_coeffs: i32, n_keep: i32, freq_lo: f64,
                             freq_hi: f64, sample_rate: f64, out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_mfcc_set_fft_precision(ctx: *mut vbx_ctx, dtype: i32) -> c_int;
        pub fn vbx_hz_to_mel(hz: f64) -> f64;
        pub fn vbx_mel_to_hz(mel: f64) -> f64;
        pub fn vbx_dct(ctx: *mut vbx_ctx, signal: *const c_void, dtype: i32, n_signals: i64, n: i32, coeffs: *mut c_void) -> c_int;
        pub fn vbx_rms(ctx: *mut vbx_ctx, x: *const c_void, dtype: i32, n_signals: i64, n: i32, stride: i64, out: *mut c_void) -> c_int;
        pub fn vbx_max_amplitude(ctx: *mut vbx_ctx, x: *const c_void, dtype: i32, n_signals: i64, n: i32, stride: i64,
                                 out: *mut c_void) -> c_int;
        pub fn vbx_normalize(ctx: *mut vbx_ctx, x_inout: *mut c_void, dtype: i32, n_signals: i64, n: i32, stride: i64,
                             maxes: *const c_void) -> c_int;
        pub fn vbx_preemphasis(ctx: *mut vbx_ctx, x_inout: *mut c_void, dtype: i32, n_signals: i64, n: i32, stride: i64,
                               factor: f64) -> c_int;
        pub fn vbx_synth_speech(ctx: *mut vbx_ctx, out: *mut c_void, dtype: i32, n_utts: i64, n_samples: i64, sample_rate: f64,
                                seed: u64, first_utt: i64) -> c_int;

        pub fn vbx_multi_create(n_devices: i32, devices: *const i32, out: *mut *mut vbx_multi) -> c_int;
        pub fn vbx_multi_destroy(m: *mut vbx_multi) -> c_int;
        pub fn vbx_multi_device_count(m: *mut vbx_multi) -> i32;
        pub fn vbx_multi_ctx(m: *mut vbx_multi, index: i32) -> *mut vbx_ctx;
        pub fn vbx_multi_last_error(m: *mut vbx_multi) -> *const c_char;
        pub fn vbx_multi_kernel_launches(m: *mut vbx_multi) -> i64;
        pub fn vbx_multi_partition(n_units: i64, n_parts: i32, part: i32, lo: *mut i64, hi: *mut i64);
        pub fn vbx_multi_lpc_host(m: *mut vbx_multi, frames: *const vbx_frames, p: i32, r_out: *mut c_void, ac_out: *mut c_void,
                                  kc_out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_multi_find_formants_host(m: *mut vbx_multi, frames: *const vbx_frames, sample_rate: f64, n_coeffs: i32,
                                            lpc_method: i32, est_inout: *mut c_void, n_formants: i32, tracks_out: *mut c_void,
                                            resonances_out: *mut c_void, nres_out: *mut i32, status_out: *mut u8, dtype: i32) -> c_int;
        pub fn vbx_multi_pitch_host(m: *mut vbx_multi, frames: *const vbx_frames, sample_rate: f64, threshold: f64, min_hz: f64,
                                    max_hz: f64, max_candidates: i32, cand_out: *mut c_void, n_cand_out: *mut i32,
                                    status_out: *mut u8, out_dtype: i32) -> c_int;
        pub fn vbx_multi_pitch_with_peaks_host(m: *mut vbx_multi, frames: *const vbx_frames, sample_rate: f64, threshold: f64,
                                               silence_threshold: f64, local_peaks: *const f64, global_peaks: *const f64,
                                               min_hz: f64, max_hz: f64, max_candidates: i32, cand_out: *mut c_void,
                                               n_cand_out: *mut i32, status_out: *mut u8, out_dtype: i32) -> c_int;
        pub fn vbx_multi_mfcc_host(m: *mut vbx_multi, frames: *const vbx_frames, num_coeffs: i32, n_keep: i32, freq_lo: f64,
                                   freq_hi: f64, sample_rate: f64, out: *mut c_void, out_dtype: i32) -> c_int;
        pub fn vbx_multi_h2d_bandwidth(m: *mut vbx_multi, bytes_per_device: usize, reps: i32, n_active: i32, gbs_out: *mut f64) -> c_int;
    }
}

// =================================================================================================
// error.rs:4-38
// =================================================================================================
pub mod error {
    use std::error::Error;
    use std::fmt;

    pub type VoxBoxResult<T> = Result<T, VoxBoxError>;

    #[derive(Debug)]
    pub enum VoxBoxError {
        /// LPC calculation error
        LPC(&'static str),
        /// Pitch calculation error
        Pitch(&'static str),
        /// Polynomial calculation error
        Polynomial(&'static str),
        /// Not enough workspace allocated
        Workspace,
        /// no reference analogue: the device / library failed (there is no CPU fallback)
        Cuda(String),
        /// sizes for which the reference would panic
        BadArg(String),
        NoMem,
    }

    impl fmt::Display for VoxBoxError {
        fn fmt(&self, fmt: &mut fmt::Formatter) -> Result<(), fmt::Error> {
            fmt.write_str(self.description())
        }
    }

    impl Error for VoxBoxError {
        fn description(&self) -> &str {
            use self::VoxBoxError::*;
            match *self {
                LPC(s) => s,
                Pitch(s) => s,
                Polynomial(s) => s,
                Workspace => "Not enough workspace allocated",
                Cuda(ref s) => s,
                BadArg(ref s) => s,
                NoMem => "out of device or pinned memory",
            }
        }
    }
}
pub use error::{VoxBoxError, VoxBoxResult};

// =================================================================================================
// element types, device context, device buffers
// =================================================================================================
mod sealed {
    pub trait Sealed {}
    impl Sealed for f32 {}
    impl Sealed for f64 {}
}

/// The two sample / coefficient types of the C ABI (the reference's generic `T: Float` / `S: Sample`).
pub trait Elem: sealed::Sealed + Copy + Default + PartialOrd + 'static {
    const DTYPE: i32;
    fn to_f64(self) -> f64;
    fn from_f64(v: f64) -> Self;
}
impl Elem for f32 {
    const DTYPE: i32 = ffi::VBX_F32;
    fn to_f64(self) -> f64 { self as f64 }
    fn from_f64(v: f64) -> f32 { v as f32 }
}
impl Elem for f64 {
    const DTYPE: i32 = ffi::VBX_F64;
    fn to_f64(self) -> f64 { self }
    fn from_f64(v: f64) -> f64 { v }
}

/// RAII wrapper of `vbx_ctx`: one device + stream + scratch arena.  Not `Sync`; one per host thread / GPU.
pub struct Context {
    raw: *mut ffi::vbx_ctx,
    owned: bool,
}

impl Context {
    pub fn new(device: i32) -> VoxBoxResult<Context> {
        let mut raw = ptr::null_mut();
        let st = unsafe { ffi::vbx_ctx_create(device, &mut raw) };
        if st != ffi::VBX_OK {
            return Err(VoxBoxError::Cuda("vbx_ctx_create failed: no usable CUDA device (no CPU fallback)".into()));
        }
        Ok(Context { raw, owned: true })
    }
    pub fn raw(&self) -> *mut ffi::vbx_ctx { self.raw }

    pub fn check(&self, st: c_int) -> VoxBoxResult<()> {
        use std::ffi::CStr;
        let msg = || unsafe { CStr::from_ptr(ffi::vbx_last_error(self.raw)).to_string_lossy().into_owned() };
        status_to_result(st, msg)
    }
    pub fn sync(&self) -> VoxBoxResult<()> { self.check(unsafe { ffi::vbx_sync(self.raw) }) }
}

impl Drop for Context {
    fn drop(&mut self) {
        if self.owned { unsafe { ffi::vbx_ctx_destroy(self.raw) }; }
    }
}

fn status_to_result<F: FnOnce() -> String>(st: c_int, msg: F) -> VoxBoxResult<()> {
    match st {
        ffi::VBX_OK => Ok(()),
        ffi::VBX_ERR_LPC => Err(VoxBoxError::LPC("Denum was <= 0.0")),              // spectrum.rs:124
        ffi::VBX_ERR_PITCH => Err(VoxBoxError::Pitch("pitch candidate strength is NaN")),
        ffi::VBX_ERR_POLYNOMIAL => Err(VoxBoxError::Polynomial("Failed to find roots")), // polynomial.rs:123
        ffi::VBX_ERR_WORKSPACE => Err(VoxBoxError::Workspace),
        ffi::VBX_ERR_NOMEM => Err(VoxBoxError::NoMem),
        ffi::VBX_ERR_BADARG => Err(VoxBoxError::BadArg(msg())),
        _ => Err(VoxBoxError::Cuda(msg())),
    }
}

thread_local! {
    static CONTEXT: RefCell<Option<Context>> = RefCell::new(None);
}

/// Runs `f` with this thread's device context (created on first use on device `$VOXBOX_B200_DEVICE`, default 0).
/// Panics if no CUDA device / library is usable: there is no CPU fallback.
pub fn with_context<R, F: FnOnce(&Context) -> R>(f: F) -> R {
    CONTEXT.with(|cell| {
        let mut slot = cell.borrow_mut();
        if slot.is_none() {
            let dev = std::env::var("VOXBOX_B200_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
            *slot = Some(Context::new(dev).expect("vox_box_b200: no usable CUDA device (there is no CPU fallback)"));
        }
        f(slot.as_ref().unwrap())
    })
}

/// Caller-owned HBM buffer (vbx_malloc / vbx_free).
pub struct DeviceBuf<T> {
    pub ptr: *mut c_void,
    pub len: usize,
    ctx: *mut ffi::vbx_ctx,
    _t: std::marker::PhantomData<T>,
}

impl<T: Copy> DeviceBuf<T> {
    pub fn new(ctx: &Context, len: usize) -> VoxBoxResult<Self> {
        let mut p = ptr::null_mut();
        ctx.check(unsafe { ffi::vbx_malloc(ctx.raw, len * std::mem::size_of::<T>(), &mut p) })?;
        Ok(DeviceBuf { ptr: p, len, ctx: ctx.raw, _t: std::marker::PhantomData })
    }
    pub fn from_host(ctx: &Context, host: &[T]) -> VoxBoxResult<Self> {
        let b = Self::new(ctx, host.len())?;
        ctx.check(unsafe { ffi::vbx_memcpy_h2d(ctx.raw, b.ptr, host.as_ptr() as *const c_void, host.len() * std::mem::size_of::<T>()) })?;
        ctx.sync()?;
        Ok(b)
    }
    /// Copies the buffer into `out` (lengths must match).
    pub fn read_into(&self, ctx: &Context, out: &mut [T]) -> VoxBoxResult<()> {
        assert!(out.len() <= self.len);
        ctx.check(unsafe { ffi::vbx_memcpy_d2h(ctx.raw, out.as_mut_ptr() as *mut c_void, self.ptr, out.len() * std::mem::size_of::<T>()) })?;
        ctx.sync()
    }
    pub fn to_host(&self, ctx: &Context, fill: T) -> VoxBoxResult<Vec<T>> {
        let mut v = vec![fill; self.len];
        self.read_into(ctx, &mut v)?;
        Ok(v)
    }
}

impl<T> Drop for DeviceBuf<T> {
    fn drop(&mut self) {
        unsafe { ffi::vbx_free(self.ctx, self.ptr) };
    }
}

fn one_frame<T: Elem>(x: &[T], window: i32) -> ffi::vbx_frames {
    ffi::vbx_frames {
        base: x.as_ptr() as *const c_void,
        n_frames: 1,
        frame_stride: x.len() as i64,
        frames_per_segment: 0,
        segment_stride: 0,
        frame_len: x.len() as i32,
        dtype: T::DTYPE,
        window,
        sample_step: 0,
    }
}

pub const MAX_RESONANCES: usize = 32; // lib.rs:26
pub const MALE_FORMANT_ESTIMATES: [f64; 4] = [320., 1440., 2760., 3200.]; // lib.rs:27
pub const FEMALE_FORMANT_ESTIMATES: [f64; 4] = [480., 1760., 3200., 3520.]; // lib.rs:28

/// lib.rs:30-32
pub fn find_formants_real_work_size(buf_len: usize, n_coeffs: usize) -> usize {
    unsafe { ffi::vbx_find_formants_real_work_size(buf_len as i64, n_coeffs as i64) as usize }
}
/// lib.rs:34-36
pub fn find_formants_complex_work_size(n_coeffs: usize) -> usize {
    unsafe { ffi::vbx_find_formants_complex_work_size(n_coeffs as i64) as usize }
}

/// lib.rs:40-116 `find_formants`: one frame; `formants` is the tracker state, in/out.
///
/// `work` / `complex_work` are not needed by the device path; `work.len()` is still checked as the reference does
/// (`Err(Workspace)`, lib.rs:46-48).  `resampled_buf.len()` selects the reference's literal buffer semantics
/// (lib.rs:54,66-75: the WHOLE resampled_buf is windowed and analysed; its tail beyond `resampled_len` is taken to be
/// zeros, as in the reference's tests) — it must be >= ceil(resample_ratio * buf.len()) or the call panics like the
/// reference's `assert!`.  Unlike the reference, `resampled_buf` and `work` are not written.
pub fn find_formants<S: Elem>(buf: &mut [S], sample_rate: S, resample_ratio: f64, resampled_buf: &mut [S], n_coeffs: usize,
                              work: &mut [S], _complex_work: &mut [Complex<S>], formants: &mut [spectrum::Resonance<S>])
                              -> VoxBoxResult<()> {
    let resampled_len = (resample_ratio * buf.len() as f64).ceil() as usize;
    if work.len() < find_formants_real_work_size(resampled_len, n_coeffs) {
        return Err(VoxBoxError::Workspace);
    }
    assert!(resampled_len <= resampled_buf.len());
    with_context(|ctx| {
        let dev = DeviceBuf::from_host(ctx, buf)?;
        let mut fr = one_frame(buf, ffi::VBX_WINDOW_NONE);
        fr.base = dev.ptr;
        let est = DeviceBuf::from_host(ctx, formants)?;
        let status = DeviceBuf::<u8>::new(ctx, 1)?;
        ctx.check(unsafe {
            ffi::vbx_find_formants_buffered(ctx.raw, &fr, sample_rate.to_f64(), resample_ratio, resampled_buf.len() as i64,
                                            n_coeffs as i32, est.ptr, formants.len() as i32, ptr::null_mut(), ptr::null_mut(),
                                            ptr::null_mut(), status.ptr as *mut u8, S::DTYPE)
        })?;
        let st = status.to_host(ctx, 0u8)?;
        ctx.check(st[0] as c_int)?; // Err(LPC("Denum was <= 0.0")) / Err(Polynomial(..)): the state is untouched
        est.read_into(ctx, formants)
    })
}

// =================================================================================================
// periodic.rs
// =================================================================================================
pub mod periodic {
    use super::*;
    use std::collections::VecDeque;

    /// periodic.rs:265-274
    pub trait Autocorrelate<T> {
        fn autocorrelate_mut(&self, coeffs: &mut [T]);
        fn autocorrelate(&self, n_coeffs: usize) -> Vec<T>;
    }

    /// periodic.rs:276-289: `r[lag] = x[0] + sum_{i>=1} x[i]·x[i+lag]` (the fold is seeded with x[0], as written).
    impl<T: Elem> Autocorrelate<T> for [T] {
        fn autocorrelate_mut(&self, coeffs: &mut [T]) {
            with_context(|ctx| {
                let fr = one_frame(self, ffi::VBX_WINDOW_NONE);
                ctx.check(unsafe {
                    ffi::vbx_autocorrelate_host(ctx.raw(), &fr, coeffs.len() as i32, coeffs.as_mut_ptr() as *mut c_void, T::DTYPE)
                }).expect("autocorrelate_mut")
            })
        }
        fn autocorrelate(&self, n_coeffs: usize) -> Vec<T> {
            let mut coeffs = vec![T::default(); n_coeffs];
            self.autocorrelate_mut(&mut coeffs[..]);
            coeffs
        }
    }

    /// periodic.rs:291-304: the same fold on a ring buffer.  The deque's two slices are uploaded as they lie in memory
    /// (ring = back ++ front with head = back.len()) and unrolled on the device.
    impl<T: Elem> Autocorrelate<T> for VecDeque<T> {
        fn autocorrelate_mut(&self, coeffs: &mut [T]) {
            with_context(|ctx| {
                let (front, back) = self.as_slices();
                let mut ring: Vec<T> = Vec::with_capacity(self.len());
                ring.extend_from_slice(back);
                ring.extend_from_slice(front);
                let heads = [back.len() as i64];
                let run = || -> VoxBoxResult<()> {
                    let dev = DeviceBuf::from_host(ctx, &ring)?;
                    let dheads = DeviceBuf::from_host(ctx, &heads)?;
                    let out = DeviceBuf::<T>::new(ctx, coeffs.len())?;
                    ctx.check(unsafe {
                        ffi::vbx_autocorrelate_ring(ctx.raw(), dev.ptr, T::DTYPE, 1, ring.len() as i64, dheads.ptr as *const i64,
                                                    ring.len() as i32, coeffs.len() as i32, out.ptr, T::DTYPE)
                    })?;
                    out.read_into(ctx, coeffs)
                };
                run().expect("autocorrelate_mut (VecDeque)")
            })
        }
        fn autocorrelate(&self, n_coeffs: usize) -> Vec<T> {
            let mut coeffs = vec![T::default(); n_coeffs];
            self.autocorrelate_mut(&mut coeffs[..]);
            coeffs
        }
    }

    /// periodic.rs:306-318
    #[repr(C)]
    #[derive(Clone, Copy, Debug, Default)]
    pub struct Pitch<T> {
        pub frequency: T,
        pub strength: T,
    }

    impl<T> Pitch<T> {
        pub fn new(frequency: T, strength: T) -> Self { Pitch { frequency, strength } }
    }

    /// periodic.rs:320-354: yields `candidates[frame][0]` (the strongest candidate) per frame; the cost fields are
    /// declared and unused in the reference.  `viterbi` is the opt-in path finder the reference documents
    /// (periodic.rs:394-395) but does not implement.
    #[allow(dead_code)]
    pub struct PitchExtractor<'a, T: 'a> {
        voiced_unvoiced_cost: T,
        voicing_threshold: T,
        candidates: &'a [&'a [Pitch<T>]],
    }

    impl<'a, T: 'a + Elem> PitchExtractor<'a, T> {
        pub fn new(candidates: &'a [&'a [Pitch<T>]], voiced_unvoiced_cost: T, voicing_threshold: T) -> Self {
            PitchExtractor { voiced_unvoiced_cost, voicing_threshold, candidates }
        }

        /// Opt-in extension: Boersma's Viterbi path over the remaining frames' candidate lists (device side).
        pub fn viterbi(&self, octave_jump_cost: f64, octave_cost: f64, ceiling_hz: f64) -> VoxBoxResult<Vec<Pitch<T>>> {
            let frames = self.candidates.len();
            let cap = self.candidates.iter().map(|c| c.len()).max().unwrap_or(0).max(1);
            let mut flat = vec![Pitch::<T>::default(); frames * cap];
            let mut counts = vec![0i32; frames];
            for (f, c) in self.candidates.iter().enumerate() {
                flat[f * cap..f * cap + c.len()].copy_from_slice(c);
                counts[f] = c.len() as i32;
            }
            with_context(|ctx| {
                let dev = DeviceBuf::from_host(ctx, &flat)?;
                let dn = DeviceBuf::from_host(ctx, &counts)?;
                let out = DeviceBuf::<Pitch<T>>::new(ctx, frames)?;
                ctx.check(unsafe {
                    ffi::vbx_pitch_viterbi(ctx.raw(), dev.ptr, T::DTYPE, dn.ptr as *const i32, 1, frames as i64, cap as i32,
                                           self.voiced_unvoiced_cost.to_f64(), octave_jump_cost, octave_cost, ceiling_hz, out.ptr,
                                           ptr::null_mut())
                })?;
                out.to_host(ctx, Pitch::<T>::default())
            })
        }
    }

    impl<'a, T: 'a + Copy> Iterator for PitchExtractor<'a, T> {
        type Item = Pitch<T>;

        fn next(&mut self) -> Option<Self::Item> {
            let n_candidates = self.candidates.len();
            if n_candidates == 0 {
                return None;
            }
            let candidate = self.candidates[0][0];
            self.candidates = if n_candidates > 1 { &self.candidates[1..] } else { &[] };
            Some(candidate)
        }
    }

    /// periodic.rs:232-252: the lag-window type parameter of `pitch`.  `Hanning` (its lag window is `HanningLag`, the
    /// Hann window's autocorrelation) is the only implementor in the reference and the one the device path implements.
    pub trait LagType {}
    pub struct Hanning;
    pub struct HanningLag;
    impl LagType for Hanning {}

    /// periodic.rs:356-358
    pub trait Pitched<S, T> {
        fn pitch<W: LagType>(&self, sample_rate: T, threshold: T, local_peak: S, global_peak: S, min: T, max: T) -> Vec<Pitch<T>>;
    }

    /// periodic.rs:377-456: Boersma autocorrelation candidates of ONE already-windowed frame, sorted by strength
    /// (descending), always containing `Pitch { 0, threshold }`.  `local_peak` / `global_peak` are ignored, as in the
    /// reference (periodic.rs:396).  A NaN strength panics, as the reference's sort does (periodic.rs:453).
    impl<S: Elem, T: Elem> Pitched<S, T> for [S] {
        fn pitch<W: LagType>(&self, sample_rate: T, threshold: T, _local_peak: S, _global_peak: S, min: T, max: T) -> Vec<Pitch<T>> {
            with_context(|ctx| {
                let fr = one_frame(self, ffi::VBX_WINDOW_NONE);
                let cap = self.len() / 4 + 2; // every other lag below N/2 a maximum, plus the unvoiced candidate
                let mut cand = vec![Pitch::<T>::default(); cap];
                let (mut n, mut st) = ([0i32; 1], [0u8; 1]);
                ctx.check(unsafe {
                    ffi::vbx_pitch_host(ctx.raw(), &fr, sample_rate.to_f64(), threshold.to_f64(), min.to_f64(), max.to_f64(),
                                        cap as i32, cand.as_mut_ptr() as *mut c_void, n.as_mut_ptr(), st.as_mut_ptr(), T::DTYPE)
                }).expect("pitch");
                assert!(st[0] == 0, "pitch: a candidate strength is NaN (the reference's sort panics here)");
                cand.truncate(n[0] as usize);
                cand
            })
        }
    }

    /// Opt-in extension of `Pitched::pitch` that honours `local_peak` / `global_peak` (the reference takes them and ignores
    /// them, periodic.rs:396): the unvoiced candidate's strength is Boersma's (1993) voiceless strength
    /// `threshold + max(0, 2 − min(local_peak / global_peak, 1)·(1 + threshold) / silence_threshold)` instead of `threshold`,
    /// so quiet frames rank it first.  `silence_threshold == 0` is exactly `pitch()` (Praat's default is 0.03 with a voicing
    /// threshold of 0.45).  The peaks are max |x| of the frame and of the whole recording, as the reference's driver computes
    /// them (examples/pitch_detection.rs:48); see `vbx_pitch_with_peaks` in include/voxbox_b200.h.  A free function rather than a
    /// method, so that the `Pitched` trait keeps the reference's surface.
    pub fn pitch_with_peaks<W: LagType, S: Elem, T: Elem>(samples: &[S], sample_rate: T, threshold: T, silence_threshold: T,
                                                          local_peak: S, global_peak: S, min: T, max: T) -> Vec<Pitch<T>> {
        with_context(|ctx| {
            let fr = one_frame(samples, ffi::VBX_WINDOW_NONE);
            let cap = samples.len() / 4 + 2; // as pitch(): every other lag below N/2 a maximum, plus the unvoiced candidate
            let mut cand = vec![Pitch::<T>::default(); cap];
            let (mut n, mut st) = ([0i32; 1], [0u8; 1]);
            let (local, global) = ([local_peak.to_f64()], [global_peak.to_f64()]);
            ctx.check(unsafe {
                ffi::vbx_pitch_with_peaks_host(ctx.raw(), &fr, sample_rate.to_f64(), threshold.to_f64(), silence_threshold.to_f64(),
                                               local.as_ptr(), global.as_ptr(), min.to_f64(), max.to_f64(), cap as i32,
                                               cand.as_mut_ptr() as *mut c_void, n.as_mut_ptr(), st.as_mut_ptr(), T::DTYPE)
            }).expect("pitch_with_peaks");
            assert!(st[0] == 0, "pitch_with_peaks: a candidate strength is NaN (the reference's sort panics here)");
            cand.truncate(n[0] as usize);
            cand
        })
    }

    /// periodic.rs:29-87
    pub fn interpolate_sinc<S: Elem>(y: &[S], offset: isize, nx: usize, x: S, max_depth: usize) -> f64 {
        let yd: Vec<f64> = y.iter().map(|v| v.to_f64()).collect();
        with_context(|ctx| {
            let run = || -> VoxBoxResult<f64> {
                let dy = DeviceBuf::from_host(ctx, &yd)?;
                let dx = DeviceBuf::from_host(ctx, &[x.to_f64()])?;
                let out = DeviceBuf::<f64>::new(ctx, 1)?;
                ctx.check(unsafe {
                    ffi::vbx_interpolate_sinc(ctx.raw(), dy.ptr as *const f64, 1, yd.len() as i64, offset as i64, nx as i64,
                                              dx.ptr as *const f64, 1, max_depth as i64, out.ptr as *mut f64)
                })?;
                Ok(out.to_host(ctx, 0f64)?[0])
            };
            run().expect("interpolate_sinc")
        })
    }

    /// periodic.rs:89-93
    pub enum Interpolation {
        None,
        Parabolic,
        Sinc(usize),
    }

    /// periodic.rs:192-230 (+ brent_maximize :103-188)
    pub fn improve_extremum<S: Elem>(y: &[S], offset: isize, nx: usize, ixmid: f64, interp: Interpolation, is_max: bool) -> (f64, f64) {
        let yd: Vec<f64> = y.iter().map(|v| v.to_f64()).collect();
        let (kind, depth) = match interp {
            Interpolation::None => (0, 0usize),
            Interpolation::Parabolic => (1, 0usize),
            Interpolation::Sinc(d) => (2, d),
        };
        with_context(|ctx| {
            let run = || -> VoxBoxResult<(f64, f64)> {
                let dy = DeviceBuf::from_host(ctx, &yd)?;
                let dx = DeviceBuf::from_host(ctx, &[ixmid])?;
                let (xm, ym) = (DeviceBuf::<f64>::new(ctx, 1)?, DeviceBuf::<f64>::new(ctx, 1)?);
                ctx.check(unsafe {
                    ffi::vbx_improve_extremum(ctx.raw(), dy.ptr as *const f64, 1, yd.len() as i64, offset as i64, nx as i64,
                                              dx.ptr as *const f64, 1, kind, depth as i64, is_max as i32, xm.ptr as *mut f64,
                                              ym.ptr as *mut f64)
                })?;
                Ok((xm.to_host(ctx, 0f64)?[0], ym.to_host(ctx, 0f64)?[0]))
            };
            run().expect("improve_extremum")
        })
    }
}

// =================================================================================================
// spectrum.rs
// =================================================================================================
pub mod spectrum {
    use super::*;
    use std::marker::PhantomData;

    /// spectrum.rs:14-48
    pub struct LPCSolver<'a, T: 'a> {
        n_coeffs: usize,
        ac: &'a mut [T],
        kc: &'a mut [T],
        tmp: &'a mut [T],
    }

    impl<'a, T: 'a + Elem> LPCSolver<'a, T> {
        /// work must be longer than `n_coeffs * 3 + 1` (spectrum.rs:26).
        pub fn new(n_coeffs: usize, work: &'a mut [T]) -> LPCSolver<'a, T> {
            assert!(work.len() > n_coeffs * 3 + 1);
            let (ac, work) = work.split_at_mut(n_coeffs + 1);
            let (kc, tmp) = work.split_at_mut(n_coeffs);
            LPCSolver { n_coeffs, ac, kc, tmp }
        }
        /// Finds the LPC coefficients for the autocorrelated buffer
        pub fn solve(&mut self, buf: &[T]) {
            buf.lpc_mut(self.n_coeffs, self.ac, self.kc, self.tmp);
        }
        pub fn lpc(&self) -> &[T] { &self.ac[..] }
    }

    /// spectrum.rs:50-55
    pub trait LPC<T> {
        fn lpc_mut(&self, n_coeffs: usize, ac: &mut [T], kc: &mut [T], tmp: &mut [T]);
        fn lpc(&self, n_coeffs: usize) -> Vec<T>;
        fn lpc_praat_mut(&self, n_coeffs: usize, coeffs: &mut [T], work: &mut [T]) -> VoxBoxResult<()>;
        fn lpc_praat(&self, n_coeffs: usize) -> VoxBoxResult<Vec<T>>;
    }

    impl<T: Elem> LPC<T> for [T] {
        /// spectrum.rs:63-84 Levinson–Durbin on the autocorrelation `self[0..=n_coeffs]`: `ac[0..=n]` (ac[0] = 1,
        /// error-filter sign) and the reflection coefficients `kc[0..n]`.  `tmp` is not needed on the device.
        fn lpc_mut(&self, n_coeffs: usize, ac: &mut [T], kc: &mut [T], _tmp: &mut [T]) {
            assert!(self.len() > n_coeffs && ac.len() > n_coeffs && kc.len() >= n_coeffs);
            with_context(|ctx| {
                let run = || -> VoxBoxResult<()> {
                    let dev = DeviceBuf::from_host(ctx, self)?;
                    let (dac, dkc) = (DeviceBuf::<T>::new(ctx, n_coeffs + 1)?, DeviceBuf::<T>::new(ctx, n_coeffs.max(1))?);
                    ctx.check(unsafe {
                        ffi::vbx_lpc_levinson(ctx.raw(), dev.ptr, T::DTYPE, 1, self.len() as i32, n_coeffs as i32, dac.ptr, dkc.ptr, T::DTYPE)
                    })?;
                    dac.read_into(ctx, &mut ac[..n_coeffs + 1])?;
                    dkc.read_into(ctx, &mut kc[..n_coeffs])
                };
                run().expect("lpc_mut")
            })
        }

        fn lpc(&self, n_coeffs: usize) -> Vec<T> {
            let mut ac = vec![T::default(); n_coeffs + 1];
            let mut kc = vec![T::default(); n_coeffs];
            let mut tmp = vec![T::default(); n_coeffs];
            self.lpc_mut(n_coeffs, &mut ac[..], &mut kc[..], &mut tmp[..]);
            ac
        }

        /// spectrum.rs:101-146 Burg (Praat form) on the frame itself; `work` is not needed on the device.
        fn lpc_praat_mut(&self, n_coeffs: usize, coeffs: &mut [T], _work: &mut [T]) -> VoxBoxResult<()> {
            with_context(|ctx| {
                let dev = DeviceBuf::from_host(ctx, self)?;
                let mut fr = one_frame(self, ffi::VBX_WINDOW_NONE);
                fr.base = dev.ptr;
                let co = DeviceBuf::<T>::new(ctx, n_coeffs)?;
                let st = DeviceBuf::<u8>::new(ctx, 1)?;
                ctx.check(unsafe { ffi::vbx_lpc_burg(ctx.raw(), &fr, n_coeffs as i32, co.ptr, st.ptr as *mut u8, T::DTYPE) })?;
                ctx.check(st.to_host(ctx, 0u8)?[0] as c_int)?; // Err(LPC("Denum was <= 0.0"))
                co.read_into(ctx, &mut coeffs[..n_coeffs])
            })
        }

        fn lpc_praat(&self, n_coeffs: usize) -> VoxBoxResult<Vec<T>> {
            let mut coeffs = vec![T::default(); n_coeffs];
            let mut work = vec![T::default(); 0];
            self.lpc_praat_mut(n_coeffs, &mut coeffs[..], &mut work[..]).map(|_| coeffs)
        }
    }

    /// spectrum.rs:149-154
    #[repr(C)]
    #[derive(Clone, Copy, Debug, Default, PartialEq)]
    pub struct Resonance<T> {
        pub frequency: T,
        pub bandwidth: T,
    }

    impl<T> Resonance<T> {
        pub fn new(f: T, b: T) -> Resonance<T> { Resonance { frequency: f, bandwidth: b } }
    }

    impl<T: Elem> Resonance<T> {
        /// spectrum.rs:166-192: `None` for roots below the real axis or inside the 50 Hz guard bands.
        pub fn from_root(root: &Complex<T>, sample_rate: T) -> Option<Resonance<T>> {
            let roots = [*root];
            let res = roots[..].to_resonance(sample_rate);
            res.first().cloned()
        }
    }

    /// spectrum.rs:195-197
    pub trait ToResonance<T> {
        fn to_resonance(&self, sample_rate: T) -> Vec<Resonance<T>>;
    }

    /// spectrum.rs:199-210: resonances of the roots with im >= 0, sorted by frequency.
    impl<T: Elem> ToResonance<T> for [Complex<T>] {
        fn to_resonance(&self, sample_rate: T) -> Vec<Resonance<T>> {
            if self.is_empty() { return Vec::new(); }
            with_context(|ctx| {
                let run = || -> VoxBoxResult<Vec<Resonance<T>>> {
                    let dev = DeviceBuf::from_host(ctx, self)?;
                    let res = DeviceBuf::<Resonance<T>>::new(ctx, self.len())?;
                    let n = DeviceBuf::<i32>::new(ctx, 1)?;
                    ctx.check(unsafe {
                        ffi::vbx_roots_to_resonances(ctx.raw(), dev.ptr, T::DTYPE, 1, self.len() as i32, sample_rate.to_f64(), 0,
                                                     res.ptr, self.len() as i32, n.ptr as *mut i32, T::DTYPE)
                    })?;
                    let mut v = res.to_host(ctx, Resonance::<T>::default())?;
                    v.truncate(n.to_host(ctx, 0i32)?[0] as usize);
                    Ok(v)
                };
                run().expect("to_resonance")
            })
        }
    }

    /// spectrum.rs:216-219
    pub trait EstimateFormants<T> {
        type FormantSlots;
        fn estimate_formants(&mut self, resonances: &[Resonance<T>]);
    }

    /// spectrum.rs:225-334: one McCandless step; `self` (<= 32 estimates) is the state, updated in place.  At most the
    /// first 32 resonances take part (find_formants passes 32 zero-padded slots, lib.rs:114).
    impl<T: Elem> EstimateFormants<T> for [Resonance<T>] {
        type FormantSlots = [Option<Resonance<T>>; 6];

        fn estimate_formants(&mut self, resonances: &[Resonance<T>]) {
            assert!(!resonances.is_empty() && resonances.len() <= MAX_RESONANCES && self.len() <= MAX_RESONANCES);
            with_context(|ctx| {
                let run = |me: &mut [Resonance<T>]| -> VoxBoxResult<()> {
                    let res = DeviceBuf::from_host(ctx, resonances)?;
                    let est = DeviceBuf::from_host(ctx, me)?;
                    ctx.check(unsafe {
                        ffi::vbx_estimate_formants(ctx.raw(), res.ptr, T::DTYPE, resonances.len() as i32, resonances.len() as i32, 1, 1,
                                                   ptr::null(), est.ptr, me.len() as i32, ptr::null_mut(), T::DTYPE)
                    })?;
                    est.read_into(ctx, me)
                };
                run(self).expect("estimate_formants")
            })
        }
    }

    /// spectrum.rs:336-369
    pub struct FormantExtractor<'a, T: 'a, I: Iterator<Item = &'a [Resonance<T>]>> {
        pub estimates: Vec<Resonance<T>>,
        #[allow(dead_code)]
        num_formants: usize,
        resonances: I,
        phantom: PhantomData<&'a T>,
    }

    impl<'a, T: 'a + Elem, I: Iterator<Item = &'a [Resonance<T>]>> FormantExtractor<'a, T, I> {
        pub fn new(num_formants: usize, resonances: I, starting_estimates: Vec<Resonance<T>>) -> Self {
            FormantExtractor { num_formants, resonances, estimates: starting_estimates, phantom: PhantomData }
        }
    }

    impl<'a, T: 'a + Elem, I: Iterator<Item = &'a [Resonance<T>]>> Iterator for FormantExtractor<'a, T, I> {
        type Item = Vec<Resonance<T>>;

        fn next(&mut self) -> Option<Self::Item> {
            let frame = self.resonances.next()?;
            self.estimates[..].estimate_formants(frame);
            Some(self.estimates.clone())
        }
    }

    /// spectrum.rs:371-373
    pub trait MFCC<T> {
        fn mfcc(&self, num_coeffs: usize, freq_bounds: (f64, f64), sample_rate: f64) -> Vec<T>;
    }

    /// spectrum.rs:401-441: `self` is a windowed frame; `num_coeffs` is both the number of mel bands and of returned
    /// DCT rows (quirk kept).  Panics where the reference panics (a filter-bank bin beyond the spectrum).
    impl<T: Elem> MFCC<T> for [T] {
        fn mfcc(&self, num_coeffs: usize, freq_bounds: (f64, f64), sample_rate: f64) -> Vec<T> {
            with_context(|ctx| {
                let fr = one_frame(self, ffi::VBX_WINDOW_NONE);
                let mut out = vec![T::default(); num_coeffs];
                ctx.check(unsafe {
                    ffi::vbx_mfcc_host(ctx.raw(), &fr, num_coeffs as i32, num_coeffs as i32, freq_bounds.0, freq_bounds.1, sample_rate,
                                       out.as_mut_ptr() as *mut c_void, T::DTYPE)
                }).expect("mfcc");
                out
            })
        }
    }

    /// spectrum.rs:375-377
    pub fn hz_to_mel(hz: f64) -> f64 { unsafe { ffi::vbx_hz_to_mel(hz) } }
    /// spectrum.rs:379-381
    pub fn mel_to_hz(mel: f64) -> f64 { unsafe { ffi::vbx_mel_to_hz(mel) } }

    /// spectrum.rs:384-388
    pub fn dct<T: Elem>(signal: &[T]) -> Vec<T> {
        let mut out = vec![T::default(); signal.len()];
        dct_mut(signal, &mut out[..]);
        out
    }

    /// spectrum.rs:391-398: `coeffs[k] = 2 sum_m signal[m] cos(pi k (2m+1) / (2n))`.
    pub fn dct_mut<T: Elem>(signal: &[T], coeffs: &mut [T]) {
        assert!(coeffs.len() >= signal.len());
        if signal.is_empty() { return; }
        with_context(|ctx| {
            let run = || -> VoxBoxResult<()> {
                let dev = DeviceBuf::from_host(ctx, signal)?;
                let out = DeviceBuf::<T>::new(ctx, signal.len())?;
                ctx.check(unsafe { ffi::vbx_dct(ctx.raw(), dev.ptr, T::DTYPE, 1, signal.len() as i32, out.ptr) })?;
                out.read_into(ctx, &mut coeffs[..signal.len()])
            };
            run().expect("dct_mut")
        })
    }
}

// =================================================================================================
// polynomial.rs
// =================================================================================================
pub mod polynomial {
    use super::*;

    /// polynomial.rs:10-21
    pub trait Polynomial<'a, T> {
        fn degree(&self) -> usize;
        fn off_low(&self) -> usize;
        fn laguerre(&self, z: Complex<T>) -> Complex<T>;

        fn find_roots_work_size(&self) -> usize;
        fn find_roots(&self) -> VoxBoxResult<Vec<Complex<T>>>;
        fn find_roots_mut<'b>(&'b mut self, work: &'b mut [Complex<T>]) -> VoxBoxResult<()>;

        fn div_polynomial(&mut self, other: Complex<T>) -> VoxBoxResult<Vec<Complex<T>>>;
        fn div_polynomial_mut(&'a mut self, other: Complex<T>, rem: &'a mut [Complex<T>]) -> VoxBoxResult<()>;
    }

    fn is_zero<T: Elem>(z: &Complex<T>) -> bool { z.re.to_f64() == 0.0 && z.im.to_f64() == 0.0 }

    impl<'a, T: Elem> Polynomial<'a, T> for [Complex<T>] {
        /// polynomial.rs:26-28: index of the highest non-zero coefficient (0 if all are zero).
        fn degree(&self) -> usize {
            self.iter().rposition(|z| !is_zero(z)).unwrap_or(0)
        }
        /// polynomial.rs:30-32: index of the lowest non-zero coefficient (0 if all are zero).
        fn off_low(&self) -> usize {
            self.iter().position(|z| !is_zero(z)).unwrap_or(0)
        }

        /// polynomial.rs:34-72: <= 20 modified-Laguerre iterations from `start`.
        fn laguerre(&self, start: Complex<T>) -> Complex<T> {
            with_context(|ctx| {
                let run = || -> VoxBoxResult<Complex<T>> {
                    let dev = DeviceBuf::from_host(ctx, self)?;
                    let out = DeviceBuf::<Complex<T>>::new(ctx, 1)?;
                    ctx.check(unsafe {
                        ffi::vbx_laguerre(ctx.raw(), dev.ptr, T::DTYPE, 1, self.len() as i32, start.re.to_f64(), start.im.to_f64(), out.ptr)
                    })?;
                    Ok(out.to_host(ctx, Complex::new(T::default(), T::default()))?[0])
                };
                run().expect("laguerre")
            })
        }

        /// polynomial.rs:75-77
        fn find_roots_work_size(&self) -> usize { self.len() * 6 + 4 }

        /// polynomial.rs:79-90
        fn find_roots(&self) -> VoxBoxResult<Vec<Complex<T>>> {
            let mut work: Vec<Complex<T>> = Vec::new();
            let mut other = self.to_vec();
            other.find_roots_mut(&mut work[..])?;
            while other.last().map_or(false, |z| is_zero(z)) {
                other.pop();
            }
            Ok(other)
        }

        /// polynomial.rs:92-152: the roots (reference order) are written back into `self`, the rest zeroed.  `work` is not
        /// needed on the device.
        fn find_roots_mut<'b>(&'b mut self, _work: &'b mut [Complex<T>]) -> VoxBoxResult<()> {
            with_context(|ctx| {
                let dev = DeviceBuf::from_host(ctx, self)?;
                let out = DeviceBuf::<Complex<T>>::new(ctx, self.len())?;
                let st = DeviceBuf::<u8>::new(ctx, 1)?;
                ctx.check(unsafe {
                    ffi::vbx_find_roots(ctx.raw(), dev.ptr, T::DTYPE, 1, self.len() as i32, out.ptr, st.ptr as *mut u8)
                })?;
                match st.to_host(ctx, 0u8)?[0] as c_int {
                    ffi::VBX_OK => {}
                    ffi::VBX_ERR_POLYNOMIAL if self.degree() < 1 => {
                        return Err(VoxBoxError::Polynomial("Zero degree polynomial: no roots to be found.")) // polynomial.rs:95
                    }
                    other => ctx.check(other)?,
                }
                out.read_into(ctx, self)
            })
        }

        /// polynomial.rs:198-204: returns the remainder.
        fn div_polynomial(&mut self, other: Complex<T>) -> VoxBoxResult<Vec<Complex<T>>> {
            let mut rem = self.to_vec();
            div_impl(self, other, &mut rem[..])?;
            Ok(rem)
        }

        /// polynomial.rs:155-195: `self /= (x + other)`, remainder in `rem[0]`.
        fn div_polynomial_mut(&'a mut self, other: Complex<T>, rem: &'a mut [Complex<T>]) -> VoxBoxResult<()> {
            div_impl(self, other, rem)
        }
    }

    fn div_impl<T: Elem>(me: &mut [Complex<T>], other: Complex<T>, rem: &mut [Complex<T>]) -> VoxBoxResult<()> {
        assert!(rem.len() >= me.len());
        with_context(|ctx| {
            let dev = DeviceBuf::from_host(ctx, me)?;
            let doth = DeviceBuf::from_host(ctx, &[other])?;
            let drem = DeviceBuf::<Complex<T>>::new(ctx, me.len())?;
            let st = DeviceBuf::<u8>::new(ctx, 1)?;
            ctx.check(unsafe {
                ffi::vbx_div_polynomial(ctx.raw(), dev.ptr, T::DTYPE, 1, me.len() as i32, doth.ptr, 0, drem.ptr, st.ptr as *mut u8)
            })?;
            match st.to_host(ctx, 0u8)?[0] as c_int {
                ffi::VBX_OK => {}
                ffi::VBX_ERR_POLYNOMIAL => return Err(VoxBoxError::Polynomial("Tried to divide by zero")), // polynomial.rs:192
                other => ctx.check(other)?,
            }
            dev.read_into(ctx, me)?;
            let n = me.len();
            drem.read_into(ctx, &mut rem[..n])
        })
    }
}

// =================================================================================================
// waves.rs
// =================================================================================================
pub mod waves {
    use super::*;

    /// waves.rs:10-12
    pub trait RMS<S> {
        fn rms(&self) -> S;
    }
    /// waves.rs:25-27
    pub trait Amplitude<S> {
        fn amplitude(self) -> S;
    }
    /// waves.rs:39-41
    pub trait MaxAmplitude<S> {
        fn max_amplitude(&self) -> S;
    }
    /// waves.rs:61-66
    pub trait Normalize<S> {
        fn normalize_with_max(&mut self, max: Option<S>);
        fn normalize(&mut self) {
            self.normalize_with_max(None);
        }
    }
    /// waves.rs:82-84
    pub trait Filter {
        fn preemphasis(&mut self, factor: f64) -> &mut Self;
    }

    fn rows_op<S: Elem>(x: &[S], max: bool) -> S {
        with_context(|ctx| {
            let run = || -> VoxBoxResult<S> {
                let dev = DeviceBuf::from_host(ctx, x)?;
                let out = DeviceBuf::<S>::new(ctx, 1)?;
                let st = unsafe {
                    if max { ffi::vbx_max_amplitude(ctx.raw(), dev.ptr, S::DTYPE, 1, x.len() as i32, x.len() as i64, out.ptr) }
                    else { ffi::vbx_rms(ctx.raw(), dev.ptr, S::DTYPE, 1, x.len() as i32, x.len() as i64, out.ptr) }
                };
                ctx.check(st)?;
                Ok(out.to_host(ctx, S::default())?[0])
            };
            run().expect("rms / max_amplitude")
        })
    }

    impl<S: Elem> RMS<S> for [S] {
        fn rms(&self) -> S { rows_op(self, false) }
    }

    impl<S: Elem> Amplitude<S> for S {
        fn amplitude(self) -> S {
            if self < S::default() { S::from_f64(-self.to_f64()) } else { self }
        }
    }

    impl<S: Elem> MaxAmplitude<S> for [S] {
        fn max_amplitude(&self) -> S {
            assert!(!self.is_empty());
            rows_op(self, true)
        }
    }

    impl<S: Elem> Normalize<S> for [S] {
        /// waves.rs:67-76: `x *= 1 / max` (no zero guard), `max` defaulting to `max_amplitude()`.
        fn normalize_with_max(&mut self, max: Option<S>) {
            with_context(|ctx| {
                let run = |me: &mut [S]| -> VoxBoxResult<()> {
                    let dev = DeviceBuf::from_host(ctx, me)?;
                    let dmax = match max {
                        Some(m) => Some(DeviceBuf::from_host(ctx, &[m])?),
                        None => None,
                    };
                    let mp = dmax.as_ref().map_or(ptr::null(), |b| b.ptr as *const c_void);
                    ctx.check(unsafe { ffi::vbx_normalize(ctx.raw(), dev.ptr, S::DTYPE, 1, me.len() as i32, me.len() as i64, mp) })?;
                    dev.read_into(ctx, me)
                };
                run(self).expect("normalize_with_max")
            })
        }
    }

    impl<S: Elem> Filter for [S] {
        /// waves.rs:86-95: `y[n-1] = x[n-1]`, `y[i] = x[i] + 2 pi factor y[i+1]` (anti-causal and additive, as written).
        fn preemphasis(&mut self, factor: f64) -> &mut [S] {
            with_context(|ctx| {
                let run = |me: &mut [S]| -> VoxBoxResult<()> {
                    let dev = DeviceBuf::from_host(ctx, me)?;
                    ctx.check(unsafe { ffi::vbx_preemphasis(ctx.raw(), dev.ptr, S::DTYPE, 1, me.len() as i32, me.len() as i64, factor) })?;
                    dev.read_into(ctx, me)
                };
                run(&mut *self).expect("preemphasis")
            });
            self
        }
    }
}

// =================================================================================================
// batched drivers (no reference analogue): the intended way to use the device
// =================================================================================================
pub mod batch {
    use super::spectrum::Resonance;
    use super::*;

    /// A batch of equally long utterances resident in HBM: one call == all frames of all utterances.
    pub struct Batch<'a> {
        ctx: &'a Context,
        audio: DeviceBuf<f32>,
        pub n_utterances: usize,
        pub samples_per_utterance: usize,
    }

    impl<'a> Batch<'a> {
        pub fn upload(ctx: &'a Context, audio: &[f32], n_utterances: usize) -> VoxBoxResult<Batch<'a>> {
            if n_utterances == 0 || audio.len() % n_utterances != 0 {
                return Err(VoxBoxError::BadArg("audio.len() must be a positive multiple of n_utterances".into()));
            }
            Ok(Batch { ctx, audio: DeviceBuf::from_host(ctx, audio)?, n_utterances, samples_per_utterance: audio.len() / n_utterances })
        }
        /// `Windower::{hanning,rectangle}(.., bin, hop)` over every utterance as one strided view.
        pub fn frames(&self, bin: usize, hop: usize, window: i32) -> ffi::vbx_frames {
            let j = if self.samples_per_utterance < bin { 0 } else { (self.samples_per_utterance - bin) / hop + 1 };
            ffi::vbx_frames {
                base: self.audio.ptr,
                n_frames: (j * self.n_utterances) as i64,
                frame_stride: hop as i64,
                frames_per_segment: j as i64,
                segment_stride: self.samples_per_utterance as i64,
                frame_len: bin as i32,
                dtype: ffi::VBX_F32,
                window,
                sample_step: 0,
            }
        }
        /// Hann -> autocorrelate(p+1) -> lpc(p) for every frame: ([F][p+1] r, [F][p+1] lpc) as fp32.
        pub fn lpc(&self, bin: usize, hop: usize, p: usize) -> VoxBoxResult<(Vec<f32>, Vec<f32>)> {
            let fr = self.frames(bin, hop, ffi::VBX_WINDOW_HANN_SYMMETRIC);
            let n = fr.n_frames as usize * (p + 1);
            let (r, ac) = (DeviceBuf::<f32>::new(self.ctx, n)?, DeviceBuf::<f32>::new(self.ctx, n)?);
            self.ctx.check(unsafe { ffi::vbx_lpc(self.ctx.raw(), &fr, p as i32, r.ptr, ac.ptr, ptr::null_mut(), ffi::VBX_F32) })?;
            Ok((r.to_host(self.ctx, 0f32)?, ac.to_host(self.ctx, 0f32)?))
        }
        /// The north-star chain (Hann -> autocorrelate -> Levinson -> Laguerre roots -> resonances -> McCandless) for every
        /// frame; `estimates` = [n_utterances][k] start state (in/out); returns the [F][k] tracks.
        pub fn formants(&self, bin: usize, hop: usize, sample_rate: f64, p: usize, estimates: &mut [Resonance<f32>]) -> VoxBoxResult<Vec<Resonance<f32>>> {
            let fr = self.frames(bin, hop, ffi::VBX_WINDOW_HANN_SYMMETRIC);
            let k = estimates.len() / self.n_utterances;
            let est = DeviceBuf::from_host(self.ctx, estimates)?;
            let trk = DeviceBuf::<Resonance<f32>>::new(self.ctx, fr.n_frames as usize * k)?;
            self.ctx.check(unsafe {
                ffi::vbx_find_formants(self.ctx.raw(), &fr, sample_rate, p as i32, ffi::VBX_LPC_AUTOCORR, est.ptr, k as i32, trk.ptr,
                                       ptr::null_mut(), ptr::null_mut(), ptr::null_mut(), ffi::VBX_F32)
            })?;
            est.read_into(self.ctx, estimates)?;
            trk.to_host(self.ctx, Resonance::default())
        }
    }

    /// The whole box behind one handle (`vbx_multi`): host slices in, host slices out, utterances sharded over the GPUs,
    /// no collective (SURVEY 8e).
    pub struct Multi {
        raw: *mut ffi::vbx_multi,
    }

    impl Multi {
        /// `n_devices = 0`: every visible device.
        pub fn new(n_devices: i32) -> VoxBoxResult<Multi> {
            let mut raw = ptr::null_mut();
            let st = unsafe { ffi::vbx_multi_create(n_devices, ptr::null(), &mut raw) };
            if st != ffi::VBX_OK {
                return Err(VoxBoxError::Cuda("vbx_multi_create failed: no usable CUDA device (no CPU fallback)".into()));
            }
            Ok(Multi { raw })
        }
        pub fn device_count(&self) -> i32 { unsafe { ffi::vbx_multi_device_count(self.raw) } }
        fn check(&self, st: c_int) -> VoxBoxResult<()> {
            use std::ffi::CStr;
            status_to_result(st, || unsafe { CStr::from_ptr(ffi::vbx_multi_last_error(self.raw)).to_string_lossy().into_owned() })
        }
        /// Formant tracks of `n_utterances` equally long utterances (`audio` = them back to back), sharded over the devices.
        pub fn formants(&self, audio: &[f32], n_utterances: usize, bin: usize, hop: usize, sample_rate: f64, p: usize,
                        estimates: &mut [Resonance<f32>]) -> VoxBoxResult<Vec<Resonance<f32>>> {
            if n_utterances == 0 || audio.len() % n_utterances != 0 {
                return Err(VoxBoxError::BadArg("audio.len() must be a positive multiple of n_utterances".into()));
            }
            let ns = audio.len() / n_utterances;
            let j = if ns < bin { 0 } else { (ns - bin) / hop + 1 };
            let k = estimates.len() / n_utterances;
            let fr = ffi::vbx_frames {
                base: audio.as_ptr() as *const c_void,
                n_frames: (j * n_utterances) as i64,
                frame_stride: hop as i64,
                frames_per_segment: j as i64,
                segment_stride: ns as i64,
                frame_len: bin as i32,
                dtype: ffi::VBX_F32,
                window: ffi::VBX_WINDOW_HANN_SYMMETRIC,
                sample_step: 0,
            };
            let mut tracks = vec![Resonance::<f32>::default(); j * n_utterances * k];
            self.check(unsafe {
                ffi::vbx_multi_find_formants_host(self.raw, &fr, sample_rate, p as i32, ffi::VBX_LPC_AUTOCORR,
                                                  estimates.as_mut_ptr() as *mut c_void, k as i32, tracks.as_mut_ptr() as *mut c_void,
                                                  ptr::null_mut(), ptr::null_mut(), ptr::null_mut(), ffi::VBX_F32)
            })?;
            Ok(tracks)
        }
    }

    impl Drop for Multi {
        fn drop(&mut self) {
            unsafe { ffi::vbx_multi_destroy(self.raw) };
        }
    }
}
