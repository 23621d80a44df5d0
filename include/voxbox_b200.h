/* voxbox_b200.h — C ABI of the B200-native vox_box hot path.
 *
 * Drop-in boundary for the framewise speech-analysis path of
 * andrewcsmith/vox_box.rs (Rust extension traits on slices; no FFI of its own).
 * Every entry point below names the reference interface it replaces
 * (file:line relative to the reference crate root).  One reference call
 * processes ONE frame slice; the entry points here are batched over frames
 * (a reference call == a batch of 1).  INTEGRATION.md shows the Rust
 * `extern "C"` block and trait impls a maintainer would add.
 *
 * Conventions
 *  - plain pointers and sizes only; `vbx_ctx` is opaque.
 *  - unless an entry point ends in `_host`, every data pointer is a DEVICE
 *    pointer (HBM resident, caller owned, never freed by the library) and the
 *    call is asynchronous on the context's stream: call vbx_sync() (or any
 *    `_host` entry point, which synchronises) before reading results.
 *  - `_host` twins take HOST pointers, stage through the context's scratch
 *    arena and return when the results are in the caller's buffers.
 *  - return value: vbx_status.  Calls that can fail per frame (Burg, root
 *    finding, pitch) also fill an optional `uint8_t status[F]` with the same
 *    codes; the call returns VBX_OK if it ran, and the Rust shim maps "any frame
 *    failed" to the matching `Err(VoxBoxError::..)`.
 *  - there is no CPU fallback: without a usable CUDA device vbx_ctx_create
 *    fails with VBX_ERR_CUDA.
 */
#ifndef VOXBOX_B200_H
#define VOXBOX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VBX_API __attribute__((visibility("default")))
#else
#define VBX_API
#endif

/* ---- status codes: error.rs:6-16 `VoxBoxError` ------------------------------ */
typedef enum vbx_status {
    VBX_OK = 0,
    VBX_ERR_LPC = 1,        /* VoxBoxError::LPC("Denum was <= 0.0")                 spectrum.rs:123-125 */
    VBX_ERR_PITCH = 2,      /* VoxBoxError::Pitch (where the reference panics on NaN, periodic.rs:453) */
    VBX_ERR_POLYNOMIAL = 3, /* VoxBoxError::Polynomial(..)                     polynomial.rs:95,123,192 */
    VBX_ERR_WORKSPACE = 4,  /* VoxBoxError::Workspace                                      lib.rs:46-48 */
    VBX_ERR_CUDA = 5,       /* CUDA runtime failure / no device (no reference analogue)                */
    VBX_ERR_BADARG = 6,     /* sizes for which the reference would panic (assert!/index)              */
    VBX_ERR_NOMEM = 7       /* device or pinned allocation failed                                      */
} vbx_status;

/* VBX_MULAW8 / VBX_ALAW8: one byte per sample, ITU-T G.711 mu-law / A-law (WAV format tags 7 / 6), accepted wherever
 * vbx_frames.dtype accepts VBX_I16 (never as out_dtype, nor by the entry points that take plain arrays).  A code decodes to
 * the 16-bit linear value of G.711 (the g711.c tables; Python's audioop.ulaw2lin / alaw2lin with width 2), range +-32124
 * (mu-law) / +-32256 (A-law):
 *   mu-law: u = ~b; t = ((u & 0x0F) << 3) + 0x84; t <<= (u & 0x70) >> 4; v = (u & 0x80) ? 0x84 - t : t - 0x84
 *   A-law:  a = b ^ 0x55; t = (a & 0x0F) << 4; seg = (a & 0x70) >> 4; t += seg ? 0x108 : 8; if (seg > 1) t <<= seg - 1;
 *           v = (a & 0x80) ? t : -t
 * The decode happens as the kernels load the samples; from there on a G.711 sample IS the VBX_I16 sample v (scaled by
 * 1/32767): every call on a G.711 view returns, bit for bit, what the same call returns on a VBX_I16 view of the decoded
 * samples. */
typedef enum vbx_dtype { VBX_F32 = 0, VBX_F64 = 1, VBX_I16 = 2, VBX_MULAW8 = 3, VBX_ALAW8 = 4 } vbx_dtype;

/* Window applied while a frame is loaded (the reference's callers window the
 * frame before calling the trait method):
 *  HANN_SYMMETRIC = sample::window::Windower::hanning (examples/pitch_detection.rs:23,
 *                   periodic.rs:493): 0.5(1-cos 2πφ), φ accumulated in steps of 1/(N-1);
 *  HANN_PERIODIC  = the in-line window of find_formants (lib.rs:66-70): φ = i/N;
 *  NONE           = frame is used as is (Windower::rectangle, tests/lib.rs:71). */
typedef enum vbx_window {
    VBX_WINDOW_NONE = 0,
    VBX_WINDOW_HANN_SYMMETRIC = 1,
    VBX_WINDOW_HANN_PERIODIC = 2,
    /* periodic.rs:232-252 HanningLag (`LagType for Hanning`): the Hann window's autocorrelation over the same
     * accumulated phases.  Only valid for vbx_window_table_host (vbx_pitch uses it internally), not as frames.window. */
    VBX_WINDOW_HANN_LAG = 3
} vbx_window;

/* A batch of frames as a strided view: frame f = base[f*frame_stride .. f*frame_stride + frame_len).
 * frame_stride == frame_len is a packed [F, N] tensor; frame_stride == hop < frame_len is the
 * overlapped view over contiguous audio that `Windower::{hanning,rectangle}(.., bin, hop)` iterates.
 * A batch of equally long utterances is a two-level view: with frames_per_segment = J > 0, frame
 * f = u*J + j starts at base[u*segment_stride + j*frame_stride] (n_frames must be a multiple of J);
 * frames_per_segment == 0 means one segment holds all frames.
 * dtype: VBX_F32 samples, VBX_I16 PCM scaled by 1/32767 on load (tests/lib.rs:17-19), VBX_MULAW8 / VBX_ALAW8 G.711 bytes
 * (decoded to int16 PCM on load, then exactly VBX_I16), or VBX_F64 samples (what the reference's f64 callers hold, e.g. a
 * frame they windowed themselves: use VBX_WINDOW_NONE; f64 samples run the same arithmetic through the general-purpose
 * kernels, the tuned batch kernels stage fp32 / int16 / G.711).  Strides are in samples whatever the sample size.
 *
 * Interleaved audio (sample_step): 0 and 1 mean contiguous frames, as above.  With s = sample_step > 1, sample i of frame
 * f = u*J + j is base[u*segment_stride + j*frame_stride + i*s]: a recording of C interleaved channels (L0 R0 L1 R1 ...) is
 * read in place with s = C, frame_stride = hop*C, segment_stride = 1 and one segment per channel (segment u = channel u,
 * J frames each; or frames_per_segment = 0 and base offset by the channel for one channel).  frame_stride must be a
 * multiple of s (every frame of a segment stays on its channel), sample_step < 0 and views whose extent overflows int64
 * are VBX_ERR_BADARG.
 * The rule that defines every result: let S = ((J-1)*frame_stride)/s + frame_len, the channel samples segment u spans
 * (J = frames_per_segment, or n_frames for a single-segment view, where u = 0).  Its PLANAR EQUIVALENT is the contiguous
 * array P[u][k] = base[u*segment_stride + k*s], k < S, laid out as rows of S' = S rounded up to a multiple of 64 samples
 * (P[u][k] at offset u*S' + k of a 256-byte-aligned buffer of the same dtype) and viewed with frame_stride/s, segment
 * stride S' and sample_step 1, everything else unchanged.  Every frame-view call on an interleaved view returns, bit for
 * bit, what the same call returns on its planar equivalent: every output, status and count, and the local and global peaks
 * of vbx_frame_peaks / vbx_pitch_with_peaks.  The library builds that planar copy on the device (a gather kernel,
 * interleave_gather_kernel, into a grow-only buffer of the context that nothing else uses) and runs the ordinary kernels
 * on it; a G.711 copy stays one byte per sample.  The _host twins upload the interleaved bytes once: when the segments
 * share memory (segment_stride below a segment's extent, the channels-as-segments layout) they cut the view into time
 * ranges of every segment rather than into whole segments.  The _multi_host twins shard such a view by segment as any
 * other, so an interleaved recording of C channels keeps at most C devices busy. */
typedef struct vbx_frames {
    const void* base;
    int64_t n_frames;
    int64_t frame_stride;       /* in samples */
    int64_t frames_per_segment; /* J, or 0 */
    int64_t segment_stride;     /* in samples; ignored when frames_per_segment == 0 */
    int32_t frame_len;          /* N */
    int32_t dtype;        /* vbx_dtype: VBX_F32, VBX_I16, VBX_MULAW8, VBX_ALAW8 or VBX_F64 */
    int32_t window;       /* vbx_window */
    union {
        int32_t reserved;    /* the field's former name: 0 is contiguous samples */
        int32_t sample_step; /* samples between consecutive samples of a frame: 0 or 1 contiguous, s > 1 interleaved */
    };
} vbx_frames;

/* #[repr(C)] Resonance<T> { frequency, bandwidth }  spectrum.rs:149-154 */
typedef struct vbx_resonance_f32 { float frequency, bandwidth; } vbx_resonance_f32;
typedef struct vbx_resonance_f64 { double frequency, bandwidth; } vbx_resonance_f64;
/* Pitch<T> { frequency, strength }  periodic.rs:306-310 */
typedef struct vbx_pitch_f32 { float frequency, strength; } vbx_pitch_f32;
typedef struct vbx_pitch_f64 { double frequency, strength; } vbx_pitch_f64;

/* lib.rs:26-28 */
#define VBX_MAX_RESONANCES 32
#define VBX_MAX_FORMANT_SLOTS 6 /* spectrum.rs:228 FormantSlots */
VBX_API extern const double VBX_MALE_FORMANT_ESTIMATES[4];
VBX_API extern const double VBX_FEMALE_FORMANT_ESTIMATES[4];

typedef struct vbx_ctx vbx_ctx;

/* ---- context, memory, errors ------------------------------------------------------ */
/* One context = one device + one stream + one scratch arena; not thread-safe (use one per host
 * thread / GPU).  The reference is pure functions on caller buffers (no context). */
VBX_API int vbx_ctx_create(int device, vbx_ctx** out);
VBX_API int vbx_ctx_destroy(vbx_ctx* ctx);
VBX_API int vbx_sync(vbx_ctx* ctx);
VBX_API void* vbx_ctx_stream(vbx_ctx* ctx);           /* the cudaStream_t the context launches on */
VBX_API const char* vbx_last_error(vbx_ctx* ctx);     /* message of the last failing call */
VBX_API const char* vbx_status_str(int status);       /* error.rs:25-32 description() strings */
VBX_API int vbx_version(void);
VBX_API int vbx_device_sm_count(vbx_ctx* ctx);
VBX_API int64_t vbx_kernel_launches(vbx_ctx* ctx);    /* kernels launched by this context so far */

VBX_API int vbx_malloc(vbx_ctx* ctx, size_t bytes, void** dev_out);
VBX_API int vbx_free(vbx_ctx* ctx, void* dev);
VBX_API int vbx_malloc_host(vbx_ctx* ctx, size_t bytes, void** host_out); /* pinned */
VBX_API int vbx_free_host(vbx_ctx* ctx, void* host);
VBX_API int vbx_memcpy_h2d(vbx_ctx* ctx, void* dev, const void* host, size_t bytes); /* async on ctx stream */
VBX_API int vbx_memcpy_d2h(vbx_ctx* ctx, void* host, const void* dev, size_t bytes); /* async on ctx stream */
VBX_API int vbx_memcpy_d2d(vbx_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
VBX_API int vbx_memset(vbx_ctx* ctx, void* dev, int value, size_t bytes);

/* Device timing on the context's stream (CUDA events), for callers without a CUDA binding. */
VBX_API int vbx_timer_start(vbx_ctx* ctx);
VBX_API int vbx_timer_stop_ms(vbx_ctx* ctx, float* ms_out); /* synchronises */

/* Per-kernel device timing for roofline reports: between begin and end an event is recorded after every kernel the
 * context launches; a kernel's time is the gap to the previous event on the stream (launches are back to back, so the
 * few memsets / small copies in between are attributed to the kernel that follows them).  end synchronises. */
VBX_API int vbx_profile_begin(vbx_ctx* ctx);
VBX_API int vbx_profile_end(vbx_ctx* ctx);
VBX_API int vbx_profile_count(vbx_ctx* ctx);
VBX_API int vbx_profile_entry(vbx_ctx* ctx, int index, char* name_out, int name_len, double* ms_total, int64_t* launches);

/* Executed-work counters of the data-dependent kernels, accumulated between vbx_profile_begin and vbx_profile_end (zero
 * outside): out[0] = Horner coefficient steps and out[1] = Laguerre rounds executed by lpc_roots_pair_kernel, summed over
 * lanes (a warp runs every round at its largest live degree, so idle lanes' steps are counted: executed, not useful, work);
 * out[2] = term-loop iterations and out[3] = interpolant evaluations executed by pitch_refine8q_kernel, summed over lanes;
 * out[4] = frames the pair kernel handed to the f64 fix-up launch (a Laguerre solve hit the 20-iteration cap unconverged).
 * bench.py turns them into executed flop for the roofline fractions of those kernels.  Synchronises.  n <= 8. */
VBX_API int vbx_profile_counters(vbx_ctx* ctx, uint64_t* out, int32_t n);

/* Measured pipe peaks of this device (dependent-free FMA loops on every SM), used as roofline
 * denominators for the FP32/FP64-bound kernels.  Values in TFLOP/s (2 flop per FMA). */
VBX_API int vbx_measure_peaks(vbx_ctx* ctx, double* fp32_tflops, double* fp64_tflops);

/* Window table exactly as the reference's callers compute it, in f64 on the host
 * (sample::window::Window phase accumulation; lib.rs:66-70).  out: n doubles (host). */
VBX_API int vbx_window_table_host(int window, int32_t n, double* out);

/* ---- periodic.rs:265-289  Autocorrelate::{autocorrelate_mut, autocorrelate} ------------ */
/* r_out[f][lag] = x[0] + Σ_{i=1}^{N-lag-1} x[i]·x[i+lag] on the (windowed) frame, lag < n_lags <= N,
 * accumulated in fp64.  r_out: [F][n_lags] of out_dtype (VBX_F32|VBX_F64). */
VBX_API int vbx_autocorrelate(vbx_ctx* ctx, const vbx_frames* frames, int32_t n_lags, void* r_out, int32_t out_dtype);
VBX_API int vbx_autocorrelate_host(vbx_ctx* ctx, const vbx_frames* frames, int32_t n_lags, void* r_out,
                                   int32_t out_dtype);

/* periodic.rs:291-304  `impl Autocorrelate for VecDeque<T>` (streaming callers keep the last n samples in a ring):
 * rings: [n_rings][capacity] of dtype (VBX_F32|VBX_F64); the logical sequence of ring b is x[i] = ring[(heads[b] + i) mod
 * capacity], i < n (heads == NULL: 0).  No window is applied (the caller's samples are used as they are).
 * r_out: [n_rings][n_lags], same fold as vbx_autocorrelate (seeded with x[0]), fp64 accumulation. */
VBX_API int vbx_autocorrelate_ring(vbx_ctx* ctx, const void* rings, int32_t dtype, int64_t n_rings, int64_t capacity,
                                   const int64_t* heads, int32_t n, int32_t n_lags, void* r_out, int32_t out_dtype);

/* ---- spectrum.rs:50-92  LPC::{lpc_mut, lpc} (Levinson–Durbin) + LPCSolver ---------------- */
/* r: [F][r_stride] of r_dtype with r_stride >= p+1.  ac_out: [F][p+1] (ac[0] = 1, error-filter
 * sign), kc_out: [F][p] reflection coefficients (may be NULL).  fp64 arithmetic. */
VBX_API int vbx_lpc_levinson(vbx_ctx* ctx, const void* r, int32_t r_dtype, int64_t n_frames, int32_t r_stride,
                             int32_t p, void* ac_out, void* kc_out, int32_t out_dtype);

/* Fused north-star chain (config C2): window → autocorrelate(p+1) → lpc(p) in one kernel.
 * Any of r_out [F][p+1], ac_out [F][p+1], kc_out [F][p] may be NULL. */
VBX_API int vbx_lpc(vbx_ctx* ctx, const vbx_frames* frames, int32_t p, void* r_out, void* ac_out, void* kc_out,
                    int32_t out_dtype);
VBX_API int vbx_lpc_host(vbx_ctx* ctx, const vbx_frames* frames, int32_t p, void* r_out, void* ac_out, void* kc_out,
                         int32_t out_dtype);

/* ---- spectrum.rs:94-146  LPC::{lpc_praat_mut, lpc_praat} (Burg, Praat form) ---------------------- */
/* coeffs_out: [F][p] (no leading 1, sign as the reference returns them).  status_out[f] (optional) =
 * VBX_ERR_LPC where the reference returns Err(LPC("Denum was <= 0.0")); such frames get NaN coefficients. */
VBX_API int vbx_lpc_burg(vbx_ctx* ctx, const vbx_frames* frames, int32_t p, void* coeffs_out, uint8_t* status_out,
                         int32_t out_dtype);

/* ---- polynomial.rs:10-205  Polynomial on [Complex<T>] ------------------------------------------------ */
/* Complex arrays are interleaved (re, im) of `dtype` (VBX_F32|VBX_F64), `len` coefficients per polynomial in
 * ascending powers, len <= 64.  One polynomial per batch entry. */
/* find_roots_mut (:92-152): roots_out[f][0..len) = the buffer after the reference's write-back (roots in the
 * reference's order, then zeros).  status_out[f] = VBX_ERR_POLYNOMIAL for "Zero degree polynomial" /
 * "Failed to find roots" (roots_out then holds the input), VBX_ERR_BADARG where the reference panics (off_low > 0). */
VBX_API int vbx_find_roots(vbx_ctx* ctx, const void* coeffs, int32_t dtype, int64_t n_polys, int32_t len, void* roots_out,
                           uint8_t* status_out);
VBX_API int64_t vbx_find_roots_work_size(int64_t len); /* polynomial.rs:75-77 (the library needs no caller workspace) */
/* laguerre (:34-72): z_out[f] = one Laguerre solve from `start`, n = len-1. */
VBX_API int vbx_laguerre(vbx_ctx* ctx, const void* coeffs, int32_t dtype, int64_t n_polys, int32_t len, double start_re,
                         double start_im, void* z_out);
/* div_polynomial_mut (:155-195): coeffs_inout /= (x + other); remainder to rem_out (optional, len entries).
 * `other`: one complex value, or one per polynomial if other_per_poly != 0.  other == 0 -> VBX_ERR_POLYNOMIAL. */
VBX_API int vbx_div_polynomial(vbx_ctx* ctx, void* coeffs_inout, int32_t dtype, int64_t n_polys, int32_t len,
                               const void* other, int32_t other_per_poly, void* rem_out, uint8_t* status_out);

/* ---- spectrum.rs:149-210  Resonance::from_root, ToResonance::to_resonance ----------------------------------- */
/* roots: [F][n_roots] complex.  res_out: [F][res_slots] resonance pairs of out_dtype, ascending frequency,
 * zero padded; nres_out[f] (optional) = count.  strict_im = 0: to_resonance (roots with im >= 0);
 * strict_im = 1: find_formants' filter (im > 0, lib.rs:95).  50 Hz guard band as the reference. */
VBX_API int vbx_roots_to_resonances(vbx_ctx* ctx, const void* roots, int32_t dtype, int64_t n_frames, int32_t n_roots,
                                    double sample_rate, int32_t strict_im, void* res_out, int32_t res_slots,
                                    int32_t* nres_out, int32_t out_dtype);

/* LPC coefficients -> roots -> resonances in one kernel (the K3+K4 stage of find_formants).
 * lpc: [F][lpc_stride], either [1, a1..ap] (lpc_has_leading_one = 1, Levinson's `ac`) or [a1..ap] (Burg).
 * precision: 0 = fp32 Laguerre/deflation + fp64 Newton polish on the original polynomial (default), 1 = fp64
 * Laguerre/deflation as the reference's f64 instantiation, -1 = library default (0).
 * roots_out (optional): [F][p] complex roots in find_roots order; without it the fp32 path divides conjugate pairs
 * out of the (real) polynomial instead of one root at a time — same resonances, no root list.  status_in
 * (optional): frames whose LPC stage failed are passed through with zero resonances. */
VBX_API int vbx_lpc_to_resonances(vbx_ctx* ctx, const void* lpc, int32_t lpc_dtype, int64_t n_frames, int32_t lpc_stride,
                                  int32_t p, int32_t lpc_has_leading_one, double sample_rate, int32_t strict_im,
                                  const uint8_t* status_in, void* res_out, int32_t res_slots, int32_t* nres_out,
                                  void* roots_out, uint8_t* status_out, int32_t out_dtype, int32_t precision);

/* ---- spectrum.rs:216-369  EstimateFormants::estimate_formants + FormantExtractor ------------------------------ */
/* Runs the McCandless step over frames, sequentially inside each segment (utterance), segments in parallel.
 * resonances: [n_segments*frames_per_segment][res_slots] pairs of res_dtype; the step sees the first
 * n_resonances entries of each frame (entries beyond res_slots read as (0,0): find_formants passes 32 zero-padded
 * slots, lib.rs:114).  est_inout: [n_segments][n_estimates] pairs of dtype: starting estimates in, final state out.
 * tracks_out (optional): [F][n_estimates] = the estimates after each frame (FormantExtractor::next).
 * status_in (optional): frames with a non-zero status leave the estimates untouched. */
VBX_API int vbx_estimate_formants(vbx_ctx* ctx, const void* resonances, int32_t res_dtype, int32_t res_slots,
                                  int32_t n_resonances, int64_t n_segments, int64_t frames_per_segment,
                                  const uint8_t* status_in, void* est_inout, int32_t n_estimates, void* tracks_out,
                                  int32_t dtype);

/* ---- lib.rs:26-116  find_formants (+ work-size helpers) -------------------------------------------------------- */
typedef enum vbx_lpc_method {
    VBX_LPC_BURG = 0,    /* lpc_praat_mut on the windowed frame: the reference's find_formants (use HANN_PERIODIC) */
    VBX_LPC_AUTOCORR = 1 /* autocorrelate(p+1) -> lpc(p): the north-star "LPC-12 + formant" chain (HANN_SYMMETRIC) */
} vbx_lpc_method;
VBX_API int64_t vbx_find_formants_real_work_size(int64_t buf_len, int64_t n_coeffs); /* lib.rs:30-32 */
VBX_API int64_t vbx_find_formants_complex_work_size(int64_t n_coeffs);               /* lib.rs:34-36 */
/* One call = find_formants applied to every frame of the view, in order, inside each segment (utterance):
 * window -> LPC -> roots -> resonances (im > 0, sorted, zero padded to 32) -> estimate_formants.
 * resample_ratio is 1 here; vbx_find_formants_resampled covers lib.rs:57-61.  With VBX_LPC_BURG the samples may also be
 * VBX_F64 (so may vbx_lpc_burg's).
 * est_inout [n_segments][n_formants] pairs (state in/out); tracks_out [F][n_formants] (optional);
 * resonances_out [F][32] pairs (optional); nres_out [F] (optional); status_out [F] (optional):
 * VBX_ERR_LPC frames leave the state untouched, exactly as the reference returns Err before the tracker. */
VBX_API int vbx_find_formants(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, int32_t n_coeffs,
                              int32_t lpc_method, void* est_inout, int32_t n_formants, void* tracks_out,
                              void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype);
VBX_API int vbx_find_formants_host(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, int32_t n_coeffs,
                                   int32_t lpc_method, void* est_inout, int32_t n_formants, void* tracks_out,
                                   void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype);

/* ---- periodic.rs:356-456  Pitched::pitch::<Hanning> (+ LocalMaxima :362-375, Pitch :306-318) --------------------- */
/* Boersma autocorrelation pitch candidates for every frame of the view (the frame is windowed by frames->window as
 * the reference's callers do, Windower::hanning => HANN_SYMMETRIC; the lag window is HanningLag, the only LagType).
 * The reference ignores its local_peak / global_peak arguments (periodic.rs:396), so they are not parameters (the opt-in
 * vbx_pitch_with_peaks below honours them).
 * cand_out: [F][max_candidates] (frequency, strength) pairs of out_dtype, sorted by strength descending exactly as
 * the returned Vec (stable; the unvoiced candidate {0, threshold} is always part of it), zero padded;
 * n_cand_out[f] (optional) = length of the reference's Vec (may exceed max_candidates: the list is truncated);
 * status_out[f] (optional) = VBX_ERR_PITCH where a strength is NaN (the reference panics in its sort) — such frames
 * return their candidates unsorted.  Everything runs in fp64: the sweep over all frame_len lags and the refinement.
 * 2 <= frame_len <= 16384 (Praat's three periods of the pitch floor: 11 520 samples for 50 Hz at 192 kHz); other lengths
 * are VBX_ERR_BADARG. */
VBX_API int vbx_pitch(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold, double min_hz,
                      double max_hz, int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out,
                      int32_t out_dtype);
VBX_API int vbx_pitch_host(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold, double min_hz,
                           double max_hz, int32_t max_candidates, void* cand_out, int32_t* n_cand_out,
                           uint8_t* status_out, int32_t out_dtype);
/* Opt-in extension: the reference's local_peak / global_peak honoured (periodic.rs:357 takes them, :396 ignores them).  In
 * Boersma (1993), the algorithm vbx_pitch implements, they make a quiet frame unvoiced: every frame is normalised (periodic.rs:404),
 * so without them a faint periodic component scores as high as loud speech.
 *  - local peak of frame f: max |x| over its frame_len samples as loaded (VBX_I16 and decoded G.711 scaled by 1/32767), before
 *    frames->window.
 *    NaN samples are ignored (a NaN never wins the max, as in max_amplitude, waves.rs:45-58); an all-NaN frame has peak 0.
 *  - global peak of segment u: the same max over every sample its frames span, [u*segment_stride, u*segment_stride +
 *    (J-1)*frame_stride + frame_len) (with hop > frame_len this includes the samples between frames); for a single-segment view,
 *    the whole extent of the view.
 *  - unvoiced strength, a = threshold, b = silence_threshold: ratio = min(local / global, 1), ratio = 0 where global <= 0 or is
 *    NaN; b > 0: R_f = a + max(0, 2 - ratio * (1 + a) / b) (Boersma 1993; Praat's voiceless strength); b == 0: R_f = a, i.e.
 *    exactly vbx_pitch (no peaks are read or computed); b < 0: VBX_ERR_BADARG.  A NaN ratio (a NaN local peak) gives R_f = a.
 * The candidate list is vbx_pitch's with the unvoiced entry's strength replaced by R_f, placed by the same stable descending
 * sort before truncation to max_candidates: it still goes after voiced candidates of equal strength, n_cand_out is unchanged,
 * and VBX_ERR_PITCH frames stay unsorted.  Praat's subtraction of the local mean and its centre-only local-peak region are not
 * implemented.
 * local_peaks [F] / global_peaks [n_segments] (device pointers for vbx_pitch_with_peaks, host pointers for the _host twins) may
 * each be NULL = computed as above from the view.  The reference takes them per call: a caller that analyses one recording over
 * several calls passes the recording-wide global peak.  The _host and _multi_host twins equal the device call bit for bit. */
VBX_API int vbx_frame_peaks(vbx_ctx* ctx, const vbx_frames* frames, double* local_out /* [F] or NULL */,
                            double* global_out /* [n_segments] or NULL */);
VBX_API int vbx_pitch_with_peaks(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold,
                                 double silence_threshold, const double* local_peaks /* [F] or NULL = computed */,
                                 const double* global_peaks /* [n_segments] or NULL = computed */, double min_hz,
                                 double max_hz, int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out,
                                 int32_t out_dtype);
VBX_API int vbx_pitch_with_peaks_host(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold,
                                      double silence_threshold, const double* local_peaks, const double* global_peaks,
                                      double min_hz, double max_hz, int32_t max_candidates, void* cand_out, int32_t* n_cand_out,
                                      uint8_t* status_out, int32_t out_dtype);
/* periodic.rs:403-408: the lag function the candidates are read from (`self_lag`: autocorrelate(N) of the windowed frame,
 * normalize(), divided by the HanningLag window) for every frame of the view: lag_out [F][frame_len] f64 (device).  The reference
 * zero-extends it to 2N (:411) before interpolating. */
VBX_API int vbx_pitch_lag_function(vbx_ctx* ctx, const vbx_frames* frames, double* lag_out);
/* periodic.rs:320-354 PitchExtractor::next: out[f] = candidates[f][0] (arg-max; the cost fields are unused). */
VBX_API int vbx_pitch_extract(vbx_ctx* ctx, const void* cand, int32_t dtype, int64_t n_frames, int32_t max_candidates,
                              void* out);
/* Opt-in extension (periodic.rs:320-335 declares `PitchExtractor::new(candidates, voiced_unvoiced_cost, voicing_threshold)` and
 * :394-395 documents the intent, the reference implements arg-max): Boersma's Viterbi path over the candidate lists of vbx_pitch,
 * sequential inside each segment (utterance).  Maximises sum(local) - sum(transition) with local = strength (- octave_cost *
 * log2(ceiling_hz / f) for voiced candidates) and transition = 0 (both unvoiced), voiced_unvoiced_cost (one voiced) or
 * octave_jump_cost * |log2(f1 / f2)| (both voiced).  All three costs 0 reproduces vbx_pitch_extract.  Only the first
 * min(n_cand[f], max_candidates, 32) candidates of a frame take part (n_cand NULL: max_candidates).
 * path_out [F] pitch pairs of dtype and/or index_out [F] chosen candidate index. */
VBX_API int vbx_pitch_viterbi(vbx_ctx* ctx, const void* cand, int32_t dtype, const int32_t* n_cand, int64_t n_segments,
                              int64_t frames_per_segment, int32_t max_candidates, double voiced_unvoiced_cost,
                              double octave_jump_cost, double octave_cost, double ceiling_hz, void* path_out, int32_t* index_out);
/* periodic.rs:29-87 interpolate_sinc(y, offset, nx, x, max_depth), batched: y [n_series][y_len] f64,
 * x [n_series][n_points] f64 -> out [n_series][n_points].  Indices the reference would panic on give NaN. */
VBX_API int vbx_interpolate_sinc(vbx_ctx* ctx, const double* y, int64_t n_series, int64_t y_len, int64_t offset,
                                 int64_t nx, const double* x, int64_t n_points, int64_t max_depth, double* out);
/* periodic.rs:192-230 improve_extremum (+ brent_maximize :103-188), batched like vbx_interpolate_sinc.
 * interpolation: 0 = Interpolation::None, 1 = Parabolic, 2 = Sinc(sinc_depth). */
VBX_API int vbx_improve_extremum(vbx_ctx* ctx, const double* y, int64_t n_series, int64_t y_len, int64_t offset,
                                 int64_t nx, const double* ixmid, int64_t n_points, int32_t interpolation,
                                 int64_t sinc_depth, int32_t is_max, double* xmid_out, double* ymid_out);

/* ---- spectrum.rs:371-441  MFCC::mfcc, hz_to_mel, mel_to_hz, dct, dct_mut ------------------------------------------ */
/* mfcc(num_coeffs, (freq_lo, freq_hi), sample_rate) on every (windowed) frame.  The reference has ONE parameter
 * `num_coeffs` that is both the number of mel bands and the number of DCT rows it returns (spectrum.rs:410-414,437-439);
 * n_keep <= num_coeffs keeps only the first n_keep DCT rows ("13 coefficients from 40 bands" = num_coeffs 40, n_keep 13;
 * n_keep == num_coeffs is the drop-in).  out: [F][n_keep]; energies_out (optional): [F][num_coeffs] log-energies before
 * the DCT.  VBX_ERR_BADARG where the reference panics (a filter-bank bin beyond the spectrum / decreasing bins).
 * The FFT (rustfft's unnormalised forward DFT) runs in fp64 by default — vbx_mfcc_set_fft_precision(ctx, VBX_F32)
 * selects an fp32 transform (faster, ~1e-6 relative error on the band sums, which can exceed the 1e-5 bound on quiet
 * frames whose band sums sit near the log10 clamp); band sums, log10 and DCT are always fp64. */
VBX_API int vbx_mfcc(vbx_ctx* ctx, const vbx_frames* frames, int32_t num_coeffs, int32_t n_keep, double freq_lo,
                     double freq_hi, double sample_rate, void* out, void* energies_out, int32_t out_dtype);
VBX_API int vbx_mfcc_host(vbx_ctx* ctx, const vbx_frames* frames, int32_t num_coeffs, int32_t n_keep, double freq_lo,
                          double freq_hi, double sample_rate, void* out, int32_t out_dtype);
VBX_API int vbx_mfcc_set_fft_precision(vbx_ctx* ctx, int32_t dtype); /* VBX_F64 (default) or VBX_F32 */
VBX_API double vbx_hz_to_mel(double hz);  /* spectrum.rs:375-377 (host) */
VBX_API double vbx_mel_to_hz(double mel); /* spectrum.rs:379-381 (host) */
/* dct / dct_mut (spectrum.rs:384-398): coeffs[s][k] = 2 Σ_m signal[s][m] cos(πk(2m+1)/(2n)), [n_signals][n] of dtype. */
VBX_API int vbx_dct(vbx_ctx* ctx, const void* signal, int32_t dtype, int64_t n_signals, int32_t n, void* coeffs);

/* ---- waves.rs:10-96  RMS, MaxAmplitude, Normalize, Filter::preemphasis ----------------------------------------------- */
/* Signals are the rows of a [n_signals][stride] device array of dtype (VBX_F32|VBX_F64), stride >= n; arithmetic in
 * fp64.  out: [n_signals] of dtype. */
VBX_API int vbx_rms(vbx_ctx* ctx, const void* x, int32_t dtype, int64_t n_signals, int32_t n, int64_t stride, void* out);
VBX_API int vbx_max_amplitude(vbx_ctx* ctx, const void* x, int32_t dtype, int64_t n_signals, int32_t n, int64_t stride,
                              void* out);
/* normalize_with_max: x *= 1/max in place; maxes: [n_signals] of dtype, or NULL = normalize() (max_amplitude of the row). */
VBX_API int vbx_normalize(vbx_ctx* ctx, void* x_inout, int32_t dtype, int64_t n_signals, int32_t n, int64_t stride,
                          const void* maxes);
/* preemphasis(factor): y[n-1] = x[n-1], y[i] = x[i] + 2π·factor·y[i+1] in place (anti-causal, additive, as written). */
VBX_API int vbx_preemphasis(vbx_ctx* ctx, void* x_inout, int32_t dtype, int64_t n_signals, int32_t n, int64_t stride,
                            double factor);

/* ---- lib.rs:40-116 find_formants with resample_ratio != 1 (lib.rs:57-61: sample::interpolate::Linear +
 * Converter::scale_sample_hz) ---------------------------------------------------------------------------------------- */
/* Every frame of the view (VBX_F32, VBX_I16, G.711 or VBX_F64 samples, frames->window = VBX_WINDOW_NONE) is resampled linearly to
 * ceil(resample_ratio * frame_len) f64 samples, then windowed with the periodic Hann of that length and run through Burg ->
 * roots -> resonances -> McCandless exactly as vbx_find_formants(.., VBX_LPC_BURG, ..).  sample_rate is passed to
 * Resonance::from_root unchanged, as the reference does (callers pass the resampled rate).  The reference analyses its whole
 * `resampled_buf`; here the buffer length equals the resampled length (what tests/lib.rs:31-32 passes).  Device pointers. */
VBX_API int vbx_find_formants_resampled(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double resample_ratio,
                                        int32_t n_coeffs, void* est_inout, int32_t n_formants, void* tracks_out,
                                        void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype);

/* The same call with the reference's literal buffer semantics (lib.rs:54,62-75; SURVEY A.10): find_formants windows and analyses
 * its WHOLE `resampled_buf`, not just the first resampled_len = ceil(resample_ratio * frame_len) entries it fills.  With
 * resampled_buf_len > resampled_len (tests/lib.rs:59,66: buf.len() = 1024, resampled_buf.len() = 2878) every frame is the resampled
 * (or, for ratio 1, copied) samples followed by the buffer's untouched tail — zeros, as in the reference's tests — the periodic
 * Hann runs at phase idx / resampled_len over the whole buffer and Burg sees resampled_buf_len samples.  resampled_buf_len = 0
 * means resampled_len (vbx_find_formants_resampled); a value below resampled_len is VBX_ERR_BADARG (the reference's assert!). */
VBX_API int vbx_find_formants_buffered(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double resample_ratio,
                                       int64_t resampled_buf_len, int32_t n_coeffs, void* est_inout, int32_t n_formants,
                                       void* tracks_out, void* resonances_out, int32_t* nres_out, uint8_t* status_out,
                                       int32_t dtype);

/* ---- the whole box behind one handle (SURVEY 8e: utterance sharding, no collective, host-side gather) ---------------------------
 * The reference is single-threaded CPU code; its callers loop over utterances.  vbx_multi owns one worker thread + one vbx_ctx per
 * device; a `_multi_host` call splits the caller's view into contiguous ranges of segments (utterances; vbx_multi_partition's
 * rule) — or of frames when the view is a single segment and the path is stateless — runs the ordinary `_host` pipeline of every
 * range on its device concurrently, and returns when all results are in the caller's (single) host buffers at their rows: the
 * host-side gather.  Workers bind to the CPUs local to their GPU (sysfs local_cpulist; VBX_MULTI_NO_BIND=1 disables).  No torch,
 * NCCL or MPI is involved.  Arguments are those of the single-device `_host` twin. */
typedef struct vbx_multi vbx_multi;
VBX_API int vbx_multi_create(int32_t n_devices /* 0 = all visible */, const int32_t* devices /* NULL = 0..n-1 */, vbx_multi** out);
VBX_API int vbx_multi_destroy(vbx_multi* m);
VBX_API int32_t vbx_multi_device_count(vbx_multi* m);
VBX_API vbx_ctx* vbx_multi_ctx(vbx_multi* m, int32_t index);   /* device `index`'s context (owned by the handle) */
VBX_API const char* vbx_multi_last_error(vbx_multi* m);
VBX_API int64_t vbx_multi_kernel_launches(vbx_multi* m);       /* kernels launched by all devices so far */
/* range [lo, hi) of `n_units` that part `part` of `n_parts` owns: lo = floor(n_units * part / n_parts) */
VBX_API void vbx_multi_partition(int64_t n_units, int32_t n_parts, int32_t part, int64_t* lo, int64_t* hi);
VBX_API int vbx_multi_lpc_host(vbx_multi* m, const vbx_frames* frames, int32_t p, void* r_out, void* ac_out, void* kc_out,
                               int32_t out_dtype);
VBX_API int vbx_multi_find_formants_host(vbx_multi* m, const vbx_frames* frames, double sample_rate, int32_t n_coeffs,
                                         int32_t lpc_method, void* est_inout, int32_t n_formants, void* tracks_out,
                                         void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype);
VBX_API int vbx_multi_pitch_host(vbx_multi* m, const vbx_frames* frames, double sample_rate, double threshold, double min_hz,
                                 double max_hz, int32_t max_candidates, void* cand_out, int32_t* n_cand_out,
                                 uint8_t* status_out, int32_t out_dtype);
VBX_API int vbx_multi_pitch_with_peaks_host(vbx_multi* m, const vbx_frames* frames, double sample_rate, double threshold,
                                            double silence_threshold, const double* local_peaks, const double* global_peaks,
                                            double min_hz, double max_hz, int32_t max_candidates, void* cand_out,
                                            int32_t* n_cand_out, uint8_t* status_out, int32_t out_dtype);
VBX_API int vbx_multi_mfcc_host(vbx_multi* m, const vbx_frames* frames, int32_t num_coeffs, int32_t n_keep, double freq_lo,
                                double freq_hi, double sample_rate, void* out, int32_t out_dtype);
/* Host->device copy bandwidth (GB/s per device, gbs_out[n_devices]) with the first n_active devices copying concurrently from
 * pinned buffers allocated by their own worker threads: which link saturates as more GPUs stage at once (tools/h2d_probe.py). */
VBX_API int vbx_multi_h2d_bandwidth(vbx_multi* m, size_t bytes_per_device, int32_t reps, int32_t n_active, double* gbs_out);

/* ---- synthetic speech-like audio, generated on the device (bench / parity-at-scale infrastructure; SURVEY 8d) ----------------
 * out: [n_utts][n_samples] of dtype (VBX_F32, or VBX_I16 = the same samples as 16-bit PCM, round(x * 32767), or VBX_MULAW8 /
 * VBX_ALAW8 = those int16 samples G.711-encoded as audioop.lin2ulaw / lin2alaw(x, 2) do: g711.c's 14-bit mu-law encoder on
 * x >> 2, its 13-bit A-law encoder on x >> 3).  Utterance u of the
 * call is global utterance first_utt + u: a function of (seed, first_utt + u, sample_rate) only.  Recipe: csrc/vbx_synth.cu. */
VBX_API int vbx_synth_speech(vbx_ctx* ctx, void* out, int32_t dtype, int64_t n_utts, int64_t n_samples, double sample_rate,
                             uint64_t seed, int64_t first_utt);

#ifdef __cplusplus
}
#endif
#endif /* VOXBOX_B200_H */
