"""ctypes binding of libvoxbox_b200.so (the C ABI in include/voxbox_b200.h).

Thin by design: the product is the CUDA library; this module only marshals
pointers for the test-suite, bench.py and Python callers.  There is no CPU
fallback — importing works anywhere (so symbol/export checks can run without a
GPU), but creating a `Context` fails loudly when the library or a CUDA device is
missing.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(_PKG))  # vox_box.rs_b200/
LIB_PATH = os.path.join(ROOT, "libvoxbox_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(ROOT), "include", "voxbox_b200.h")

OK, ERR_LPC, ERR_PITCH, ERR_POLYNOMIAL, ERR_WORKSPACE, ERR_CUDA, ERR_BADARG, ERR_NOMEM = range(8)
F32, F64, I16, MULAW8, ALAW8 = 0, 1, 2, 3, 4  # MULAW8 / ALAW8: G.711 bytes, decoded to int16 PCM on load
WINDOW_NONE, WINDOW_HANN_SYMMETRIC, WINDOW_HANN_PERIODIC, WINDOW_HANN_LAG = 0, 1, 2, 3
INTERP_NONE, INTERP_PARABOLIC, INTERP_SINC = 0, 1, 2
MAX_RESONANCES = 32
LPC_BURG, LPC_AUTOCORR = 0, 1
_NP = {F32: np.float32, F64: np.float64, I16: np.int16, MULAW8: np.uint8, ALAW8: np.uint8}


class VoxBoxError(RuntimeError):
    """Mirror of error.rs VoxBoxError + the CUDA/BADARG/NOMEM codes of the C ABI."""

    def __init__(self, status, message):
        super().__init__(f"vbx status {status}: {message}")
        self.status = status


class Frames(C.Structure):
    """struct vbx_frames.  sample_step (0 / 1 contiguous, C for C interleaved channels) shares its int32 with the field's
    former name `reserved`, which stays as an alias."""
    _fields_ = [("base", C.c_void_p), ("n_frames", C.c_int64), ("frame_stride", C.c_int64),
                ("frames_per_segment", C.c_int64), ("segment_stride", C.c_int64), ("frame_len", C.c_int32), ("dtype", C.c_int32), ("window", C.c_int32), ("sample_step", C.c_int32)]

    reserved = property(lambda self: self.sample_step, lambda self, v: setattr(self, "sample_step", v))


def channel_view(n_frames, stride, frames_per_segment=0, segment_stride=0, channels=1):
    """(n_frames, frame_stride, frames_per_segment, segment_stride, sample_step) of the view a `_host` helper builds.
    channels=1: the arguments as given.  channels=C > 1: the buffer holds C interleaved channels (the WAV layout, n_samples*C
    samples), n_frames and stride count the frames and the hop of ONE channel, and the view has one segment per channel
    (segment u = channel u, sample_step C), so the helper returns C*n_frames rows, channel-major."""
    channels = int(channels)
    if channels < 1:
        raise ValueError(f"channels must be >= 1, not {channels}")
    if channels == 1:
        return n_frames, stride, frames_per_segment, segment_stride, 0
    if frames_per_segment:
        raise ValueError("channels > 1 views the buffer as one segment per channel: frames_per_segment must be 0")
    return channels * n_frames, stride * channels, n_frames, 1, channels


_lib = None


def load_library():
    """Load libvoxbox_b200.so; raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VoxBoxError(ERR_CUDA, f"{LIB_PATH} not built — run `python __graft_entry__.py` "
                                        "(make -C vox_box.rs_b200); there is no CPU fallback")
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


_vp, _i32, _i64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
_frp = C.POINTER(Frames)


def _declare(L):
    def sig(name, res, *args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = list(args)

    sig("vbx_ctx_create", C.c_int, C.c_int, C.POINTER(_vp))
    sig("vbx_ctx_destroy", C.c_int, _vp)
    sig("vbx_sync", C.c_int, _vp)
    sig("vbx_ctx_stream", _vp, _vp)
    sig("vbx_last_error", C.c_char_p, _vp)
    sig("vbx_status_str", C.c_char_p, C.c_int)
    sig("vbx_version", C.c_int)
    sig("vbx_device_sm_count", C.c_int, _vp)
    sig("vbx_kernel_launches", _i64, _vp)
    sig("vbx_malloc", C.c_int, _vp, _sz, C.POINTER(_vp))
    sig("vbx_free", C.c_int, _vp, _vp)
    sig("vbx_malloc_host", C.c_int, _vp, _sz, C.POINTER(_vp))
    sig("vbx_free_host", C.c_int, _vp, _vp)
    sig("vbx_memcpy_h2d", C.c_int, _vp, _vp, _vp, _sz)
    sig("vbx_memcpy_d2h", C.c_int, _vp, _vp, _vp, _sz)
    sig("vbx_memcpy_d2d", C.c_int, _vp, _vp, _vp, _sz)
    sig("vbx_memset", C.c_int, _vp, _vp, C.c_int, _sz)
    sig("vbx_timer_start", C.c_int, _vp)
    sig("vbx_timer_stop_ms", C.c_int, _vp, C.POINTER(C.c_float))
    sig("vbx_measure_peaks", C.c_int, _vp, C.POINTER(C.c_double), C.POINTER(C.c_double))
    sig("vbx_profile_begin", C.c_int, _vp)
    sig("vbx_profile_end", C.c_int, _vp)
    sig("vbx_profile_count", C.c_int, _vp)
    sig("vbx_profile_entry", C.c_int, _vp, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_double), C.POINTER(_i64))
    sig("vbx_profile_counters", C.c_int, _vp, C.POINTER(C.c_uint64), _i32)
    sig("vbx_window_table_host", C.c_int, C.c_int, _i32, C.POINTER(C.c_double))
    sig("vbx_autocorrelate", C.c_int, _vp, _frp, _i32, _vp, _i32)
    sig("vbx_autocorrelate_host", C.c_int, _vp, _frp, _i32, _vp, _i32)
    sig("vbx_autocorrelate_ring", C.c_int, _vp, _vp, _i32, _i64, _i64, _vp, _i32, _i32, _vp, _i32)
    sig("vbx_lpc_levinson", C.c_int, _vp, _vp, _i32, _i64, _i32, _i32, _vp, _vp, _i32)
    sig("vbx_lpc", C.c_int, _vp, _frp, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_lpc_host", C.c_int, _vp, _frp, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_lpc_burg", C.c_int, _vp, _frp, _i32, _vp, _vp, _i32)
    sig("vbx_find_roots", C.c_int, _vp, _vp, _i32, _i64, _i32, _vp, _vp)
    sig("vbx_find_roots_work_size", _i64, _i64)
    sig("vbx_laguerre", C.c_int, _vp, _vp, _i32, _i64, _i32, C.c_double, C.c_double, _vp)
    sig("vbx_div_polynomial", C.c_int, _vp, _vp, _i32, _i64, _i32, _vp, _i32, _vp, _vp)
    sig("vbx_roots_to_resonances", C.c_int, _vp, _vp, _i32, _i64, _i32, C.c_double, _i32, _vp, _i32, _vp, _i32)
    sig("vbx_lpc_to_resonances", C.c_int, _vp, _vp, _i32, _i64, _i32, _i32, _i32, C.c_double, _i32, _vp, _vp, _i32, _vp,
        _vp, _vp, _i32, _i32)
    sig("vbx_estimate_formants", C.c_int, _vp, _vp, _i32, _i32, _i32, _i64, _i64, _vp, _vp, _i32, _vp, _i32)
    sig("vbx_find_formants_real_work_size", _i64, _i64, _i64)
    sig("vbx_find_formants_complex_work_size", _i64, _i64)
    sig("vbx_find_formants", C.c_int, _vp, _frp, C.c_double, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i32)
    sig("vbx_find_formants_host", C.c_int, _vp, _frp, C.c_double, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i32)
    _d = C.c_double
    sig("vbx_find_formants_resampled", C.c_int, _vp, _frp, _d, _d, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i32)
    sig("vbx_pitch", C.c_int, _vp, _frp, _d, _d, _d, _d, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_pitch_host", C.c_int, _vp, _frp, _d, _d, _d, _d, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_pitch_lag_function", C.c_int, _vp, _frp, _vp)
    sig("vbx_frame_peaks", C.c_int, _vp, _frp, _vp, _vp)
    sig("vbx_pitch_with_peaks", C.c_int, _vp, _frp, _d, _d, _d, _vp, _vp, _d, _d, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_pitch_with_peaks_host", C.c_int, _vp, _frp, _d, _d, _d, _vp, _vp, _d, _d, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_pitch_extract", C.c_int, _vp, _vp, _i32, _i64, _i32, _vp)
    sig("vbx_pitch_viterbi", C.c_int, _vp, _vp, _i32, _vp, _i64, _i64, _i32, _d, _d, _d, _d, _vp, _vp)
    sig("vbx_interpolate_sinc", C.c_int, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _i64, _vp)
    sig("vbx_improve_extremum", C.c_int, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _i32, _i64, _i32, _vp, _vp)
    sig("vbx_mfcc", C.c_int, _vp, _frp, _i32, _i32, _d, _d, _d, _vp, _vp, _i32)
    sig("vbx_mfcc_host", C.c_int, _vp, _frp, _i32, _i32, _d, _d, _d, _vp, _i32)
    sig("vbx_mfcc_set_fft_precision", C.c_int, _vp, _i32)
    sig("vbx_hz_to_mel", _d, _d)
    sig("vbx_mel_to_hz", _d, _d)
    sig("vbx_dct", C.c_int, _vp, _vp, _i32, _i64, _i32, _vp)
    sig("vbx_rms", C.c_int, _vp, _vp, _i32, _i64, _i32, _i64, _vp)
    sig("vbx_max_amplitude", C.c_int, _vp, _vp, _i32, _i64, _i32, _i64, _vp)
    sig("vbx_normalize", C.c_int, _vp, _vp, _i32, _i64, _i32, _i64, _vp)
    sig("vbx_preemphasis", C.c_int, _vp, _vp, _i32, _i64, _i32, _i64, _d)
    sig("vbx_find_formants_buffered", C.c_int, _vp, _frp, _d, _d, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i32)
    sig("vbx_synth_speech", C.c_int, _vp, _vp, _i32, _i64, _i64, _d, C.c_uint64, _i64)
    sig("vbx_multi_create", C.c_int, _i32, C.POINTER(_i32), C.POINTER(_vp))
    sig("vbx_multi_destroy", C.c_int, _vp)
    sig("vbx_multi_device_count", _i32, _vp)
    sig("vbx_multi_ctx", _vp, _vp, _i32)
    sig("vbx_multi_last_error", C.c_char_p, _vp)
    sig("vbx_multi_kernel_launches", _i64, _vp)
    sig("vbx_multi_partition", None, _i64, _i32, _i32, C.POINTER(_i64), C.POINTER(_i64))
    sig("vbx_multi_lpc_host", C.c_int, _vp, _frp, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_multi_find_formants_host", C.c_int, _vp, _frp, C.c_double, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i32)
    sig("vbx_multi_pitch_host", C.c_int, _vp, _frp, _d, _d, _d, _d, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_multi_pitch_with_peaks_host", C.c_int, _vp, _frp, _d, _d, _d, _vp, _vp, _d, _d, _i32, _vp, _vp, _vp, _i32)
    sig("vbx_multi_mfcc_host", C.c_int, _vp, _frp, _i32, _i32, _d, _d, _d, _vp, _i32)
    sig("vbx_multi_h2d_bandwidth", C.c_int, _vp, _sz, _i32, _i32, C.POINTER(_d))


def window_table(window, n):
    out = np.empty(n, dtype=np.float64)
    st = load_library().vbx_window_table_host(window, n, out.ctypes.data_as(C.POINTER(C.c_double)))
    if st:
        raise VoxBoxError(st, "vbx_window_table_host")
    return out


class DeviceArray:
    """Caller-owned HBM buffer (vbx_malloc) with numpy shape/dtype metadata."""

    def __init__(self, ctx, shape, dtype):
        self.ctx, self.shape, self.dtype = ctx, tuple(int(s) for s in np.atleast_1d(shape)), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = _vp()
        ctx._check(ctx.lib.vbx_malloc(ctx.h, max(self.nbytes, 1), C.byref(p)), "vbx_malloc")
        self.ptr = p.value

    def upload(self, host):
        host = np.ascontiguousarray(host, dtype=self.dtype)
        assert host.nbytes == self.nbytes
        self.ctx._check(self.ctx.lib.vbx_memcpy_h2d(self.ctx.h, self.ptr, host.ctypes.data, self.nbytes), "h2d")
        self.ctx.sync()  # `host` may be a temporary
        return self

    def to_host(self):
        out = np.empty(self.shape, dtype=self.dtype)
        self.ctx._check(self.ctx.lib.vbx_memcpy_d2h(self.ctx.h, out.ctypes.data, self.ptr, self.nbytes), "d2h")
        self.ctx.sync()
        return out

    def free(self):
        if self.ptr:
            self.ctx.lib.vbx_free(self.ctx.h, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """vbx_ctx: one device + stream + scratch arena.  Fails loudly without the library / a GPU."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = _vp()
        st = self.lib.vbx_ctx_create(device, C.byref(h))
        if st != OK:
            raise VoxBoxError(st, "vbx_ctx_create failed: no usable CUDA device (there is no CPU fallback)")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.vbx_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, st, what):
        if st != OK:
            raise VoxBoxError(st, f"{what}: {self.lib.vbx_last_error(self.h).decode()} "
                                  f"[{self.lib.vbx_status_str(st).decode()}]")

    # -- plumbing ---------------------------------------------------------------------------
    def sync(self):
        self._check(self.lib.vbx_sync(self.h), "vbx_sync")

    def empty(self, shape, dtype):
        return DeviceArray(self, shape, dtype)

    def to_device(self, host):
        host = np.ascontiguousarray(host)
        return DeviceArray(self, host.shape, host.dtype).upload(host)

    def timer_start(self):
        self._check(self.lib.vbx_timer_start(self.h), "vbx_timer_start")

    def timer_stop_ms(self):
        ms = C.c_float(0)
        self._check(self.lib.vbx_timer_stop_ms(self.h, C.byref(ms)), "vbx_timer_stop_ms")
        return ms.value

    @property
    def kernel_launches(self):
        return self.lib.vbx_kernel_launches(self.h)

    @property
    def sm_count(self):
        return self.lib.vbx_device_sm_count(self.h)

    def profile_begin(self):
        self._check(self.lib.vbx_profile_begin(self.h), "vbx_profile_begin")

    def profile_end(self):
        """Returns {kernel name: (total ms, launches)} for the launches since profile_begin."""
        self._check(self.lib.vbx_profile_end(self.h), "vbx_profile_end")
        out = {}
        for i in range(self.lib.vbx_profile_count(self.h)):
            name = C.create_string_buffer(128)
            ms, n = C.c_double(0), _i64(0)
            self._check(self.lib.vbx_profile_entry(self.h, i, name, 128, C.byref(ms), C.byref(n)), "vbx_profile_entry")
            out[name.value.decode()] = (ms.value, n.value)
        return out

    def profile_counters(self):
        """Executed-work counters of the last profile_begin..profile_end window (vbx_profile_counters)."""
        out = (C.c_uint64 * 8)()
        self._check(self.lib.vbx_profile_counters(self.h, out, 8), "vbx_profile_counters")
        return dict(roots_horner_steps=out[0], roots_rounds=out[1], refine_terms=out[2], refine_evals=out[3], roots_fixup_frames=out[4])

    def measure_peaks(self):
        a, b = C.c_double(0), C.c_double(0)
        self._check(self.lib.vbx_measure_peaks(self.h, C.byref(a), C.byref(b)), "vbx_measure_peaks")
        return dict(fp32_tflops=a.value, fp64_tflops=b.value)

    @staticmethod
    def frames(base_ptr, n_frames, frame_len, frame_stride, window=WINDOW_NONE, dtype=F32, frames_per_segment=0,
               segment_stride=0, sample_step=0):
        """vbx_frames: sample i of frame f = u*J + j is base[u*segment_stride + j*frame_stride + i*sample_step]
        (J = frames_per_segment; sample_step 0 or 1 = contiguous frames)."""
        return Frames(base_ptr, n_frames, frame_stride, frames_per_segment, segment_stride, frame_len, dtype, window, sample_step)

    @staticmethod
    def _host_view(base_ptr, n_frames, frame_len, stride, window, dtype, frames_per_segment=0, segment_stride=0, channels=1):
        """The view of a `_host` helper (channel_view) and its number of frames."""
        F, fst, J, seg, step = channel_view(n_frames, stride, frames_per_segment, segment_stride, channels)
        return Context.frames(base_ptr, F, frame_len, fst, window, dtype, J, seg, step), F

    @staticmethod
    def n_frames_of(n_samples, frame_len, hop):
        """Windower::{hanning,rectangle}: a frame while bin <= remaining, advance by hop."""
        return 0 if n_samples < frame_len else (n_samples - frame_len) // hop + 1

    # -- device-pointer ops -------------------------------------------------------------------
    def autocorrelate(self, frames, n_lags, out_dtype=F64, out=None):
        r = out if out is not None else self.empty((frames.n_frames, n_lags), _NP[out_dtype])
        self._check(self.lib.vbx_autocorrelate(self.h, C.byref(frames), n_lags, r.ptr, out_dtype), "vbx_autocorrelate")
        return r

    def lpc(self, frames, p, out_dtype=F64, want_r=True, want_kc=True, out=None):
        """Fused window→autocorrelate(p+1)→lpc(p).  Returns (r, ac, kc) device arrays (None if not wanted)."""
        F = frames.n_frames
        if out is not None:
            r, ac, kc = out
        else:
            r = self.empty((F, p + 1), _NP[out_dtype]) if want_r else None
            ac = self.empty((F, p + 1), _NP[out_dtype])
            kc = self.empty((F, p), _NP[out_dtype]) if want_kc else None
        self._check(self.lib.vbx_lpc(self.h, C.byref(frames), p, r.ptr if r else None, ac.ptr if ac else None,
                                     kc.ptr if kc else None, out_dtype), "vbx_lpc")
        return r, ac, kc

    def lpc_levinson(self, r, p, out_dtype=F64):
        F, stride = r.shape
        ac = self.empty((F, p + 1), _NP[out_dtype])
        kc = self.empty((F, p), _NP[out_dtype])
        rd = F64 if r.dtype == np.float64 else F32
        self._check(self.lib.vbx_lpc_levinson(self.h, r.ptr, rd, F, stride, p, ac.ptr, kc.ptr, out_dtype),
                    "vbx_lpc_levinson")
        return ac, kc

    # -- host-pointer twins (H2D + kernels + D2H inside the call) ------------------------------
    def autocorrelate_host(self, audio, n_frames, frame_len, stride, window, n_lags, out_dtype=F64, sample_dtype=None, channels=1):
        audio = np.ascontiguousarray(audio)
        fr, n_frames = self._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, _sample_dtype(audio, sample_dtype),
                                       channels=channels)
        r = np.empty((n_frames, n_lags), dtype=_NP[out_dtype])
        self._check(self.lib.vbx_autocorrelate_host(self.h, C.byref(fr), n_lags, r.ctypes.data, out_dtype),
                    "vbx_autocorrelate_host")
        return r

    def lpc_host(self, audio, n_frames, frame_len, stride, window, p, out_dtype=F64, out=None, sample_dtype=None, channels=1):
        audio = np.ascontiguousarray(audio)
        fr, n_frames = self._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, _sample_dtype(audio, sample_dtype),
                                       channels=channels)
        if out is None:
            out = (np.empty((n_frames, p + 1), dtype=_NP[out_dtype]), np.empty((n_frames, p + 1), dtype=_NP[out_dtype]),
                   np.empty((n_frames, p), dtype=_NP[out_dtype]))
        r, ac, kc = out
        self._check(self.lib.vbx_lpc_host(self.h, C.byref(fr), p, r.ctypes.data if r is not None else None,
                                          ac.ctypes.data if ac is not None else None,
                                          kc.ctypes.data if kc is not None else None, out_dtype), "vbx_lpc_host")
        return r, ac, kc


# ---- formant path (appended to Context) ---------------------------------------------------------
def _dt_of(a):
    return F64 if np.dtype(a.dtype) in (np.dtype(np.float64), np.dtype(np.complex128)) else F32


def _lpc_burg(self, frames, p, out_dtype=F64):
    """spectrum.rs:94-146 lpc_praat over frames → (coeffs [F][p], status [F]) device arrays."""
    co = self.empty((frames.n_frames, p), _NP[out_dtype])
    st = self.empty((frames.n_frames,), np.uint8)
    self._check(self.lib.vbx_lpc_burg(self.h, C.byref(frames), p, co.ptr, st.ptr, out_dtype), "vbx_lpc_burg")
    return co, st


def _find_roots(self, coeffs):
    """polynomial.rs:92-152 find_roots_mut on host complex arrays [F][len] → (buffer after write-back, status)."""
    c = np.ascontiguousarray(coeffs)
    assert c.dtype in (np.complex64, np.complex128) and c.ndim == 2
    d = self.to_device(c)
    out = self.empty(c.shape, c.dtype)
    st = self.empty((c.shape[0],), np.uint8)
    self._check(self.lib.vbx_find_roots(self.h, d.ptr, _dt_of(c), c.shape[0], c.shape[1], out.ptr, st.ptr), "vbx_find_roots")
    return out.to_host(), st.to_host()


def _laguerre(self, coeffs, start):
    c = np.ascontiguousarray(coeffs)
    assert c.dtype in (np.complex64, np.complex128) and c.ndim == 2
    d = self.to_device(c)
    z = self.empty((c.shape[0],), c.dtype)
    self._check(self.lib.vbx_laguerre(self.h, d.ptr, _dt_of(c), c.shape[0], c.shape[1], start.real, start.imag, z.ptr),
                "vbx_laguerre")
    return z.to_host()


def _div_polynomial(self, coeffs, other):
    c = np.ascontiguousarray(coeffs)
    assert c.dtype in (np.complex64, np.complex128) and c.ndim == 2
    d = self.to_device(c)
    o = self.to_device(np.asarray([other], dtype=c.dtype))
    rem = self.empty(c.shape, c.dtype)
    st = self.empty((c.shape[0],), np.uint8)
    self._check(self.lib.vbx_div_polynomial(self.h, d.ptr, _dt_of(c), c.shape[0], c.shape[1], o.ptr, 0, rem.ptr, st.ptr),
                "vbx_div_polynomial")
    return d.to_host(), rem.to_host(), st.to_host()


def _roots_to_resonances(self, roots, fs, strict_im=False, res_slots=None, out_dtype=F64):
    r = np.ascontiguousarray(roots)
    assert r.dtype in (np.complex64, np.complex128) and r.ndim == 2
    slots = res_slots or max(r.shape[1], 1)
    d = self.to_device(r)
    res = self.empty((r.shape[0], slots, 2), _NP[out_dtype])
    n = self.empty((r.shape[0],), np.int32)
    self._check(self.lib.vbx_roots_to_resonances(self.h, d.ptr, _dt_of(r), r.shape[0], r.shape[1], fs, int(strict_im),
                                                 res.ptr, slots, n.ptr, out_dtype), "vbx_roots_to_resonances")
    return res.to_host(), n.to_host()


def _lpc_to_resonances(self, lpc, p, has_one, fs, strict_im=True, res_slots=None, out_dtype=F64, precision=-1,
                       status_in=None, want_roots=False):
    """lpc: DeviceArray [F][stride].  Returns dict of device arrays."""
    F, stride = lpc.shape
    slots = res_slots or p
    res = self.empty((F, slots, 2), _NP[out_dtype])
    n = self.empty((F,), np.int32)
    st = self.empty((F,), np.uint8)
    roots = self.empty((F, p, 2), _NP[out_dtype]) if want_roots else None
    self._check(self.lib.vbx_lpc_to_resonances(self.h, lpc.ptr, _dt_of(lpc), F, stride, p, int(has_one), fs, int(strict_im),
                                               status_in.ptr if status_in is not None else None, res.ptr, slots, n.ptr,
                                               roots.ptr if roots else None, st.ptr, out_dtype, precision),
                "vbx_lpc_to_resonances")
    return dict(resonances=res, n_res=n, status=st, roots=roots)


def _estimate_formants(self, resonances, estimates, n_segments=1, n_resonances=None, dtype=F64):
    """FormantExtractor over host arrays: resonances [F][slots][2], estimates [n_segments][k][2] (or [k][2]).
    Returns (tracks [F][k][2], final estimates)."""
    res = np.ascontiguousarray(resonances, dtype=_NP[dtype])
    est = np.ascontiguousarray(estimates, dtype=_NP[dtype]).reshape(n_segments, -1, 2)
    F, slots = res.shape[0], res.shape[1]
    k = est.shape[1]
    d_res, d_est = self.to_device(res), self.to_device(est)
    tracks = self.empty((F, k, 2), _NP[dtype])
    self._check(self.lib.vbx_estimate_formants(self.h, d_res.ptr, dtype, slots, n_resonances or slots, n_segments,
                                               F // n_segments, None, d_est.ptr, k, tracks.ptr, dtype),
                "vbx_estimate_formants")
    return tracks.to_host(), d_est.to_host()


def _find_formants(self, frames, fs, p, method, estimates, dtype=F64, want_resonances=True):
    """Device-pointer find_formants.  estimates: host [n_segments][k][2].  Returns dict of host arrays."""
    F = frames.n_frames
    J = frames.frames_per_segment or F
    segs = F // J if J else 0
    est = np.ascontiguousarray(estimates, dtype=_NP[dtype])
    k = est.shape[-2]
    est = est.reshape(segs, k, 2)
    d_est = self.to_device(est)
    tracks = self.empty((F, k, 2), _NP[dtype])
    res = self.empty((F, MAX_RESONANCES, 2), _NP[dtype]) if want_resonances else None
    nres = self.empty((F,), np.int32)
    st = self.empty((F,), np.uint8)
    self._check(self.lib.vbx_find_formants(self.h, C.byref(frames), fs, p, method, d_est.ptr, k, tracks.ptr,
                                           res.ptr if res else None, nres.ptr, st.ptr, dtype), "vbx_find_formants")
    return dict(tracks=tracks.to_host(), estimates=d_est.to_host(), resonances=res.to_host() if res else None,
                n_res=nres.to_host(), status=st.to_host())


def _find_formants_host(self, audio, n_frames, frame_len, stride, window, fs, p, method, estimates, dtype=F64,
                        frames_per_segment=0, segment_stride=0, sample_dtype=None, channels=1):
    """estimates: [n_segments][k][2] (one row per channel with channels=C)."""
    audio = np.ascontiguousarray(audio)
    fr, n_frames = self._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, _sample_dtype(audio, sample_dtype),
                                   frames_per_segment, segment_stride, channels)
    J = fr.frames_per_segment or n_frames
    segs = n_frames // J if J else 0
    est = np.ascontiguousarray(estimates, dtype=_NP[dtype]).reshape(segs, -1, 2).copy()
    k = est.shape[1]
    tracks = np.zeros((n_frames, k, 2), dtype=_NP[dtype])
    res = np.zeros((n_frames, MAX_RESONANCES, 2), dtype=_NP[dtype])
    nres = np.zeros(n_frames, dtype=np.int32)
    st = np.zeros(n_frames, dtype=np.uint8)
    self._check(self.lib.vbx_find_formants_host(self.h, C.byref(fr), fs, p, method, est.ctypes.data, k, tracks.ctypes.data,
                                                res.ctypes.data, nres.ctypes.data, st.ctypes.data, dtype),
                "vbx_find_formants_host")
    return dict(tracks=tracks, estimates=est, resonances=res, n_res=nres, status=st)


Context.lpc_burg = _lpc_burg
Context.find_roots = _find_roots
Context.laguerre = _laguerre
Context.div_polynomial = _div_polynomial
Context.roots_to_resonances = _roots_to_resonances
Context.lpc_to_resonances = _lpc_to_resonances
Context.estimate_formants = _estimate_formants
Context.find_formants = _find_formants
Context.find_formants_host = _find_formants_host


# ---- pitch path (appended to Context) -------------------------------------------------------------
def _pitch(self, frames, fs, threshold, fmin, fmax, max_cand=16, out_dtype=F64):
    """periodic.rs:356-456 pitch::<Hanning> over frames → dict of device arrays
    (candidates [F][max_cand][2] sorted by strength desc, n_cand [F], status [F])."""
    F = frames.n_frames
    cand = self.empty((F, max_cand, 2), _NP[out_dtype])
    n = self.empty((F,), np.int32)
    st = self.empty((F,), np.uint8)
    self._check(self.lib.vbx_pitch(self.h, C.byref(frames), fs, threshold, fmin, fmax, max_cand, cand.ptr, n.ptr, st.ptr,
                                   out_dtype), "vbx_pitch")
    return dict(candidates=cand, n_cand=n, status=st)


def _pitch_host(self, audio, n_frames, frame_len, stride, window, fs, threshold, fmin, fmax, max_cand=16, out_dtype=F64,
                frames_per_segment=0, segment_stride=0, sample_dtype=None, channels=1):
    audio = np.ascontiguousarray(audio)
    fr, n_frames = self._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, _sample_dtype(audio, sample_dtype),
                                   frames_per_segment, segment_stride, channels)
    cand = np.zeros((n_frames, max_cand, 2), dtype=_NP[out_dtype])
    n = np.zeros(n_frames, dtype=np.int32)
    st = np.zeros(n_frames, dtype=np.uint8)
    self._check(self.lib.vbx_pitch_host(self.h, C.byref(fr), fs, threshold, fmin, fmax, max_cand, cand.ctypes.data,
                                        n.ctypes.data, st.ctypes.data, out_dtype), "vbx_pitch_host")
    return dict(candidates=cand, n_cand=n, status=st)


def _pitch_extract(self, cand):
    """periodic.rs:320-354 PitchExtractor: strongest candidate per frame."""
    F, max_cand = cand.shape[0], cand.shape[1]
    out = self.empty((F, 2), cand.dtype)
    self._check(self.lib.vbx_pitch_extract(self.h, cand.ptr, _dt_of(cand), F, max_cand, out.ptr), "vbx_pitch_extract")
    return out


def _interpolate_sinc(self, y, offset, nx, x, max_depth):
    """periodic.rs:29-87 on host arrays: y [S][y_len] (or [y_len]), x [S][M] (or [M]) → values [S][M]."""
    y = np.atleast_2d(np.ascontiguousarray(y, dtype=np.float64))
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(y.shape[0], -1)
    dy, dx = self.to_device(y), self.to_device(x)
    out = self.empty(x.shape, np.float64)
    self._check(self.lib.vbx_interpolate_sinc(self.h, dy.ptr, y.shape[0], y.shape[1], offset, nx, dx.ptr, x.shape[1],
                                              max_depth, out.ptr), "vbx_interpolate_sinc")
    return out.to_host()


def _improve_extremum(self, y, offset, nx, ixmid, interp=INTERP_SINC, depth=1200, is_max=True):
    y = np.atleast_2d(np.ascontiguousarray(y, dtype=np.float64))
    x = np.ascontiguousarray(ixmid, dtype=np.float64).reshape(y.shape[0], -1)
    dy, dx = self.to_device(y), self.to_device(x)
    xm, ym = self.empty(x.shape, np.float64), self.empty(x.shape, np.float64)
    self._check(self.lib.vbx_improve_extremum(self.h, dy.ptr, y.shape[0], y.shape[1], offset, nx, dx.ptr, x.shape[1],
                                              interp, depth, int(is_max), xm.ptr, ym.ptr), "vbx_improve_extremum")
    return xm.to_host(), ym.to_host()


def _pitch_lag_function(self, frames):
    """periodic.rs:403-408 self_lag for every frame → device array [F][N] f64."""
    out = self.empty((frames.n_frames, frames.frame_len), np.float64)
    self._check(self.lib.vbx_pitch_lag_function(self.h, C.byref(frames), out.ptr), "vbx_pitch_lag_function")
    return out


def _n_segments(n_frames, frames_per_segment):
    return n_frames // frames_per_segment if frames_per_segment else 1


def _g711_law(audio, sample_dtype):
    """sample_dtype of uint8 host samples: G.711 codes carry no mark of their law, so the caller names it (MULAW8 / ALAW8);
    None for other samples, which must then not claim a law."""
    if audio.dtype == np.uint8:
        if sample_dtype not in (MULAW8, ALAW8):
            raise ValueError("uint8 samples are G.711 codes of an unknown law: pass sample_dtype=MULAW8 or sample_dtype=ALAW8")
        return sample_dtype
    if sample_dtype in (MULAW8, ALAW8):
        raise ValueError(f"sample_dtype {sample_dtype} (G.711) needs uint8 samples, not {audio.dtype}")
    return None


def _sample_dtype(audio, sample_dtype=None):
    """vbx dtype of the host samples of the int16 / float32 `_host` wrappers: int16 PCM, uint8 G.711 codes, anything else
    float32."""
    law = _g711_law(audio, sample_dtype)
    return law if law is not None else (I16 if audio.dtype == np.int16 else F32)


def _host_audio(audio, sample_dtype=None):
    """Host samples and their vbx dtype: int16 PCM, uint8 G.711 codes (sample_dtype MULAW8 / ALAW8), float64, or anything
    else as float32."""
    audio = np.asarray(audio)
    law = _g711_law(audio, sample_dtype)
    if law is not None:
        return np.ascontiguousarray(audio), law
    if audio.dtype == np.int16:
        return np.ascontiguousarray(audio), I16
    if audio.dtype == np.float64:
        return np.ascontiguousarray(audio), F64
    return np.ascontiguousarray(audio, dtype=np.float32), F32


def _host_peaks(a, n):
    """Caller-supplied peaks for a `_host` twin: None, or a contiguous float64 array of n values."""
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1)
    assert a.size == n, (a.size, n)
    return a


def _frame_peaks(self, frames):
    """Local peak per frame [F] and global peak per segment [n_segments] (max |x| before the window; vbx_frame_peaks) →
    (local, global) device arrays of float64."""
    local = self.empty((frames.n_frames,), np.float64)
    glob = self.empty((_n_segments(frames.n_frames, frames.frames_per_segment),), np.float64)
    self._check(self.lib.vbx_frame_peaks(self.h, C.byref(frames), local.ptr, glob.ptr), "vbx_frame_peaks")
    return local, glob


def _pitch_with_peaks(self, frames, fs, threshold, silence_threshold, fmin, fmax, max_cand=16, out_dtype=F64, local_peaks=None,
                      global_peaks=None):
    """vbx_pitch with Boersma's voiceless strength as the unvoiced candidate's strength (vbx_pitch_with_peaks).  local_peaks [F] /
    global_peaks [n_segments]: float64 device arrays, or None = computed from the view.  → dict of device arrays as pitch()."""
    F = frames.n_frames
    cand = self.empty((F, max_cand, 2), _NP[out_dtype])
    n = self.empty((F,), np.int32)
    st = self.empty((F,), np.uint8)
    self._check(self.lib.vbx_pitch_with_peaks(self.h, C.byref(frames), fs, threshold, silence_threshold,
                                              local_peaks.ptr if local_peaks is not None else None,
                                              global_peaks.ptr if global_peaks is not None else None, fmin, fmax, max_cand,
                                              cand.ptr, n.ptr, st.ptr, out_dtype), "vbx_pitch_with_peaks")
    return dict(candidates=cand, n_cand=n, status=st)


def _pitch_with_peaks_host(self, audio, n_frames, frame_len, stride, window, fs, threshold, silence_threshold, fmin, fmax,
                           max_cand=16, out_dtype=F64, frames_per_segment=0, segment_stride=0, local_peaks=None,
                           global_peaks=None, sample_dtype=None, channels=1):
    """Host twin of pitch_with_peaks: audio int16 / float32 / float64 samples (or uint8 G.711 codes with sample_dtype), peaks
    host arrays or None (local [F], global [n_segments]: one per channel with channels=C)."""
    audio, dt = _host_audio(audio, sample_dtype)
    fr, n_frames = self._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, dt, frames_per_segment, segment_stride,
                                   channels)
    lp = _host_peaks(local_peaks, n_frames)
    gp = _host_peaks(global_peaks, _n_segments(n_frames, fr.frames_per_segment))
    cand = np.zeros((n_frames, max_cand, 2), dtype=_NP[out_dtype])
    n = np.zeros(n_frames, dtype=np.int32)
    st = np.zeros(n_frames, dtype=np.uint8)
    self._check(self.lib.vbx_pitch_with_peaks_host(self.h, C.byref(fr), fs, threshold, silence_threshold,
                                                   lp.ctypes.data if lp is not None else None,
                                                   gp.ctypes.data if gp is not None else None, fmin, fmax, max_cand,
                                                   cand.ctypes.data, n.ctypes.data, st.ctypes.data, out_dtype),
                "vbx_pitch_with_peaks_host")
    return dict(candidates=cand, n_cand=n, status=st)


Context.pitch = _pitch
Context.frame_peaks = _frame_peaks
Context.pitch_with_peaks = _pitch_with_peaks
Context.pitch_with_peaks_host = _pitch_with_peaks_host
Context.pitch_lag_function = _pitch_lag_function
Context.pitch_host = _pitch_host
Context.pitch_extract = _pitch_extract
Context.interpolate_sinc = _interpolate_sinc
Context.improve_extremum = _improve_extremum


# ---- MFCC and waves.rs helpers (appended to Context) -------------------------------------------------
def hz_to_mel(hz):
    return load_library().vbx_hz_to_mel(hz)


def mel_to_hz(mel):
    return load_library().vbx_mel_to_hz(mel)


def _mfcc(self, frames, num_coeffs, f_lo, f_hi, fs, n_keep=None, out_dtype=F64, want_energies=False):
    """spectrum.rs:410-440 mfcc over frames → device array [F][n_keep] (and the log-energies [F][num_coeffs])."""
    n_keep = num_coeffs if n_keep is None else n_keep
    out = self.empty((frames.n_frames, n_keep), _NP[out_dtype])
    en = self.empty((frames.n_frames, num_coeffs), _NP[out_dtype]) if want_energies else None
    self._check(self.lib.vbx_mfcc(self.h, C.byref(frames), num_coeffs, n_keep, f_lo, f_hi, fs, out.ptr,
                                  en.ptr if en else None, out_dtype), "vbx_mfcc")
    return (out, en) if want_energies else out


def _mfcc_host(self, audio, n_frames, frame_len, stride, window, num_coeffs, f_lo, f_hi, fs, n_keep=None, out_dtype=F64,
               frames_per_segment=0, segment_stride=0, sample_dtype=None, channels=1):
    audio = np.ascontiguousarray(audio)
    n_keep = num_coeffs if n_keep is None else n_keep
    fr, n_frames = self._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, _sample_dtype(audio, sample_dtype),
                                   frames_per_segment, segment_stride, channels)
    out = np.zeros((n_frames, n_keep), dtype=_NP[out_dtype])
    self._check(self.lib.vbx_mfcc_host(self.h, C.byref(fr), num_coeffs, n_keep, f_lo, f_hi, fs, out.ctypes.data, out_dtype),
                "vbx_mfcc_host")
    return out


def _dct(self, signal):
    x = np.atleast_2d(np.ascontiguousarray(signal))
    d = self.to_device(x)
    out = self.empty(x.shape, x.dtype)
    self._check(self.lib.vbx_dct(self.h, d.ptr, _dt_of(x), x.shape[0], x.shape[1], out.ptr), "vbx_dct")
    return out.to_host()


def _rows_op(self, name, x):
    x = np.atleast_2d(np.ascontiguousarray(x))
    d = self.to_device(x)
    out = self.empty((x.shape[0],), x.dtype)
    self._check(getattr(self.lib, name)(self.h, d.ptr, _dt_of(x), x.shape[0], x.shape[1], x.shape[1], out.ptr), name)
    return out.to_host()


def _normalize(self, x, maxes=None):
    x = np.atleast_2d(np.ascontiguousarray(x))
    d = self.to_device(x)
    m = self.to_device(np.ascontiguousarray(maxes, dtype=x.dtype)) if maxes is not None else None
    self._check(self.lib.vbx_normalize(self.h, d.ptr, _dt_of(x), x.shape[0], x.shape[1], x.shape[1], m.ptr if m else None),
                "vbx_normalize")
    return d.to_host()


def _preemphasis(self, x, factor):
    x = np.atleast_2d(np.ascontiguousarray(x))
    d = self.to_device(x)
    self._check(self.lib.vbx_preemphasis(self.h, d.ptr, _dt_of(x), x.shape[0], x.shape[1], x.shape[1], factor),
                "vbx_preemphasis")
    return d.to_host()


Context.mfcc = _mfcc
Context.mfcc_set_fft_precision = lambda self, dtype: self._check(self.lib.vbx_mfcc_set_fft_precision(self.h, dtype),
                                                                 "vbx_mfcc_set_fft_precision")
Context.mfcc_host = _mfcc_host
Context.dct = _dct
Context.rms = lambda self, x: _rows_op(self, "vbx_rms", x)
Context.max_amplitude = lambda self, x: _rows_op(self, "vbx_max_amplitude", x)
Context.normalize = _normalize
Context.preemphasis = _preemphasis


def _find_formants_resampled(self, frames, fs, ratio, p, estimates, dtype=F64):
    """lib.rs:40-116 with resample_ratio != 1 over a device view.  estimates: host [n_segments][k][2]."""
    F = frames.n_frames
    J = frames.frames_per_segment or F
    segs = F // J if J else 0
    est = np.ascontiguousarray(estimates, dtype=_NP[dtype])
    k = est.shape[-2]
    d_est = self.to_device(est.reshape(segs, k, 2))
    tracks = self.empty((F, k, 2), _NP[dtype])
    res = self.empty((F, MAX_RESONANCES, 2), _NP[dtype])
    nres = self.empty((F,), np.int32)
    st = self.empty((F,), np.uint8)
    self._check(self.lib.vbx_find_formants_resampled(self.h, C.byref(frames), fs, ratio, p, d_est.ptr, k, tracks.ptr, res.ptr,
                                                     nres.ptr, st.ptr, dtype), "vbx_find_formants_resampled")
    return dict(tracks=tracks.to_host(), estimates=d_est.to_host(), resonances=res.to_host(), n_res=nres.to_host(),
                status=st.to_host())


Context.find_formants_resampled = _find_formants_resampled


def _autocorrelate_ring(self, rings, heads, n, n_lags, out_dtype=F64):
    """periodic.rs:291-304 Autocorrelate for VecDeque: rings host [B][capacity], heads [B] → r [B][n_lags]."""
    rings = np.atleast_2d(np.ascontiguousarray(rings))
    d = self.to_device(rings)
    h = self.to_device(np.ascontiguousarray(heads, dtype=np.int64))
    r = self.empty((rings.shape[0], n_lags), _NP[out_dtype])
    self._check(self.lib.vbx_autocorrelate_ring(self.h, d.ptr, _dt_of(rings), rings.shape[0], rings.shape[1], h.ptr, n, n_lags,
                                                r.ptr, out_dtype), "vbx_autocorrelate_ring")
    return r.to_host()


Context.autocorrelate_ring = _autocorrelate_ring


def _pitch_viterbi(self, cand, n_cand, n_segments, voiced_unvoiced_cost=0.14, octave_jump_cost=0.35, octave_cost=0.01, ceiling_hz=600.0):
    """Viterbi path over vbx_pitch's candidate lists (device arrays) → (path [F][2], index [F]) device arrays."""
    F, K = cand.shape[0], cand.shape[1]
    path = self.empty((F, 2), cand.dtype)
    idx = self.empty((F,), np.int32)
    self._check(self.lib.vbx_pitch_viterbi(self.h, cand.ptr, _dt_of(cand), n_cand.ptr if n_cand is not None else None, n_segments,
                                           F // n_segments, K, voiced_unvoiced_cost, octave_jump_cost, octave_cost, ceiling_hz,
                                           path.ptr, idx.ptr), "vbx_pitch_viterbi")
    return path, idx


Context.pitch_viterbi = _pitch_viterbi


def _find_formants_buffered(self, frames, fs, ratio, resampled_buf_len, p, estimates, dtype=F64):
    """lib.rs:40-116 with the literal resampled_buf semantics (SURVEY A.10) over a device view."""
    F = frames.n_frames
    J = frames.frames_per_segment or F
    segs = F // J if J else 0
    est = np.ascontiguousarray(estimates, dtype=_NP[dtype])
    k = est.shape[-2]
    d_est = self.to_device(est.reshape(segs, k, 2))
    tracks = self.empty((F, k, 2), _NP[dtype])
    res = self.empty((F, MAX_RESONANCES, 2), _NP[dtype])
    nres = self.empty((F,), np.int32)
    st = self.empty((F,), np.uint8)
    self._check(self.lib.vbx_find_formants_buffered(self.h, C.byref(frames), fs, ratio, resampled_buf_len, p, d_est.ptr, k,
                                                    tracks.ptr, res.ptr, nres.ptr, st.ptr, dtype), "vbx_find_formants_buffered")
    return dict(tracks=tracks.to_host(), estimates=d_est.to_host(), resonances=res.to_host(), n_res=nres.to_host(),
                status=st.to_host())


def _synth_speech(self, n_utts, n_samples, fs, seed=0x5EED, first_utt=0, dtype=F32, out=None):
    """Synthetic speech-like corpus generated on the device → DeviceArray [n_utts][n_samples] (csrc/vbx_synth.cu): dtype F32,
    I16, or MULAW8 / ALAW8 (the I16 samples G.711-encoded, uint8)."""
    d = out if out is not None else self.empty((n_utts, n_samples), _NP[dtype])
    self._check(self.lib.vbx_synth_speech(self.h, d.ptr, dtype, n_utts, n_samples, float(fs), seed, first_utt), "vbx_synth_speech")
    return d


Context.find_formants_buffered = _find_formants_buffered
Context.synth_speech = _synth_speech


def multi_partition(n_units, n_parts, part):
    lo, hi = _i64(0), _i64(0)
    load_library().vbx_multi_partition(n_units, n_parts, part, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


class _BorrowedContext(Context):
    """A device context owned by a Multi handle (never destroyed from Python)."""

    def __init__(self, lib, handle):
        self.lib, self.h = lib, _vp(handle)

    def close(self):
        self.h = None


class Multi:
    """vbx_multi: one worker thread + context per device; `_host` calls sharded by utterance, results gathered into the
    caller's single host arrays (no torch / NCCL).  Fails loudly without the library / a GPU."""

    def __init__(self, n_devices=0, devices=None):
        self.lib = load_library()
        h = _vp()
        arr = (C.c_int32 * len(devices))(*devices) if devices else None
        st = self.lib.vbx_multi_create(n_devices if not devices else len(devices), arr, C.byref(h))
        if st != OK:
            raise VoxBoxError(st, "vbx_multi_create failed: no usable CUDA device (there is no CPU fallback)")
        self.h = h
        self.n = self.lib.vbx_multi_device_count(h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.vbx_multi_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def ctx(self, i=0):
        return _BorrowedContext(self.lib, self.lib.vbx_multi_ctx(self.h, i))

    @property
    def kernel_launches(self):
        return self.lib.vbx_multi_kernel_launches(self.h)

    def _check(self, st, what):
        if st != OK:
            raise VoxBoxError(st, f"{what}: {self.lib.vbx_multi_last_error(self.h).decode()} [{self.lib.vbx_status_str(st).decode()}]")

    def h2d_bandwidth(self, bytes_per_device, reps=8, n_active=0):
        out = (C.c_double * self.n)()
        self._check(self.lib.vbx_multi_h2d_bandwidth(self.h, bytes_per_device, reps, n_active, out), "vbx_multi_h2d_bandwidth")
        return list(out)

    @staticmethod
    def _view(audio, n_frames, frame_len, stride, window, frames_per_segment, segment_stride, sample_dtype=None, channels=1):
        """(audio, view, number of frames) of a `_host` call (channel_view); an interleaved recording shards by channel, so
        at most `channels` devices get work."""
        audio = np.ascontiguousarray(audio)
        fr, F = Context._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, _sample_dtype(audio, sample_dtype),
                                   frames_per_segment, segment_stride, channels)
        return audio, fr, F

    def lpc_host(self, audio, n_frames, frame_len, stride, window, p, out_dtype=F64, frames_per_segment=0, segment_stride=0,
                 sample_dtype=None, channels=1):
        audio, fr, n_frames = self._view(audio, n_frames, frame_len, stride, window, frames_per_segment, segment_stride,
                                         sample_dtype, channels)
        r = np.zeros((n_frames, p + 1), dtype=_NP[out_dtype])
        ac = np.zeros((n_frames, p + 1), dtype=_NP[out_dtype])
        kc = np.zeros((n_frames, p), dtype=_NP[out_dtype])
        self._check(self.lib.vbx_multi_lpc_host(self.h, C.byref(fr), p, r.ctypes.data, ac.ctypes.data, kc.ctypes.data, out_dtype),
                    "vbx_multi_lpc_host")
        return r, ac, kc

    def find_formants_host(self, audio, n_frames, frame_len, stride, window, fs, p, method, estimates, dtype=F64,
                           frames_per_segment=0, segment_stride=0, sample_dtype=None, channels=1):
        audio, fr, n_frames = self._view(audio, n_frames, frame_len, stride, window, frames_per_segment, segment_stride,
                                         sample_dtype, channels)
        J = fr.frames_per_segment or n_frames
        segs = n_frames // J if J else 0
        est = np.ascontiguousarray(estimates, dtype=_NP[dtype]).reshape(segs, -1, 2).copy()
        k = est.shape[1]
        tracks = np.zeros((n_frames, k, 2), dtype=_NP[dtype])
        res = np.zeros((n_frames, MAX_RESONANCES, 2), dtype=_NP[dtype])
        nres = np.zeros(n_frames, dtype=np.int32)
        st = np.zeros(n_frames, dtype=np.uint8)
        self._check(self.lib.vbx_multi_find_formants_host(self.h, C.byref(fr), fs, p, method, est.ctypes.data, k, tracks.ctypes.data,
                                                          res.ctypes.data, nres.ctypes.data, st.ctypes.data, dtype),
                    "vbx_multi_find_formants_host")
        return dict(tracks=tracks, estimates=est, resonances=res, n_res=nres, status=st)

    def pitch_host(self, audio, n_frames, frame_len, stride, window, fs, threshold, fmin, fmax, max_cand=16, out_dtype=F64,
                   frames_per_segment=0, segment_stride=0, sample_dtype=None, channels=1):
        audio, fr, n_frames = self._view(audio, n_frames, frame_len, stride, window, frames_per_segment, segment_stride,
                                         sample_dtype, channels)
        cand = np.zeros((n_frames, max_cand, 2), dtype=_NP[out_dtype])
        n = np.zeros(n_frames, dtype=np.int32)
        st = np.zeros(n_frames, dtype=np.uint8)
        self._check(self.lib.vbx_multi_pitch_host(self.h, C.byref(fr), fs, threshold, fmin, fmax, max_cand, cand.ctypes.data,
                                                  n.ctypes.data, st.ctypes.data, out_dtype), "vbx_multi_pitch_host")
        return dict(candidates=cand, n_cand=n, status=st)

    def pitch_with_peaks_host(self, audio, n_frames, frame_len, stride, window, fs, threshold, silence_threshold, fmin, fmax,
                              max_cand=16, out_dtype=F64, frames_per_segment=0, segment_stride=0, local_peaks=None,
                              global_peaks=None, sample_dtype=None, channels=1):
        """Context.pitch_with_peaks_host sharded over the devices (vbx_multi_pitch_with_peaks_host)."""
        audio, dt = _host_audio(audio, sample_dtype)
        fr, n_frames = Context._host_view(audio.ctypes.data, n_frames, frame_len, stride, window, dt, frames_per_segment,
                                          segment_stride, channels)
        lp = _host_peaks(local_peaks, n_frames)
        gp = _host_peaks(global_peaks, _n_segments(n_frames, fr.frames_per_segment))
        cand = np.zeros((n_frames, max_cand, 2), dtype=_NP[out_dtype])
        n = np.zeros(n_frames, dtype=np.int32)
        st = np.zeros(n_frames, dtype=np.uint8)
        self._check(self.lib.vbx_multi_pitch_with_peaks_host(self.h, C.byref(fr), fs, threshold, silence_threshold,
                                                             lp.ctypes.data if lp is not None else None,
                                                             gp.ctypes.data if gp is not None else None, fmin, fmax, max_cand,
                                                             cand.ctypes.data, n.ctypes.data, st.ctypes.data, out_dtype),
                    "vbx_multi_pitch_with_peaks_host")
        return dict(candidates=cand, n_cand=n, status=st)

    def mfcc_host(self, audio, n_frames, frame_len, stride, window, num_coeffs, f_lo, f_hi, fs, n_keep=None, out_dtype=F64,
                  frames_per_segment=0, segment_stride=0, sample_dtype=None, channels=1):
        audio, fr, n_frames = self._view(audio, n_frames, frame_len, stride, window, frames_per_segment, segment_stride,
                                         sample_dtype, channels)
        n_keep = num_coeffs if n_keep is None else n_keep
        out = np.zeros((n_frames, n_keep), dtype=_NP[out_dtype])
        self._check(self.lib.vbx_multi_mfcc_host(self.h, C.byref(fr), num_coeffs, n_keep, f_lo, f_hi, fs, out.ctypes.data, out_dtype),
                    "vbx_multi_mfcc_host")
        return out
