"""Interleaved multi-channel views (vbx_frames.sample_step) on the GPU.  The header defines every result by the planar
equivalent of the view: each test builds that array in numpy exactly as the header states it (interleave_util), uploads it,
and asserts np.array_equal between the call on the interleaved view and the same call on the planar view.  Covered: every
entry point that takes a vbx_frames, C = 1 (step 0 against step 1), 2, 3 and 6 channels, f32 / i16 / mu-law / A-law samples
(and f64 where the path takes them), the telephone framing (8 kHz, 200 / 80), the C3 framing (44.1 kHz, 1102 / 441) and the
400-sample MFCC framing of mfcc_lane5_kernel, the `_host` twins with per-frame time chunks and with the default chunking, the
`Multi` twins on every visible device, the argument checks, a stereo mu-law recording of real speech against the f64 oracle,
and the kernels a contiguous view launches."""
import ctypes as C
import os

import numpy as np
import pytest

from g711_codec import DECODE, ENCODE
from gpu_util import ctx, normwise, synth, vb
from interleave_util import planar_equivalent

pytestmark = pytest.mark.gpu
MALE = np.array([[f, 1.0] for f in (320., 1440., 2760., 3200.)])
DTYPES = {"f32": vb.F32, "i16": vb.I16, "mulaw": vb.MULAW8, "alaw": vb.ALAW8, "f64": vb.F64}
NP = {vb.F32: np.float32, vb.I16: np.int16, vb.MULAW8: np.uint8, vb.ALAW8: np.uint8, vb.F64: np.float64}
# (fs, N, hop): the telephone framing, C3's framing, and the 400-sample framing of mfcc_lane5_kernel
TEL, C3, LANE5 = (8000.0, 200, 80), (44100.0, 1102, 441), (16000.0, 400, 160)


def _recording(n, channels, dtype, fs, seed=0):
    """[n][channels] samples (the WAV layout) of synthetic speech, a different utterance per channel."""
    x = np.stack([synth.utterance(seed + 11 * ch, fs, seconds=n / fs + 0.01)[:n] for ch in range(channels)], axis=1)
    x = x.astype(np.float64) / np.max(np.abs(x))
    if dtype in (vb.F32, vb.F64):
        return (0.7 * x).astype(NP[dtype])
    pcm = np.round(x * 30000).astype(np.int16)
    if dtype == vb.I16:
        return pcm
    return ENCODE["mulaw" if dtype == vb.MULAW8 else "alaw"](pcm)


def _host(v):
    if isinstance(v, vb.DeviceArray):
        return v.to_host()
    if isinstance(v, dict):
        return {k: _host(x) for k, x in v.items()}
    if isinstance(v, (tuple, list)):
        return [_host(x) for x in v]
    return v


def assert_same(a, b, what=""):
    a, b = _host(a), _host(b)
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            assert_same(a[k], b[k], f"{what}.{k}")
    elif isinstance(a, list):
        assert len(a) == len(b)
        for i, (x, y) in enumerate(zip(a, b)):
            assert_same(x, y, f"{what}[{i}]")
    elif a is None:
        assert b is None, what
    else:
        assert np.array_equal(a, b, equal_nan=True), what


class Rec:
    """One interleaved recording on the device, and the views of one framing over it: the interleaved view with a segment per
    channel (or, with `channel`, a single-segment view of that channel) and its planar equivalent, uploaded as the header
    defines it."""

    def __init__(self, c, x, dtype):
        self.c, self.x, self.dt = c, x, dtype
        self.flat = np.ascontiguousarray(x).reshape(-1)
        self.d = c.to_device(self.flat)
        self.n, self.C = x.shape
        self._keep = []

    def views(self, N, hop, window, channel=None, step=None):
        c, C_ = self.c, self.C
        J = c.n_frames_of(self.n, N, hop)
        s = C_ if step is None else step
        es = np.dtype(NP[self.dt]).itemsize
        if channel is None:
            kw = dict(n_frames=C_ * J, frame_len=N, frame_stride=hop * s, frames_per_segment=J, segment_stride=1, sample_step=s)
            base, buf = self.d.ptr, self.flat
        else:
            kw = dict(n_frames=J, frame_len=N, frame_stride=hop * s, sample_step=s)
            base, buf = self.d.ptr + channel * es, self.flat[channel:]
        inter = c.frames(base, kw["n_frames"], N, kw["frame_stride"], window, self.dt, kw.get("frames_per_segment", 0),
                         kw.get("segment_stride", 0), s)
        P, pv = planar_equivalent(buf, **kw)
        dp = c.to_device(P)
        self._keep.append(dp)
        planar = c.frames(dp.ptr, pv["n_frames"], N, pv["frame_stride"], window, self.dt, pv["frames_per_segment"],
                          pv["segment_stride"])
        return inter, planar


def _segments(fr):
    return fr.n_frames // fr.frames_per_segment if fr.frames_per_segment else 1


def _same(fn, rec, N, hop, window, what, **kw):
    inter, planar = rec.views(N, hop, window, **kw)
    assert_same(fn(inter), fn(planar), what)


def _device_paths(rec, fs, N, hop, f64):
    """Every frame-view entry point on one framing."""
    c = rec.c
    _same(lambda fr: c.autocorrelate(fr, 13), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "autocorrelate")
    _same(lambda fr: c.lpc(fr, 12), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "lpc")
    _same(lambda fr: c.lpc(fr, 30), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "lpc-30")
    if not f64:  # the autocorrelation formant chain stages fp32 / integer samples
        _same(lambda fr: c.find_formants(fr, fs, 12, vb.LPC_AUTOCORR, np.repeat(MALE[None], _segments(fr), 0)), rec, N, hop,
              vb.WINDOW_HANN_SYMMETRIC, "find_formants autocorr")
    _same(lambda fr: c.lpc_burg(fr, 12), rec, N, hop, vb.WINDOW_HANN_PERIODIC, "lpc_burg")
    _same(lambda fr: c.find_formants(fr, fs, 12, vb.LPC_BURG, np.repeat(MALE[None], _segments(fr), 0)), rec, N, hop,
          vb.WINDOW_HANN_PERIODIC, "find_formants burg")
    _same(lambda fr: c.find_formants_resampled(fr, 10000.0, 10000.0 / fs, 10, np.repeat(MALE[None], _segments(fr), 0)), rec, N,
          hop, vb.WINDOW_NONE, "find_formants_resampled")
    _same(lambda fr: c.find_formants_buffered(fr, fs, 1.0, N + 37, 10, np.repeat(MALE[None], _segments(fr), 0)), rec, N, hop,
          vb.WINDOW_NONE, "find_formants_buffered")
    _same(lambda fr: c.pitch(fr, fs, 0.45, 75.0, 600.0, 16), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "pitch")
    _same(lambda fr: c.pitch_with_peaks(fr, fs, 0.45, 0.03, 75.0, 600.0, 16), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC,
          "pitch_with_peaks computed")
    _same(lambda fr: c.frame_peaks(fr), rec, N, hop, vb.WINDOW_NONE, "frame_peaks")
    _same(lambda fr: c.pitch_lag_function(fr), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "pitch_lag_function")
    # caller-given peaks (half the computed ones, so that the voiceless strength changes)
    inter, planar = rec.views(N, hop, vb.WINDOW_HANN_SYMMETRIC)
    loc, glo = (c.to_device(0.5 * a.to_host()) for a in c.frame_peaks(planar))
    assert_same(c.pitch_with_peaks(inter, fs, 0.45, 0.03, 75.0, 600.0, 16, local_peaks=loc, global_peaks=glo),
                c.pitch_with_peaks(planar, fs, 0.45, 0.03, 75.0, 600.0, 16, local_peaks=loc, global_peaks=glo), "pitch_with_peaks given")
    hi = min(6855.0, 0.45 * fs)
    _same(lambda fr: c.mfcc(fr, 26, 100.0, hi, fs, n_keep=13, want_energies=True), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "mfcc")


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("channels", [2, 3, 6])
@pytest.mark.parametrize("framing", [TEL, C3], ids=["tel", "c3"])
def test_device_paths_equal_planar(framing, channels, dt):
    fs, N, hop = framing
    dtype = DTYPES[dt]
    rec = Rec(ctx(), _recording(int(0.3 * fs), channels, dtype, fs, seed=channels), dtype)
    _device_paths(rec, fs, N, hop, dtype == vb.F64)


@pytest.mark.parametrize("dt", ["f32", "i16", "mulaw"])
def test_single_segment_channel_view(dt):
    """One channel of a 3-channel recording as a single-segment view (base offset by the channel)."""
    fs, N, hop = C3
    dtype = DTYPES[dt]
    rec = Rec(ctx(), _recording(int(0.3 * fs), 3, dtype, fs, seed=5), dtype)
    c = rec.c
    for ch in (0, 2):
        _same(lambda fr: c.lpc(fr, 12), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "lpc", channel=ch)
        _same(lambda fr: c.find_formants(fr, fs, 12, vb.LPC_BURG, MALE[None]), rec, N, hop, vb.WINDOW_HANN_PERIODIC, "ff", channel=ch)
        _same(lambda fr: c.pitch_with_peaks(fr, fs, 0.45, 0.03, 75.0, 600.0, 16), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "pwp",
              channel=ch)
        _same(lambda fr: c.mfcc(fr, 26, 100.0, 6855.0, fs, n_keep=13), rec, N, hop, vb.WINDOW_HANN_SYMMETRIC, "mfcc", channel=ch)


@pytest.mark.parametrize("dt", list(DTYPES))
def test_one_channel_step_one_is_step_zero(dt):
    """C = 1: sample_step 1 and 0 are the same contiguous view, with the same kernels."""
    fs, N, hop = C3
    dtype = DTYPES[dt]
    rec = Rec(ctx(), _recording(int(0.3 * fs), 1, dtype, fs, seed=1), dtype)
    c = rec.c
    J = c.n_frames_of(rec.n, N, hop)
    for win, fn in ((vb.WINDOW_HANN_PERIODIC, lambda fr: c.find_formants(fr, fs, 12, vb.LPC_BURG, MALE[None])),
                    (vb.WINDOW_HANN_SYMMETRIC, lambda fr: c.pitch_with_peaks(fr, fs, 0.45, 0.03, 75.0, 600.0, 16)),
                    (vb.WINDOW_HANN_SYMMETRIC, lambda fr: c.mfcc(fr, 26, 100.0, 6855.0, fs, n_keep=13))):
        outs, names = [], []
        for step in (0, 1):
            c.profile_begin()
            outs.append(_host(fn(c.frames(rec.d.ptr, J, N, hop, win, dtype, sample_step=step))))
            names.append(sorted(c.profile_end()))
        assert_same(outs[0], outs[1])
        assert names[0] == names[1] and not any("interleave" in k for k in names[0]), names


def test_mfcc_lane5_framing():
    """400 / 160 at 16 kHz: the planar rows keep mfcc_lane5_kernel's alignment, and the interleaved view takes it too."""
    fs, N, hop = LANE5
    c = ctx()
    for dtype in (vb.F32, vb.I16, vb.MULAW8, vb.ALAW8):
        for channels in (2, 3):
            rec = Rec(c, _recording(int(0.5 * fs), channels, dtype, fs, seed=9), dtype)
            inter, planar = rec.views(N, hop, vb.WINDOW_HANN_SYMMETRIC)
            c.profile_begin()
            a = c.mfcc(inter, 40, 133.0, 6855.0, fs, n_keep=13).to_host()
            names = c.profile_end()
            assert_same(a, c.mfcc(planar, 40, 133.0, 6855.0, fs, n_keep=13))
            assert "mfcc_lane5_kernel" in names and "interleave_gather_kernel" in names, names


def test_strided_gather_geometry():
    """Segments that do not share memory (channel 1 of a batch of equally long stereo files): the strided gather kernel."""
    fs, N, hop = TEL
    c = ctx()
    files = np.stack([_recording(4000, 2, vb.I16, fs, seed=20 + k) for k in range(3)])  # [file][time][channel]
    flat = files.reshape(-1)
    d = c.to_device(flat)
    J = c.n_frames_of(4000, N, hop)
    inter = c.frames(d.ptr + 2, 3 * J, N, hop * 2, vb.WINDOW_HANN_SYMMETRIC, vb.I16, J, 8000, 2)
    P, pv = planar_equivalent(flat[1:], 3 * J, N, hop * 2, J, 8000, 2)
    dp = c.to_device(P)
    planar = c.frames(dp.ptr, 3 * J, N, pv["frame_stride"], vb.WINDOW_HANN_SYMMETRIC, vb.I16, J, pv["segment_stride"])
    c.profile_begin()
    a = c.lpc(inter, 12)
    names = c.profile_end()
    assert "interleave_gather_strided_kernel" in names, names
    assert_same(a, c.lpc(planar, 12))
    assert_same(c.find_formants(inter, fs, 12, vb.LPC_BURG, np.repeat(MALE[None], 3, 0)),
                c.find_formants(planar, fs, 12, vb.LPC_BURG, np.repeat(MALE[None], 3, 0)))


# ---- host twins ----------------------------------------------------------------------------------------------------------------
# channels=1 is the contiguous single-segment view, whose frame chunks are uploaded as they are (their alignment follows the
# chunk start); it is checked on the telephone framing, whose hop keeps every chunk at the same 16-sample alignment
@pytest.mark.parametrize("chunk_mb", ["0", None], ids=["frame-chunks", "default"])
@pytest.mark.parametrize("dt", ["f32", "i16", "mulaw", "alaw"])
@pytest.mark.parametrize("framing,channels", [(TEL, 1), (TEL, 2), (TEL, 3), (TEL, 6), (C3, 2), (C3, 3), (C3, 6)],
                         ids=["tel-1", "tel-2", "tel-3", "tel-6", "c3-2", "c3-3", "c3-6"])
def test_host_twins_equal_planar_device(monkeypatch, framing, channels, dt, chunk_mb):
    """The `_host` helpers with channels=C against the device call on the planar equivalent.  VBX_HOST_CHUNK_MB=0 cuts the
    view into one frame time per chunk, so the tracker state (est_inout) carries across every chunk; with C3's odd hop of 441
    samples every chunk starts at a different alignment, which the pipeline's gather restores."""
    if chunk_mb is not None:
        monkeypatch.setenv("VBX_HOST_CHUNK_MB", chunk_mb)
    else:
        monkeypatch.delenv("VBX_HOST_CHUNK_MB", raising=False)
    fs, N, hop = framing
    dtype = DTYPES[dt]
    c = ctx()
    x = _recording(int(0.4 * fs), channels, dtype, fs, seed=30 + channels)
    rec = Rec(c, x, dtype)
    J = c.n_frames_of(rec.n, N, hop)
    sd = dtype if dtype in (vb.MULAW8, vb.ALAW8) else None
    kw = dict(sample_dtype=sd, channels=channels)
    _, pl = rec.views(N, hop, vb.WINDOW_HANN_SYMMETRIC)
    assert_same(c.lpc_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, 12, **kw), c.lpc(pl, 12), "lpc_host")
    assert_same(c.autocorrelate_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, 13, **kw), c.autocorrelate(pl, 13), "ac_host")
    assert_same(c.mfcc_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, 26, 100.0, 0.45 * fs, fs, n_keep=13, **kw),
                c.mfcc(pl, 26, 100.0, 0.45 * fs, fs, n_keep=13), "mfcc_host")
    assert_same(c.pitch_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 75.0, 600.0, 16, **kw),
                c.pitch(pl, fs, 0.45, 75.0, 600.0, 16), "pitch_host")
    assert_same(c.pitch_with_peaks_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 0.03, 75.0, 600.0, 16, **kw),
                c.pitch_with_peaks(pl, fs, 0.45, 0.03, 75.0, 600.0, 16), "pitch_with_peaks_host computed")
    loc, glo = (0.5 * a.to_host() for a in c.frame_peaks(pl))
    assert_same(c.pitch_with_peaks_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 0.03, 75.0, 600.0, 16, local_peaks=loc,
                                        global_peaks=glo, **kw),
                c.pitch_with_peaks(pl, fs, 0.45, 0.03, 75.0, 600.0, 16, local_peaks=c.to_device(loc), global_peaks=c.to_device(glo)),
                "pitch_with_peaks_host given")
    est = np.repeat(MALE[None], channels, 0)
    for method, win in ((vb.LPC_BURG, vb.WINDOW_HANN_PERIODIC), (vb.LPC_AUTOCORR, vb.WINDOW_HANN_SYMMETRIC)):
        _, plw = rec.views(N, hop, win)
        assert_same(c.find_formants_host(x, J, N, hop, win, fs, 12, method, est, **kw), c.find_formants(plw, fs, 12, method, est),
                    f"find_formants_host {method}")


def test_host_twin_f64_pitch_with_peaks(monkeypatch):
    monkeypatch.setenv("VBX_HOST_CHUNK_MB", "0")
    fs, N, hop = TEL
    c = ctx()
    x = _recording(3000, 2, vb.F64, fs, seed=3)
    rec = Rec(c, x, vb.F64)
    _, pl = rec.views(N, hop, vb.WINDOW_HANN_SYMMETRIC)
    J = c.n_frames_of(rec.n, N, hop)
    assert_same(c.pitch_with_peaks_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 0.03, 75.0, 600.0, 16, channels=2),
                c.pitch_with_peaks(pl, fs, 0.45, 0.03, 75.0, 600.0, 16))


@pytest.mark.parametrize("channels", [2, 6])
def test_multi_every_device(channels):
    fs, N, hop = TEL
    m = vb.Multi()
    try:
        c = m.ctx(0)
        x = _recording(int(0.4 * fs), channels, vb.MULAW8, fs, seed=40 + channels)
        rec = Rec(c, x, vb.MULAW8)
        J = c.n_frames_of(rec.n, N, hop)
        kw = dict(sample_dtype=vb.MULAW8, channels=channels)
        _, pl = rec.views(N, hop, vb.WINDOW_HANN_SYMMETRIC)
        _, plp = rec.views(N, hop, vb.WINDOW_HANN_PERIODIC)
        assert_same(m.lpc_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, 12, **kw), c.lpc(pl, 12))
        assert_same(m.mfcc_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, 26, 100.0, 3600.0, fs, n_keep=13, **kw),
                    c.mfcc(pl, 26, 100.0, 3600.0, fs, n_keep=13))
        assert_same(m.pitch_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 75.0, 600.0, 16, **kw),
                    c.pitch(pl, fs, 0.45, 75.0, 600.0, 16))
        assert_same(m.pitch_with_peaks_host(x, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 0.03, 75.0, 600.0, 16, **kw),
                    c.pitch_with_peaks(pl, fs, 0.45, 0.03, 75.0, 600.0, 16))
        est = np.repeat(MALE[None], channels, 0)
        assert_same(m.find_formants_host(x, J, N, hop, vb.WINDOW_HANN_PERIODIC, fs, 12, vb.LPC_BURG, est, **kw),
                    c.find_formants(plp, fs, 12, vb.LPC_BURG, est))
    finally:
        m.close()


# ---- argument checks -------------------------------------------------------------------------------------------------------------
def test_bad_steps_are_badarg():
    c = ctx()
    d = c.to_device(np.zeros(8192, dtype=np.float32))
    h = np.zeros(8192, dtype=np.float32)
    out = c.empty((1 << 16,), np.float64)
    o, st, n = out.ptr, c.empty((64,), np.uint8).ptr, c.empty((64,), np.int32).ptr
    ho, hn, hst = np.zeros(1 << 16), np.zeros(64, np.int32), np.zeros(64, np.uint8)
    est = c.to_device(np.repeat(MALE[None], 2, 0))
    hest = np.repeat(MALE[None], 2, 0).copy()
    L, mh = c.lib, None
    bads = [dict(step=-1, fst=80), dict(step=2, fst=81), dict(step=3, fst=80)]
    for b in bads:
        for base, host in ((d.ptr, False), (h.ctypes.data, True)):
            fr = C.byref(c.frames(base, 4, 100, b["fst"], vb.WINDOW_HANN_SYMMETRIC, vb.F32, 2, 1, b["step"]))
            frn = C.byref(c.frames(base, 4, 100, b["fst"], vb.WINDOW_NONE, vb.F32, 2, 1, b["step"]))
            if host:
                calls = [L.vbx_autocorrelate_host(c.h, fr, 8, ho.ctypes.data, vb.F64),
                         L.vbx_lpc_host(c.h, fr, 8, ho.ctypes.data, ho.ctypes.data, None, vb.F64),
                         L.vbx_find_formants_host(c.h, fr, 8000.0, 8, vb.LPC_BURG, hest.ctypes.data, 4, ho.ctypes.data, None, None,
                                                  None, vb.F64),
                         L.vbx_pitch_host(c.h, fr, 8000.0, 0.45, 75.0, 600.0, 4, ho.ctypes.data, hn.ctypes.data, hst.ctypes.data, vb.F64),
                         L.vbx_pitch_with_peaks_host(c.h, fr, 8000.0, 0.45, 0.03, None, None, 75.0, 600.0, 4, ho.ctypes.data, None,
                                                     None, vb.F64),
                         L.vbx_mfcc_host(c.h, fr, 13, 13, 100.0, 3600.0, 8000.0, ho.ctypes.data, vb.F64)]
            else:
                calls = [L.vbx_autocorrelate(c.h, fr, 8, o, vb.F64), L.vbx_lpc(c.h, fr, 8, o, o, None, vb.F64),
                         L.vbx_lpc_burg(c.h, fr, 8, o, st, vb.F64),
                         L.vbx_find_formants(c.h, fr, 8000.0, 8, vb.LPC_BURG, est.ptr, 4, o, None, None, None, vb.F64),
                         L.vbx_find_formants(c.h, fr, 8000.0, 8, vb.LPC_AUTOCORR, est.ptr, 4, o, None, None, None, vb.F64),
                         L.vbx_find_formants_resampled(c.h, frn, 8000.0, 0.5, 8, est.ptr, 4, o, o, n, st, vb.F64),
                         L.vbx_find_formants_buffered(c.h, frn, 8000.0, 1.0, 150, 8, est.ptr, 4, o, o, n, st, vb.F64),
                         L.vbx_pitch(c.h, fr, 8000.0, 0.45, 75.0, 600.0, 4, o, n, st, vb.F64),
                         L.vbx_pitch_with_peaks(c.h, fr, 8000.0, 0.45, 0.03, None, None, 75.0, 600.0, 4, o, n, st, vb.F64),
                         L.vbx_frame_peaks(c.h, frn, o, o),
                         L.vbx_pitch_lag_function(c.h, fr, o),
                         L.vbx_mfcc(c.h, fr, 13, 13, 100.0, 3600.0, 8000.0, o, None, vb.F64)]
            assert calls == [vb.ERR_BADARG] * len(calls), (b, host, calls)
    # an extent past int64
    big = C.byref(c.frames(d.ptr, 4, 100, 1 << 61, vb.WINDOW_NONE, vb.F32, 2, 1, 2))
    assert L.vbx_frame_peaks(c.h, big, o, o) == vb.ERR_BADARG
    m = vb.Multi()
    try:
        fr = C.byref(c.frames(h.ctypes.data, 4, 100, 81, vb.WINDOW_HANN_SYMMETRIC, vb.F32, 2, 1, 2))
        assert m.lib.vbx_multi_lpc_host(m.h, fr, 8, ho.ctypes.data, ho.ctypes.data, None, vb.F64) == vb.ERR_BADARG
        assert m.lib.vbx_multi_mfcc_host(m.h, fr, 13, 13, 100.0, 3600.0, 8000.0, ho.ctypes.data, vb.F64) == vb.ERR_BADARG
        assert m.lib.vbx_multi_pitch_host(m.h, fr, 8000.0, 0.45, 75.0, 600.0, 4, ho.ctypes.data, None, None, vb.F64) == vb.ERR_BADARG
        assert m.lib.vbx_multi_pitch_with_peaks_host(m.h, fr, 8000.0, 0.45, 0.03, None, None, 75.0, 600.0, 4, ho.ctypes.data, None,
                                                     None, vb.F64) == vb.ERR_BADARG
        assert m.lib.vbx_multi_find_formants_host(m.h, fr, 8000.0, 8, vb.LPC_BURG, hest.ctypes.data, 4, ho.ctypes.data, None, None,
                                                  None, vb.F64) == vb.ERR_BADARG
    finally:
        m.close()


# ---- real speech, stereo mu-law ----------------------------------------------------------------------------------------------
def test_stereo_mulaw_real_speech_vs_oracle(oracle, fixtures_dir):
    """Channel 0: tests/fixtures/sample-two_vowels.wav, channel 1: a synthetic utterance; both mu-law, interleaved, analysed by
    the `_host` helpers with channels=2.  Each channel's formants, pitch list and MFCC match the f64 oracle on that channel's
    decoded samples at the tolerances of test_gpu_real_speech.py."""
    x, fs = oracle.read_wav(os.path.join(fixtures_dir, "sample-two_vowels.wav"))
    other = synth.utterance(77, fs, seconds=x.size / fs + 0.01)[:x.size].astype(np.float64)
    other = 0.6 * other / np.max(np.abs(other))
    codes = np.stack([ENCODE["mulaw"](np.round(ch * 32767.0).astype(np.int16)) for ch in (x, other)], axis=1)  # [time][2]
    xs = DECODE["mulaw"](codes).astype(np.float64) / 32767.0
    c = ctx()
    kw = dict(sample_dtype=vb.MULAW8, channels=2)
    # formants: Burg on the 1102 / 441 framing
    N, hop = 1102, 441
    J = c.n_frames_of(x.size, N, hop)
    est = np.repeat(MALE[None], 2, 0)
    out = c.find_formants_host(codes, J, N, hop, vb.WINDOW_HANN_PERIODIC, fs, 12, vb.LPC_BURG, est, **kw)
    m = c.mfcc_host(codes, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, 40, 133.0, 6855.0, fs, n_keep=13, **kw)
    w = oracle.hanning_window(N)
    for ch in range(2):
        rows = slice(ch * J, (ch + 1) * J)
        state = MALE.copy()
        for f in range(J):
            o = oracle.find_formants(xs[f * hop:f * hop + N, ch].copy(), fs, 12, state)
            assert o["status"] == out["status"][ch * J + f] and o["n_res"] == out["n_res"][ch * J + f], (ch, f)
            if o["status"] == 0:
                state = o["formants"]
            assert np.max(np.abs(out["tracks"][ch * J + f] - state)) < 0.5, (ch, f)
        mo = np.stack([oracle.mfcc(xs[f * hop:f * hop + N, ch] * w, 40, 133.0, 6855.0, fs)[:13] for f in range(J)])
        assert np.max(normwise(m[rows], mo)) < 1e-5, ch
    # pitch: three periods of 75 Hz, 10 ms hop, every list position
    N, K = 1764, 48
    J = c.n_frames_of(x.size, N, hop)
    res = c.pitch_host(codes, J, N, hop, vb.WINDOW_HANN_SYMMETRIC, fs, 0.45, 75.0, 600.0, K, **kw)
    w = oracle.hanning_window(N)
    for ch in range(2):
        voiced = 0
        for f in range(J):
            rs, rc, extra = oracle.pitch(xs[f * hop:f * hop + N, ch] * w, fs, 0.45, 75.0, 600.0, max_cand=K)
            g = ch * J + f
            cand = res["candidates"][g]
            assert rs == res["status"][g] and extra["n_cand"] == res["n_cand"][g], (ch, f)
            k = rc.shape[0]
            assert (cand[0, 0] != 0) == (rc[0, 0] != 0), (ch, f)
            assert np.max(np.abs(cand[:k, 0] - rc[:, 0])) < 0.1 and np.max(np.abs(cand[:k, 1] - rc[:, 1])) < 1e-6, (ch, f)
            voiced += int(cand[0, 0] != 0)
        assert voiced > J // 4, ch
