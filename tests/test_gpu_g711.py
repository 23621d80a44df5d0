"""G.711 mu-law / A-law input (VBX_MULAW8 / VBX_ALAW8) on the GPU.  The header promises that every call on a G.711 view returns,
bit for bit, what the same call returns on a VBX_I16 view of the decoded samples; every device entry point that takes a frame
view is checked that way (np.array_equal) at shapes that reach each of its kernels, on input that holds all 256 codes.  The
`_host` twins equal the device call, vbx_synth_speech's G.711 output is the numpy encoder applied to its int16 output, the entry
points that take plain arrays reject the new dtypes, and real speech stored as mu-law matches the f64 oracle on the decoded
samples at the tolerances of test_gpu_real_speech.py."""
import ctypes as C
import os

import numpy as np
import pytest

from g711_codec import DECODE, ENCODE
from gpu_util import ctx, normwise, synth, vb

pytestmark = pytest.mark.gpu
LAWS = {"mulaw": vb.MULAW8, "alaw": vb.ALAW8}
MALE = np.array([[f, 1.0] for f in (320., 1440., 2760., 3200.)])


def _codes(law, n, seed=70, fs=16000):
    """n G.711 codes of synthetic speech, with every one of the 256 codes (in shuffled order) a third of the way in."""
    x = synth.utterance(seed, fs, seconds=n / fs + 0.01)[:n].astype(np.float64)
    assert x.size == n
    codes = ENCODE[law](np.round(x / np.max(np.abs(x)) * 30000).astype(np.int16))
    codes[n // 3:n // 3 + 256] = np.random.default_rng(seed).permutation(256).astype(np.uint8)
    return codes


class Pair:
    """The same samples on the device twice: as G.711 codes and as the int16 values they decode to."""

    def __init__(self, c, law, codes):
        self.c, self.dt = c, LAWS[law]
        self.d8, self.d16 = c.to_device(codes), c.to_device(DECODE[law](codes))

    def views(self, n_frames, N, hop, window, off=0, J=0, seg_stride=0):
        g = self.c.frames(self.d8.ptr + off, n_frames, N, hop, window, self.dt, J, seg_stride)
        i = self.c.frames(self.d16.ptr + 2 * off, n_frames, N, hop, window, vb.I16, J, seg_stride)
        return g, i


def _host(v):
    if isinstance(v, vb.DeviceArray):
        return v.to_host()
    if isinstance(v, dict):
        return {k: _host(x) for k, x in v.items()}
    if isinstance(v, (tuple, list)):
        return [_host(x) for x in v]
    return v


def assert_same(a, b):
    a, b = _host(a), _host(b)
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            assert_same(a[k], b[k])
    elif isinstance(a, list):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert_same(x, y)
    elif a is None:
        assert b is None
    else:
        assert np.array_equal(a, b, equal_nan=True)


def _both(fn, pair, *view_args, **view_kw):
    g, i = pair.views(*view_args, **view_kw)
    assert_same(fn(g), fn(i))


@pytest.fixture(scope="module", params=list(LAWS))
def law(request):
    return request.param


@pytest.fixture(scope="module")
def pair(law):
    return Pair(ctx(), law, _codes(law, 48000))


# ---- LPC / autocorrelation: every kernel plan_lpc can pick for integer samples ------------------------------------------
@pytest.mark.parametrize("off", [0, 5, 16])
def test_lpc_fused16(pair, off):
    """400 / 160 / LPC-12 (the C2 shape): lpc_fused16_kernel, 16-byte staging when the base is aligned, scalar otherwise."""
    c = pair.c
    F = c.n_frames_of(48000 - off, 400, 160)
    _both(lambda fr: c.lpc(fr, 12), pair, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, off)
    _both(lambda fr: c.autocorrelate(fr, 16), pair, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, off)


@pytest.mark.parametrize("off", list(range(16)))
def test_lpc_aligned(pair, off):
    """1102 / 441 / LPC-12 (the C3 shape): lpc_fuseda_kernel, whose walk starts every frame at its 4-sample alignment: base
    offsets of 0..15 bytes put the G.711 span at every position of a 16-byte load."""
    c = pair.c
    F = c.n_frames_of(48000 - off, 1102, 441)
    _both(lambda fr: c.lpc(fr, 12), pair, F, 1102, 441, vb.WINDOW_HANN_SYMMETRIC, off)
    _both(lambda fr: c.autocorrelate(fr, 13, out_dtype=vb.F32), pair, F, 1102, 441, vb.WINDOW_HANN_PERIODIC, off)


@pytest.mark.parametrize("seg_stride", [20 * 441 + 7, 20 * 441 + 1, 20 * 441 + 446])
def test_lpc_aligned_segments_odd_strides(pair, seg_stride):
    c = pair.c
    J, U = 20, 4
    assert (U - 1) * seg_stride + (J - 1) * 441 + 1102 + 3 <= 48000
    _both(lambda fr: c.lpc(fr, 12), pair, U * J, 1102, 441, vb.WINDOW_HANN_SYMMETRIC, 3, J, seg_stride)


@pytest.mark.parametrize("p", [13, 18, 24])
def test_lpc_general(pair, p):
    """14..25 lags on the 1102 / 441 framing: lpc_fused_kernel."""
    c = pair.c
    F = c.n_frames_of(48000 - 1, 1102, 441)
    _both(lambda fr: c.lpc(fr, p), pair, F, 1102, 441, vb.WINDOW_HANN_SYMMETRIC, 1)


def test_lpc_generic(pair, monkeypatch):
    """More than 25 lags, and every view with VBX_LPC_FORCE_GENERIC=1: autocorr_generic_kernel + Levinson."""
    c = pair.c
    F = c.n_frames_of(48000 - 3, 1102, 441)
    _both(lambda fr: c.lpc(fr, 30), pair, F, 1102, 441, vb.WINDOW_HANN_SYMMETRIC, 3)
    _both(lambda fr: c.autocorrelate(fr, 40), pair, F, 1102, 441, vb.WINDOW_NONE, 3)
    monkeypatch.setenv("VBX_LPC_FORCE_GENERIC", "1")
    _both(lambda fr: c.lpc(fr, 12), pair, F, 1102, 441, vb.WINDOW_HANN_SYMMETRIC, 3)
    F2 = c.n_frames_of(48000, 400, 160)
    _both(lambda fr: c.lpc(fr, 12), pair, F2, 400, 160, vb.WINDOW_HANN_SYMMETRIC)


# ---- MFCC -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("off", [0, 2, 1])
def test_mfcc_lane5(pair, off):
    """400-sample frames: mfcc_lane5_kernel on sample pairs; an odd base offset sends the view to mfcc_warp_kernel."""
    c = pair.c
    F = c.n_frames_of(48000 - off, 400, 160)
    _both(lambda fr: c.mfcc(fr, 40, 133.0, 6855.0, 16000.0, n_keep=13, want_energies=True), pair, F, 400, 160,
          vb.WINDOW_HANN_SYMMETRIC, off)


@pytest.mark.parametrize("N", [160, 200, 512, 441])
def test_mfcc_warp_and_generic(pair, N):
    """mfcc_warp_kernel (160, 200, 512) and the any-length mfcc_kernel (441), fp64 and fp32 transforms."""
    c = pair.c
    hi = 7000.0 if N >= 256 else 6000.0
    F = min(c.n_frames_of(48000 - 1, N, N // 2), 150)
    _both(lambda fr: c.mfcc(fr, 26, 100.0, hi, 16000.0, n_keep=13), pair, F, N, N // 2, vb.WINDOW_HANN_SYMMETRIC, 1)
    c.mfcc_set_fft_precision(vb.F32)
    try:
        _both(lambda fr: c.mfcc(fr, 26, 100.0, hi, 16000.0, n_keep=13), pair, F, N, N // 2, vb.WINDOW_HANN_SYMMETRIC, 1)
    finally:
        c.mfcc_set_fft_precision(vb.F64)


# ---- pitch --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,hop", [(240, 160), (640, 160), (9000, 4000)])
def test_pitch(pair, N, hop):
    c = pair.c
    F = c.n_frames_of(48000 - 1, N, hop)
    args = (F, N, hop, vb.WINDOW_HANN_SYMMETRIC, 1)
    _both(lambda fr: c.pitch(fr, 16000.0, 0.45, 75.0, 600.0, 16), pair, *args)
    _both(lambda fr: c.pitch_with_peaks(fr, 16000.0, 0.45, 0.03, 75.0, 600.0, 16), pair, *args)
    _both(lambda fr: c.frame_peaks(fr), pair, *args)
    _both(lambda fr: c.pitch_lag_function(fr), pair, *args)
    # the local peak is max |decoded| / 32767, as for int16
    g, _ = pair.views(*args)
    loc, _ = c.frame_peaks(g)
    dec = pair.d16.to_host().astype(np.float64)
    ref = np.array([np.max(np.abs(dec[1 + f * hop:1 + f * hop + N])) / 32767.0 for f in range(F)])
    assert np.array_equal(loc.to_host(), ref)


# ---- Burg and the formant paths ------------------------------------------------------------------------------------------------
def test_burg_and_formants(pair):
    c = pair.c
    F = c.n_frames_of(48000 - 7, 1102, 441)
    args = (F, 1102, 441, vb.WINDOW_HANN_PERIODIC, 7)
    _both(lambda fr: c.lpc_burg(fr, 12), pair, *args)
    _both(lambda fr: c.find_formants(fr, 44100.0, 12, vb.LPC_BURG, MALE[None]), pair, *args)
    _both(lambda fr: c.find_formants(fr, 44100.0, 12, vb.LPC_AUTOCORR, MALE[None]), pair, F, 1102, 441, vb.WINDOW_HANN_SYMMETRIC, 7)
    # several utterances (segments) with an odd segment stride
    J, U, S = 16, 5, 16 * 441 + 661
    _both(lambda fr: c.find_formants(fr, 44100.0, 12, vb.LPC_AUTOCORR, np.repeat(MALE[None], U, 0)), pair, U * J, 1102, 441,
          vb.WINDOW_HANN_SYMMETRIC, 1, J, S)


def test_formants_resampled_and_buffered(pair):
    c = pair.c
    F = min(c.n_frames_of(48000 - 3, 1024, 512), 60)
    args = (F, 1024, 512, vb.WINDOW_NONE, 3)
    _both(lambda fr: c.find_formants_resampled(fr, 10000.0, 10000.0 / 44100.0, 10, MALE[None]), pair, *args)
    _both(lambda fr: c.find_formants_resampled(fr, 16000.0, 1.0, 10, MALE[None]), pair, *args)
    _both(lambda fr: c.find_formants_buffered(fr, 16000.0, 0.9, 1500, 10, MALE[None]), pair, *args)


# ---- host twins ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("off", [0, 3])
def test_host_twins_equal_device(law, monkeypatch, off):
    """Many chunks (1 MB each) from a host array at an odd byte offset; framings whose kernels do not depend on where a chunk
    lands in device memory (the device call runs on a 256-byte-aligned copy, as the chunks do)."""
    monkeypatch.setenv("VBX_HOST_CHUNK_MB", "1")
    c = ctx()
    dt = LAWS[law]
    buf = _codes(law, 16000 * 200 + 3, seed=71)
    host = buf[off:off + 16000 * 200]
    assert host.ctypes.data % 2 == off % 2
    d = c.to_device(host)
    n = host.size
    F = c.n_frames_of(n, 400, 160)
    fr = c.frames(d.ptr, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, dt)
    assert_same(c.lpc_host(host, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 12, sample_dtype=dt), c.lpc(fr, 12))
    assert_same(c.autocorrelate_host(host, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 13, sample_dtype=dt), c.autocorrelate(fr, 13))
    assert_same(c.mfcc_host(host, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 40, 133.0, 6855.0, 16000.0, n_keep=13, sample_dtype=dt),
                c.mfcc(fr, 40, 133.0, 6855.0, 16000.0, n_keep=13))
    Fp = c.n_frames_of(n, 640, 160)
    frp = c.frames(d.ptr, Fp, 640, 160, vb.WINDOW_HANN_SYMMETRIC, dt)
    assert_same(c.pitch_host(host, Fp, 640, 160, vb.WINDOW_HANN_SYMMETRIC, 16000.0, 0.45, 75.0, 600.0, 16, sample_dtype=dt),
                c.pitch(frp, 16000.0, 0.45, 75.0, 600.0, 16))
    assert_same(c.pitch_with_peaks_host(host, Fp, 640, 160, vb.WINDOW_HANN_SYMMETRIC, 16000.0, 0.45, 0.03, 75.0, 600.0, 16,
                                        sample_dtype=dt),
                c.pitch_with_peaks(frp, 16000.0, 0.45, 0.03, 75.0, 600.0, 16))
    # utterances as segments: Burg find_formants, one utterance per chunk boundary region
    J, U = 98, 20
    S = n // U
    frs = c.frames(d.ptr, U * J, 400, 160, vb.WINDOW_HANN_PERIODIC, dt, J, S)
    est = np.repeat(MALE[None], U, 0)
    assert_same(c.find_formants_host(host, U * J, 400, 160, vb.WINDOW_HANN_PERIODIC, 16000.0, 12, vb.LPC_BURG, est,
                                     frames_per_segment=J, segment_stride=S, sample_dtype=dt),
                c.find_formants(frs, 16000.0, 12, vb.LPC_BURG, est))
    with pytest.raises(ValueError):
        c.lpc_host(host, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 12)


def test_multi_two_devices(law):
    m = vb.Multi()
    try:
        if m.n < 2:
            pytest.skip("needs two visible GPUs")
        dt = LAWS[law]
        host = _codes(law, 16000 * 60, seed=72)
        c = m.ctx(0)
        d = c.to_device(host)
        F = c.n_frames_of(host.size, 400, 160)
        fr = c.frames(d.ptr, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, dt)
        assert_same(m.lpc_host(host, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 12, sample_dtype=dt), c.lpc(fr, 12))
        assert_same(m.mfcc_host(host, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 40, 133.0, 6855.0, 16000.0, n_keep=13, sample_dtype=dt),
                    c.mfcc(fr, 40, 133.0, 6855.0, 16000.0, n_keep=13))
        Fp = c.n_frames_of(host.size, 640, 160)
        frp = c.frames(d.ptr, Fp, 640, 160, vb.WINDOW_HANN_SYMMETRIC, dt)
        assert_same(m.pitch_host(host, Fp, 640, 160, vb.WINDOW_HANN_SYMMETRIC, 16000.0, 0.45, 75.0, 600.0, 16, sample_dtype=dt),
                    c.pitch(frp, 16000.0, 0.45, 75.0, 600.0, 16))
        assert_same(m.pitch_with_peaks_host(host, Fp, 640, 160, vb.WINDOW_HANN_SYMMETRIC, 16000.0, 0.45, 0.03, 75.0, 600.0, 16,
                                            sample_dtype=dt),
                    c.pitch_with_peaks(frp, 16000.0, 0.45, 0.03, 75.0, 600.0, 16))
        J, U = 98, 8
        S = host.size // U
        frs = c.frames(d.ptr, U * J, 400, 160, vb.WINDOW_HANN_PERIODIC, dt, J, S)
        est = np.repeat(MALE[None], U, 0)
        assert_same(m.find_formants_host(host, U * J, 400, 160, vb.WINDOW_HANN_PERIODIC, 16000.0, 12, vb.LPC_BURG, est,
                                         frames_per_segment=J, segment_stride=S, sample_dtype=dt),
                    c.find_formants(frs, 16000.0, 12, vb.LPC_BURG, est))
    finally:
        m.close()


# ---- synth, rejections ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fs", [8000.0, 16000.0])
def test_synth_speech_g711(law, fs):
    c = ctx()
    pcm = c.synth_speech(3, 12345, fs, seed=9, first_utt=4, dtype=vb.I16).to_host()
    codes = c.synth_speech(3, 12345, fs, seed=9, first_utt=4, dtype=LAWS[law]).to_host()
    assert codes.dtype == np.uint8 and np.array_equal(codes, ENCODE[law](pcm))


def test_rejections():
    c = ctx()
    d = c.to_device(np.zeros(1024, dtype=np.uint8))
    r = c.empty((64,), np.float64)
    for dt in (vb.MULAW8, vb.ALAW8):
        assert c.lib.vbx_autocorrelate_ring(c.h, d.ptr, dt, 1, 64, None, 64, 8, r.ptr, vb.F64) == vb.ERR_BADARG
        assert c.lib.vbx_rms(c.h, d.ptr, dt, 1, 64, 64, r.ptr) == vb.ERR_BADARG
        fr = c.frames(d.ptr, 4, 64, 64, vb.WINDOW_NONE, vb.MULAW8)
        assert c.lib.vbx_autocorrelate(c.h, C.byref(fr), 8, r.ptr, dt) == vb.ERR_BADARG
        assert c.lib.vbx_lpc(c.h, C.byref(fr), 4, None, r.ptr, None, dt) == vb.ERR_BADARG
    bad = c.frames(d.ptr, 4, 64, 64, vb.WINDOW_NONE, 5)
    assert c.lib.vbx_autocorrelate(c.h, C.byref(bad), 8, r.ptr, vb.F64) == vb.ERR_BADARG
    assert c.lib.vbx_mfcc(c.h, C.byref(bad), 13, 13, 100.0, 4000.0, 16000.0, r.ptr, None, vb.F64) == vb.ERR_BADARG


# ---- real speech, mu-law ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def speech_mulaw(oracle, fixtures_dir):
    x, fs = oracle.read_wav(os.path.join(fixtures_dir, "sample-two_vowels.wav"))
    codes = ENCODE["mulaw"](np.round(x * 32767.0).astype(np.int16))
    return codes, DECODE["mulaw"](codes).astype(np.float64) / 32767.0, fs


def test_real_speech_mulaw_vs_oracle(oracle, speech_mulaw):
    codes, xs, fs = speech_mulaw
    c = ctx()
    d = c.to_device(codes)
    # formants: Burg on the 1102 / 441 framing, tracker from the MALE estimates
    N, hop = 1102, 441
    F = c.n_frames_of(codes.size, N, hop)
    out = c.find_formants(c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_PERIODIC, vb.MULAW8), fs, 12, vb.LPC_BURG, MALE[None])
    state = MALE.copy()
    for f in range(F):
        res = oracle.find_formants(xs[f * hop:f * hop + N].copy(), fs, 12, state)
        assert res["status"] == out["status"][f] and res["n_res"] == out["n_res"][f], f
        if res["status"] == 0:
            state = res["formants"]
        assert np.max(np.abs(out["tracks"][f] - state)) < 0.5, f
    # MFCC on the same framing
    w = oracle.hanning_window(N)
    m = c.mfcc(c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, vb.MULAW8), 40, 133.0, 6855.0, fs, n_keep=13).to_host()
    mo = np.stack([oracle.mfcc(xs[f * hop:f * hop + N] * w, 40, 133.0, 6855.0, fs)[:13] for f in range(F)])
    assert np.max(normwise(m, mo)) < 1e-5
    # pitch: three periods of 75 Hz, 10 ms hop, every list position
    N, K = 1764, 48
    F = c.n_frames_of(codes.size, N, hop)
    w = oracle.hanning_window(N)
    res = c.pitch(c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, vb.MULAW8), fs, 0.45, 75.0, 600.0, K)
    cand, n, st = res["candidates"].to_host(), res["n_cand"].to_host(), res["status"].to_host()
    voiced = 0
    for f in range(F):
        rs, rc, extra = oracle.pitch(xs[f * hop:f * hop + N] * w, fs, 0.45, 75.0, 600.0, max_cand=K)
        assert rs == st[f] and extra["n_cand"] == n[f], f
        k = rc.shape[0]
        assert (cand[f, 0, 0] != 0) == (rc[0, 0] != 0), f
        assert np.max(np.abs(cand[f, :k, 0] - rc[:, 0])) < 0.1 and np.max(np.abs(cand[f, :k, 1] - rc[:, 1])) < 1e-6, f
        voiced += int(cand[f, 0, 0] != 0)
    assert voiced > F // 4
