"""GPU tests of the opt-in peaks extension of the pitch path: vbx_frame_peaks, vbx_pitch_with_peaks and its `_host` /
`_multi_host` twins (the reference's local_peak / global_peak honoured as Boersma's voiceless strength).

Tolerances are test_gpu_pitch.py's: status and counts equal, no voiced/unvoiced flips, top frequency within 0.1 Hz, strengths
within 1e-6; the peaks themselves are exact."""
import numpy as np
import pytest

from gpu_util import ctx, synth, vb

pytestmark = pytest.mark.gpu
TOL_HZ = 0.1
TOL_STRENGTH = 1e-6
A, B = 0.45, 0.03  # Praat's voicing and silence thresholds
FS = 16000


def _peak(x, dtype):
    """max |x| as the library defines it: int16 scaled by 1/32767, NaN ignored, 0 for no (non-NaN) samples."""
    v = x.astype(np.float64) / 32767.0 if dtype == vb.I16 else x.astype(np.float64)
    a = np.abs(v)
    a = a[~np.isnan(a)]
    return float(a.max()) if a.size else 0.0


def _voiceless(local, glob, a=A, b=B):
    """R_f from the definition, in f64 and in the device's order of operations: ratio = min(local/global, 1) (0 where
    global <= 0 or is NaN), a + max(0, 2 − ratio·(1 + a)/b), a NaN ratio giving a."""
    local = np.asarray(local, dtype=np.float64)
    glob = np.broadcast_to(np.asarray(glob, dtype=np.float64), local.shape)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(glob > 0, local / np.where(glob > 0, glob, 1.0), 0.0)
        ratio = np.where(ratio > 1.0, 1.0, ratio)
        v = 2.0 - ratio * (1.0 + a) / b
    return a + np.where(v > 0.0, v, 0.0)


def _ref_pitch_with_peaks(oracle, audio, F, N, hop, window, fs, a, b, fmin, fmax, max_cand, local_peaks=None, global_peak=None):
    """The reference's per-frame pitch() with the unvoiced candidate's strength replaced by R_f, then its stable sort.  pitch()
    appends {0, threshold} before it sorts, and the threshold is used nowhere else (periodic.rs:452-453), so the oracle's
    pitch run with threshold = R_f, one frame at a time, is exactly that list.  Peaks left None are max |x| of each frame /
    of the view's extent.  Returns (candidates [F][max_cand][2], counts, status, R_f [F])."""
    audio = np.ascontiguousarray(audio, dtype=np.float32)
    if local_peaks is None:
        local_peaks = [_peak(audio[f * hop:f * hop + N], vb.F32) for f in range(F)]
    if global_peak is None:
        global_peak = _peak(audio[:(F - 1) * hop + N], vb.F32)
    unv = _voiceless(local_peaks, global_peak, a, b) if b > 0 else np.full(F, float(a))
    cand = np.zeros((F, max_cand, 2))
    n = np.zeros(F, dtype=np.int32)
    st = np.zeros(F, dtype=np.uint8)
    for f in range(F):
        c, nc, s = oracle.batch_pitch(audio[f * hop:f * hop + N], 1, N, N, window, fs, float(unv[f]), fmin, fmax, max_cand)
        cand[f], n[f], st[f] = c[0], nc[0], s[0]
    return cand, n, st, unv


def _corpus(seconds=3.0, seed=5):
    """One recording with an amplitude ramp, silent gaps (near-silent noise and exact zeros) and a quiet periodic tail.
    Returns (audio float32, slice of the quiet tail in samples)."""
    x = synth.utterance(seed, FS, seconds=seconds).astype(np.float64)
    n = x.size
    env = np.ones(n)
    q = n // 6
    env[:q] = np.linspace(0.05, 1.0, q)                # ramp up
    env[2 * q:3 * q] = 1e-3                             # near-silent gap
    env[3 * q:3 * q + q // 4] = 0.0                     # exact silence
    env[3 * q + q // 4:4 * q] = np.linspace(1.0, 0.1, q - q // 4)  # ramp down
    x = x * env
    tail = slice(5 * q, n)                              # quiet periodic tail: a 150 Hz tone at 1 % of the peak
    t = np.arange(n - 5 * q) / FS
    x[tail] = 0.01 * np.max(np.abs(x[:5 * q])) * np.sin(2 * np.pi * 150.0 * t)
    return x.astype(np.float32), tail


def _compare(res, ref_cand, ref_n, ref_st, max_cand):
    cand, n, st = res["candidates"], res["n_cand"], res["status"]
    if hasattr(cand, "to_host"):
        cand, n, st = cand.to_host(), n.to_host(), st.to_host()
    assert np.array_equal(st, ref_st)
    assert np.array_equal(n, ref_n), f"candidate-count mismatches in {np.count_nonzero(n != ref_n)} frames"
    voiced, voiced_ref = cand[:, 0, 0] != 0, ref_cand[:, 0, 0] != 0
    assert np.array_equal(voiced, voiced_ref), f"{np.count_nonzero(voiced != voiced_ref)} voiced/unvoiced flips"
    assert np.max(np.abs(cand[:, 0, 0] - ref_cand[:, 0, 0])) < TOL_HZ
    k = np.minimum(n, max_cand)
    mask = np.arange(max_cand)[None, :] < k[:, None]
    ds = np.abs(cand[..., 1] - ref_cand[..., 1])[mask]
    assert ds.max() < TOL_STRENGTH, ds.max()
    return cand


def _equal(a, b):
    for key in ("candidates", "n_cand", "status"):
        x, y = a[key], b[key]
        x = x.to_host() if hasattr(x, "to_host") else x
        y = y.to_host() if hasattr(y, "to_host") else y
        assert np.array_equal(x, y), key


# ---- 1. peaks are exact -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [vb.F32, vb.I16, vb.F64])
@pytest.mark.parametrize("hop", [160, 400, 530])
@pytest.mark.parametrize("segmented", [False, True])
def test_frame_peaks_exact(dtype, hop, segmented):
    c = ctx()
    rng = np.random.default_rng(hop + 7 * dtype + (100 if segmented else 0))
    N, L = 400, 9000
    U = 3 if segmented else 1
    row = L + 700  # padding after every utterance: samples outside every frame
    J = c.n_frames_of(L, N, hop)
    ext = (J - 1) * hop + N
    x = rng.standard_normal((U, row)) * np.linspace(0.2, 1.0, row)
    for u in range(U):
        x[u, ext:] = 50.0 + u        # beyond the last frame: in no peak
        if hop > N:
            x[u, N + 3] = 20.0 + u   # in the gap after frame 0: the global peak only
    if dtype == vb.I16:
        x = np.clip(np.round(x * 3000), -32768, 32767).astype(np.int16)
        x[0, 5] = -32768
    else:
        x = x.astype(np.float32 if dtype == vb.F32 else np.float64)
        x[0, rng.integers(0, ext, 40)] = np.nan
        x[0, 2 * hop:2 * hop + N] = np.nan  # an all-NaN frame
    flat = np.ascontiguousarray(x).reshape(-1)
    d = c.to_device(flat)
    if segmented:
        F = U * J
        fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, dtype=dtype, frames_per_segment=J, segment_stride=row)
    else:  # one segment: the frames of the first row
        F = J
        fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, dtype=dtype)
    local, glob = c.frame_peaks(fr)
    local, glob = local.to_host(), glob.to_host()
    ref_local = np.array([_peak(flat[(f // J) * row + (f % J) * hop:][:N], dtype) for f in range(F)])
    ref_glob = np.array([_peak(flat[u * row:u * row + ext], dtype) for u in range(F // J)])
    assert np.array_equal(local, ref_local), np.flatnonzero(local != ref_local)[:10]
    assert np.array_equal(glob, ref_glob), (glob, ref_glob)
    if dtype != vb.I16:
        assert local[2] == 0.0  # the all-NaN frame
    if hop > N and dtype != vb.I16:  # (int16 clips the gap sample to the range of the frames' samples)
        assert np.all(glob > local.max())  # the gap sample counts for the segment only


# ---- 2. an extension, not a change --------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,hop,fmin,fmax,window", [
    (640, 160, 75.0, 600.0, vb.WINDOW_HANN_SYMMETRIC),   # C4
    (400, 160, 100.0, 500.0, vb.WINDOW_HANN_SYMMETRIC),
    (2048, 1024, 100.0, 500.0, vb.WINDOW_HANN_SYMMETRIC),
    (333, 100, 120.0, 800.0, vb.WINDOW_HANN_SYMMETRIC),
    (512, 256, 75.0, 600.0, vb.WINDOW_NONE),
])
@pytest.mark.parametrize("out_dtype", [vb.F32, vb.F64])
def test_zero_silence_threshold_is_vbx_pitch(N, hop, fmin, fmax, window, out_dtype):
    c = ctx()
    audio = synth.utterance(11, FS, seconds=2.0)
    F = min(c.n_frames_of(audio.size, N, hop), 150)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, N, hop, window)
    ref = c.pitch(fr, float(FS), A, fmin, fmax, max_cand=40, out_dtype=out_dtype)
    got = c.pitch_with_peaks(fr, float(FS), A, 0.0, fmin, fmax, max_cand=40, out_dtype=out_dtype)
    _equal(got, ref)


def test_zero_silence_threshold_segments_and_slabs(monkeypatch):
    c = ctx()
    N, hop = 640, 160
    audio = synth.corpus(3, FS, seconds=1.0, first=20)
    J = c.n_frames_of(audio.shape[1], N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, 3 * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=audio.shape[1])
    monkeypatch.setenv("VBX_PITCH_SLAB_MB", "1")  # ~100 frames per slab
    for out_dtype in (vb.F32, vb.F64):
        _equal(c.pitch_with_peaks(fr, float(FS), A, 0.0, 75.0, 600.0, 16, out_dtype),
               c.pitch(fr, float(FS), A, 75.0, 600.0, 16, out_dtype))


def test_slabs_do_not_change_the_peaks_path(monkeypatch):
    """The voiceless strength is indexed by the frame of the batch: slabs smaller than the batch give the same lists."""
    c = ctx()
    audio, _ = _corpus()
    F = c.n_frames_of(audio.size, 640, 160)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, 640, 160, vb.WINDOW_HANN_SYMMETRIC)
    whole = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, 16)
    monkeypatch.setenv("VBX_PITCH_SLAB_MB", "1")
    _equal(c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, 16), whole)


def test_negative_silence_threshold_is_badarg():
    c = ctx()
    d = c.to_device(np.zeros(1280, dtype=np.float32))
    fr = c.frames(d.ptr, 2, 640, 640, vb.WINDOW_HANN_SYMMETRIC)
    with pytest.raises(vb.VoxBoxError) as e:
        c.pitch_with_peaks(fr, float(FS), A, -0.01, 75.0, 600.0, 16)
    assert e.value.status == vb.ERR_BADARG


# ---- 3. oracle parity, 4. truncation, 5. behaviour ------------------------------------------------------------------------
def test_oracle_parity_computed_peaks(oracle):
    c = ctx()
    audio, _ = _corpus()
    N, hop, K = 640, 160, 40
    F = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC)
    res = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K)
    ref_cand, ref_n, ref_st, ref_unv = _ref_pitch_with_peaks(oracle, audio, F, N, hop, oracle.WIN_HANN_SYMMETRIC, float(FS), A, B,
                                                                  75.0, 600.0, K)
    cand = _compare(res, ref_cand, ref_n, ref_st, K)
    # the unvoiced entry carries R_f (computed here from the definition) to 1e-12 relative
    local, glob = c.frame_peaks(fr)
    rf = _voiceless(local.to_host(), glob.to_host()[0])
    assert np.allclose(ref_unv, rf, rtol=1e-12, atol=0)
    n = res["n_cand"].to_host()
    for f in np.flatnonzero(n <= K):
        unv = cand[f, :n[f]][cand[f, :n[f], 0] == 0.0, 1]
        assert np.any(np.abs(unv - rf[f]) <= 1e-12 * rf[f]), (f, unv, rf[f])
    assert np.count_nonzero(rf > A) > 20 and np.count_nonzero(rf == A) > 20  # both regimes are exercised


def test_oracle_parity_caller_peaks(oracle):
    c = ctx()
    audio, _ = _corpus(seed=9)
    N, hop, K = 640, 160, 40
    F = c.n_frames_of(audio.size, N, hop)
    rng = np.random.default_rng(1)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC)
    local, glob = c.frame_peaks(fr)
    lp = local.to_host() * rng.uniform(0.5, 1.5, F)
    gp = 2.0 * float(glob.to_host()[0])  # the peak of a longer recording this view is part of
    res = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K, local_peaks=c.to_device(lp),
                             global_peaks=c.to_device(np.array([gp])))
    ref_cand, ref_n, ref_st, ref_unv = _ref_pitch_with_peaks(oracle, audio, F, N, hop, oracle.WIN_HANN_SYMMETRIC, float(FS), A, B,
                                                                  75.0, 600.0, K, local_peaks=lp, global_peak=gp)
    _compare(res, ref_cand, ref_n, ref_st, K)
    assert np.allclose(ref_unv, _voiceless(lp, gp), rtol=1e-12, atol=0)


def test_truncation(oracle):
    c = ctx()
    audio, _ = _corpus(seed=13)
    N, hop, K = 640, 160, 3
    F = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC)
    res = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K)
    full, ref_n, ref_st, ref_unv = _ref_pitch_with_peaks(oracle, audio, F, N, hop, oracle.WIN_HANN_SYMMETRIC, float(FS), A, B,
                                                              75.0, 600.0, 200)
    # where the unvoiced entry sits in the full list
    rank = np.array([int(np.flatnonzero((full[f, :ref_n[f], 0] == 0.0) & (full[f, :ref_n[f], 1] == ref_unv[f]))[0])
                     for f in range(F)])
    top = (rank == 0) & (ref_n > K)
    below = rank >= K  # left below the cut, as in vbx_pitch
    assert top.sum() > 10 and below.sum() > 10, (top.sum(), below.sum())
    cand = _compare(res, full[:, :K], ref_n, ref_st, K)
    assert np.all(cand[top, 0, 0] == 0.0) and np.all(cand[top, 0, 1] == ref_unv[top])
    assert not np.any(cand[below, :, 0] == 0.0)  # truncated away, as the reference's list truncated


def test_quiet_frames_are_unvoiced():
    c = ctx()
    audio, tail = _corpus(seed=17)
    N, hop, K = 640, 160, 16
    F = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC)
    plain = c.pitch(fr, float(FS), A, 75.0, 600.0, K)
    peaks = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K)
    quiet = np.arange(F)[(np.arange(F) * hop >= tail.start) & (np.arange(F) * hop + N <= tail.stop)]
    assert quiet.size > 40
    # a clean 150 Hz tone: voiced with strength > 0.9 without peaks; at 1 % of the peak, R_f = 0.45 + 2 − 0.01·1.45/0.03 > 1,
    # above any voiced strength (those are <= 1, periodic.rs:446)
    pc = plain["candidates"].to_host()
    assert np.all(pc[quiet, 0, 0] > 0.0) and np.all(pc[quiet, 0, 1] > 0.9)
    kc = peaks["candidates"].to_host()
    assert np.all(kc[quiet, 0, 0] == 0.0) and np.all(kc[quiet, 0, 1] > 1.0)
    # chained into the Viterbi path finder: the quiet frames' path is unvoiced
    path, _ = c.pitch_viterbi(peaks["candidates"], peaks["n_cand"], 1)
    assert np.all(path.to_host()[quiet, 0] == 0.0)
    path0, _ = c.pitch_viterbi(plain["candidates"], plain["n_cand"], 1)
    assert np.all(path0.to_host()[quiet, 0] > 0.0)


# ---- 6. twins -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [vb.F32, vb.I16])
def test_host_twin_single_segment(monkeypatch, dtype):
    """One long recording, cut into frame ranges by the host pipeline: the global peak must be the whole view's."""
    c = ctx()
    parts = [_corpus(seconds=4.0, seed=s)[0] * g for s, g in ((21, 1.0), (22, 0.3), (23, 0.05), (24, 0.01))]
    audio = np.concatenate(parts).astype(np.float32)
    if dtype == vb.I16:
        audio = np.round(audio / np.max(np.abs(audio)) * 30000).astype(np.int16)
    N, hop, K = 640, 160, 16
    F = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, dtype=dtype)
    dev = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K)
    monkeypatch.setenv("VBX_HOST_CHUNK_MB", "0")  # the smallest chunks: a few frames each
    host = c.pitch_with_peaks_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K)
    _equal(host, dev)
    monkeypatch.setenv("VBX_HOST_CHUNK_MB", "1")
    host = c.pitch_with_peaks_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K)
    _equal(host, dev)
    # caller-supplied peaks reach every chunk at their rows
    local, glob = c.frame_peaks(fr)
    lp, gp = local.to_host()[::-1].copy(), glob.to_host() * 1.5
    dev = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K, local_peaks=c.to_device(lp), global_peaks=c.to_device(gp))
    host = c.pitch_with_peaks_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K,
                                   local_peaks=lp, global_peaks=gp)
    _equal(host, dev)
    # the chunk-local global peak would differ: quiet frames of the last part are judged against the loud first part
    assert np.count_nonzero(dev["candidates"].to_host()[:, 0, 0] == 0.0) > F // 8


def test_host_twin_segmented(monkeypatch):
    c = ctx()
    gains = np.linspace(1.0, 0.02, 12)
    audio = np.stack([_corpus(seconds=2.0, seed=30 + u)[0] * g for u, g in enumerate(gains)]).astype(np.float32)
    N, hop, K = 640, 160, 16
    U, ns = audio.shape
    J = c.n_frames_of(ns, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)
    dev = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K, out_dtype=vb.F32)
    monkeypatch.setenv("VBX_HOST_CHUNK_MB", "0")  # one utterance per chunk
    host = c.pitch_with_peaks_host(audio, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K, vb.F32, J, ns)
    _equal(host, dev)
    gp = np.full(U, float(np.max(np.abs(audio))))  # one global peak for all utterances: the recording-wide one
    dev = c.pitch_with_peaks(fr, float(FS), A, B, 75.0, 600.0, K, out_dtype=vb.F32, global_peaks=c.to_device(gp))
    host = c.pitch_with_peaks_host(audio, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K, vb.F32, J, ns,
                                   global_peaks=gp)
    _equal(host, dev)


def test_multi_twin():
    c = ctx()
    N, hop, K = 640, 160, 16
    audio = np.concatenate([_corpus(seconds=3.0, seed=40 + s)[0] * g for s, g in enumerate((1.0, 0.1, 0.02))]).astype(np.float32)
    F = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    dev = c.pitch_with_peaks(c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC), float(FS), A, B, 75.0, 600.0, K)
    utts = np.stack([_corpus(seconds=2.0, seed=50 + u)[0] * g for u, g in enumerate(np.linspace(1.0, 0.05, 5))]).astype(np.float32)
    U, ns = utts.shape
    J = c.n_frames_of(ns, N, hop)
    du = c.to_device(utts)
    dev_seg = c.pitch_with_peaks(c.frames(du.ptr, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns),
                                 float(FS), A, B, 75.0, 600.0, K)
    with vb.Multi() as m:
        got = m.pitch_with_peaks_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K)
        _equal(got, dev)
        got = m.pitch_with_peaks_host(utts, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(FS), A, B, 75.0, 600.0, K,
                                      frames_per_segment=J, segment_stride=ns)
        _equal(got, dev_seg)
