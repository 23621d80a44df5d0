"""GPU parity of the pitch path at every frame length vbx_pitch accepts (2 <= frame_len <= 16 384) vs the f64 oracle.

launch_pitch sizes the lag sweep from the frame length: G = ceil(N / 16) lag groups on (G + 1) / 2 lanes per frame, as many
frames per CTA as fill about 160 threads within 56 KB of shared memory, and the smallest CTA-size class of
pitch_lag64_kernel (160, 256 or 512 threads) that holds them.  `_plan` restates that arithmetic; the lengths below sit on
every boundary it has (one lag group, every residue mod 16, the change from two frames per CTA to one at 2 560 / 2 561, the
class changes at 5 120 / 5 121 and 8 192 / 8 193, the limit 16 384).  The refinement's windowed-sinc depth is
min(1200, lag + 1), so only lags above 1 200 (96 kHz and 192 kHz audio here) run it at its cap, where the Hann factors'
recurrence is at its design limit.

Candidate lists follow the acceptance rules of test_pitch_full_list_parity_10k_frames: identical status and n_cand,
identical voiced/unvoiced decisions, every list position within 0.1 Hz, strengths within 1e-6.  Mismatch counts are
reported, never masked."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from gpu_util import ctx, normwise, synth, vb

pytestmark = pytest.mark.gpu
TOL_HZ = 0.1
TOL_STRENGTH = 1e-6
# Lag function vs the oracle's: norm-wise per frame over the lags the candidate search reads (below ixmax), and past ixmax
# element-wise relative to Σ|x_i·x_{i+lag}| / (Σ x_i² · lag window), the size of the terms that lag sums (a lag whose sum
# cancels is not held to more digits than its terms carry).  Largest errors on a B200: 6.2e-15 below ixmax (I16 without a
# window: the oracle scales the samples by 1/32767 before the window, the device folds the scale into it) and 2.1e-15 past.
LAG_TOL_BELOW = 2e-14
LAG_TOL_ABOVE = 2e-14

DTYPES = {"f32": vb.F32, "i16": vb.I16, "f64": vb.F64}
WINDOWS = {"none": vb.WINDOW_NONE, "hann": vb.WINDOW_HANN_SYMMETRIC}
LAG_LENGTHS = list(range(2, 81)) + [2047, 2048, 2560, 2561, 5120, 5121, 8192, 8193, 11520, 16383, 16384]


def _plan(n):
    """(lanes per frame, frames per CTA, threads per CTA) of the lag sweep, as launch_pitch computes them."""
    n16 = (n + 15) // 16 * 16
    lpf = (n16 // 16 + 1) // 2
    frame_bytes = (n16 + 48) * 9 // 8 * 8
    fpc = max(160 // lpf, 1)
    while fpc > 1 and fpc * frame_bytes > 56 * 1024:
        fpc -= 1
    return lpf, fpc, max((fpc * lpf + 31) // 32 * 32, 64)


def test_plan_covers_every_lag_kernel_class():
    """The lengths of this file reach every CTA shape of the sweep, including the 512-thread class."""
    assert _plan(16)[1:] == (99, 128) and _plan(2560)[1] == 2 and _plan(2561)[1] == 1
    assert _plan(5120)[2] == 160 and _plan(5121)[2] == 192 and _plan(8192)[2] == 256
    assert _plan(8193)[2] == 288 and _plan(16384)[2] == 512


def _pool_map(fn, items):
    """The oracle calls release the GIL: run them on every core."""
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        return list(ex.map(fn, items))


@pytest.fixture(scope="module")
def sources():
    """The same 96 000 samples as f32, as int16 PCM and as f64 values no f32 can hold, on the host and on the device; and
    the f64 value of every sample as the reference's caller sees it (int16 PCM scaled by 1/32767)."""
    c = ctx()
    a = synth.utterance(31, 48000, seconds=2.0)
    pcm = np.round(a.astype(np.float64) * 32767.0).astype(np.int16)
    a64 = a.astype(np.float64) + 1e-9 * np.sin(np.arange(a.size))
    host = {"f32": a, "i16": pcm, "f64": a64}
    value = {"f32": a.astype(np.float64), "i16": pcm.astype(np.float64) / 32767.0, "f64": a64}
    return {k: (host[k], c.to_device(host[k]), value[k]) for k in host}


def _window(window, n, oracle):
    return oracle.hanning_window(n) if window == vb.WINDOW_HANN_SYMMETRIC else np.ones(n)


def _oracle_lag(oracle, xw):
    """The oracle's self_lag (periodic.rs:403-408) of one windowed frame, and the scale of each lag's terms.  No candidate
    passes the (0, 0) filter, so the oracle skips the refinement."""
    st, _, ex = oracle.pitch(xw, 1.0, 0.0, 0.0, 0.0, 1, want_lag=True)
    assert st == 0
    n = xw.size
    ax = np.abs(xw)
    terms = np.correlate(ax, ax, "full")[n - 1:] + ax[0]  # the fold seeds every lag with x[0] (periodic.rs:284)
    scale = terms / (max(terms[0], 1e-300) * np.abs(oracle.hanning_lag_window(n)))
    return ex["lag"][:n], scale


def _lag_mismatches(got, ref, scale):
    """(description of every disagreement, norm-wise error below ixmax, worst scaled error past ixmax) of one frame."""
    n = ref.size
    ixmax = n // 2
    bad = []
    for name, test in (("NaN", np.isnan), ("+Inf", np.isposinf), ("-Inf", np.isneginf)):
        if not np.array_equal(test(got), test(ref)):
            bad.append(f"{name} at {np.flatnonzero(test(got) != test(ref))[:8].tolist()}")
    fin = np.isfinite(ref) & np.isfinite(got)
    lo = fin[:ixmax]
    below = float(normwise(got[:ixmax][lo], ref[:ixmax][lo])) if lo.any() else 0.0
    hi = fin[ixmax:]
    d = np.abs(got[ixmax:] - ref[ixmax:])[hi] / np.maximum(scale[ixmax:][hi], 1e-300)
    above = float(d.max()) if d.size else 0.0
    if below > LAG_TOL_BELOW:
        bad.append(f"norm-wise error below ixmax {below:.2e}")
    if above > LAG_TOL_ABOVE:
        bad.append(f"error past ixmax {above:.2e} (at lag {ixmax + int(np.flatnonzero(hi)[np.argmax(d)])})")
    return bad, below, above


@pytest.mark.parametrize("window", list(WINDOWS), ids=list(WINDOWS))
@pytest.mark.parametrize("dtype", list(DTYPES), ids=list(DTYPES))
def test_lag_function_every_kernel_shape(oracle, sources, dtype, window):
    """vbx_pitch_lag_function at every length of LAG_LENGTHS: a batch of (frames per CTA + 1) overlapping frames, whose
    last CTA holds one frame, and a single frame.  WINDOW_NONE keeps x[0] != 0, where the fold-seed quirk is live."""
    c = ctx()
    host, dev, value = sources[dtype]
    wkind = WINDOWS[window]
    jobs = []
    for n in LAG_LENGTHS:
        F = _plan(n)[1] + 1
        hop = max(n - n // 3, 1)
        jobs += [(n, f, hop) for f in range(F)]
    refs = dict(zip(jobs, _pool_map(lambda j: _oracle_lag(oracle, value[j[1] * j[2]: j[1] * j[2] + j[0]] * _window(wkind, j[0], oracle)), jobs)))
    failures, worst_below, worst_above = [], 0.0, 0.0
    for n in LAG_LENGTHS:
        F = _plan(n)[1] + 1
        hop = max(n - n // 3, 1)
        batch = c.pitch_lag_function(c.frames(dev.ptr, F, n, hop, wkind, dtype=DTYPES[dtype])).to_host()
        single = c.pitch_lag_function(c.frames(dev.ptr, 1, n, hop, wkind, dtype=DTYPES[dtype])).to_host()
        for f, got in [(f, batch[f]) for f in range(F)] + [(0, single[0])]:
            ref, scale = refs[(n, f, hop)]
            bad, below, above = _lag_mismatches(got, ref, scale)
            worst_below, worst_above = max(worst_below, below), max(worst_above, above)
            if bad:
                failures.append(f"N={n} frame {f}: " + "; ".join(bad))
    print(f"lag function {dtype}/{window}: worst norm-wise error below ixmax {worst_below:.2e}, past ixmax {worst_above:.2e}")
    assert not failures, f"{len(failures)} frames differ from the oracle:\n" + "\n".join(failures[:40])


@pytest.mark.parametrize("n", [17, 640, 2561, 5121, 8193, 16384])
def test_lag_function_segments_and_silence(oracle, sources, n):
    """A two-level view with an odd segment_stride (I16 samples: segments start at odd sample offsets), and an all-zero frame
    between two others, whose lag function is NaN exactly where the oracle's is (0 / 0 in normalize, waves.rs:70)."""
    c = ctx()
    host, dev, value = sources["i16"]
    w = oracle.hanning_window(n)
    J, hop = 2, n // 2 + 1
    ss = (J - 1) * hop + n + 1
    ss += 1 - ss % 2
    assert 2 * ss + (J - 1) * hop + n <= host.size
    got = c.pitch_lag_function(c.frames(dev.ptr, 3 * J, n, hop, vb.WINDOW_HANN_SYMMETRIC, dtype=vb.I16, frames_per_segment=J,
                                        segment_stride=ss)).to_host()
    starts = [u * ss + j * hop for u in range(3) for j in range(J)]
    refs = _pool_map(lambda s: _oracle_lag(oracle, value[s:s + n] * w), starts)
    failures = [f"frame {f}: " + "; ".join(b) for f, (g, (r, s)) in enumerate(zip(got, refs)) if (b := _lag_mismatches(g, r, s)[0])]
    assert not failures, failures

    audio = np.concatenate([host[:n], np.zeros(n, np.int16), host[n:2 * n]])
    d = c.to_device(audio)
    got = c.pitch_lag_function(c.frames(d.ptr, 3, n, n, vb.WINDOW_HANN_SYMMETRIC, dtype=vb.I16)).to_host()
    ref, scale = _oracle_lag(oracle, np.zeros(n))
    assert np.all(np.isnan(ref)) and np.all(np.isnan(got[1])), int(np.count_nonzero(~np.isnan(got[1])))
    for f in (0, 2):
        r, s = _oracle_lag(oracle, audio[f * n:(f + 1) * n].astype(np.float64) / 32767.0 * w)
        assert not _lag_mismatches(got[f], r, s)[0]


def _list_audio(fs, n, hop, F, noise_frames, seed):
    """Speech-like audio for F frames of n samples, hop apart, with white noise over the frames in `noise_frames` (hundreds
    of candidates each: refine tiles of 256 entries then fall inside one frame, and n_cand exceeds any small max_cand)."""
    a = synth.utterance(seed, fs, seconds=((F - 1) * hop + n) / fs + 0.01)[: (F - 1) * hop + n].copy()
    rng = np.random.default_rng(seed)
    for f in noise_frames:
        a[f * hop:f * hop + n] = (0.3 * rng.standard_normal(n)).astype(np.float32)
    return a


def _compare_lists(res, ref, what):
    cand, n, st = res
    rc, rn, rs = ref
    assert np.array_equal(st, rs), f"{what}: status differs in {np.count_nonzero(st != rs)} frames"
    assert np.array_equal(n, rn), f"{what}: n_cand differs in {np.count_nonzero(n != rn)} frames"
    voiced, rvoiced = cand[:, 0, 0] != 0, rc[:, 0, 0] != 0
    assert np.array_equal(voiced, rvoiced), f"{what}: {np.count_nonzero(voiced != rvoiced)} voiced/unvoiced flips"
    K = cand.shape[1]
    mask = np.arange(K)[None, :] < np.minimum(n, K)[:, None]
    df = np.abs(cand[..., 0] - rc[..., 0])[mask]
    ds = np.abs(cand[..., 1] - rc[..., 1])[mask]
    bad_f, bad_s = int(np.count_nonzero(~(df <= TOL_HZ))), int(np.count_nonzero(~(ds <= TOL_STRENGTH)))
    assert bad_f == 0 and bad_s == 0, (f"{what}: of {int(mask.sum())} list positions {bad_f} differ by > {TOL_HZ} Hz (max "
                                       f"{np.nanmax(df):.3e}) and {bad_s} by > {TOL_STRENGTH} in strength (max {np.nanmax(ds):.3e})")
    return int(mask.sum())


LIST_SHAPES = [  # fs, N, fmin, fmax, frames
    (96000, 3840, 75.0, 600.0, 60),     # three periods of 75 Hz: lags 160 .. 1 280, the sinc depth reaches its cap of 1 200
    (96000, 5760, 50.0, 600.0, 60),     # the 256-thread class
    (192000, 11520, 50.0, 600.0, 40),   # the 512-thread class; three periods of 50 Hz at 192 kHz
    (192000, 16384, 30.0, 600.0, 40),   # the longest frame
    (48000, 2560, 75.0, 600.0, 80),     # two frames per CTA
    (48000, 2561, 75.0, 600.0, 80),     # one frame per CTA
    (16000, 17, 10.0, 8000.0, 100),     # candidates from lag 2 up to ixmax − 2
    (16000, 33, 10.0, 8000.0, 100),
]


@pytest.mark.parametrize("fs,n,fmin,fmax,F", LIST_SHAPES, ids=[f"{s[0] // 1000}k-N{s[1]}" for s in LIST_SHAPES])
def test_full_candidate_lists(oracle, fs, n, fmin, fmax, F):
    """Every position of every frame's list (max_cand holds the longest possible list) vs the oracle; a call with a short
    max_cand returns the same lists truncated, bit for bit."""
    c = ctx()
    hop = max(n // 4, 1)
    noise = [F // 3, F // 3 + 4 * (n > 40), F - 1]
    audio = _list_audio(fs, n, hop, F, noise, seed=n)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, n, hop, vb.WINDOW_HANN_SYMMETRIC)
    K = n // 4 + 2  # local maxima below ixmax = N/2 are at least two lags apart, plus the unvoiced candidate
    res = c.pitch(fr, float(fs), 0.45, fmin, fmax, max_cand=K)
    got = tuple(res[k].to_host() for k in ("candidates", "n_cand", "status"))
    ref = oracle.batch_pitch(audio, F, n, hop, oracle.WIN_HANN_SYMMETRIC, float(fs), 0.45, fmin, fmax, K, n_threads=0)
    positions = _compare_lists(got, ref, f"fs {fs} N {n}")
    assert np.all(got[1] <= K)
    if n > 2000:
        assert got[1][noise].min() >= 100, got[1][noise]
    print(f"fs {fs} N {n}: {positions} list positions match; n_cand of the noise frames {got[1][noise].tolist()}")
    short = c.pitch(fr, float(fs), 0.45, fmin, fmax, max_cand=4)
    assert np.array_equal(short["candidates"].to_host(), got[0][:, :4]) and np.array_equal(short["n_cand"].to_host(), got[1])
    assert np.array_equal(short["status"].to_host(), got[2])


@pytest.mark.parametrize("fs,n,fmin", [(96000, 5760, 50.0), (192000, 11520, 50.0)])
def test_one_frame_slabs_match_one_slab(monkeypatch, fs, n, fmin):
    """VBX_PITCH_SLAB_MB=0: one frame per slab (a launch sequence per frame) gives the single-slab results bit for bit."""
    c = ctx()
    F, hop = 12, n // 4
    audio = _list_audio(fs, n, hop, F, [5], seed=n + 1)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, n, hop, vb.WINDOW_HANN_SYMMETRIC)

    def run():
        r = c.pitch(fr, float(fs), 0.45, fmin, 600.0, max_cand=64)
        return [r[k].to_host() for k in ("candidates", "n_cand", "status")] + [c.pitch_lag_function(fr).to_host()]

    whole = run()
    monkeypatch.setenv("VBX_PITCH_SLAB_MB", "0")
    sliced = run()
    for name, a, b in zip(("candidates", "n_cand", "status", "lag function"), whole, sliced):
        assert np.array_equal(a, b, equal_nan=a.dtype.kind == "f"), name


def test_twins_at_11520(monkeypatch):
    """N = 11 520: the host twin in one-frame chunks, and pitch_with_peaks with silence_threshold 0, equal vbx_pitch bit for bit."""
    c = ctx()
    fs, n, F = 192000, 11520, 12
    hop = n // 4
    audio = _list_audio(fs, n, hop, F, [7], seed=11)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, F, n, hop, vb.WINDOW_HANN_SYMMETRIC)
    dev = c.pitch(fr, float(fs), 0.45, 50.0, 600.0, max_cand=32)
    dev = {k: v.to_host() for k, v in dev.items()}
    peaks = c.pitch_with_peaks(fr, float(fs), 0.45, 0.0, 50.0, 600.0, max_cand=32)
    for k in dev:
        assert np.array_equal(peaks[k].to_host(), dev[k]), k
    monkeypatch.setenv("VBX_HOST_CHUNK_MB", "0")
    host = c.pitch_host(audio, F, n, hop, vb.WINDOW_HANN_SYMMETRIC, float(fs), 0.45, 50.0, 600.0, 32)
    for k in dev:
        assert np.array_equal(host[k], dev[k]), k


def test_frame_length_limits():
    """frame_len 2 .. 16 384 is accepted (include/voxbox_b200.h); 1 and 16 385 are VBX_ERR_BADARG on every pitch entry."""
    c = ctx()
    d = c.to_device(synth.utterance(4, 48000, seconds=1.0))
    for n in (1, 16385):
        fr = c.frames(d.ptr, 1, n, n, vb.WINDOW_HANN_SYMMETRIC)
        for call in (lambda: c.pitch(fr, 48000.0, 0.45, 50.0, 600.0), lambda: c.pitch_lag_function(fr),
                     lambda: c.pitch_with_peaks(fr, 48000.0, 0.45, 0.03, 50.0, 600.0)):
            with pytest.raises(vb.VoxBoxError) as e:
                call()
            assert e.value.status == vb.ERR_BADARG, (n, e.value)
    for n in (8193, 16384):
        fr = c.frames(d.ptr, 2, n, n, vb.WINDOW_HANN_SYMMETRIC)
        res = c.pitch(fr, 48000.0, 0.45, 50.0, 600.0)
        assert np.all(res["n_cand"].to_host() >= 1) and np.all(res["status"].to_host() == vb.OK)
        assert np.all(np.isfinite(c.pitch_lag_function(fr).to_host()[:, : n // 2]))
