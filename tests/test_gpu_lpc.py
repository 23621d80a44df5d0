"""GPU parity: windowed autocorrelation + Levinson (north-star chain C2) through the C ABI vs the
f64 oracle.  Tolerance (BASELINE.json north_star): autocorrelation and LPC within 1e-5 relative,
measured norm-wise per frame vector (SURVEY §8d)."""
import numpy as np
import pytest

from gpu_util import ctx, normwise, synth, vb

pytestmark = pytest.mark.gpu
TOL = 1e-5  # north_star: "autocorrelation, LPC ... within 1e-5 relative (fp32)"


def _run_lpc(audio, N, hop, window, p, out_dtype):
    c = ctx()
    F = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    r, ac, kc = c.lpc(c.frames(d.ptr, F, N, hop, window), p, out_dtype=out_dtype)
    return F, r.to_host(), ac.to_host(), kc.to_host()


@pytest.mark.parametrize("fs,N,hop", [(16000, 400, 160), (44100, 1102, 441)])
@pytest.mark.parametrize("out_dtype", [vb.F64, vb.F32])
def test_lpc12_synthetic_speech(oracle, fs, N, hop, out_dtype):
    """C2 / C3 shapes on the synthetic corpus (−40 dB noise floor), order 12."""
    audio = synth.utterance(3, fs, seconds=2.0)
    p = 12
    F, r, ac, kc = _run_lpc(audio, N, hop, vb.WINDOW_HANN_SYMMETRIC, p, out_dtype)
    r_ref, ac_ref, kc_ref = oracle.batch_lpc(audio, F, N, hop, oracle.WIN_HANN_SYMMETRIC, p, n_threads=0, want_kc=True)
    assert r.shape == r_ref.shape and ac.shape == ac_ref.shape and kc.shape == kc_ref.shape
    assert np.max(normwise(r, r_ref)) < TOL
    assert np.max(normwise(ac, ac_ref)) < TOL
    assert np.max(normwise(kc, kc_ref)) < TOL
    if out_dtype == vb.F64:  # fp64 accumulation: far inside the tolerance
        assert np.max(normwise(r, r_ref)) < 1e-12
        assert np.max(normwise(ac, ac_ref)) < 1e-7


@pytest.mark.parametrize("window", [vb.WINDOW_NONE, vb.WINDOW_HANN_SYMMETRIC, vb.WINDOW_HANN_PERIODIC])
@pytest.mark.parametrize("N,hop,n_lags", [(400, 160, 13), (64, 64, 9), (101, 37, 5), (1102, 441, 13), (30, 7, 30),
                                           (512, 512, 17), (257, 300, 11), (2048, 1024, 25), (640, 160, 2)])
def test_autocorrelate_shapes(oracle, window, N, hop, n_lags):
    """Overlapped, packed and gapped views, odd sizes, every fused lag count class, incl. the
    reference's `x[0] +` seed quirk (visible with WINDOW_NONE where x[0] != 0)."""
    rng = np.random.default_rng(N * 1000 + hop)
    F = 37
    audio = rng.standard_normal((F - 1) * hop + N).astype(np.float32)
    c = ctx()
    d = c.to_device(audio)
    r = c.autocorrelate(c.frames(d.ptr, F, N, hop, window), n_lags, out_dtype=vb.F64).to_host()
    r_ref = oracle.batch_autocorrelate(audio, F, N, hop, window, n_lags)
    assert np.max(normwise(r, r_ref)) < 1e-12


def test_autocorrelate_generic_fallback(oracle):
    """n_lags above the fused range (pitch-style full-lag call) takes the generic kernel."""
    rng = np.random.default_rng(5)
    N, hop, F = 300, 100, 9
    audio = rng.standard_normal((F - 1) * hop + N).astype(np.float32)
    c = ctx()
    d = c.to_device(audio)
    for n_lags in (1, 26, 300):
        r = c.autocorrelate(c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC), n_lags).to_host()
        r_ref = oracle.batch_autocorrelate(audio, F, N, hop, oracle.WIN_HANN_SYMMETRIC, n_lags)
        assert np.max(normwise(r, r_ref)) < 1e-12


def test_doc_example_quirk(oracle):  # periodic.rs:262-263 (doc is wrong; code gives [2.5, 1.5])
    c = ctx()
    x = np.array([1.0, 0.5, 0.0, -0.5, -1.0], dtype=np.float32)
    r = c.autocorrelate_host(x, 1, 5, 5, vb.WINDOW_NONE, 2)
    assert r.tolist() == [[2.5, 1.5]]


def test_lpc_kat_through_gpu(oracle):  # spectrum.rs:471-487 test_lpc: sine(8) → autocorrelate(8) → normalize → lpc(4)
    c = ctx()
    s = oracle.sine(8).astype(np.float32)
    r = c.autocorrelate_host(s, 1, 8, 8, vb.WINDOW_NONE, 8)[0]
    auto = r / np.max(np.abs(r))
    assert np.all(np.abs(auto - [1.0, 0.7071, 0.1250, -0.3536, -0.5, -0.3536, -0.1250, 0.0]) < 1e-4)
    ac, kc = c.lpc_levinson(c.to_device(auto[None, :]), 4)
    assert np.all(np.abs(ac.to_host()[0] - [1.0, -1.3122, 0.8660, -0.0875, -0.0103]) < 1e-4)


@pytest.mark.parametrize("p", [1, 2, 7, 12, 16, 24, 32])
def test_levinson_orders(oracle, p):
    rng = np.random.default_rng(p)
    F = 50
    x = rng.standard_normal((F, 256))
    r = np.stack([oracle.autocorrelate(x[f] * oracle.hanning_window(256), p + 1) for f in range(F)])
    c = ctx()
    ac, kc = c.lpc_levinson(c.to_device(r), p)
    ref = [oracle.lpc(r[f], p, with_kc=True) for f in range(F)]
    assert np.max(normwise(ac.to_host(), np.stack([a for a, _ in ref]))) < 1e-9
    assert np.max(normwise(kc.to_host(), np.stack([k for _, k in ref]))) < 1e-9


def test_lpc_host_twin_matches_device(oracle):
    audio = synth.utterance(1, 16000, seconds=1.0)
    c = ctx()
    F = c.n_frames_of(audio.size, 400, 160)
    r, ac, kc = c.lpc_host(audio, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 12)
    _, r2, ac2, kc2 = _run_lpc(audio, 400, 160, vb.WINDOW_HANN_SYMMETRIC, 12, vb.F64)
    assert np.array_equal(r, r2) and np.array_equal(ac, ac2) and np.array_equal(kc, kc2)


def test_ragged_and_empty_inputs(oracle):
    c = ctx()
    assert c.n_frames_of(399, 400, 160) == 0  # Windower drops a short tail entirely
    d = c.to_device(np.zeros(400, dtype=np.float32))
    r, ac, kc = c.lpc(c.frames(d.ptr, 0, 400, 160, vb.WINDOW_HANN_SYMMETRIC), 12)  # zero frames: no-op
    assert r.shape == (0, 13)
    with pytest.raises(vb.VoxBoxError) as e:  # lag >= len: the reference's `self.len() - lag` underflows
        c.autocorrelate(c.frames(d.ptr, 1, 10, 10, vb.WINDOW_NONE), 11)
    assert e.value.status == vb.ERR_BADARG
    # silent frame: r = 0, Levinson divides by err = 0 → NaN propagates exactly like the reference
    r, ac, kc = c.lpc(c.frames(d.ptr, 1, 400, 160, vb.WINDOW_HANN_SYMMETRIC), 12)
    assert np.all(r.to_host() == 0.0) and np.isnan(ac.to_host()[0, 1])


def test_full_size_properties(oracle):
    """BASELINE C2 at full size (1 h of 16 kHz audio, 359 280 frames): size-independent properties
    (r[0] = frame energy >= |r[lag]|, ac[0] = 1, |kc| < 1 for a valid autocorrelation, linearity of r in
    gain²) plus oracle parity on a random subset of frames."""
    fs, N, hop, p, n_utts = 16000, 400, 160, 12, 360
    base = synth.corpus(6, fs)  # 6 distinct utterances tiled to 1 h (generation cost only)
    audio = np.tile(base, (n_utts // 6, 1))
    c = ctx()
    d = c.to_device(audio)
    n_samp = audio.shape[1]
    f_per = c.n_frames_of(n_samp, N, hop)
    assert f_per == 998 and f_per * n_utts == 359280
    # one two-level view over the whole [n_utts, n_samp] tensor: frame u*J + j starts at u*n_samp + j*hop
    fr = c.frames(d.ptr, n_utts * f_per, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=f_per, segment_stride=n_samp)
    r_all, a_all, k_all = c.lpc(fr, p, out_dtype=vb.F64)
    r, a, k = r_all.to_host(), a_all.to_host(), k_all.to_host()
    assert np.all(np.isfinite(r)) and np.all(np.isfinite(a))
    assert np.all(r[:, 0] > 0) and np.all(np.abs(r[:, 1:]) <= r[:, :1] * (1 + 1e-12))
    assert np.all(a[:, 0] == 1.0) and np.all(np.abs(k) < 1.0)
    # tiling: utterance u and u+6 are identical inputs → identical outputs (determinism across CTAs)
    assert np.array_equal(r[: 6 * f_per], r[6 * f_per: 12 * f_per])
    rng = np.random.default_rng(0)
    pick = np.sort(rng.choice(6 * f_per, 400, replace=False))
    flat = audio[:6].reshape(-1)
    for f in pick:
        u, j = divmod(int(f), f_per)
        seg = flat[u * n_samp + j * hop: u * n_samp + j * hop + N]
        r_ref, a_ref = oracle.batch_lpc(np.ascontiguousarray(seg), 1, N, N, oracle.WIN_HANN_SYMMETRIC, p)
        assert normwise(r[f], r_ref[0]) < 1e-12 and normwise(a[f], a_ref[0]) < TOL


def test_autocorrelate_ring_vecdeque(oracle):
    """periodic.rs:291-304 `impl Autocorrelate for VecDeque`: wrap-around rings give the same lags as the unrolled slice."""
    c = ctx()
    rng = np.random.default_rng(8)
    cap, n = 700, 512
    rings = rng.standard_normal((5, cap))
    heads = np.array([0, 1, 188, 350, 699])
    r = c.autocorrelate_ring(rings, heads, n, 16)
    for b in range(5):
        x = np.roll(rings[b], -heads[b])[:n]
        assert np.max(np.abs(r[b] - oracle.autocorrelate(x, 16))) < 1e-12 * np.max(np.abs(r[b]))
    r32 = c.autocorrelate_ring(rings.astype(np.float32), heads, n, 16, out_dtype=vb.F32)
    assert r32.dtype == np.float32 and np.allclose(r32, r, rtol=1e-5)
    with pytest.raises(vb.VoxBoxError) as e:
        c.autocorrelate_ring(rings, heads, n, n + 1)
    assert e.value.status == vb.ERR_BADARG


@pytest.mark.parametrize("N,hop,n_lags", [(400, 160, 13), (16, 16, 2), (16, 16, 16), (32, 16, 9), (48, 16, 16), (64, 64, 13),
                                           (512, 128, 11), (512, 512, 16), (400, 480, 13), (1024, 256, 15), (2048, 1024, 14),
                                           (640, 160, 3)])
@pytest.mark.parametrize("F", [1, 7, 333])
def test_autocorrelate_16_aligned_kernel(oracle, N, hop, n_lags, F):
    """The 16-sample-chunk kernel (frame length and hop multiples of 16, <= 16 lags): odd / even chunk counts (one or two
    pre-roll chunks for the second half-frame lane), a single chunk, packed and gapped views, partial last CTA, the
    x[0]-seed quirk (WINDOW_NONE), float and int16 samples, a base pointer that is not 16-byte aligned."""
    rng = np.random.default_rng(N * 131 + hop * 7 + n_lags)
    total = (F - 1) * hop + N
    audio = rng.standard_normal(total + 3).astype(np.float32)
    c = ctx()
    d = c.to_device(audio)
    for off in (0, 3):  # off = 3: staging takes the scalar path
        for window in (vb.WINDOW_NONE, vb.WINDOW_HANN_SYMMETRIC):
            r = c.autocorrelate(c.frames(d.ptr + 4 * off, F, N, hop, window), n_lags, out_dtype=vb.F64).to_host()
            r_ref = oracle.batch_autocorrelate(audio[off:off + total], F, N, hop, window, n_lags)
            assert np.max(normwise(r, r_ref)) < 1e-12, (off, window)
    pcm = np.clip(np.round(audio * 8000.0), -32767, 32767).astype(np.int16)
    dp = c.to_device(pcm)
    r = c.autocorrelate(c.frames(dp.ptr, F, N, hop, vb.WINDOW_HANN_PERIODIC, dtype=vb.I16), n_lags, out_dtype=vb.F64).to_host()
    # int16 samples are scaled by 1/32767 on load (folded into the window table): compare with the oracle on the integer
    # values (exact in fp32) scaled afterwards
    r_ref = oracle.batch_autocorrelate(pcm[:total].astype(np.float32), F, N, hop, vb.WINDOW_HANN_PERIODIC, n_lags) / 32767.0 ** 2
    assert np.max(normwise(r, r_ref)) < 1e-12


def test_lpc_16_aligned_kernel_segments(oracle):
    """Segmented batch (utterances) through the 16-aligned kernel: CTAs never straddle segments."""
    fs, N, hop, p = 16000, 400, 160, 12
    utts = np.stack([synth.utterance(u, fs, seconds=1.0) for u in range(5)])
    J = (utts.shape[1] - N) // hop + 1
    c = ctx()
    d = c.to_device(utts)
    fr = c.frames(d.ptr, 5 * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=utts.shape[1])
    r, ac, kc = c.lpc(fr, p, out_dtype=vb.F64)
    r, ac = r.to_host(), ac.to_host()
    for u in range(5):
        r_ref, ac_ref = oracle.batch_lpc(utts[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, p)
        assert np.max(normwise(r[u * J:(u + 1) * J], r_ref)) < 1e-12
        assert np.max(normwise(ac[u * J:(u + 1) * J], ac_ref)) < 1e-7


@pytest.mark.parametrize("ns,dtype", [(16000, "f32"), (16001, "f32"), (16003, "i16"), (24000, "i16"), (8000, "f32")])
def test_lpc_16_aligned_kernel_straddles_utterances(oracle, ns, dtype):
    """CTAs of the 16-aligned kernel take 64 consecutive frames of the batch, so most of them cross from one utterance into
    the next and stage their span as two pieces; an odd utterance length makes the second piece's source unaligned
    (scalar staging path).  Utterances shorter than one CTA's 64 frames (ns = 8000: 48 frames) take the per-segment mode,
    one utterance per CTA.  Results must equal the per-utterance oracle in both modes."""
    fs, N, hop, p, U = 16000, 400, 160, 12, 7
    rng = np.random.default_rng(ns)
    audio = (rng.standard_normal((U, ns)) * 0.1).astype(np.float32)
    J = (ns - N) // hop + 1
    c = ctx()
    if dtype == "i16":
        pcm = np.clip(np.round(audio * 20000.0), -32767, 32767).astype(np.int16)
        d = c.to_device(pcm)
        ref_in = pcm.astype(np.float32)          # exact in fp32; the 1/32767 scale is applied to r afterwards
        scale = 1.0 / 32767.0 ** 2
        fr = c.frames(d.ptr, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, dtype=vb.I16, frames_per_segment=J, segment_stride=ns)
    else:
        d = c.to_device(audio)
        ref_in, scale = audio, 1.0
        fr = c.frames(d.ptr, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)
    c.profile_begin()
    r = c.autocorrelate(fr, p + 1, out_dtype=vb.F64).to_host()
    assert "lpc_fused16_kernel" in c.profile_end()
    for u in range(U):
        r_ref = oracle.batch_autocorrelate(ref_in[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, p + 1) * scale
        assert np.max(normwise(r[u * J:(u + 1) * J], r_ref)) < 1e-12, u
