"""GPU tests of the round-2 additions, all through the C ABI vs the f64 oracle:
  * full pitch candidate LIST parity on >= 10 k frames (fp64 lag sweep; periodic.rs:403-453),
  * f64 sample input on every path (the reference's f64 callers; a frame windowed by the caller),
  * find_formants with the literal resampled_buf semantics (lib.rs:54,62-75; tests/lib.rs:44-90),
  * the LPC stage's scratch inside find_formants (Burg rows in global memory, non-fused autocorrelation),
  * the on-device synthetic corpus (determinism, statistics), executed-work counters,
  * vbx_multi: one handle drives the visible devices, results gathered into one host buffer."""
import os

import numpy as np
import pytest

from gpu_util import ctx, normwise, synth, vb

pytestmark = pytest.mark.gpu
MALE = np.array([[f, 1.0] for f in (320., 1440., 2760., 3200.)])


# ------------------------------------------------------------------------------------- pitch list parity
def test_pitch_full_list_parity_10k_frames(oracle):
    """Every position of the returned Vec<Pitch> (not only the top candidate) within 0.1 Hz / 1e-6 strength on 11 964
    frames of the on-device corpus: the fp32 lag sweep of round 1 left 0.3 % of the weak entries off by > 0.1 Hz."""
    c = ctx()
    fs, N, hop, K, U = 16000, 640, 160, 40, 12
    ns = fs * 10
    d = c.synth_speech(U, ns, fs, seed=0x5EED, first_utt=7000)
    audio = d.to_host()
    J = c.n_frames_of(ns, N, hop)
    F = U * J
    assert F >= 10000
    res = c.pitch(c.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns), float(fs), 0.45, 75.0,
                  600.0, K)
    cand, n, st = res["candidates"].to_host(), res["n_cand"].to_host(), res["status"].to_host()
    refs = [oracle.batch_pitch(audio[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, float(fs), 0.45, 75.0, 600.0, K, n_threads=0) for u in range(U)]
    rc, rn, rs = (np.concatenate([r[i] for r in refs]) for i in range(3))
    assert np.array_equal(st, rs)
    assert np.array_equal(n, rn)
    assert np.array_equal(cand[:, 0, 0] != 0, rc[:, 0, 0] != 0)
    mask = np.arange(K)[None, :] < np.minimum(n, K)[:, None]
    df = np.abs(cand[..., 0] - rc[..., 0])[mask]
    ds = np.abs(cand[..., 1] - rc[..., 1])[mask]
    n_bad = int(np.count_nonzero(df > 0.1))
    assert n_bad == 0, f"{n_bad} of {mask.sum()} list positions differ by > 0.1 Hz (max {df.max():.3e} Hz)"
    assert ds.max() < 1e-6, ds.max()


# ------------------------------------------------------------------------------------- f64 samples
def test_f64_samples_every_path(oracle):
    """A frame the caller windowed in f64 (what `for frame in Windower::hanning(..)` yields in the reference) goes in as
    VBX_F64 samples with VBX_WINDOW_NONE; results equal the oracle on the same f64 values."""
    c = ctx()
    fs, N, hop = 16000, 640, 160
    a32 = synth.utterance(9, fs, seconds=1.0)
    F = min(c.n_frames_of(a32.size, N, hop), 40)
    w = oracle.hanning_window(N)
    frames64 = np.stack([a32[f * hop:f * hop + N].astype(np.float64) * w for f in range(F)])  # packed, windowed in f64
    frames64 += 1e-9 * np.sin(np.arange(N))[None, :]  # not representable in fp32: narrowing would be visible
    d = c.to_device(frames64)
    fr = c.frames(d.ptr, F, N, N, vb.WINDOW_NONE, dtype=vb.F64)
    # autocorrelate + lpc
    r, ac, _ = c.lpc(fr, 12)
    rr = np.stack([oracle.autocorrelate(frames64[f], 13) for f in range(F)])
    ra = np.stack([oracle.lpc(rr[f], 12) for f in range(F)])
    assert np.max(normwise(r.to_host(), rr)) < 1e-12
    assert np.max(normwise(ac.to_host(), ra)) < 1e-8
    # pitch: full lists
    res = c.pitch(fr, float(fs), 0.45, 75.0, 600.0, 24)
    cand, n = res["candidates"].to_host(), res["n_cand"].to_host()
    for f in range(F):
        _, pc, ex = oracle.pitch(frames64[f], float(fs), 0.45, 75.0, 600.0, 24)
        assert n[f] == ex["n_cand"]
        k = min(n[f], 24)
        assert np.max(np.abs(cand[f, :k, 0] - pc[:k, 0])) < 0.1 and np.max(np.abs(cand[f, :k, 1] - pc[:k, 1])) < 1e-6
    # mfcc
    m = c.mfcc(fr, 40, 133.0, 6855.0, float(fs), n_keep=13).to_host()
    mo = np.stack([np.asarray(oracle.mfcc(frames64[f], 40, 133.0, 6855.0, float(fs)))[:13] for f in range(F)])
    assert np.max(normwise(m, mo)) < 1e-10


def test_f64_host_twin_lpc(oracle):
    import ctypes as C
    c = ctx()
    x = np.cumsum(np.random.default_rng(3).standard_normal(4000)) * 1e-2
    F = c.n_frames_of(x.size, 400, 160)
    fr = c.frames(x.ctypes.data, F, 400, 160, vb.WINDOW_HANN_SYMMETRIC, dtype=vb.F64)
    r = np.zeros((F, 13))
    ac = np.zeros((F, 13))
    c._check(c.lib.vbx_lpc_host(c.h, C.byref(fr), 12, r.ctypes.data, ac.ctypes.data, None, vb.F64), "vbx_lpc_host")
    w = oracle.hanning_window(400)
    rr = np.stack([oracle.autocorrelate(x[f * 160:f * 160 + 400] * w, 13) for f in range(F)])
    ra = np.stack([oracle.lpc(rr[f], 12) for f in range(F)])
    assert np.max(normwise(r, rr)) < 1e-12 and np.max(normwise(ac, ra)) < 1e-8


# ------------------------------------------------------------------------------------- literal buffer semantics
def test_find_formants_literal_buffer_semantics(oracle, fixtures_dir):
    """tests/lib.rs:44-90 as written: buf = 1024-sample frames (hop 1024, rectangle), resampled_buf.len() = the file
    length (2878), resample_ratio 1, 10 coefficients: Burg sees 1024 windowed samples followed by 1854 zeros."""
    c = ctx()
    x, fs = oracle.read_wav(os.path.join(fixtures_dir, "short_sample.wav"))
    xf = x.astype(np.float32)
    assert xf.size == 2878
    F = c.n_frames_of(xf.size, 1024, 1024)
    d = c.to_device(xf)
    fr = c.frames(d.ptr, F, 1024, 1024, vb.WINDOW_NONE)
    out = c.find_formants_buffered(fr, fs, 1.0, xf.size, 10, MALE[None])
    est = MALE.copy()
    for f in range(F):
        rbuf = np.zeros(xf.size)
        o = oracle.find_formants(xf[f * 1024:(f + 1) * 1024].astype(np.float64), fs, 10, est, resampled_buf=rbuf)
        assert o["status"] == 0
        est = o["formants"]
        assert np.max(np.abs(out["tracks"][f] - est)) < 0.5, (f, out["tracks"][f], est)
    # and the assert! of lib.rs:54
    with pytest.raises(vb.VoxBoxError) as e:
        c.find_formants_buffered(fr, fs, 1.0, 1000, 10, MALE[None])
    assert e.value.status == vb.ERR_BADARG
    # resampled AND buffered
    out2 = c.find_formants_buffered(fr, fs, 0.9, 1500, 10, MALE[None])
    est = MALE.copy()
    for f in range(F):
        rbuf = np.zeros(1500)
        o = oracle.find_formants(xf[f * 1024:(f + 1) * 1024].astype(np.float64), fs, 10, est, resample_ratio=0.9, resampled_buf=rbuf)
        est = o["formants"]
        assert np.max(np.abs(out2["tracks"][f] - est)) < 0.5


# ------------------------------------------------------------------------------------- nested scratch (ADVICE r1)
def test_find_formants_burg_global_scratch(oracle, monkeypatch):
    """Burg rows that do not fit shared memory come out of find_formants' own reservation (no arena growth under the
    caller's pointers): forced here with VBX_BURG_FORCE_GLOBAL on a batch large enough to move the arena."""
    c = ctx()
    fs, N, hop = 16000, 400, 160
    audio = synth.corpus(2, fs, seconds=2.0, first=40)
    ns = audio.shape[1]
    J = c.n_frames_of(ns, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, 2 * J, N, hop, vb.WINDOW_HANN_PERIODIC, frames_per_segment=J, segment_stride=ns)
    ref = c.find_formants(fr, float(fs), 12, vb.LPC_BURG, np.tile(MALE, (2, 1, 1)))
    monkeypatch.setenv("VBX_BURG_FORCE_GLOBAL", "1")
    c2 = vb.Context(0)  # a fresh context: its arena starts empty, so the call below sizes it in one reservation
    d2 = c2.to_device(audio)
    fr2 = c2.frames(d2.ptr, 2 * J, N, hop, vb.WINDOW_HANN_PERIODIC, frames_per_segment=J, segment_stride=ns)
    c2.profile_begin()
    out = c2.find_formants(fr2, float(fs), 12, vb.LPC_BURG, np.tile(MALE, (2, 1, 1)))
    names = c2.profile_end()
    assert "burg_block_kernel" in names
    c2.close()
    assert np.array_equal(out["n_res"], ref["n_res"]) and np.array_equal(out["status"], ref["status"])
    assert np.max(np.abs(out["tracks"] - ref["tracks"])) < 1e-6
    assert np.max(np.abs(out["resonances"] - ref["resonances"])) < 1e-6


def test_find_formants_generic_autocorrelation_scratch(oracle, monkeypatch):
    c = ctx()
    fs, N, hop = 16000, 400, 160
    audio = synth.utterance(41, fs, seconds=2.0)
    J = c.n_frames_of(audio.size, N, hop)
    d = c.to_device(audio)
    fr = c.frames(d.ptr, J, N, hop, vb.WINDOW_HANN_SYMMETRIC)
    ref = c.find_formants(fr, float(fs), 12, vb.LPC_AUTOCORR, MALE[None])
    monkeypatch.setenv("VBX_LPC_FORCE_GENERIC", "1")
    c2 = vb.Context(0)
    d2 = c2.to_device(audio)
    c2.profile_begin()
    out = c2.find_formants(c2.frames(d2.ptr, J, N, hop, vb.WINDOW_HANN_SYMMETRIC), float(fs), 12, vb.LPC_AUTOCORR, MALE[None])
    names = c2.profile_end()
    assert "autocorr_generic_kernel" in names and "levinson_kernel" in names
    c2.close()
    assert np.array_equal(out["n_res"], ref["n_res"])
    assert np.max(np.abs(out["tracks"] - ref["tracks"])) < 1e-3


# ------------------------------------------------------------------------------------- synthetic corpus + counters
def test_synth_speech_deterministic_and_speech_like():
    c = ctx()
    fs, ns = 16000, 32000
    a = c.synth_speech(6, ns, fs, seed=1234, first_utt=10).to_host()
    b = c.synth_speech(3, ns, fs, seed=1234, first_utt=13).to_host()
    assert np.array_equal(a[3:], b), "utterance u must depend on (seed, u) only"
    assert not np.array_equal(a[0], a[1])
    assert np.all(np.isfinite(a)) and np.all(np.abs(a) < 0.6)
    peak = np.max(np.abs(a), axis=1)
    assert np.all(peak > 0.4)  # scaled to peak 0.5 (+ the -40 dB floor)
    pcm = c.synth_speech(6, ns, fs, seed=1234, first_utt=10, dtype=vb.I16).to_host()
    assert pcm.dtype == np.int16
    assert np.max(np.abs(pcm / 32767.0 - a)) < 1.0 / 32767.0
    # a different seed gives a different corpus
    assert not np.array_equal(a, c.synth_speech(6, ns, fs, seed=1235, first_utt=10).to_host())


def test_profile_counters_count_executed_work():
    c = ctx()
    fs, N, hop = 16000, 400, 160
    d = c.synth_speech(2, fs * 2, fs, first_utt=50)
    J = c.n_frames_of(fs * 2, N, hop)
    fr = c.frames(d.ptr, 2 * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=fs * 2)
    c.profile_begin()
    c.find_formants(fr, float(fs), 12, vb.LPC_AUTOCORR, np.tile(MALE, (2, 1, 1)))
    names = c.profile_end()
    w = c.profile_counters()
    assert "lpc_roots_pair_kernel" in names
    F = 2 * J
    # 5 solves over degrees 12, 10, 8, 6, 4 with >= 2 rounds each: at least 80 Horner steps per frame
    assert w["roots_horner_steps"] >= 80 * F and w["roots_rounds"] >= 10 * F
    assert w["roots_horner_steps"] <= 20 * 40 * 32 * ((F + 31) // 32) * 1.01  # the 20-iteration cap bounds it
    Fp = 2 * c.n_frames_of(fs * 2, 640, hop)
    frp = c.frames(d.ptr, Fp, 640, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=Fp // 2, segment_stride=fs * 2)
    c.profile_begin()
    c.pitch(frp, float(fs), 0.45, 75.0, 600.0, 16)
    names = c.profile_end()
    w = c.profile_counters()
    assert "pitch_lag64_kernel" in names and "pitch_refine8q_kernel" in names
    assert w["refine_evals"] > 0 and w["refine_terms"] > w["refine_evals"]
    assert w["roots_horner_steps"] == 0  # zeroed by profile_begin


# ------------------------------------------------------------------------------------- vbx_multi
def test_multi_matches_single_context(oracle):
    """vbx_multi over every visible device (1 on the test box): sharded by utterance, gathered into one host buffer;
    results equal the single-context host twins bit for bit."""
    c = ctx()
    fs, N, hop, U = 16000, 400, 160, 7
    ns = fs * 2
    audio = c.synth_speech(U, ns, fs, first_utt=300).to_host()
    J = c.n_frames_of(ns, N, hop)
    F = U * J
    with vb.Multi(0) as m:
        assert m.n >= 1
        r, ac, kc = m.lpc_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, 12, vb.F64, J, ns)
        ff = m.find_formants_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(fs), 12, vb.LPC_AUTOCORR, np.tile(MALE, (U, 1, 1)),
                                  vb.F64, J, ns)
        pt = m.pitch_host(audio, U * c.n_frames_of(ns, 640, hop), 640, hop, vb.WINDOW_HANN_SYMMETRIC, float(fs), 0.45, 75.0, 600.0, 16,
                          vb.F64, c.n_frames_of(ns, 640, hop), ns)
        mf = m.mfcc_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, 40, 133.0, 6855.0, float(fs), 13, vb.F64, J, ns)
        assert m.kernel_launches > 0
        bw = m.h2d_bandwidth(32 << 20, 2)
        assert len(bw) == m.n and bw[0] > 1.0
    ff1 = c.find_formants_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, float(fs), 12, vb.LPC_AUTOCORR, np.tile(MALE, (U, 1, 1)), vb.F64, J, ns)
    for k in ("tracks", "estimates", "resonances", "n_res", "status"):
        assert np.array_equal(ff[k], ff1[k]), k
    Jp = c.n_frames_of(ns, 640, hop)
    pt1 = c.pitch_host(audio, U * Jp, 640, hop, vb.WINDOW_HANN_SYMMETRIC, float(fs), 0.45, 75.0, 600.0, 16, vb.F64, Jp, ns)
    assert np.array_equal(pt["candidates"], pt1["candidates"]) and np.array_equal(pt["n_cand"], pt1["n_cand"])
    mf1 = c.mfcc_host(audio, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, 40, 133.0, 6855.0, float(fs), 13, vb.F64, J, ns)
    assert np.array_equal(mf, mf1)
    rr = np.concatenate([oracle.batch_lpc(audio[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, 12)[0] for u in range(U)])
    assert np.max(normwise(r, rr)) < 1e-12


def test_multi_partition_rule():
    lo_hi = [vb.multi_partition(4500, 8, p) for p in range(8)]
    assert lo_hi[0][0] == 0 and lo_hi[-1][1] == 4500
    assert all(a[1] == b[0] for a, b in zip(lo_hi, lo_hi[1:]))
    assert max(h - l for l, h in lo_hi) - min(h - l for l, h in lo_hi) <= 1


# ------------------------------------------------------------------------------------- frame-chunk pipelining of find_formants
@pytest.mark.parametrize("method,window", [(vb.LPC_AUTOCORR, vb.WINDOW_HANN_SYMMETRIC), (vb.LPC_BURG, vb.WINDOW_HANN_PERIODIC)])
@pytest.mark.parametrize("segmented", [True, False])
def test_find_formants_frame_chunks_identical(monkeypatch, method, window, segmented):
    """vbx_find_formants processes the frames of every utterance in chunks (LPC + roots of chunk c + 1 on the main stream while
    the tracker steps through chunk c on the side stream): any chunk count gives bit-identical tracks, state, resonances,
    counts and status."""
    c = ctx()
    fs, N, hop, U = 16000, 400, 160, 5
    ns = fs * 2
    d = c.synth_speech(U, ns, fs, first_utt=900)
    J = c.n_frames_of(ns, N, hop)
    if segmented:
        fr = c.frames(d.ptr, U * J, N, hop, window, frames_per_segment=J, segment_stride=ns)
        est = np.tile(MALE, (U, 1, 1))
    else:
        fr = c.frames(d.ptr, c.n_frames_of(U * ns, N, hop), N, hop, window)
        est = MALE[None]
    monkeypatch.setenv("VBX_FORMANT_CHUNKS", "1")
    ref = c.find_formants(fr, float(fs), 12, method, est)
    ref_tracks_only = c.find_formants(fr, float(fs), 12, method, est, want_resonances=False)
    for k in ("3", "5", "8", "1000"):
        monkeypatch.setenv("VBX_FORMANT_CHUNKS", k)
        c.profile_begin()
        out = c.find_formants(fr, float(fs), 12, method, est)
        names = c.profile_end()
        assert names["tracker_idx_kernel"][1] == min(int(k), fr.frames_per_segment or fr.n_frames)
        for key in ("tracks", "estimates", "resonances", "n_res", "status"):
            assert np.array_equal(out[key], ref[key]), (k, key)
        out2 = c.find_formants(fr, float(fs), 12, method, est, want_resonances=False)
        assert np.array_equal(out2["tracks"], ref_tracks_only["tracks"]) and np.array_equal(out2["estimates"], ref_tracks_only["estimates"])
    assert np.array_equal(ref_tracks_only["tracks"], ref["tracks"])


# ------------------------------------------------------------------------------------- the aligned-down LPC kernel (vbx_lpca.cuh)
@pytest.mark.parametrize("N,hop,p,window", [(1102, 441, 12, vb.WINDOW_HANN_SYMMETRIC), (1102, 441, 12, vb.WINDOW_NONE), (333, 100, 12, vb.WINDOW_HANN_SYMMETRIC),
                                             (257, 100, 8, vb.WINDOW_HANN_PERIODIC), (64, 64, 4, vb.WINDOW_NONE), (17, 5, 12, vb.WINDOW_NONE),
                                             (50, 50, 1, vb.WINDOW_HANN_SYMMETRIC), (2047, 1, 12, vb.WINDOW_HANN_SYMMETRIC)])
@pytest.mark.parametrize("plan", ["32:8", "16:8", "32:4", "8:4"])
def test_lpc_aligned_kernel_shapes(oracle, monkeypatch, N, hop, p, window, plan):
    c = ctx()
    monkeypatch.setenv("VBX_LPCA_PLAN", plan)
    monkeypatch.setenv("VBX_LPC16", "0")
    audio = synth.utterance(77, 16000, seconds=1.0)
    F = min(c.n_frames_of(audio.size, N, hop), 300)
    d = c.to_device(audio)
    c.profile_begin()
    r, ac, kc = c.lpc(c.frames(d.ptr, F, N, hop, window), p)
    names = c.profile_end()
    if plan.startswith("32:"):  # smaller CTAs may not reach a whole warp once K shrinks for a short frame: general kernel then
        assert "lpc_fuseda_kernel" in names, names
    rr, ra, rk = oracle.batch_lpc(audio, F, N, hop, window, p, want_kc=True)
    assert np.max(normwise(r.to_host(), rr)) < 1e-12
    assert np.max(normwise(ac.to_host(), ra)) < 1e-8
    assert np.max(normwise(kc.to_host(), rk)) < 1e-8


def test_lpc_aligned_kernel_unaligned_base_segments_pcm_and_nonfinite(oracle):
    c = ctx()
    fs, N, hop, p = 44100, 1102, 441, 12
    audio = synth.corpus(3, fs, seconds=1.0, first=60)  # 3 utterances x 44100 samples
    ns = audio.shape[1]
    J = c.n_frames_of(ns, N, hop)
    # (1) every base alignment, segmented view
    flat = np.concatenate([np.zeros(8, np.float32), audio.reshape(-1), np.zeros(8, np.float32)])
    d = c.to_device(flat)
    for off in range(8):
        x = flat[off:off + 3 * ns].reshape(3, ns)
        c.profile_begin()
        r, ac, _ = c.lpc(c.frames(d.ptr + 4 * off, 3 * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns), p)
        assert "lpc_fuseda_kernel" in c.profile_end()
        rr = np.concatenate([oracle.batch_lpc(np.ascontiguousarray(x[u]), J, N, hop, oracle.WIN_HANN_SYMMETRIC, p)[0] for u in range(3)])
        assert np.max(normwise(r.to_host(), rr)) < 1e-12, off
    # (2) int16 PCM, odd sample offsets
    pcm = np.clip(np.round(audio[0].astype(np.float64) * 32767), -32768, 32767).astype(np.int16)
    dp = c.to_device(np.concatenate([np.zeros(8, np.int16), pcm]))
    for off in (0, 1, 3, 5, 7):
        fr = c.frames(dp.ptr + 2 * (8 - off), c.n_frames_of(ns - 8, N, hop), N, hop, vb.WINDOW_HANN_SYMMETRIC, dtype=vb.I16)
        r, ac, _ = c.lpc(fr, p)
        x = np.concatenate([np.zeros(off, np.int16), pcm])[: ns].astype(np.float32) / np.float32(1.0)
        xs = (np.concatenate([np.zeros(off), pcm.astype(np.float64)]) / 32767.0)
        w = oracle.hanning_window(N)
        rr = np.stack([oracle.autocorrelate(xs[f * hop:f * hop + N] * w, p + 1) for f in range(fr.n_frames)])
        assert np.max(normwise(r.to_host(), rr)) < 1e-9, off  # sample/32767·w vs sample·(w/32767): an ulp of f64
    # (3) non-finite samples: a NaN / Inf poisons exactly the frames that contain it (the zero-weight neighbours do not)
    bad = audio[0].copy()
    bad[5000] = np.nan
    bad[20000] = np.inf
    bad[20001] = -np.inf
    db = c.to_device(bad)
    r, ac, _ = c.lpc(c.frames(db.ptr, J, N, hop, vb.WINDOW_HANN_SYMMETRIC), p)
    rr, ra = oracle.batch_lpc(bad, J, N, hop, oracle.WIN_HANN_SYMMETRIC, p)
    rg = r.to_host()
    assert np.array_equal(np.isnan(rg), np.isnan(rr))
    ok = ~np.isnan(rr).any(axis=1)
    assert ok.sum() > J // 2 and np.max(normwise(rg[ok], rr[ok])) < 1e-12


def test_find_formants_c3_uses_aligned_kernel(oracle):
    c = ctx()
    fs, N, hop = 44100, 1102, 441
    d = c.synth_speech(4, fs * 2, fs, first_utt=1234)
    audio = d.to_host()
    J = c.n_frames_of(fs * 2, N, hop)
    fr = c.frames(d.ptr, 4 * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=fs * 2)
    c.profile_begin()
    out = c.find_formants(fr, float(fs), 12, vb.LPC_AUTOCORR, np.tile(MALE, (4, 1, 1)))
    names = c.profile_end()
    assert "lpc_fuseda_kernel" in names
    for u in range(4):
        o = oracle.batch_formants(audio[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, 1, float(fs), 12, np.array([0, J]), MALE)
        sl = slice(u * J, (u + 1) * J)
        assert np.array_equal(out["n_res"][sl], o["n_res"])
        assert np.max(np.abs(out["tracks"][sl] - o["tracks"])) < 0.5


# ------------------------------------------------------------------------------------- the persistent TMA-fed LPC kernel
@pytest.mark.parametrize("N,hop,p,fs", [(1102, 441, 12, 44100), (400, 100, 12, 16000), (333, 333, 5, 16000), (1000, 30, 12, 16000)])
def test_lpc_persistent_kernel(oracle, monkeypatch, N, hop, p, fs):
    """Batches with at least two tiles of 32 frames per SM take lpc_fusedp_kernel (warp-specialised, TMA + mbarrier ring);
    same arithmetic as the one-shot aligned kernel: bit-identical to it, and within rounding of the oracle.  Covers ragged
    last tiles of a segment, every base alignment, a non-finite sample, and fewer parts."""
    c = ctx()
    monkeypatch.setenv("VBX_LPC16", "0")
    ns = fs * 3 + 7  # odd utterance length: segment starts walk through the alignments
    U = max(14, -(-2 * c.sm_count // ((c.n_frames_of(ns, N, hop) + 31) // 32)) + 1)  # at least two tiles per SM
    d = c.synth_speech(U, ns, fs, first_utt=4242)
    audio = d.to_host()
    J = c.n_frames_of(ns, N, hop)
    tiles = U * ((J + 31) // 32)
    sm = c.sm_count
    fr = c.frames(d.ptr, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)
    c.profile_begin()
    r, ac, kc = c.lpc(fr, p)
    names = c.profile_end()
    assert tiles >= 2 * sm and "lpc_fusedp_kernel" in names, (names, tiles)
    rg, ag, kg = r.to_host(), ac.to_host(), kc.to_host()
    monkeypatch.setenv("VBX_LPCP", "0")
    c.profile_begin()
    r2, ac2, kc2 = c.lpc(fr, p)
    assert "lpc_fuseda_kernel" in c.profile_end()
    monkeypatch.delenv("VBX_LPCP")
    assert np.array_equal(rg, r2.to_host()) and np.array_equal(ag, ac2.to_host()) and np.array_equal(kg, kc2.to_host())
    for u in (0, 5, U - 1):
        rr, ra = oracle.batch_lpc(audio[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, p)
        assert np.max(normwise(rg[u * J:(u + 1) * J], rr)) < 1e-12
        assert np.max(normwise(ag[u * J:(u + 1) * J], ra)) < 1e-8
    # fewer parts, fp32 outputs, r only
    monkeypatch.setenv("VBX_LPCP_K", "4")
    r4, a4, _ = c.lpc(fr, p, out_dtype=vb.F32, want_kc=False)
    monkeypatch.delenv("VBX_LPCP_K")
    assert np.max(normwise(r4.to_host(), rg)) < 1e-6 and np.max(normwise(a4.to_host(), ag)) < 1e-5


def test_lpc_persistent_kernel_nonfinite_and_alignment(oracle, monkeypatch):
    c = ctx()
    fs, N, hop, p = 44100, 1102, 441, 12
    U, ns = 32, 44100 * 3  # 32 x 10 tiles >= 2 per SM
    base = c.synth_speech(U, ns, fs, first_utt=99).to_host()
    for off in range(4):
        flat = np.concatenate([np.zeros(off, np.float32), base.reshape(-1), np.zeros(16, np.float32)])
        x = flat[off:off + U * ns].reshape(U, ns).copy()
        if off == 1:
            flat[off + 5000] = np.nan            # inside frames
            flat[off + 2 * ns + 441 * 7 - 1] = np.inf  # one sample before frame 7 of utterance 2: a zero-weight neighbour for a = 1..3
            x = flat[off:off + U * ns].reshape(U, ns).copy()
        d = c.to_device(flat)
        J = c.n_frames_of(ns, N, hop)
        fr = c.frames(d.ptr + 4 * off, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)
        c.profile_begin()
        r, ac, _ = c.lpc(fr, p)
        assert "lpc_fusedp_kernel" in c.profile_end()
        rg = r.to_host()
        for u in (0, 2, U - 1):
            rr, _ = oracle.batch_lpc(np.ascontiguousarray(x[u]), J, N, hop, oracle.WIN_HANN_SYMMETRIC, p)
            sl = rg[u * J:(u + 1) * J]
            assert np.array_equal(np.isnan(sl), np.isnan(rr)), (off, u)
            ok = np.isfinite(rr).all(axis=1)
            assert np.max(normwise(sl[ok], rr[ok])) < 1e-12, (off, u)


# ------------------------------------------------------------------------------------- roots fix-up launch
def test_roots_fixup_redoes_flagged_frames_in_f64(oracle, monkeypatch):
    """Frames on which the pair-deflation kernel's Laguerre solve runs into the 20-iteration cap without converging are redone by
    the f64 reference-order kernel.  VBX_ROOTS_FORCE_HARD=7 flags every 7th frame: those rows must equal the precision = 1 path bit
    for bit, the others the unflagged pair result."""
    c = ctx()
    fs, N, hop = 44100, 1102, 441
    d = c.synth_speech(2, fs * 2, fs, first_utt=3131)
    J = c.n_frames_of(fs * 2, N, hop)
    fr = c.frames(d.ptr, 2 * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=fs * 2)
    r, ac, _ = c.lpc(fr, 12)
    pair = c.lpc_to_resonances(ac, 12, True, float(fs))
    f64 = c.lpc_to_resonances(ac, 12, True, float(fs), precision=1)
    monkeypatch.setenv("VBX_ROOTS_FORCE_HARD", "7")
    c.profile_begin()
    mixed = c.lpc_to_resonances(ac, 12, True, float(fs))
    names = c.profile_end()
    assert "lpc_roots_pair_kernel" in names and "lpc_roots_rt_kernel<double> (fix-up launch)" in names
    a, b, m = pair["resonances"].to_host(), f64["resonances"].to_host(), mixed["resonances"].to_host()
    flagged = (np.arange(2 * J) % 7) == 0
    assert np.array_equal(m[flagged], b[flagged])
    assert np.array_equal(m[~flagged], a[~flagged])
    assert np.array_equal(mixed["n_res"].to_host(), pair["n_res"].to_host())
    assert np.max(np.abs(a - b)) < 1e-3  # and the two solvers agree anyway


def test_lpc_persistent_kernel_repeatable_under_load(monkeypatch):
    """The persistent kernel's hand-offs are mbarriers (TMA completion, part buffers) — primitives compute-sanitizer's racecheck does
    not model, so it reports them as hazards.  A real race would show as run-to-run differences: 12 repetitions on a batch of ~40
    tiles per SM, also with other work queued on the device, must be bit-identical to the one-shot kernel's result."""
    c = ctx()
    fs, N, hop, p = 44100, 1102, 441, 12
    U, ns = 200, fs * 3
    d = c.synth_speech(U, ns, fs, first_utt=777)
    J = c.n_frames_of(ns, N, hop)
    fr = c.frames(d.ptr, U * J, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)
    monkeypatch.setenv("VBX_LPCP", "0")
    r0, a0, k0 = (x.to_host() for x in c.lpc(fr, p))
    monkeypatch.delenv("VBX_LPCP")
    other = vb.Context(0)  # a second context keeps the device busy with another stream's kernels
    d2 = other.synth_speech(64, 16000 * 10, 16000, first_utt=1)
    fr2 = other.frames(d2.ptr, 64 * 997, 640, 160, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=997, segment_stride=160000)
    for rep in range(12):
        if rep % 2:
            other.pitch(fr2, 16000.0, 0.45, 75.0, 600.0, 16)  # asynchronous on the other context's stream
        c.profile_begin()
        r, a, k = c.lpc(fr, p)
        assert "lpc_fusedp_kernel" in c.profile_end()
        assert np.array_equal(r.to_host(), r0) and np.array_equal(a.to_host(), a0) and np.array_equal(k.to_host(), k0), rep
    other.sync()
    other.close()
