#!/usr/bin/env python
"""Cost of the peaks extension on the C4 workload (16 kHz, N=640, hop=160, 75-600 Hz, bench.py's 360 x 10 s utterances,
synthesised on the device): vbx_pitch and vbx_pitch_with_peaks (Praat's thresholds 0.45 / 0.03, peaks computed) alternated in
one process, the vbx_frame_peaks kernel time from vbx_profile_begin/end, and its unique bytes over that time as a fraction of
the B200's 7.7 TB/s.  GPU only.  Usage: python tools/bench_pitch_peaks.py [--reps R] [--out FILE.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vox_box.rs_b200", "python"))
import voxbox_b200 as vb  # noqa: E402

HBM_TBS = 7.7  # HGX B200 data sheet, one GPU


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers below are still device measurements; say that the query failed
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="alternating (vbx_pitch, vbx_pitch_with_peaks) pairs")
    ap.add_argument("--utts", type=int, default=360)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    fs, N, hop, K, seconds = 16000, 640, 160, 16, 10.0
    ctx = vb.Context(0)
    L, h = ctx.lib, ctx.h
    U, ns = args.utts, int(fs * seconds)
    J = ctx.n_frames_of(ns, N, hop)
    F = U * J
    audio = ctx.synth_speech(U, ns, fs, 0x5EED, 0)
    fr = ctx.frames(audio.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)
    cand, nc, st = ctx.empty((F, K, 2), np.float32), ctx.empty((F,), np.int32), ctx.empty((F,), np.uint8)
    local, glob = ctx.empty((F,), np.float64), ctx.empty((U,), np.float64)

    def plain():
        ctx._check(L.vbx_pitch(h, C.byref(fr), float(fs), 0.45, 75.0, 600.0, K, cand.ptr, nc.ptr, st.ptr, vb.F32), "vbx_pitch")

    def peaks():
        ctx._check(L.vbx_pitch_with_peaks(h, C.byref(fr), float(fs), 0.45, 0.03, None, None, 75.0, 600.0, K, cand.ptr, nc.ptr,
                                          st.ptr, vb.F32), "vbx_pitch_with_peaks")

    def frame_peaks():
        ctx._check(L.vbx_frame_peaks(h, C.byref(fr), local.ptr, glob.ptr), "vbx_frame_peaks")

    def timed(fn, n=1):
        ctx.sync()
        ctx.timer_start()
        for _ in range(n):
            fn()
        return ctx.timer_stop_ms() / n  # device events around the calls; stop synchronises

    for fn in (plain, peaks, plain, peaks):  # warm-up: modules, arena, window tables
        fn()
    t_plain, t_peaks = [], []
    for _ in range(args.reps):
        t_plain.append(timed(plain))
        t_peaks.append(timed(peaks))
    ctx.profile_begin()
    peaks()
    prof = ctx.profile_end()
    ms_kernel_prof = prof.get("frame_peaks_kernel", (float("nan"), 0))[0]
    frame_peaks()
    ms_kernel_loop = timed(frame_peaks, 50)  # the stand-alone call (memset + kernel), 50 back-to-back launches
    extent = (J - 1) * hop + N
    unique_bytes = U * extent * 4  # every sample the view spans, read once from HBM (frames overlap: the rest hits L2)

    def stats(v):
        v = np.asarray(v)
        return dict(mean=float(v.mean()), min=float(v.min()), max=float(v.max()), std=float(v.std()))

    name, power = gpu_info()
    s_plain, s_peaks = stats(t_plain), stats(t_peaks)
    rec = dict(
        workload=f"C4 shape: {U} utt x {J} frames = {F} frames, 16 kHz f32, N={N} hop={hop}, 75-600 Hz, {K} candidates, fp32 out",
        gpu=name, power_limit=power, reps=args.reps,
        ms_vbx_pitch=s_plain, ms_vbx_pitch_with_peaks=s_peaks,
        overhead_ms=s_peaks["mean"] - s_plain["mean"], overhead_pct=100.0 * (s_peaks["mean"] / s_plain["mean"] - 1.0),
        frame_peaks_kernel_ms_profiled=ms_kernel_prof,
        frame_peaks_call_ms=ms_kernel_loop,
        frame_peaks_kernel_share_pct=100.0 * ms_kernel_prof / s_peaks["mean"],
        unique_bytes=unique_bytes,
        hbm_fraction_profiled=unique_bytes / (ms_kernel_prof * 1e-3) / (HBM_TBS * 1e12),
        hbm_fraction_call=unique_bytes / (ms_kernel_loop * 1e-3) / (HBM_TBS * 1e12),
        profile={k: dict(ms=v[0], launches=v[1]) for k, v in prof.items()},
        note="hbm fractions: unique bytes (the samples the view spans) over kernel time, against 7.7 TB/s; the audio "
             "(230 MB) is larger than the 126 MB L2, but the back-to-back loop re-reads part of it from L2",
    )
    line = json.dumps(rec, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
