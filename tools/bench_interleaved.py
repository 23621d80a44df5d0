"""Interleaved multi-channel input (vbx_frames.sample_step) vs its planar equivalent, on the sizes a user runs: one hour of
8 kHz stereo G.711 mu-law (the two-channel call-centre recording) and one hour of 44.1 kHz stereo int16 on C3's framing.

Reports, per recording:
 - gather: interleave_gather_kernel's time per call (vbx_profile_*) and the HBM bytes it moves (each interleaved byte read
   once, each planar byte written once) over that time.  The kernel is a copy: HBM bandwidth is what bounds it.
 - device-resident frames/s of LPC-12, LPC-12 + formants, MFCC and pitch on the interleaved view (samples in HBM, the gather
   included) and on its planar equivalent (already deinterleaved in HBM); the difference is the gather's cost.
 - end to end: the `_host` call on the interleaved buffer (channels as segments, staged once) against numpy deinterleaving
   the same buffer on one CPU thread into a planar buffer plus the planar `_host` call; both buffers are pinned.  The
   deinterleave is timed on its own as well.
Outputs are checked equal between the interleaved and planar calls before anything is timed.  The card's name, power limit
and clocks are read in the same run.  Writes one JSON file (--out).

    python tools/bench_interleaved.py --out bench_interleaved.json
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402  (Pinned, MALE, SEED)
from bench_g711 import gpu_info  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "vox_box.rs_b200", "python"))
import voxbox_b200 as vb  # noqa: E402

NP = {vb.I16: np.int16, vb.MULAW8: np.uint8}
RECORDINGS = {
    "tel_stereo_mulaw_1h": dict(fs=8000, seconds=3600.0, channels=2, dtype=vb.MULAW8, n=200, hop=80, pitch_n=320,
                                mfcc=(26, 100.0, 3800.0)),
    "c3_stereo_i16_1h": dict(fs=44100, seconds=3600.0, channels=2, dtype=vb.I16, n=1102, hop=441, pitch_n=1764,
                             mfcc=(40, 133.0, 6855.0)),
}
PATHS = ("lpc12", "lpc12_formants", "mfcc", "pitch")


def calls(ctx, rec, fr, outs, host):
    """The call of every path on view `fr`: device pointers (host=False) or the `_host` twin (host=True)."""
    L, h, fs = ctx.lib, ctx.h, float(rec["fs"])
    M, lo, hi = rec["mfcc"]
    o = outs["h" if host else "d"]
    est = outs["est_h" if host else "est_d"]
    U = rec["channels"]

    def ck(st, what):
        ctx._check(st, what)

    def formants(f):
        if host:
            est.a[...] = outs["est0"].reshape(U, 8)
            ck(L.vbx_find_formants_host(h, C.byref(f), fs, 12, vb.LPC_AUTOCORR, est.ptr, 4, o["tracks"].ptr, None, None, None, vb.F32),
               "vbx_find_formants_host")
        else:
            ck(L.vbx_memcpy_d2d(h, est.ptr, outs["est0_d"].ptr, outs["est0"].nbytes), "d2d")
            ck(L.vbx_find_formants(h, C.byref(f), fs, 12, vb.LPC_AUTOCORR, est.ptr, 4, o["tracks"].ptr, None, None, None, vb.F32),
               "vbx_find_formants")

    sfx = "_host" if host else ""
    lpc = getattr(L, "vbx_lpc" + sfx)
    mfcc = getattr(L, "vbx_mfcc" + sfx)
    pitch = getattr(L, "vbx_pitch" + sfx)
    return {
        "lpc12": lambda f: ck(lpc(h, C.byref(f), 12, None, o["ac"].ptr, None, vb.F32), "lpc"),
        "lpc12_formants": formants,
        "mfcc": (lambda f: ck(mfcc(h, C.byref(f), M, 13, lo, hi, fs, o["mfcc"].ptr, vb.F32), "mfcc")) if host else
                (lambda f: ck(mfcc(h, C.byref(f), M, 13, lo, hi, fs, o["mfcc"].ptr, None, vb.F32), "mfcc")),
        "pitch": lambda f: ck(pitch(h, C.byref(f), fs, 0.45, 75.0, 600.0, 8, o["cand"].ptr, None, None, vb.F32), "pitch"),
    }


def run(ctx, key, rec, steps, e2e_steps):
    fs, U, dt = rec["fs"], rec["channels"], rec["dtype"]
    ns = int(round(fs * rec["seconds"]))
    npt = NP[dt]
    es = np.dtype(npt).itemsize
    pinned = []

    def pin(shape, dtype):
        b = bench.Pinned(ctx, shape, dtype)
        pinned.append(b)
        return b

    # channel u = utterance u of bench.py's seeded synthetic corpus; planar [U][ns] on the device, interleaved [ns][U] both places
    d_plan = ctx.synth_speech(U, ns, float(fs), bench.SEED, 0, dtype=dt)
    h_plan = pin((U, ns), npt)
    ctx._check(ctx.lib.vbx_memcpy_d2h(ctx.h, h_plan.ptr, d_plan.ptr, h_plan.nbytes), "d2h")
    ctx.sync()
    h_int = pin((ns, U), npt)
    h_int.a[...] = h_plan.a.T
    d_int = ctx.to_device(h_int.a)
    h_dst = pin((U, ns), npt)  # where the numpy deinterleave writes
    out = {"fs": fs, "seconds": rec["seconds"], "channels": U, "dtype": {vb.I16: "i16", vb.MULAW8: "mulaw8"}[dt],
           "interleaved_bytes": int(h_int.nbytes), "paths": {}}
    est0 = np.tile(np.array([[f, 1.0] for f in bench.MALE], dtype=np.float32), (U, 1, 1))
    for path in PATHS:
        N = rec["pitch_n"] if path == "pitch" else rec["n"]
        hop = rec["hop"]
        J = bench.n_frames_of(ns, N, hop)
        F = U * J
        win = vb.WINDOW_HANN_SYMMETRIC
        # the interleaved view (one segment per channel, step U) and the planar [U][ns] a deinterleaving caller holds: its rows
        # are a multiple of 64 samples like the planar equivalent's, so both put every segment at the same alignment
        assert ns % 64 == 0 and (J - 1) * hop + N <= ns
        inter = ctx.frames(d_int.ptr, F, N, hop * U, win, dt, J, 1, U)
        plan = ctx.frames(d_plan.ptr, F, N, hop, win, dt, J, ns)
        hinter = ctx.frames(h_int.ptr, F, N, hop * U, win, dt, J, 1, U)
        hplan = ctx.frames(h_dst.ptr, F, N, hop, win, dt, J, ns)
        shapes = dict(ac=(F, 13), tracks=(F, 8), mfcc=(F, 13), cand=(F, 8, 2))
        need = {"lpc12": "ac", "lpc12_formants": "tracks", "mfcc": "mfcc", "pitch": "cand"}[path]
        outs = dict(d={need: ctx.empty(shapes[need], np.float32)}, h={need: pin(shapes[need], np.float32)},
                    est_d=ctx.empty((U, 4, 2), np.float32), est_h=pin((U, 8), np.float32), est0=est0, est0_d=ctx.to_device(est0))
        dev = calls(ctx, rec, None, outs, host=False)[path]
        host = calls(ctx, rec, None, outs, host=True)[path]
        # equality first: the interleaved call returns what the planar call returns
        dev(inter)
        a = outs["d"][need].to_host()
        dev(plan)
        assert np.array_equal(a, outs["d"][need].to_host(), equal_nan=True), (key, path, "device")
        host(hinter)
        b = outs["h"][need].a.copy()
        h_dst.a[...] = h_int.a.T
        host(hplan)
        assert np.array_equal(b, outs["h"][need].a, equal_nan=True) and np.array_equal(a.reshape(b.shape), b, equal_nan=True), \
            (key, path, "host")
        r = {"frame_len": N, "hop": hop, "frames_per_step": F}
        for name, fr in (("interleaved", inter), ("planar", plan)):
            for _ in range(2):
                dev(fr)
            ctx.sync()
            ctx.timer_start()
            for _ in range(steps):
                dev(fr)
            ms = ctx.timer_stop_ms()
            r[f"device_{name}_ms_per_step"] = ms / steps
            r[f"device_{name}_frames_per_s"] = F * steps / (ms * 1e-3)
        r["device_interleaved_vs_planar"] = r["device_interleaved_frames_per_s"] / r["device_planar_frames_per_s"]
        # the gather alone, from the per-kernel profile of the interleaved device call
        ctx.profile_begin()
        for _ in range(steps):
            dev(inter)
        prof = ctx.profile_end()
        g_ms, g_n = prof.get("interleave_gather_kernel", (0.0, 0))
        S = (J - 1) * hop + N
        g_bytes = (U * S + U * (-(-S // 64) * 64)) * es  # interleaved span read + planar rows written
        r["gather_ms_per_call"] = g_ms / max(g_n, 1)
        r["gather_bytes_per_call"] = int(g_bytes)
        r["gather_hbm_gb_per_s"] = g_bytes / (r["gather_ms_per_call"] * 1e-3) / 1e9 if g_n else None
        # end to end: interleaved `_host` vs numpy deinterleave + planar `_host`, pinned buffers both
        for _ in range(1):
            host(hinter)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host(hinter)
        t_int = (time.perf_counter() - t0) / e2e_steps
        t_de, t_tot = 0.0, 0.0
        for _ in range(e2e_steps):
            t0 = time.perf_counter()
            np.copyto(h_dst.a, h_int.a.T)
            t1 = time.perf_counter()
            host(hplan)
            t2 = time.perf_counter()
            t_de += t1 - t0
            t_tot += t2 - t0
        t_de /= e2e_steps
        t_tot /= e2e_steps
        r.update(e2e_interleaved_ms=1e3 * t_int, e2e_interleaved_frames_per_s=F / t_int, e2e_deinterleave_plus_planar_ms=1e3 * t_tot,
                 e2e_deinterleave_plus_planar_frames_per_s=F / t_tot, numpy_deinterleave_ms=1e3 * t_de,
                 e2e_planar_host_call_ms=1e3 * (t_tot - t_de), e2e_interleaved_vs_deinterleave=t_tot / t_int,
                 h2d_bytes_interleaved=int(h_int.nbytes), steps=steps, e2e_steps=e2e_steps)
        out["paths"][path] = r
        print(f"{key:22s} {path:15s} device inter {r['device_interleaved_frames_per_s']:.3e} planar {r['device_planar_frames_per_s']:.3e}"
              f" f/s | gather {r['gather_ms_per_call']:.3f} ms {r['gather_hbm_gb_per_s'] or 0:.0f} GB/s | e2e inter "
              f"{r['e2e_interleaved_ms']:.1f} ms, numpy+planar {r['e2e_deinterleave_plus_planar_ms']:.1f} ms "
              f"(deinterleave {r['numpy_deinterleave_ms']:.1f} ms)", flush=True)
        for k in ("est_d", "est0_d"):
            outs[k].free()
        outs["d"][need].free()
    d_int.free()
    d_plan.free()
    for b in pinned:
        b.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", default=",".join(RECORDINGS))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=None, help="override the recording length (rehearsal)")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    ctx = vb.Context(0)
    result = {"gpu_before": gpu_info(), "sm_count": ctx.sm_count, "recordings": {}}
    for key in args.recordings.split(","):
        rec = dict(RECORDINGS[key])
        if args.seconds:
            rec["seconds"] = args.seconds
        result["recordings"][key] = run(ctx, key, rec, args.steps, args.e2e_steps)
    result["gpu_after"] = gpu_info()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
