"""Input format vs throughput: the C2 (LPC-12), C3 (LPC-12 + formants) and C5 (MFCC) workloads of bench.py, plus LPC-12 and
MFCC on one 8 kHz telephone shape (200 / 80), each fed f32, int16 PCM (VBX_I16) and G.711 mu-law (VBX_MULAW8) samples.

Per format: the device-resident rate (samples already in HBM, device-pointer call) and the end-to-end rate (samples in pinned
host memory, the `_host` call: chunked H2D / kernels / D2H).  The audio is bench.py's seeded synthetic corpus, generated on the
device in each format (vbx_synth_speech: the mu-law corpus is the int16 corpus G.711-encoded).  The card's name, power limit and
clocks are read in the same run.  Writes one JSON file (--out).

    python tools/bench_g711.py --out bench_g711.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload definitions: CONFIGS, n_frames_of, Pinned, MALE, SEED)

sys.path.insert(0, os.path.join(ROOT, "vox_box.rs_b200", "python"))
import voxbox_b200 as vb  # noqa: E402

MFCC_ARGS = {16000: (40, 133.0, 6855.0), 8000: (26, 100.0, 3800.0)}  # (bands, lo, hi); 13 coefficients kept
WORKLOADS = {
    "c2": dict(bench.CONFIGS["c2"]),
    "c3": dict(bench.CONFIGS["c3"], utts=1500),
    "c5": dict(bench.CONFIGS["c5"]),
    "tel_lpc": dict(bench.CONFIGS["c2"], fs=8000, n=200, hop=80, utts=720),
    "tel_mfcc": dict(bench.CONFIGS["c5"], fs=8000, n=200, hop=80, utts=3600),
}
FORMATS = {"f32": (vb.F32, np.float32), "i16": (vb.I16, np.int16), "mulaw8": (vb.MULAW8, np.uint8)}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem,temperature.gpu"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:  # the rates stay valid; say that the card could not be read
        return {"error": repr(e)}


def steps_for(ctx, cfg, fr, outs):
    """(device call, host call) of a workload on one view: same C entry points and arguments as bench.py's Workload."""
    L, h, fs, kind = ctx.lib, ctx.h, float(cfg["fs"]), cfg["kind"]
    if kind == "lpc":
        p = cfg["p"]
        return (lambda f=fr: ctx._check(L.vbx_lpc(h, C.byref(f), p, outs["d0"].ptr, outs["d1"].ptr, None, vb.F32), "vbx_lpc"),
                lambda f: ctx._check(L.vbx_lpc_host(h, C.byref(f), p, outs["h0"].ptr, outs["h1"].ptr, None, vb.F32), "vbx_lpc_host"))
    if kind == "formants":
        p, U = cfg["p"], cfg["utts"]
        est0 = outs["est0"]

        def dev(f=fr):
            ctx._check(L.vbx_memcpy_d2d(h, outs["d1"].ptr, outs["d_est0"].ptr, est0.nbytes), "vbx_memcpy_d2d")
            ctx._check(L.vbx_find_formants(h, C.byref(f), fs, p, vb.LPC_AUTOCORR, outs["d1"].ptr, 4, outs["d0"].ptr, None, None, None,
                                           vb.F32), "vbx_find_formants")

        def host(f):
            outs["h1"].a[...] = est0.reshape(U, 8)
            ctx._check(L.vbx_find_formants_host(h, C.byref(f), fs, p, vb.LPC_AUTOCORR, outs["h1"].ptr, 4, outs["h0"].ptr, None, None,
                                                None, vb.F32), "vbx_find_formants_host")
        return dev, host
    M, lo, hi = MFCC_ARGS[cfg["fs"]]
    return (lambda f=fr: ctx._check(L.vbx_mfcc(h, C.byref(f), M, 13, lo, hi, fs, outs["d0"].ptr, None, vb.F32), "vbx_mfcc"),
            lambda f: ctx._check(L.vbx_mfcc_host(h, C.byref(f), M, 13, lo, hi, fs, outs["h0"].ptr, vb.F32), "vbx_mfcc_host"))


def run(ctx, key, cfg, steps, e2e_steps):
    U, fs, N, hop = cfg["utts"], cfg["fs"], cfg["n"], cfg["hop"]
    ns = int(round(fs * cfg["seconds"]))
    J = bench.n_frames_of(ns, N, hop)
    F = U * J
    kind = cfg["kind"]
    pinned = []

    def pin(shape, dtype):
        b = bench.Pinned(ctx, shape, dtype)
        pinned.append(b)
        return b

    outs = {}
    if kind == "lpc":
        outs.update(d0=ctx.empty((F, 13), np.float32), d1=ctx.empty((F, 13), np.float32), h0=pin((F, 13), np.float32),
                    h1=pin((F, 13), np.float32))
    elif kind == "formants":
        est0 = np.tile(np.array([[f, 1.0] for f in bench.MALE], dtype=np.float32), (U, 1, 1))
        outs.update(est0=est0, d_est0=ctx.to_device(est0), d0=ctx.empty((F, 4, 2), np.float32), d1=ctx.empty((U, 4, 2), np.float32),
                    h0=pin((F, 8), np.float32), h1=pin((U, 8), np.float32))
    else:
        outs.update(d0=ctx.empty((F, 13), np.float32), h0=pin((F, 13), np.float32))
    rec = {"workload": key, "fs": fs, "frame_len": N, "hop": hop, "utterances": U, "seconds_per_utterance": cfg["seconds"],
           "frames_per_step": F, "kind": kind}
    for name, (dt, npt) in FORMATS.items():
        d = ctx.synth_speech(U, ns, fs, bench.SEED, 0, dtype=dt)
        hbuf = pin((U, ns), npt)
        ctx._check(ctx.lib.vbx_memcpy_d2h(ctx.h, hbuf.ptr, d.ptr, hbuf.nbytes), "vbx_memcpy_d2h")
        ctx.sync()
        fr = ctx.frames(d.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, dt, J, ns)
        hfr = ctx.frames(hbuf.ptr, F, N, hop, vb.WINDOW_HANN_SYMMETRIC, dt, J, ns)
        dev, host = steps_for(ctx, cfg, fr, outs)
        for _ in range(3):
            dev()
        ctx.sync()
        ctx.timer_start()
        for _ in range(steps):
            dev()
        ms = ctx.timer_stop_ms()
        for _ in range(2):
            host(hfr)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host(hfr)
        e2e_s = time.perf_counter() - t0
        rec[name] = {"device_resident_frames_per_s": F * steps / (ms * 1e-3), "device_ms_per_step": ms / steps, "steps": steps,
                     "e2e_frames_per_s": F * e2e_steps / e2e_s, "e2e_ms_per_step": 1e3 * e2e_s / e2e_steps, "e2e_steps": e2e_steps,
                     "h2d_bytes_per_step": int(hbuf.nbytes)}
        d.free()
        print(f"{key:9s} {name:7s} device {rec[name]['device_resident_frames_per_s']:.3e} frames/s   "
              f"e2e {rec[name]['e2e_frames_per_s']:.3e} frames/s   ({hbuf.nbytes / 1e6:.0f} MB in)", flush=True)
    for b in pinned:
        b.free()
    for k in ("d0", "d1", "d_est0"):
        if k in outs:
            outs[k].free()
    for name in ("i16", "mulaw8"):
        rec[name]["e2e_vs_f32"] = rec[name]["e2e_frames_per_s"] / rec["f32"]["e2e_frames_per_s"]
    rec["mulaw8"]["e2e_vs_i16"] = rec["mulaw8"]["e2e_frames_per_s"] / rec["i16"]["e2e_frames_per_s"]
    rec["mulaw8"]["device_vs_i16"] = rec["mulaw8"]["device_resident_frames_per_s"] / rec["i16"]["device_resident_frames_per_s"]
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    ctx = vb.Context(0)
    result = {"gpu_before": gpu_info(), "sm_count": ctx.sm_count, "workloads": {}}
    for key in args.workloads.split(","):
        result["workloads"][key] = run(ctx, key, WORKLOADS[key], args.steps, args.e2e_steps)
    result["gpu_after"] = gpu_info()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: {f: round(v[f]["e2e_frames_per_s"]) for f in FORMATS} for k, v in result["workloads"].items()}))


if __name__ == "__main__":
    main()
