#!/usr/bin/env python
"""bench.py — throughput of the vox_box hot path on B200 (BASELINE.json metric: "LPC+formant and pitch frames/sec").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config all|c1|c2|c3|c4|c5] [--utts U]
                    [--dump-outputs DIR]

The headline record (the keys at the top level of the ONE JSON line rank 0 prints) is C3 = BASELINE.json configs[2], the
config the metric is quoted on: LPC-12 + formant extraction (Hann -> autocorrelate(13) -> Levinson -> Laguerre roots ->
resonances -> McCandless tracker) on synthetic 44.1 kHz speech, ONE GPU's share of the 100 h corpus (4500 utterances x
10 s = 4.49 M frames per GPU per step).  With the default --config all the same line carries the other BASELINE configs as
complete sub-records under "configs": c2 (LPC-12 on 1 h of 16 kHz audio), c4 (Boersma pitch 75-600 Hz), c5 (MFCC 13/40)
— each with value, e2e, roofline, kernels, clocks, sustained and (N = 1) cpu_baseline — and c1
(examples/pitch_detection.rs as shipped, CPU-timed).  A "step" is one pass of the hot path over the config's batch.

One process per GPU under torchrun (weak scaling: every rank owns its own batch of distinct utterances; the path shards
by utterance with no data-path collective; torch.distributed/NCCL only carries the barrier and the max-over-ranks of the
timings).  Without torchrun, --gpus N > 1 runs the N devices from ONE process (a thread and a vbx_ctx per device, no torch).
At N > 1, "multi" is the in-library multi-GPU leg: rank 0 drives all N GPUs through vbx_multi_find_formants_host (one
host buffer in, one out; no torch / NCCL on that path).

`value` = device-resident throughput (CUDA events on the library's stream, max over ranks); `e2e` = the same work through
the host-pointer C-ABI call (pinned host buffers; H2D + kernels + D2H inside the timed region); `sustained` = the
device-resident loop run for >= 2 s with clocks and power sampled inside; `roofline` = the dominant kernel against the
pipe that bounds it (FMA peaks measured on this device in this run; executed-work counters for the data-dependent
kernels), `roofline_hbm` against MEASURED_PEAKS.json's copy bandwidth; `cpu_baseline` = the CPU oracle (a C++ port of the
Rust reference — no Rust toolchain in this image) on this box's host cores, single-threaded as shipped and on all threads.
`--impl reference` times that CPU port alone on the same configs.  Audio is synthesised on the device (vbx_synth_speech:
every utterance distinct); the CPU legs of the GPU arm read those very samples back.

--steps K sets the timed steps behind `value` / `ms_per_step` of every config (and C1's repetitions); the sustained leg runs
the same loop for >= 2 s and the end-to-end legs their own small count, each reported next to its value.  The seeded synthesis
gives every run with the same arguments the same inputs, so --dump-outputs DIR (what the last timed step computed, see
dump_outputs) lets two builds be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import re
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "vox_box.rs_b200", "python"))
sys.path.insert(0, ROOT)

MALE = (320., 1440., 2760., 3200.)  # lib.rs:27
SEED = 0x5EED

CONFIGS = {
    "c2": dict(kind="lpc", fs=16000, n=400, hop=160, seconds=10.0, utts=360, p=12,
               metric="LPC-12 frames/sec (autocorrelation + Levinson)", dtype="f64",
               workload="C2: LPC-12 (Hann -> autocorrelate(13) fp64 -> Levinson) on 1 h synthetic 16 kHz audio, "
                        "N=400 hop=160, {utts} utt x {J} frames = {F} frames per GPU"),
    "c3": dict(kind="formants", fs=44100, n=1102, hop=441, seconds=10.0, utts=4500, p=12,
               metric="LPC-12 + formant frames/sec (autocorrelation + Levinson -> Laguerre roots -> McCandless)", dtype="f64",
               workload="C3: formant extraction (Hann -> autocorrelate(13) -> Levinson -> Laguerre roots -> resonances -> "
                        "McCandless tracker) on synthetic 44.1 kHz speech, N=1102 hop=441, {utts} utt x {J} frames = {F} frames "
                        "per GPU per step (4500 utterances = one GPU's share of 100 h over 8 GPUs; every utterance distinct)"),
    "c4": dict(kind="pitch", fs=16000, n=640, hop=160, seconds=10.0, utts=360,
               metric="Boersma pitch frames/sec (75-600 Hz)", dtype="f64",
               workload="C4: Boersma pitch 75-600 Hz (Hann -> all-lag autocorrelation fp64 -> candidates -> Brent/sinc refinement) "
                        "on synthetic 16 kHz audio, N=640 hop=160, {utts} utt x {J} frames = {F} frames per GPU per step "
                        "(1 h of the 1000 h corpus per step; every utterance distinct)"),
    "c5": dict(kind="mfcc", fs=16000, n=400, hop=160, seconds=10.0, utts=3600,
               metric="MFCC frames/sec (13 coefficients from 40 mel bands)", dtype="f64",
               workload="C5: MFCC (Hann -> FFT -> 40 mel bands -> log10 -> DCT, 13 kept) on synthetic 16 kHz audio, N=400 "
                        "hop=160, {utts} utt x {J} frames = {F} frames per GPU per step (every utterance distinct)"),
}
C1 = dict(metric="Boersma pitch frames/sec, examples/pitch_detection.rs as shipped (CPU)",
          workload="C1: examples/pitch_detection.rs as shipped: 150 Hz unit sine, fs 44100, 2049 samples, Windower::hanning(2048, 1024) "
                   "= 1 frame, pitch::<Hanning>(44100, 0.2, ., ., 100, 500); and the same call at fs 11025 over tests/short_sample.wav")
DEFAULT_STEPS = {"lpc": 200, "formants": 20, "pitch": 10, "mfcc": 20}


def n_frames_of(n_samples, frame_len, hop):
    return 0 if n_samples < frame_len else (n_samples - frame_len) // hop + 1


def config_dict(cfg, U, world):
    """`config` of a record: identical for the GPU arm and the reference arm of the same workload."""
    ns = int(round(cfg["fs"] * cfg["seconds"]))
    J = n_frames_of(ns, cfg["n"], cfg["hop"])
    in_mb = U * ns * 4 / 1e6
    outputs = {"lpc": "r[13], ac[13] fp32", "formants": "4 formant (frequency, bandwidth) tracks per frame, fp32",
               "pitch": "up to 16 (frequency, strength) candidates per frame fp32 + count + status",
               "mfcc": "13 MFCC per frame fp32"}[cfg["kind"]]
    return {"workload": cfg["workload"].format(utts=U, J=J, F=U * J), "frames_per_gpu": U * J, "window": "hann_symmetric",
            "outputs": outputs,
            "l2": f"inputs larger than L2 ({in_mb:.0f} MB audio per step), no flush" if in_mb > 130 else
                  f"inputs ({in_mb:.0f} MB) fit L2: compute-bound kernels, no flush",
            "parallelism": f"utterance-sharded x{world}, no collective"}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def _ncu_traffic(profile_name):
    """dram read+write bytes per launch from a committed `ncu --set full` summary under profiles/ (or None)."""
    try:
        txt = open(os.path.join(ROOT, "profiles", profile_name)).read()
        tot = 0.0
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            m = re.search(key + r" = ([0-9.]+) (\w+)", txt)
            tot += float(m.group(1)) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[m.group(2)]
        return tot
    except Exception:
        return None


_NCU_KEYS = {"smsp__issue_active.avg.pct_of_peak_sustained_active": "issue_slots_pct",
             "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active": "pipe_fp64_pct",
             "sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active": "pipe_fma_pct",
             "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active": "pipe_lsu_pct",
             "sm__warps_active.avg.pct_of_peak_sustained_active": "warps_active_pct",
             "launch__registers_per_thread": "registers",
             "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum": "smem_wavefronts",
             "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum": "smem_bank_conflict_wavefronts",
             "gpu__time_duration.sum": "duration"}


def _ncu_counters(profile_name):
    """Key counters of a committed `ncu --set full` summary under profiles/ (tools/ncu_summary.sh): what the kernel's pipes
    did in that capture — the cross-check of the fractions this run computes from its own timings (or None)."""
    try:
        out = {"profile": "profiles/" + profile_name}
        for line in open(os.path.join(ROOT, "profiles", profile_name)):
            m = re.match(r"([\w.]+) = ([0-9.]+) ?(\S*)", line)
            if m and m.group(1) in _NCU_KEYS:
                v = float(m.group(2))
                out[_NCU_KEYS[m.group(1)]] = (v, m.group(3)) if m.group(1) == "gpu__time_duration.sum" else v
        return out if len(out) > 1 else None
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock, power and throttle reasons of one GPU while the timed regions run (NVML; falls back to the
    nvidia-smi query line of /opt/skills/guides/B200_PROFILING.md).  Samples are time-stamped so that a leg can be
    summarised on its own (`window`)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        self.index, self.samples, self.max_mhz = index, [], None  # samples: (t, mhz, watts, reason mask)
        self._stop = threading.Event()
        self._t = None
        self.how = None

    def _run_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        self.how = "nvml"
        reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                w = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
            except Exception:
                w = None
            self.samples.append((time.perf_counter(), pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), w, int(reasons(h))))
            time.sleep(0.002)

    def _run_smi(self):
        import subprocess
        self.how = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        bits = [0x8, 0x40, 0x20, 0x4]
        p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                              "-lms", "100"], stdout=subprocess.PIPE, text=True)
        try:
            while not self._stop.is_set():
                line = p.stdout.readline()
                if not line:
                    break
                f = [x.strip() for x in line.split(",")]
                self.max_mhz = int(f[1])
                mask = sum(b for b, v in zip(bits, f[3:]) if v.lower().startswith("active"))
                try:
                    w = float(f[2])
                except ValueError:
                    w = None
                self.samples.append((time.perf_counter(), int(f[0]), w, mask))
        finally:
            p.terminate()

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            try:
                self._run_smi()
            except Exception:
                self.how = "unavailable"

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=5)

    def summary(self, t0=None, t1=None):
        rows = [r for r in self.samples if (t0 is None or r[0] >= t0) and (t1 is None or r[0] <= t1)]
        s = sorted(r[1] for r in rows)
        # "under load": drop samples below half the maximum seen (idle gaps between regions)
        hot = [x for x in s if x >= 0.5 * s[-1]] if s else []
        mask = 0
        for r in rows:
            mask |= r[3]
        watts = [r[2] for r in rows if r[2] is not None]
        return {"sm_mhz": hot[len(hot) // 2] if hot else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if mask & b), "samples": len(s), "how": self.how,
                "power_w_max": max(watts) if watts else None, "power_w_mean": sum(watts) / len(watts) if watts else None}


# ------------------------------------------------------------------------------------------------
# ranks: torchrun processes (NCCL barrier / max), threads of one process, or a single rank
# ------------------------------------------------------------------------------------------------
class NullComm:
    rank, world = 0, 1

    def barrier(self):
        pass

    def max(self, x):
        return x

    def close(self):
        pass


class TorchComm:
    """One process per GPU (torchrun): torch.distributed over NCCL for the barrier and the max-over-ranks only."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        self.rank, self.world, self.torch, self.dist = rank, world, torch, dist
        torch.cuda.set_device(local_rank)
        # NCCL may print its version banner on stdout while the communicator is created: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            t = torch.zeros(1, device="cuda")
            dist.all_reduce(t)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier(self):
        self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        self.dist.destroy_process_group()


class ThreadComm:
    """N devices driven from one process: a thread (and a vbx_ctx) per device, no torch."""

    class _Shared:
        def __init__(self, world):
            self.bar = threading.Barrier(world)
            self.vals = [0.0] * world

    def __init__(self, shared, rank, world):
        self.s, self.rank, self.world = shared, rank, world

    def barrier(self):
        self.s.bar.wait()

    def max(self, x):
        self.s.vals[self.rank] = x
        self.s.bar.wait()
        m = max(self.s.vals)
        self.s.bar.wait()
        return m

    def close(self):
        pass


def numa_bind(gpu_index):
    """Bind the calling thread to the CPUs NVML reports as local to the GPU; returns the previous mask (or None)."""
    try:
        import pynvml
        before = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_words = (os.cpu_count() + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= before
        if cpus and cpus != before:
            os.sched_setaffinity(0, cpus)
            return before
    except Exception:
        pass
    return None


def host_threads():
    """Host threads for the CPU arm: every core this process may run on (torchrun exports OMP_NUM_THREADS=1, which
    would silently make the "all host threads" baseline single-threaded, so the count is passed explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------------
# CPU port (oracle) of each config: used by --impl reference and by the cpu_baseline leg
# ------------------------------------------------------------------------------------------------
CPU_FRAMES_PER_THREAD_S = {"lpc": 3.0e5, "formants": 2.2e4, "pitch": 280.0, "mfcc": 1.6e4}  # rough, only sizes the samples


def cpu_pass(cfg, audio_rows, J, n_threads):
    """One pass of the reference's per-frame loop over the given utterances on the CPU oracle (n_threads: 1 = as
    shipped, >1 = OpenMP over frames / utterances: the rayon-wrapper stand-in)."""
    import oracle
    N, hop, fs = cfg["n"], cfg["hop"], float(cfg["fs"])
    kind = cfg["kind"]
    for row in audio_rows:
        if kind == "lpc":
            oracle.batch_lpc(row, J, N, hop, oracle.WIN_HANN_SYMMETRIC, cfg["p"], n_threads=n_threads)
        elif kind == "pitch":
            oracle.batch_pitch(row, J, N, hop, oracle.WIN_HANN_SYMMETRIC, fs, 0.45, 75.0, 600.0, 16, n_threads=n_threads)
        elif kind == "mfcc":
            oracle.batch_mfcc(row, J, N, hop, oracle.WIN_HANN_SYMMETRIC, 40, 133.0, 6855.0, fs, n_keep=13, n_threads=n_threads)
    if kind == "formants":
        # utterances in parallel (the tracker is sequential inside an utterance); frame f of the flattened batch
        # starts at f*hop, so utterance u owns frames [u*ns/hop, u*ns/hop + J) when hop divides the utterance length
        rows = np.ascontiguousarray(np.stack(audio_rows))
        U, ns = rows.shape
        est = np.array([[f, 1.0] for f in MALE])
        if ns % hop == 0:
            starts = np.arange(U, dtype=np.int64) * (ns // hop)
            offs = np.stack([starts, starts + J], axis=1).reshape(-1)
            oracle.batch_formants(rows.reshape(-1), int(offs[-1]), N, hop, oracle.WIN_HANN_SYMMETRIC, 1, fs, cfg["p"], offs, est,
                                  n_threads=n_threads)
        else:
            for u in range(U):
                oracle.batch_formants(rows[u], J, N, hop, oracle.WIN_HANN_SYMMETRIC, 1, fs, cfg["p"],
                                      np.array([0, J], dtype=np.int64), est, n_threads=n_threads)


def cpu_sample_utts(cfg, J, threads, seconds):
    """Utterances whose pass costs about `seconds` of wall time on `threads` threads."""
    frames = seconds * threads * CPU_FRAMES_PER_THREAD_S[cfg["kind"]]
    lo = threads if cfg["kind"] == "formants" else 1  # the formant loop parallelises over utterances
    return int(max(lo, min(cfg["utts"], round(frames / J))))


def host_corpus(cfg, n_utts, first=0):
    """Host-synthesised utterances (numpy/scipy recipe of voxbox_b200.synth) for the reference arm, which must not touch
    the GPU: a bounded number of distinct utterances, tiled."""
    from voxbox_b200 import synth
    distinct = min(n_utts, 48 if cfg["fs"] <= 16000 else 24)
    base = synth.corpus(distinct, cfg["fs"], cfg["seconds"], first=first)
    reps = -(-n_utts // distinct)
    return np.ascontiguousarray(np.tile(base, (reps, 1))[:n_utts]), distinct


def c1_record(args, reps=None):
    """BASELINE configs[0]: examples/pitch_detection.rs as shipped, timed on the CPU oracle (one thread, as shipped)."""
    import oracle
    reps = reps or (args.steps if args.steps is not None else 20)
    out = {"metric": C1["metric"], "unit": "frames/s", "higher_is_better": True, "dtype": "f64", "data": "synthetic sine + tests/fixtures/short_sample.wav",
           "config": {"workload": C1["workload"]}, "impl_note": "CPU oracle (C++ f64 port of the Rust reference), 1 thread, as shipped"}
    cases = {}
    # (i) exactly the example (examples/pitch_detection.rs:15-33,47-49; expected 150 +- 0.01 Hz, periodic.rs:497)
    fs = 44100.0
    x = oracle.sine_signal(fs, 150.0, 2049)[:2048] * oracle.hanning_window(2048)
    for _ in range(2):
        oracle.pitch(x, fs, 0.2, 100.0, 500.0)
    t0 = time.perf_counter()
    for _ in range(reps):
        _, cand, _ = oracle.pitch(x, fs, 0.2, 100.0, 500.0)
    dt = (time.perf_counter() - t0) / reps
    cases["sine_150hz_44100"] = {"frames_per_s": 1.0 / dt, "ms_per_frame": 1e3 * dt, "top_candidate_hz": float(cand[0][0]),
                                 "top_candidate_strength": float(cand[0][1]), "expected_hz": "150 +- 0.01 (periodic.rs:497)",
                                 "ok": bool(abs(cand[0][0] - 150.0) < 0.01)}
    # (ii) BASELINE's wording "on tests/short_sample.wav": the same call at fs 11025 over the fixture (1 frame of 2048)
    wav = os.path.join(ROOT, "tests", "fixtures", "short_sample.wav")
    if os.path.exists(wav):
        y, fs2 = oracle.read_wav(wav)
        xw = np.asarray(y[:2048], dtype=np.float64) * oracle.hanning_window(2048)
        oracle.pitch(xw, float(fs2), 0.2, 100.0, 500.0)
        t0 = time.perf_counter()
        for _ in range(reps):
            _, cand2, _ = oracle.pitch(xw, float(fs2), 0.2, 100.0, 500.0)
        dt2 = (time.perf_counter() - t0) / reps
        cases["short_sample_wav_11025"] = {"frames_per_s": 1.0 / dt2, "ms_per_frame": 1e3 * dt2, "top_candidate_hz": float(cand2[0][0]),
                                           "top_candidate_strength": float(cand2[0][1]),
                                           "expected_hz": "100.22727800116024 (SURVEY 8d restatement)"}
    out["cases"] = cases
    out["value"] = cases["sine_150hz_44100"]["frames_per_s"]
    out["ms_per_step"] = cases["sine_150hz_44100"]["ms_per_frame"]
    out["steps"] = reps
    out["cpu_baseline"] = {"value": out["value"], "unit": "frames/s", "cores": 1, "kind": "port",
                           "sample": f"{reps} repetitions of the example's single 2048-sample frame"}
    return out


def reference_record(args, key, cfg, world):
    """CPU arm of one config: the oracle port of the reference's per-frame loop, frame-parallel over all host threads (the
    "rayon wrapper" stand-in); every step is a bounded sample of the config's workload."""
    import oracle
    threads = host_threads()
    ns = int(round(cfg["fs"] * cfg["seconds"]))
    J = n_frames_of(ns, cfg["n"], cfg["hop"])
    n_s = cpu_sample_utts(cfg, J, threads, 0.5)
    audio, distinct = host_corpus(cfg, n_s)
    rows = list(audio)
    for _ in range(args.warmup):
        cpu_pass(cfg, rows, J, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_pass(cfg, rows, J, threads)
    dt = time.perf_counter() - t0
    value = len(rows) * J * args.steps / dt
    # single thread, as shipped
    n1 = max(1, cpu_sample_utts(cfg, J, 1, 1.0))
    t0 = time.perf_counter()
    cpu_pass(cfg, rows[:n1], J, 1)
    t1 = time.perf_counter() - t0
    sample = (f"C++ f64 port of the Rust reference (no cargo in this image): each step = {len(rows)} of the config's {cfg['utts']} "
              f"utterances ({distinct} distinct, host-synthesised) x {J} frames, {args.steps} steps, OpenMP over frames on {threads} threads; "
              f"single thread as shipped: {min(n1, len(rows))} utterances")
    return {"impl": "reference", "metric": cfg["metric"], "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(cfg, cfg["utts"], world),
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port",
                             "single_thread_value": min(n1, len(rows)) * J / t1, "sample": sample},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def run_reference(args, keys, rank, world):
    if rank != 0:
        return
    head = keys[0]
    line = reference_record(args, head, CONFIGS[head], world)
    subs = {}
    for k in keys[1:]:
        subs[k] = reference_record(args, k, CONFIGS[k], world)
    if args.config == "all":
        c1 = c1_record(args)
        c1["impl"] = "reference"
        subs["c1"] = c1
    if subs:
        line["configs"] = subs
    print(json.dumps(line), flush=True)


def cpu_baseline(cfg, rows, J):
    """Bounded CPU sample on rank 0 (N=1 only): oracle port, single thread as shipped + all threads, on the very samples the
    GPU processed (copied device -> host)."""
    threads = host_threads()
    n_all = min(cpu_sample_utts(cfg, J, threads, 0.6), len(rows))
    n_one = max(1, min(n_all, cpu_sample_utts(cfg, J, 1, 1.0)))
    rows = [np.array(r, dtype=np.float32) for r in rows[:n_all]]  # off the pinned buffer
    t0 = time.perf_counter()
    cpu_pass(cfg, rows[:n_one], J, 1)
    t1 = time.perf_counter() - t0
    reps = 0
    t0 = time.perf_counter()
    while True:
        cpu_pass(cfg, rows, J, threads)
        reps += 1
        if time.perf_counter() - t0 > 3.0 or reps >= 50:
            break
    tn = time.perf_counter() - t0
    return {"value": n_all * J * reps / tn, "unit": "frames/s", "cores": threads, "kind": "port",
            "single_thread_value": n_one * J / t1,
            "sample": f"C++ f64 port of the Rust reference (no cargo here): {n_all} of this run's utterances x {J} frames x {reps} "
                      f"passes on {threads} OpenMP threads; single thread as shipped: {n_one} utterances"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Pinned:
    """Pinned host buffer (vbx_malloc_host) viewed as a numpy array."""

    def __init__(self, ctx, shape, dtype):
        self.ctx, self.shape, self.dtype = ctx, tuple(shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        self.p = C.c_void_p()
        ctx._check(ctx.lib.vbx_malloc_host(ctx.h, max(self.nbytes, 1), C.byref(self.p)), "vbx_malloc_host")
        ct = {np.dtype(np.float32): C.c_float, np.dtype(np.int16): C.c_int16, np.dtype(np.int32): C.c_int32,
              np.dtype(np.uint8): C.c_uint8}[self.dtype]
        self.a = np.ctypeslib.as_array(C.cast(self.p, C.POINTER(ct)), shape=self.shape)

    @property
    def ptr(self):
        return self.p.value

    def free(self):
        if self.p:
            self.a = None
            self.ctx.lib.vbx_free_host(self.ctx.h, self.p)
            self.p = None


class Workload:
    """Device buffers + the device-pointer step and the host-pointer (e2e) step of one config.  The audio is synthesised
    on the device (utterances first_utt … first_utt + U − 1 of the seeded corpus) and copied to pinned host memory for the
    end-to-end legs."""

    def __init__(self, ctx, vb, cfg, first_utt, want_host=True):
        self.ctx, self.vb, self.cfg = ctx, vb, cfg
        L, h = ctx.lib, ctx.h
        U, fs = cfg["utts"], cfg["fs"]
        ns = int(round(fs * cfg["seconds"]))
        N, hop = cfg["n"], cfg["hop"]
        J = n_frames_of(ns, N, hop)
        F = U * J
        self.U, self.J, self.F, self.ns = U, J, F, ns
        self._pinned = []
        self.d_audio = ctx.synth_speech(U, ns, fs, SEED, first_utt)
        win = vb.WINDOW_HANN_SYMMETRIC
        fr = ctx.frames(self.d_audio.ptr, F, N, hop, win, frames_per_segment=J, segment_stride=ns)
        kind = cfg["kind"]

        def pinned(shape, dtype):
            b = Pinned(ctx, shape, dtype)
            self._pinned.append(b)
            return b

        hfr = hfr16 = None
        self.h_audio = None
        if want_host:
            self.h_audio = pinned((U, ns), np.float32)
            ctx._check(L.vbx_memcpy_d2h(h, self.h_audio.ptr, self.d_audio.ptr, self.h_audio.nbytes), "vbx_memcpy_d2h")
            # the same utterances as 16-bit PCM (the format the reference's WAV drivers read, tests/lib.rs:15-19)
            d16 = ctx.synth_speech(U, ns, fs, SEED, first_utt, dtype=vb.I16)
            h16 = pinned((U, ns), np.int16)
            ctx._check(L.vbx_memcpy_d2h(h, h16.ptr, d16.ptr, h16.nbytes), "vbx_memcpy_d2h")
            ctx.sync()
            d16.free()
            hfr = ctx.frames(self.h_audio.ptr, F, N, hop, win, frames_per_segment=J, segment_stride=ns)
            hfr16 = ctx.frames(h16.ptr, F, N, hop, win, dtype=vb.I16, frames_per_segment=J, segment_stride=ns)
            self.h2d, self.h2d16 = self.h_audio.nbytes, h16.nbytes
        self.hfr16 = hfr16
        fsd = float(fs)

        if kind == "lpc":
            p = cfg["p"]
            d_r, d_ac = ctx.empty((F, p + 1), np.float32), ctx.empty((F, p + 1), np.float32)
            self.step = lambda: ctx._check(L.vbx_lpc(h, C.byref(fr), p, d_r.ptr, d_ac.ptr, None, vb.F32), "vbx_lpc")
            self.outputs = lambda: {"r": d_r.to_host(), "lpc": d_ac.to_host()}
            self._keep = (d_r, d_ac)
            if want_host:
                h_r, h_ac = pinned((F, p + 1), np.float32), pinned((F, p + 1), np.float32)
                self.e2e_step = lambda fr_=hfr: ctx._check(L.vbx_lpc_host(h, C.byref(fr_), p, h_r.ptr, h_ac.ptr, None, vb.F32), "vbx_lpc_host")
                self.d2h = h_r.nbytes + h_ac.nbytes
                self.api = "vbx_lpc_host (pinned host buffers)"
                self.check = lambda: float(np.sum(h_r.a[::max(1, F // 1000), 0], dtype=np.float64))
        elif kind == "formants":
            p = cfg["p"]
            est0 = np.tile(np.array([[f, 1.0] for f in MALE], dtype=np.float32), (U, 1, 1))
            d_est0 = ctx.to_device(est0)
            d_est = ctx.empty((U, 4, 2), np.float32)
            d_trk = ctx.empty((F, 4, 2), np.float32)

            def step():
                # the tracker state is in/out: every step starts from the MALE estimates (tests/lib.rs:36,60)
                ctx._check(L.vbx_memcpy_d2d(h, d_est.ptr, d_est0.ptr, est0.nbytes), "vbx_memcpy_d2d")
                ctx._check(L.vbx_find_formants(h, C.byref(fr), fsd, p, vb.LPC_AUTOCORR, d_est.ptr, 4, d_trk.ptr, None, None, None,
                                               vb.F32), "vbx_find_formants")

            self.step = step
            self.outputs = lambda: {"tracks": d_trk.to_host(), "estimates": d_est.to_host()}
            self._keep = (d_est0, d_est, d_trk, est0)
            if want_host:
                h_trk, h_est = pinned((F, 8), np.float32), pinned((U, 8), np.float32)

                def e2e_step(fr_=hfr):
                    h_est.a[...] = est0.reshape(U, 8)
                    ctx._check(L.vbx_find_formants_host(h, C.byref(fr_), fsd, p, vb.LPC_AUTOCORR, h_est.ptr, 4, h_trk.ptr, None, None, None,
                                                        vb.F32), "vbx_find_formants_host")

                self.e2e_step = e2e_step
                self.h2d += int(est0.nbytes)
                self.h2d16 += int(est0.nbytes)
                self.d2h = h_trk.nbytes + int(est0.nbytes)
                self.api = "vbx_find_formants_host (pinned host buffers)"
                self.check = lambda: float(np.sum(h_trk.a[::max(1, F // 1000)], dtype=np.float64))
        elif kind == "pitch":
            K = 16
            d_c, d_n, d_s = ctx.empty((F, K, 2), np.float32), ctx.empty((F,), np.int32), ctx.empty((F,), np.uint8)
            self.step = lambda: ctx._check(L.vbx_pitch(h, C.byref(fr), fsd, 0.45, 75.0, 600.0, K, d_c.ptr, d_n.ptr, d_s.ptr, vb.F32), "vbx_pitch")
            self.outputs = lambda: {"candidates": d_c.to_host(), "n_cand": d_n.to_host(), "status": d_s.to_host()}
            self._keep = (d_c, d_n, d_s)
            if want_host:
                h_c, h_n, h_s = pinned((F, K * 2), np.float32), pinned((F,), np.int32), pinned((F,), np.uint8)
                self.e2e_step = lambda fr_=hfr: ctx._check(L.vbx_pitch_host(h, C.byref(fr_), fsd, 0.45, 75.0, 600.0, K, h_c.ptr, h_n.ptr, h_s.ptr, vb.F32), "vbx_pitch_host")
                self.d2h = h_c.nbytes + h_n.nbytes + h_s.nbytes
                self.api = "vbx_pitch_host (pinned host buffers)"
                self.check = lambda: float(np.sum(h_c.a[::max(1, F // 1000), 0], dtype=np.float64))
        elif kind == "mfcc":
            d_o = ctx.empty((F, 13), np.float32)
            self.step = lambda: ctx._check(L.vbx_mfcc(h, C.byref(fr), 40, 13, 133.0, 6855.0, fsd, d_o.ptr, None, vb.F32), "vbx_mfcc")
            self.outputs = lambda: {"mfcc": d_o.to_host()}
            self._keep = (d_o,)
            if want_host:
                h_o = pinned((F, 13), np.float32)
                self.e2e_step = lambda fr_=hfr: ctx._check(L.vbx_mfcc_host(h, C.byref(fr_), 40, 13, 133.0, 6855.0, fsd, h_o.ptr, vb.F32), "vbx_mfcc_host")
                self.d2h = h_o.nbytes
                self.api = "vbx_mfcc_host (pinned host buffers)"
                self.check = lambda: float(np.sum(h_o.a[::max(1, F // 1000), 0], dtype=np.float64))

    def free(self):
        self.step = self.e2e_step = self.check = self.outputs = None
        for b in self._pinned:
            b.free()
        for d in (self.d_audio,) + tuple(x for x in self._keep if hasattr(x, "free")):
            d.free()

    def kernel_table(self, counters, steps):
        """Work per frame of every kernel of the step: name -> (pipe that bounds it, flop per frame, HBM bytes per frame,
        committed ncu summary or None, how the flop figure was obtained).  Deterministic kernels carry SURVEY §8d's
        algorithmic figure (which is what they execute); the data-dependent ones (Laguerre roots, Brent refinement) carry
        the work they EXECUTED in this run's timed region, from the library's in-kernel counters."""
        cfg, N, hop, F = self.cfg, self.cfg["n"], self.cfg["hop"], self.F
        p = cfg.get("p", 12)
        alg = "algorithmic (SURVEY 8d) = executed: the kernel's work does not depend on the data"
        lpc_flop = 2 * (p + 1) * N + N + 350
        # one Horner coefficient step = 3 complex FMA (P, P', P''/2) = 12 FFMA = 24 flop; one Laguerre round ~ 60 flop
        roots_flop = (24.0 * counters["roots_horner_steps"] + 60.0 * counters["roots_rounds"]) / max(1, steps * F)
        # one term-loop iteration ~ 22 fp64 flop per lane (2 products, shared reciprocal = 3 DFMA, 2 Hann recurrences,
        # accumulate); one evaluation ~ 300 fp64 flop of setup per lane (3 sincospi, 2 reciprocals, Brent update)
        refine_flop = (22.0 * counters["refine_terms"] + 300.0 * counters["refine_evals"]) / max(1, steps * F)
        cnt = "executed: in-kernel counters of this run (vbx_profile_counters), lane-summed incl. idle lanes; fp32 Horner + Laguerre only"
        cnt_r = "executed: in-kernel counters of this run (vbx_profile_counters), lane-summed; 22 flop per term iteration + 300 per evaluation (instruction-count estimate)"
        return {
            "lpc": {"lpc_fused16_kernel": ("fp64", lpc_flop, 4 * hop + 2 * 4 * (p + 1), "r1_lpc16_final_full.txt", alg),
                    "lpc_fused_kernel": ("fp64", lpc_flop, 4 * hop + 2 * 4 * (p + 1), "r1_lpc_final_full.txt", alg),
                    "lpc_fuseda_kernel": ("fp64", lpc_flop, 4 * hop + 2 * 4 * (p + 1), None, alg),
                    "lpc_fusedp_kernel": ("fp64", lpc_flop, 4 * hop + 2 * 4 * (p + 1), "r2_lpcp_v1_full.txt", alg)},
            "formants": {
                "lpc_fused_kernel": ("fp64", lpc_flop, 4 * hop + 8 * (p + 1), "r1_lpc_final_full.txt", alg),
                "lpc_fuseda_kernel": ("fp64", lpc_flop, 4 * hop + 8 * (p + 1), "r2_lpca_v1_full.txt", alg),
                "lpc_fusedp_kernel": ("fp64", lpc_flop, 4 * hop + 8 * (p + 1), "r2_lpcp_v1_full.txt", alg),
                "lpc_fused16_kernel": ("fp64", lpc_flop, 4 * hop + 8 * (p + 1), "r1_lpc16_final_full.txt", alg),
                "lpc_roots_pair_kernel": ("fp32", roots_flop, 8 * (p + 1) + 8 * p + 5, "r2_roots_v2_full.txt", cnt),
                "lpc_roots_rt_kernel": ("fp32", roots_flop, 8 * (p + 1) + 8 * p + 5, None, cnt),
                # latency-bound by construction (998 sequential steps per utterance): no pipe fraction is meaningful
                "tracker_idx_kernel": (None, None, 8 * p + 4 + 4 * 8, "r1_tracker_final_full.txt", "latency-bound: sequential over the frames of an utterance"),
            },
            "pitch": {
                "pitch_lag64_kernel": ("fp64", 2.0 * N * (N + 1) / 2, 4 * hop + 8 * N, "r2_lag64_v2_full.txt", alg),
                "pitch_lag_kernel": ("fp32", 2.0 * N * (N + 1) / 2, 4 * hop + 8 * N, "r1_lag_final_full.txt", alg),
                "pitch_refine8q_kernel": ("fp64", refine_flop, 8 * N, "r2_refine2_v1_full.txt", cnt_r),
                "pitch_finalize_kernel": (None, None, 16 * 16 + 140, None, "small"),
            },
            # mfcc_lane5_kernel: the fp64 instructions it EXECUTES (ncu source counters of profiles/r2_mfcc_lane5_v5_full.txt: 390
            # warp-wide DFMA / DADD / DMUL per frame, the same for every frame), each charged as one FMA issue slot of 32 lanes —
            # i.e. the fraction is the fp64 pipe's utilisation; the kernel's other limit is the shared-memory data path (DESIGN K8)
            "mfcc": {"mfcc_lane5_kernel": ("fp64", 390.0 * 64, 4 * hop + 4 * 13, "r2_mfcc_lane5_v5_full.txt",
                                           "executed: 390 fp64 warp instructions per frame (ncu), each an FMA issue slot"),
                     "mfcc_warp_kernel": ("fp64", 19.5e3, 4 * hop + 4 * 13, "r1_mfcc_final_full.txt", alg),
                     "mfcc_kernel": ("fp64", 19.5e3, 4 * hop + 4 * 13, None, alg)},
        }[cfg["kind"]]

    def roofline(self, prof, counters, steps, peaks, hbm_peak, hbm_src):
        """Per-kernel roofline from the per-kernel device times measured over the timed region (vbx_profile_*):
        achieved = flop (or bytes) per launch / average launch duration.  Returns (dominant kernel's roofline object, its
        HBM view, the per-kernel table)."""
        table = self.kernel_table(counters, steps)
        total_ms = sum(ms for ms, _ in prof.values()) or 1e-9
        kernels = {}
        for name, (ms, n) in sorted(prof.items(), key=lambda kv: -kv[1][0]):
            entry = {"ms_per_step": ms / steps, "launches_per_step": n / steps, "share": ms / total_ms}
            if name in table:
                pipe, flop, byts, prof_file, how = table[name]
                if prof_file:
                    entry["ncu"] = _ncu_counters(prof_file)
                sec = ms * 1e-3 / steps
                entry.update({"gbs": byts * self.F / sec / 1e9, "frac_hbm": byts * self.F / sec / 1e9 / hbm_peak, "work": how})
                if pipe:
                    entry.update({"bound": pipe, "flop_per_frame": flop, "tflops": flop * self.F / sec / 1e12,
                                  "frac": flop * self.F / sec / 1e12 / peaks[pipe + "_tflops"]})
                else:
                    entry.update({"bound": "latency", "frac": None})
            kernels[name] = entry
        dom = next((k for k in kernels if k in table and table[k][0]), None)
        if dom is None:
            return None, None, kernels
        pipe, flop, byts, profile, how = table[dom]
        k = kernels[dom]
        launches = max(1.0, k["launches_per_step"])
        roof = {"bound": pipe, "achieved": k["tflops"], "peak": peaks[pipe + "_tflops"], "unit": "TFLOP/s", "frac": k["frac"],
                "traffic": _ncu_traffic(profile) if profile else None,
                "traffic_note": f"dram read+write of one ncu --set full capture (profiles/{profile}); that capture's batch may be smaller "
                                "than this run's — compare per frame" if profile else None,
                "kernel": dom, "flop_per_frame": flop, "work": how,
                "flop_per_launch": flop * self.F / launches, "avg_launch_ms": k["ms_per_step"] / launches, "share_of_step": k["share"],
                "peak_source": "vbx_measure_peaks: dependent-free FMA loop on this device, this run",
                "timing": "CUDA events on the library's stream around every launch of the timed region (vbx_profile_begin/end)"}
        roof_hbm = {"bound": "hbm", "achieved": k["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": k["frac_hbm"],
                    "bytes_per_frame": byts, "kernel": dom, "peak_source": hbm_src}
        return roof, roof_hbm, kernels


DUMP_ROWS = 1 << 16  # rows kept per array by --dump-outputs: every config together stays below 64 MB


def dump_outputs(out_dir, key, arrays):
    """--dump-outputs: writes each output of the last timed step as out_dir/<config>_<name>.npy in float32 (float64 stays
    float64).  An array with more than DUMP_ROWS rows (frames or utterances) keeps a fixed, seeded sample of its rows in
    ascending order, and out_dir/<config>_<name>_rows.npy lists their indices, so that runs of two builds on the same
    arguments compare output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.shape[0] > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(SEED).choice(a.shape[0], DUMP_ROWS, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, f"{key}_{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{key}_{name}.npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def gpu_record(ctx, vb, key, cfg, args, comm, clocks, peaks):
    """All legs of one config on this rank's GPU; returns the record on rank 0 (None elsewhere)."""
    rank, world = comm.rank, comm.world
    steps = args.steps if args.steps is not None else DEFAULT_STEPS[cfg["kind"]]
    warmup = max(args.warmup, 3)
    wl = Workload(ctx, vb, cfg, first_utt=rank * cfg["utts"], want_host=not args.device_only)
    F = wl.F
    ctx.sync()
    # ---- device-resident throughput -------------------------------------------------------
    for _ in range(warmup):
        wl.step()
    ctx.sync()
    comm.barrier()
    t_a = time.perf_counter()
    l0 = ctx.kernel_launches
    ctx.profile_begin()  # an event after every launch: per-kernel device times for the roofline
    ctx.timer_start()
    for _ in range(steps):
        wl.step()
    ms = ctx.timer_stop_ms()
    prof = ctx.profile_end()
    counters = ctx.profile_counters()
    launches = ctx.kernel_launches - l0
    t_b = time.perf_counter()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, key, wl.outputs())
    comm.barrier()
    ms = comm.max(ms)
    rec = None
    if args.device_only:
        if rank == 0:
            mp = _peaks()
            _, _, kernels = wl.roofline(prof, counters, steps, peaks, mp["hbm_gbs"] if mp else 6650.0, "")
            rec = {"device_only": True, "config": key, "value": F * world * steps / (ms * 1e-3), "unit": "frames/s",
                   "ms_per_step": ms / steps, "gpu_launches": launches, "kernel_share": {k: v["share"] for k, v in kernels.items()}}
        wl.free()
        return rec
    # ---- sustained: the same loop for >= 2 s, clocks and power sampled inside ---------------------------------
    sus_steps = int(min(max(steps, np.ceil(2000.0 * steps / max(ms, 1e-3))), 200000))
    comm.barrier()
    t_s0 = time.perf_counter()
    ctx.timer_start()
    for _ in range(sus_steps):
        wl.step()
    sus_ms = comm.max(ctx.timer_stop_ms())
    t_s1 = time.perf_counter()
    comm.barrier()
    # ---- end to end through the host-pointer C-ABI call ------------------------------------------
    e2e_steps = max(3, min(steps, 20 if wl.h2d < (1 << 30) else 5))
    for _ in range(3 if wl.h2d < (1 << 30) else 2):
        wl.e2e_step()
    comm.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        wl.e2e_step()
    e2e_s = comm.max(time.perf_counter() - t0)
    comm.barrier()
    checksum = wl.check()
    # the same call fed with 16-bit PCM host samples (scaled by 1/32767 on load)
    for _ in range(2):
        wl.e2e_step(wl.hfr16)
    comm.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        wl.e2e_step(wl.hfr16)
    e2e16_s = comm.max(time.perf_counter() - t0)
    comm.barrier()
    if rank == 0:
        total_frames = F * world
        mp = _peaks()
        hbm_peak = mp["hbm_gbs"] if mp else 6650.0
        hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if mp else "fallback 6650 GB/s (of fallback)"
        roof, roof_hbm, kernels = wl.roofline(prof, counters, steps, peaks, hbm_peak, hbm_src)
        rec = {
            "metric": cfg["metric"], "value": total_frames * steps / (ms * 1e-3), "unit": "frames/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
            "config": config_dict(cfg, wl.U, world),
            "e2e": {"value": total_frames * e2e_steps / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": wl.h2d,
                    "d2h_bytes_per_step": int(wl.d2h), "steps": e2e_steps, "api": wl.api},
            "e2e_pcm16": {"value": total_frames * e2e_steps / e2e16_s, "unit": "frames/s", "h2d_bytes_per_step": wl.h2d16,
                          "d2h_bytes_per_step": int(wl.d2h), "steps": e2e_steps,
                          "note": "same call, host samples as int16 PCM (vbx_frames.dtype = VBX_I16)"},
            "gpu_launches": int(launches),
            "roofline": roof, "roofline_hbm": roof_hbm, "kernels": kernels, "pipe_peaks": peaks, "work_counters": counters,
            "clocks": clocks.summary(t_a, t_b),
            "sustained": {"value": total_frames * sus_steps / (sus_ms * 1e-3), "unit": "frames/s", "steps": sus_steps,
                          "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / sus_steps, "clocks": clocks.summary(t_s0, t_s1)},
            "checksum": checksum,
        }
        if world == 1 and not args.no_cpu:
            mine = os.sched_getaffinity(0)
            if getattr(args, "cpus_before", None):
                os.sched_setaffinity(0, args.cpus_before)  # all host cores for the CPU leg
            rec["cpu_baseline"] = cpu_baseline(cfg, wl.h_audio.a, wl.J)
            os.sched_setaffinity(0, mine)
    wl.free()
    return rec


def multi_record(vb, cfg, world, args):
    """The in-library multi-GPU leg (rank 0 only, the other ranks' contexts idle): ONE host buffer of world x U'
    utterances -> vbx_multi_find_formants_host -> ONE host result buffer; no torch / NCCL on this path."""
    ns = int(round(cfg["fs"] * cfg["seconds"]))
    J = n_frames_of(ns, cfg["n"], cfg["hop"])
    # bound the pinned host buffer to ~12 GB for the whole box
    u_per = int(max(8, min(cfg["utts"], (12 << 30) // (world * ns * 4))))
    U = u_per * world
    F = U * J
    with vb.Multi(world) as m:
        c0 = m.ctx(0)
        h_audio = Pinned(c0, (U, ns), np.float32)
        # synthesise on device 0 in slices and copy to the host buffer
        sl = max(1, min(U, (2 << 30) // (ns * 4)))
        for u0 in range(0, U, sl):
            n = min(sl, U - u0)
            d = c0.synth_speech(n, ns, cfg["fs"], SEED, 1_000_000 + u0)
            c0._check(c0.lib.vbx_memcpy_d2h(c0.h, h_audio.ptr + u0 * ns * 4, d.ptr, n * ns * 4), "vbx_memcpy_d2h")
            c0.sync()
            d.free()
        h_trk, h_est = Pinned(c0, (F, 8), np.float32), Pinned(c0, (U, 8), np.float32)
        est0 = np.tile(np.array([[f, 1.0] for f in MALE], dtype=np.float32).reshape(1, 8), (U, 1))
        fr = c0.frames(h_audio.ptr, F, cfg["n"], cfg["hop"], vb.WINDOW_HANN_SYMMETRIC, frames_per_segment=J, segment_stride=ns)

        def step():
            h_est.a[...] = est0
            m._check(m.lib.vbx_multi_find_formants_host(m.h, C.byref(fr), float(cfg["fs"]), cfg["p"], vb.LPC_AUTOCORR, h_est.ptr, 4,
                                                        h_trk.ptr, None, None, None, vb.F32), "vbx_multi_find_formants_host")

        for _ in range(2):
            step()
        l0 = m.kernel_launches
        steps = 5
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
        rec = {"api": "vbx_multi_find_formants_host (one pinned host buffer in, one out; one worker thread + context per device; no torch / NCCL)",
               "value": F * steps / dt, "unit": "frames/s", "n_gpus": world, "steps": steps, "utterances": U, "frames": F,
               "h2d_bytes_per_step": int(h_audio.nbytes + est0.nbytes), "d2h_bytes_per_step": int(h_trk.nbytes + est0.nbytes),
               "gpu_launches": int(m.kernel_launches - l0),
               "h2d_probe_gbs": {str(k): m.h2d_bandwidth(256 << 20, 4, k) for k in sorted({1, min(2, world), world})},
               "checksum": float(np.sum(h_trk.a[::max(1, F // 1000)], dtype=np.float64))}
        for b in (h_audio, h_trk, h_est):
            b.free()
    return rec


def run_rank(args, keys, comm, local_rank, out):
    import voxbox_b200 as vb
    # Run this rank on the CPUs next to its GPU while the pinned host buffers are allocated and the end-to-end legs run
    # (NUMA-local staging memory).  gpu_record lifts the binding for its CPU-baseline leg, which uses every host core.
    args.cpus_before = numa_bind(local_rank) if not isinstance(comm, ThreadComm) else None
    ctx = vb.Context(local_rank)  # raises without the CUDA library / a device: no CPU fallback
    peaks = ctx.measure_peaks()   # FP32/FP64 FMA pipe peaks of this device (roofline denominators)
    recs = {}
    with ClockSampler(local_rank) as clocks:
        for k in keys:
            cfg = dict(CONFIGS[k])
            if args.utts and k == args.head:
                cfg["utts"] = args.utts
            recs[k] = gpu_record(ctx, vb, k, cfg, args, comm, clocks, peaks)
    ctx.close()
    if comm.rank == 0:
        out["recs"] = recs
        out["vb"] = vb


def run_ours(args, keys, rank, world, local_rank):
    out = {}
    if world > 1:
        comm = TorchComm(rank, world, local_rank)
        run_rank(args, keys, comm, local_rank, out)
    elif args.gpus > 1:
        shared = ThreadComm._Shared(args.gpus)
        errs = []

        def body(r):
            try:
                run_rank(args, keys, ThreadComm(shared, r, args.gpus), r, out)
            except BaseException as e:  # noqa: BLE001
                errs.append(e)
                shared.bar.abort()

        ts = [threading.Thread(target=body, args=(r,)) for r in range(args.gpus)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]
        comm = NullComm()
        comm.world = args.gpus
    else:
        comm = NullComm()
        run_rank(args, keys, comm, local_rank, out)
    n_gpus = comm.world
    if rank == 0:
        recs = out["recs"]
        head = keys[0]
        line = recs[head]
        if args.device_only:
            print(json.dumps({"device_only": True, "configs": recs}), flush=True)
        else:
            subs = {k: recs[k] for k in keys[1:]}
            if args.config == "all" and not args.no_cpu:
                c1 = c1_record(args)
                subs["c1"] = c1
            if subs:
                line["configs"] = subs
    if world > 1:
        comm.barrier()
    if rank == 0 and not args.device_only:
        if n_gpus > 1 and not args.no_multi and "c3" in keys:
            try:
                line["multi"] = multi_record(out["vb"], CONFIGS["c3"], n_gpus, args)
            except Exception as e:  # noqa: BLE001 — the leg is reported, never fatal for the contract line
                line["multi"] = {"error": str(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        comm.barrier()
        comm.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of every config (default: a count per config, DEFAULT_STEPS)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="all", choices=["all", "c1"] + sorted(CONFIGS),
                    help="all = headline C3 + C2/C4/C5/C1 sub-records (default); cX = that config alone")
    ap.add_argument("--utts", type=int, default=None, help="utterances per GPU per step of the headline config (default: the config's)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs (and C1)")
    ap.add_argument("--no-multi", action="store_true", help="skip the in-library multi-GPU leg at N > 1")
    ap.add_argument("--device-only", action="store_true",
                    help="device-resident steps only (no e2e / cpu legs): the command the ncu launch lists under profiles/ are taken with")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<config>_<name>.npy (rank 0's GPU; "
                         "a fixed, seeded sample of the rows of a larger output)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "c1"):
        ap.error("--dump-outputs writes the outputs of the GPU path: it needs --impl ours and a GPU config")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config == "c1":
        if rank == 0:
            if args.steps is None:
                args.steps = 10
            print(json.dumps(c1_record(args)), flush=True)
        return
    keys = ["c3", "c2", "c4", "c5"] if args.config == "all" else [args.config]
    args.head = keys[0]
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 3
        run_reference(args, keys, rank, world)
    else:
        run_ours(args, keys, rank, world, local_rank)


if __name__ == "__main__":
    main()
