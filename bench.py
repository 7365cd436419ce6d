#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 Silero-VAD stream engine.

Metric (BASELINE.json): audio-seconds per wall-second over N concurrent 16 kHz streams (Silero v5), plus p99 latency
of one batched frame step.  Headline workload = configs[1]: 4,096 concurrent 16 kHz streams per GPU, every step advances
every stream by `--frames-per-step` 512-sample frames (hop 512).  Weak scaling: streams per GPU fixed.

  python bench.py [--gpus N] [--steps K] [--warmup W]              our arm
  python bench.py [...] --dump-outputs DIR                          ... and DIR/<name>.npy = what its last timed step returned
  python bench.py --impl reference [...]                            CPU arm (oracle port, all host threads)

One JSON line on stdout (rank 0).  Besides the contract's keys (DESIGN.md "Measurement"):
  value / ms_per_step      one timed region of exactly K steps (barrier + synchronize on both sides, max over ranks) after
                           0.5 s of untimed steps, an engine reset and max(W, input pool size) warm-up steps
  e2e                      the public host-buffer call with the wire format (int16 PCM, CVAD_PCM_S16_32767) in pinned host
                           buffers, H2D + D2H inside the timed region of K steps; e2e.f32 = the same with float32 PCM
  value_fp32               the same workload on the FP32-FMA build of the kernels (same-precision anchor)
  extra                    the other configurations of BASELINE.json, each with its own roofline:
                             configs2  v4 behind the 8 kHz resampler, 16,384 streams (N = 1 only)
                             configs3  v5, 8,192 streams per GPU, 24 / 48 kHz mixed, resampled on the GPU (every N: the
                                       65,536-stream configuration is 8 of these), device-resident and e2e (int16 wire)
                             configs4  10,000 live streams through BatchedVADManager, 30 ms int16 messages with jitter,
                                       p50 / p99 of one tick (N = 1 only)
                             configs0  one stream, 60 s of audio in one VADWrapper.process_audio_data call (N = 1 only)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from collections import deque
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "cutter-vad_b200"))

FLOP_V5 = 1_127_936             # v5/16k nominal FLOP per 512-sample frame (SURVEY.md 8a, BASELINE.md 3)
FLOP_V5_FE = 865_536            # STFT + encoder.0-3 share (432,768 MAC)
FLOP_V5_REC = 262_400           # LSTM + decoder share (131,200 MAC)
FLOP_V4 = 1_379_280             # v4/16k nominal (dense STFT counted as the graph states it)
SMS, FP32_LANES = 148, 128
# FFT resampler, algorithmic FLOP per chunk: 2.5 N log2 N (real forward) + 2.5 * 512 * 9 (real inverse)
FLOP_RESAMPLE = {8000: 16_640, 24000: 29_900, 48000: 52_160, 16000: 0}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


def ncu_traffic_bytes(kernel: str):
    """DRAM read+write bytes per launch of `kernel` from the newest committed ncu --set full summary
    (profiles/*.json, written by tools/ncu_summary.py from the same bench command); None if absent."""
    best = None
    for f in sorted((ROOT / "profiles").glob("*.json")):
        if "warm_caches" in f.name:      # --cache-control none captures re-read the replayed inputs from L2: not a DRAM figure
            continue
        try:
            d = json.loads(f.read_text())
            for k in d.get("full_capture", []):
                if kernel in k.get("kernel", ""):
                    tot = 0.0
                    for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                        val, _, unit = k.get(key, "0 byte").partition(" ")
                        mult = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit.strip(), 1)
                        tot += float(val) * mult
                    best = {"bytes": tot, "source": f"profiles/{f.name}"}
        except Exception:
            continue
    return best


def synth_audio(n_streams: int, n_samples: int, seed: int) -> np.ndarray:
    """Vectorised version of the tests' signal recipe: per-stream noise floor plus gated
    harmonic 'voice' bursts (reference examples/probability_demo.py:60-67), float32."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_samples, dtype=np.float32) / 16000.0
    sigma = np.array([0.005, 0.02, 0.1], np.float32)[np.arange(n_streams) % 3][:, None]
    level = np.array([0.3, 0.7], np.float32)[(np.arange(n_streams) // 3) % 2][:, None]
    f0 = rng.uniform(110, 220, size=(n_streams, 1)).astype(np.float32)
    out = rng.standard_normal((n_streams, n_samples), dtype=np.float32) * sigma
    ph = 2 * np.pi * f0 * t[None, :]
    voice = level * (0.4 * np.sin(ph) + 0.3 * np.sin(2 * ph) + 0.2 * np.sin(4 * ph))
    period = rng.uniform(1.0, 4.0, size=(n_streams, 1)).astype(np.float32)
    phase = rng.uniform(0, 1, size=(n_streams, 1)).astype(np.float32)
    gate = (((t[None, :] / period) + phase) % 1.0) < 0.5
    out += np.where(gate, voice, 0.0).astype(np.float32)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the measurement (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """index of the next sample: lets a caller cut out the samples taken during one leg"""
        return len(self.lines)

    def stop(self, lo: int = 0, hi: int = None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        return self.summary(lo, hi)

    def summary(self, lo: int = 0, hi: int = None):
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[lo:hi]:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU arm

def cpu_port(native=True):
    sys.path.insert(0, str(ROOT / "oracle"))
    from vad_oracle import RefLib, RefV5, v5_blob
    # compiled for this host at run time, so outside the tree (which may be read-only); the loaded library outlives its file
    with tempfile.TemporaryDirectory(prefix="cvad_bench_") as tmp:
        lib = RefLib(native=native, build_dir=tmp)
    blob = v5_blob(str(ROOT / "cutter-vad_b200" / "real_time_vad" / "models" / "silero_vad_v5.onnx"))
    return lib, RefV5(blob, lib)


def cpu_baseline_sample(n_streams: int, target_s: float = 12.0):
    """Oracle port (plain C + OpenMP, every host thread) on a bounded sample of the workload."""
    lib, ref = cpu_port()
    cores = host_threads()
    n = min(n_streams, 1024)
    audio = synth_audio(n, 512 * 8, seed=99)
    t0 = time.perf_counter()
    ref.run(audio, 8, nthreads=cores)
    dt = time.perf_counter() - t0
    rate = n * 8 / dt
    frames = int(max(8, min(4000, rate * target_s / n)))
    audio = synth_audio(n, 512 * frames, seed=100)
    t0 = time.perf_counter()
    ref.run(audio, frames, nthreads=cores)
    dt = time.perf_counter() - t0
    fps = n * frames / dt
    return {"value": fps * 0.032, "unit": "audio-s/s", "cores": cores, "kind": "port",
            "frames_per_s": fps,
            "sample": f"{n} streams x {frames} frames (hop 512) of the same synthetic recipe, {dt:.1f} s, "
                      f"oracle/silero_ref.c -O3 -march=native + OpenMP; CPU restatement, not onnxruntime"}


def workload_config(model: str, streams: int, frames_per_step: int, rate: int = 16000, mixed: bool = False):
    """`config` of the JSON line: the workload only, identical in both arms (arithmetic and cache notes are separate keys)."""
    what = f"Silero {model}, {streams} concurrent {rate // 1000} kHz streams per GPU batched per frame step"
    if (model, rate, mixed) == ("v5", 16000, False):
        what += " (BASELINE.json configs[1])"
    elif mixed:
        what = (f"Silero {model}, {streams} concurrent streams per GPU, 24 / 48 kHz by stream parity, resampled to 16 kHz on the "
                "GPU and stepped one frame per call (BASELINE.json configs[3] per-GPU share)")
    elif rate != 16000:
        what += ", resampled to 16 kHz on the GPU"
    return {"workload": what, "model": model, "src_rate": rate, "streams_per_gpu": streams,
            "frames_per_step": frames_per_step, "hop": 512, "frame_len": 512, "denoise": True, "state_machine": True}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    lib, ref = cpu_port()
    cores = host_threads()
    n, F = args.streams, args.frames_per_step
    pool = [synth_audio(n, 512 * F, seed=1000 + i) for i in range(4)]
    h = np.zeros((n, 128), np.float32)
    c = np.zeros((n, 128), np.float32)
    for i in range(args.warmup):
        ref.run(pool[i % 4], F, h=h, c=c, nthreads=cores)
    lat = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        t1 = time.perf_counter()
        ref.run(pool[i % 4], F, h=h, c=c, nthreads=cores)
        lat.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    value = n * F * args.steps * 0.032 / dt
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config("v5", n, F),
        "p99_step_ms": 1e3 * float(np.percentile(lat, 99)),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port",
                         "sample": f"every step = full workload ({n} streams x {F} frames); oracle/silero_ref.c "
                                   f"(plain C, OpenMP, {cores} threads); CPU restatement of the reference's "
                                   "onnxruntime path, onnxruntime itself is absent from this image"},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------- GPU arm

def pin_to_gpu_numa_node(local: int):
    """Bind this rank's host threads to the CPUs of its GPU's NUMA node BEFORE any pinned buffer is allocated, so that the
    pages the H2D copies read are local to the GPU's PCIe root (every rank on node 0 halves the copy rate at 8 GPUs)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                   # nvml prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        if node < 0:
            return {"numa_node": None, "note": "the platform reports no NUMA affinity for this GPU"}
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return {"numa_node": node, "note": "no allowed CPU on the GPU's node"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as exc:                              # measurement aid only: never fail the bench over it
        return {"numa_node": None, "note": f"not pinned: {exc}"}


class Workload:
    """Synthetic inputs of one configuration: a pool of distinct step buffers (> 126 MB L2 in total) on the device, and,
    for the e2e legs, the same in pinned host memory as float32 and as int16 PCM."""

    def __init__(self, torch, local, rank, model, n, F, rate, mixed, want_host=True, pool_bytes=300e6):
        from real_time_vad.engine import capi
        self.torch, self.capi, self.local = torch, capi, local
        self.model, self.n, self.F, self.rate, self.mixed = model, n, F, rate, mixed
        self.n_in = 1536 if mixed else rate * 512 // 16000          # row length per frame (24 kHz rows use the first half)
        self.step_samples = self.n_in * F
        self.step_bytes_f32 = n * self.step_samples * 4
        self.pool_n = int(min(64, max(2, np.ceil(pool_bytes / self.step_bytes_f32))))
        self.rates_np = np.where(np.arange(n) & 1, 48000, 24000).astype(np.int32) if mixed else None
        cu = f"cuda:{local}"
        self.host_f32, self.host_s16, self.dev = [], [], []
        for i in range(self.pool_n):
            x = synth_audio(n, self.step_samples, seed=rank * 7919 + i + (17 if mixed else 0) + rate)
            if want_host:
                t = torch.empty((n, self.step_samples), dtype=torch.float32).pin_memory()
                t.numpy()[:] = x
                self.host_f32.append(t)
                if i < 8:
                    q = torch.empty((n, self.step_samples), dtype=torch.int16).pin_memory()
                    q.numpy()[:] = np.clip(np.rint(x * 32767.0), -32768, 32767).astype(np.int16)
                    self.host_s16.append(q)
                self.dev.append(t.to(cu))
            else:
                self.dev.append(torch.from_numpy(x).to(cu))
        self.d_probs = torch.zeros((n, F), dtype=torch.float32, device=cu)
        self.d_flags = torch.zeros((n, F), dtype=torch.uint8, device=cu)
        self.max_events = max(16, 2 * n * F)
        self.d_events = torch.zeros((self.max_events * 24,), dtype=torch.uint8, device=cu)
        self.d_nev = torch.zeros((1,), dtype=torch.int32, device=cu)
        self.d_rates = torch.from_numpy(self.rates_np).to(cu) if mixed else None
        self.dargs = [self._dev_args(b) for b in self.dev]
        self.rate_kw = {"src_rates": self.rates_np, "max_frames": F} if mixed else {"src_rate": rate}

    def _dev_args(self, buf):
        a = self.capi.StepArgs()
        a.n_streams = self.n
        a.audio = buf.data_ptr()
        a.pcm_format = self.capi.PCM_F32
        a.stream_stride = self.step_samples
        a.max_frames = self.F
        a.frame_len = a.hop = self.n_in
        a.src_rate = 48000 if self.mixed else self.rate
        if self.mixed:
            a.src_rates = self.d_rates.data_ptr()
        a.probs_out = self.d_probs.data_ptr()
        a.flags_out = self.d_flags.data_ptr()
        a.events_out = self.d_events.data_ptr()
        a.max_events = self.max_events
        a.n_events_out = self.d_nev.data_ptr()
        return a

    @property
    def audio_s_per_step(self):
        return self.n * self.F * 0.032

    def outputs(self):
        """What a caller of the last device step received: probabilities [n][F], flags [n][F] and the event records
        [events][stream, slot, frame, kind, stream_frame], sorted (the kernel appends events in no fixed order)."""
        n_ev = min(int(self.d_nev.item()), self.max_events)
        rec = np.dtype([("stream", "<i4"), ("slot", "<i4"), ("frame", "<i4"), ("kind", "<i4"), ("stream_frame", "<i8")])
        ev = self.d_events[:n_ev * rec.itemsize].cpu().numpy().view(rec)
        ev = np.stack([ev[k].astype(np.float64) for k in rec.names], axis=1).reshape(n_ev, len(rec.names))
        ev = ev[np.lexsort(ev.T[::-1])]
        return self.d_probs.cpu().numpy(), self.d_flags.cpu().numpy(), ev


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, outputs):
    """DIR/<name>.npy: probs, flags (float32), events and streams (float64, the stream index of each row).  Over DUMP_BYTES
    in the worst case (one event per stream and frame) the rows are a fixed seeded sample of the streams."""
    probs, flags, ev = outputs
    n, F = probs.shape
    rows = np.arange(n)
    per_row = 8 * F + 8 + 40 * F
    if n * per_row > DUMP_BYTES - 4096:                     # (room for the four .npy headers)
        k = (DUMP_BYTES - 4096) // per_row
        rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
        ev = ev[np.isin(ev[:, 0], rows)]
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "probs.npy", probs[rows].astype(np.float32))
    np.save(d / "flags.npy", flags[rows].astype(np.float32))
    np.save(d / "events.npy", ev)
    np.save(d / "streams.npy", rows.astype(np.float64))


def settle(step, barrier, seconds=0.5):
    """Untimed steps for `seconds` of wall time: GPU clocks and host threads reach the state of a service under sustained
    load.  The caller resets the engine afterwards, so that what is timed and returned depends on the arguments only."""
    i, t_end = 0, time.perf_counter() + seconds
    while time.perf_counter() < t_end:
        step(i)
        i += 1
    barrier()


def time_device(torch, dist, world, eng, wl, stream, steps, warmup, keep_outputs=False):
    """`value` leg: inputs resident in HBM, cvad_step_device, CUDA events on the engine's stream.  After `warmup` untimed
    steps, ONE region of exactly `steps` steps is timed (barrier + synchronize on both sides; the max over ranks).
    -> dict(region_ms, launches in the region, per-step latency p50 / p99, per-kernel ms from a separate pass, and with
    `keep_outputs` what the region's last step returned)"""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    settle(lambda i: eng.step_device(wl.dargs[i % wl.pool_n]), barrier)
    eng.reset()
    # the warm-up steps every buffer of the pool at least once: a buffer's first read pays address-translation misses
    # that a running service never sees
    warmup = max(warmup, wl.pool_n)
    for i in range(warmup):
        eng.step_device(wl.dargs[i % wl.pool_n])
    eng.sync()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    l0 = eng.launch_count()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for i in range(steps):
            eng.step_device(wl.dargs[(warmup + i) % wl.pool_n])
        e1.record(stream)
    barrier()
    launches = eng.launch_count() - l0
    outputs = wl.outputs() if keep_outputs else None
    ms_t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=f"cuda:{wl.local}")
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    region_ms = float(ms_t[0])
    # per-kernel durations for the roofline: the same K steps again with events around the kernels
    # (kept out of the passes above: events between the kernels would serialise their overlap)
    eng.set_timing(True)
    with torch.cuda.stream(stream):
        for i in range(steps):
            eng.step_device(wl.dargs[(warmup + i) % wl.pool_n])
    barrier()
    fe_ms, rec_ms, n_timed = eng.read_timing()
    eng.set_timing(False)
    lat = []
    for i in range(steps):
        a0 = torch.cuda.Event(enable_timing=True)
        a1 = torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        eng.step_device(wl.dargs[i % wl.pool_n])
        a1.record(stream)
        a1.synchronize()
        lat.append(a0.elapsed_time(a1))
    return {"region_ms": region_ms, "launches": int(launches), "outputs": outputs, "warmup": warmup,
            "fe_ms": fe_ms / max(n_timed, 1), "rec_ms": rec_ms / max(n_timed, 1),
            "p50_step_ms": float(np.percentile(lat, 50)), "p99_step_ms": float(np.percentile(lat, 99))}


def time_e2e(torch, dist, world, eng, wl, steps, warmup, pcm: str, depth=4):
    """`e2e` leg: the public host-buffer call (StreamEngine.submit / collect -> cvad_step_submit / _collect) with `depth`
    steps in flight; every step's H2D of its inputs and D2H of its results is inside the timed region of exactly `steps`
    steps (wall clock, max over ranks).  A short region mostly measures the fill and drain of the pipeline."""
    capi = wl.capi
    pool = [t.numpy() for t in (wl.host_s16 if pcm == "s16" else wl.host_f32)]
    kw = dict(wl.rate_kw)
    if pcm == "s16":
        kw["pcm_format"] = capi.PCM_S16_32767

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def pipelined(k):
        inflight = deque()
        for i in range(k):
            inflight.append(eng.submit(pool[i % len(pool)], **kw))
            if len(inflight) == depth:
                r = inflight.popleft().collect()
        while inflight:
            r = inflight.popleft().collect()
        return r

    settle(lambda i: pipelined(32), barrier)
    eng.reset()
    pipelined(max(warmup, depth))          # the warm-up runs every lane of the pipeline the timed region uses
    barrier()
    t0 = time.perf_counter()
    r = pipelined(steps)
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=f"cuda:{wl.local}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t[0])
    events = len(r.events)
    # one call at a time: latency distribution of the blocking form
    lat = []
    for i in range(steps):
        t1 = time.perf_counter()
        eng.step(pool[i % len(pool)], **kw)
        lat.append(time.perf_counter() - t1)
    es = 2 if pcm == "s16" else 4
    return {"value": wl.audio_s_per_step * steps * world / dt, "unit": "audio-s/s",
            "h2d_bytes_per_step": wl.n * wl.step_samples * es, "d2h_bytes_per_step": wl.n * wl.F * 5 + wl.n * 4 + 4,
            "ms_per_step": 1e3 * dt / steps,
            "p50_call_ms": 1e3 * float(np.percentile(lat, 50)), "p99_call_ms": 1e3 * float(np.percentile(lat, 99)),
            "pcm": ("int16 (the websocket wire format, vad_websocket_server.py:341), / 32767.0f in the frame loader"
                    if pcm == "s16" else "float32"),
            "events_last_step": events}


def pinned_copy_rate(torch, wl):
    h0 = torch.cuda.Event(enable_timing=True)
    h1 = torch.cuda.Event(enable_timing=True)
    h0.record()
    for i in range(10):
        wl.dev[i % wl.pool_n].copy_(wl.host_f32[i % wl.pool_n], non_blocking=True)
    h1.record()
    torch.cuda.synchronize()
    return 10 * wl.step_bytes_f32 / (h0.elapsed_time(h1) * 1e-3) / 1e9


def single_stream_call(seconds=60, repeats=5):
    """BASELINE.json configs[0] on the engine: ONE 16 kHz stream, `seconds` of synthetic audio through
    VADWrapper.process_audio_data (512-sample frames, hop 256 as the reference frames them, vad_wrapper.py:626-629), callbacks
    attached.  The recurrent part is strictly sequential (one stream): this is the latency floor of the drop-in call, not a
    throughput figure."""
    from real_time_vad import VADConfig, VADWrapper
    audio = synth_audio(1, 16000 * seconds, seed=3)[0]
    w = VADWrapper(VADConfig())
    n_ev = [0]
    w.set_callbacks(voice_start_callback=lambda: n_ev.__setitem__(0, n_ev[0] + 1),
                    voice_end_callback=lambda b: n_ev.__setitem__(0, n_ev[0] + 1))
    w.process_audio_data(audio[:16000])                       # warm-up (engine creation, first launches)
    ms = []
    for _ in range(repeats):
        w.reset()
        t0 = time.perf_counter()
        w.process_audio_data(audio)
        ms.append(1e3 * (time.perf_counter() - t0))
    frames = (len(audio) - 512) // 256 + 1
    w.cleanup()
    med = float(np.median(ms))
    return {"workload": f"one 16 kHz stream, {seconds} s of audio in one VADWrapper.process_audio_data call (BASELINE.json configs[0])",
            "frames": frames, "call_ms_p50": med, "call_ms_min": float(min(ms)), "value": seconds / (med * 1e-3), "unit": "audio-s/s",
            "us_per_frame": 1e3 * med / frames, "events": n_ev[0] // repeats}


def service_tick(n_streams=10000, ticks=120):
    """BASELINE.json configs[4]: `n_streams` live clients through BatchedVADManager -- 480-sample int16 messages (30 ms) with
    arrival jitter, the websocket server's thresholds, 10 % of the streams with start / end callbacks.  Timed: the
    manager's calls of one tick (pushes + step).  tools/bench_service.py is the long form of this."""
    from real_time_vad import BatchedVADManager, VADConfig
    from real_time_vad.engine import capi
    n = n_streams
    mgr = BatchedVADManager(max_streams=n, frame_len=480, hop=480, pcm_format=capi.PCM_S16_32767)
    cfg = VADConfig(buffer_size=480, vad_start_probability=0.4, vad_end_probability=0.3,
                    voice_start_frame_count=6, voice_end_frame_count=12)
    fired = [0, 0]
    ids = []
    for s in range(n):
        if s < n // 10:
            ids.append(mgr.open_stream(cfg, on_voice_start=lambda: fired.__setitem__(0, fired[0] + 1),
                                       on_voice_end=lambda b: fired.__setitem__(1, fired[1] + 1)))
        else:
            ids.append(mgr.open_stream(cfg))
    ids = np.array(ids)
    rng = np.random.default_rng(0)
    sec = 3
    audio = np.clip(np.round(synth_audio(n, 16000 * sec, seed=1) * 32767.0), -32768, 32767).astype(np.int16)
    pos = np.zeros(n, np.int64)
    lat_tick, lat_step, lat_push, frames, events, phases, host = [], [], [], 0, 0, [], []
    for t in range(ticks + 10):
        k = rng.choice([0, 1, 1, 1, 1, 1, 1, 2], size=n)               # jitter: late / on time / catching up
        t_push = 0.0
        for m in (1, 2):
            sel = np.flatnonzero(k >= m)
            if sel.size == 0:
                continue
            start = pos[sel] % (16000 * sec - 480)
            block = audio[sel[:, None], start[:, None] + np.arange(480)[None, :]]   # the clients' side: not timed
            t0 = time.perf_counter()
            mgr.push_many(ids[sel], block)
            t_push += time.perf_counter() - t0
            pos[sel] += 480
        t1 = time.perf_counter()
        out = mgr.step()
        t2 = time.perf_counter()
        if t >= 10:
            lat_tick.append(t_push + t2 - t1)
            lat_step.append(t2 - t1)
            lat_push.append(t_push)
            phases.append(getattr(out, "phase_ms", (0.0, 0.0, 0.0)))
            host.append(getattr(out, "host_ms", (0.0,) * 5))
            frames += out.frames
            events += len(out.events)
    mgr.close()
    total = sum(lat_tick)
    return {"workload": f"{n} live streams through BatchedVADManager, 480-sample int16 messages with jitter, websocket thresholds, "
                        "10 % of the streams with callbacks (BASELINE.json configs[4])",
            "ticks": ticks, "budget_ms": 30.0,
            "tick_ms_p50": 1e3 * float(np.percentile(lat_tick, 50)), "tick_ms_p99": 1e3 * float(np.percentile(lat_tick, 99)),
            "step_ms_p50": 1e3 * float(np.percentile(lat_step, 50)), "step_ms_p99": 1e3 * float(np.percentile(lat_step, 99)),
            "push_ms_p50": 1e3 * float(np.percentile(lat_push, 50)), "push_ms_p99": 1e3 * float(np.percentile(lat_push, 99)),
            "native_step_ms_p50": dict(zip(("gather", "cvad_step", "deliver"), [float(x) for x in np.percentile(np.array(phases), 50, axis=0)])),
            "python_step_ms_p50": dict(zip(("native_call", "unpack", "event_tuples", "callbacks_wav", "result"),
                                           [float(x) for x in np.percentile(np.array(host), 50, axis=0)])),
            "value": frames * 0.030 / total, "unit": "audio-s/s", "frames": frames, "events": events, "callbacks_fired": fired,
            "timed": "the manager's calls only (push_many + step); building the synthetic clients' messages is outside"}


def simple_roofline(kernel, bound, flop_per_frame, frames_per_step, step_ms, peak, peak_src):
    tf = frames_per_step * flop_per_frame / (step_ms * 1e-3) / 1e12
    return {"bound": bound, "kernel": kernel, "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
            "traffic": None, "algorithmic_flop_per_frame": flop_per_frame, "frames_per_launch": frames_per_step,
            "step_ms": step_ms, "peak_source": peak_src,
            "note": "whole step (every kernel of it) against the peak of the pipe its dominant kernel runs on"}


def dev_pool_mb(n, F, rate, mixed):
    n_in = 1536 if mixed else rate * 512 // 16000
    step_bytes = n * n_in * F * 4
    return int(min(64, max(2, np.ceil(300e6 / step_bytes)))) * step_bytes / 1e6


def transfer_bound(n, F, rate, mixed, world, h2d_gbs):
    """audio-s/s the measured pinned-copy rate allows for int16 input (context for e2e: the path is PCIe-bound)"""
    n_in = 1536 if mixed else rate * 512 // 16000
    return n * F * 0.032 * world / (n * n_in * F * 2 / (h2d_gbs * 1e9))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from real_time_vad.engine.stream_engine import StreamEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this engine has no CPU fallback)")
    numa = pin_to_gpu_numa_node(local)            # before the first pinned allocation
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks, peaks_src = load_peaks()
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    peak_fp32 = SMS * FP32_LANES * 2 * sm_max * 1e6 / 1e12
    peak_bf16 = float(peaks.get("bf16_tflops", 1645.0))
    peak_bf16_src = f"{peaks_src} MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)"
    peak_fp32_src = f"148 SMs x 128 FP32 lanes x 2 x sm_max_mhz {sm_max:.0f} ({peaks_src} MEASURED_PEAKS.json clock)"

    n, F = args.streams, args.frames_per_step
    mixed = bool(args.mixed_rates)
    rate = 48000 if mixed else args.src_rate
    model, math = args.model, args.math
    stream = torch.cuda.Stream(device=local)
    sampler = ClockSampler(local)

    # ================= headline configuration
    wl = Workload(torch, local, rank, model, n, F, rate, mixed)
    eng = StreamEngine(model, max_streams=n, device=local)
    eng.set_math(math)
    eng.configure(enable_denoising=True)
    eng.set_stream(stream.cuda_stream)
    sampler.start()
    time.sleep(0.12)
    c_lo = sampler.mark()
    dev = time_device(torch, dist, world, eng, wl, stream, args.steps, args.warmup, keep_outputs=bool(args.dump_outputs))
    c_hi = sampler.mark()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dev["outputs"])
    e2e = time_e2e(torch, dist, world, eng, wl, args.steps, args.warmup, "s16")
    e2e_f32 = time_e2e(torch, dist, world, eng, wl, args.steps, args.warmup, "f32")
    h2d_gbs = pinned_copy_rate(torch, wl)
    eng.close()

    region_ms = dev["region_ms"]
    total_audio = wl.audio_s_per_step * args.steps * world
    value = total_audio / (region_ms * 1e-3)
    frames_per_step = n * F
    step_ms = region_ms / args.steps

    extras = {}
    value_fp32 = None
    run_extras = not args.no_extras and (model, rate, mixed, F) == ("v5", 16000, False, 1)
    # ================= same workload, FP32-FMA build (same-precision anchor) -- N = 1 only
    if run_extras and world == 1:
        e32 = StreamEngine(model, max_streams=n, device=local)
        e32.set_math("fp32")
        e32.configure(enable_denoising=True)
        e32.set_stream(stream.cuda_stream)
        d32 = time_device(torch, dist, world, e32, wl, stream, args.steps, args.warmup)
        e32.close()
        m32 = d32["region_ms"]
        value_fp32 = {"value": total_audio / (m32 * 1e-3), "unit": "audio-s/s", "ms_per_step": m32 / args.steps,
                      "math": "fp32 (packed FP32 FMA on the CUDA cores, ascending-k accumulation)",
                      "roofline": simple_roofline("v5_frontend_kernel + v5_recurrent_kernel", "fp32_ffma", FLOP_V5, frames_per_step,
                                                  m32 / args.steps, peak_fp32, peak_fp32_src)}
    del wl
    torch.cuda.empty_cache()

    # ================= configs[3] per-GPU share: 8,192 streams, 24 / 48 kHz mixed -- every N
    if run_extras:
        w3 = Workload(torch, local, rank, "v5", 8192, 1, 48000, True, pool_bytes=200e6)
        e3 = StreamEngine("v5", max_streams=8192, device=local)
        e3.configure(enable_denoising=True)
        e3.set_stream(stream.cuda_stream)
        d3 = time_device(torch, dist, world, e3, w3, stream, args.steps, args.warmup)
        x3 = time_e2e(torch, dist, world, e3, w3, args.steps, args.warmup, "s16")
        e3.close()
        m3 = d3["region_ms"]
        flop3 = FLOP_V5 + (FLOP_RESAMPLE[24000] + FLOP_RESAMPLE[48000]) // 2
        extras["configs3"] = {
            "config": workload_config("v5", 8192, 1, 48000, True), "n_gpus": world,
            "value": w3.audio_s_per_step * args.steps * world / (m3 * 1e-3), "unit": "audio-s/s", "ms_per_step": m3 / args.steps,
            "p99_step_ms": d3["p99_step_ms"], "gpu_launches": d3["launches"],
            "e2e": x3,
            "roofline": simple_roofline("rate_lists + 2 x resample_fft_kernel + v5tc_frontend_kernel<FUSED,H16>", "tensor", flop3,
                                        8192, m3 / args.steps, peak_bf16, peak_bf16_src)}
        del w3
        torch.cuda.empty_cache()

    # ================= configs[2]: v4 behind the 8 kHz resampler, 16,384 streams -- N = 1 only
    if run_extras and world == 1:
        w2 = Workload(torch, local, rank, "v4", 16384, 1, 8000, False, want_host=False, pool_bytes=200e6)
        e2 = StreamEngine("v4", max_streams=16384, device=local)
        e2.configure(enable_denoising=True)
        e2.set_stream(stream.cuda_stream)
        d2 = time_device(torch, dist, world, e2, w2, stream, args.steps, args.warmup)
        m2 = d2["region_ms"] / args.steps
        extras["configs2"] = {
            "config": workload_config("v4", 16384, 1, 8000), "math": e2.math, "n_gpus": 1,
            "value": w2.audio_s_per_step / (m2 * 1e-3), "unit": "audio-s/s", "ms_per_step": m2,
            "p99_step_ms": d2["p99_step_ms"], "gpu_launches": d2["launches"],
            "kernel_ms": {"frontend_kernels": d2["fe_ms"], "v4_recurrent_kernel": d2["rec_ms"]},
            "roofline": simple_roofline("resample_fft<1> + v4_stft_fft + v4tc_stft<CORR> + v4_frontend + v4_recurrent", "fp32_ffma",
                                        FLOP_V4 + FLOP_RESAMPLE[8000], 16384, m2, peak_fp32, peak_fp32_src)}
        e2.close()
        del w2
        torch.cuda.empty_cache()

    # ================= configs[4]: the manager's tick at 10,000 live streams; configs[0]: one stream, one call -- N = 1 only
    if run_extras and world == 1:
        try:
            extras["configs4"] = service_tick()
        except Exception as exc:                       # the service leg must not take the headline line down with it
            extras["configs4"] = {"error": f"{type(exc).__name__}: {exc}"}
        try:
            extras["configs0"] = single_stream_call()
        except Exception as exc:
            extras["configs0"] = {"error": f"{type(exc).__name__}: {exc}"}
    sampler.stop()
    clocks = sampler.summary(c_lo, max(c_hi, c_lo + 1))
    clocks["whole_run"] = sampler.summary()

    if rank == 0:
        tc = math in ("tc", "tc16")
        fused = tc and model == "v5" and F == 1 and os.environ.get("CVAD_FUSE", "1") != "0"
        h16 = fused and math == "tc16"      # FP16 two-way split: 3 tensor-core products per MAC (BF16 split: 6)
        # chained one-frame steps (cvad_step_device on 16 kHz input): the timed region holds K launches of ONE kernel and
        # nothing else -- no memset, no event -- each scheduled by programmatic dependent launch while its predecessor
        # drains, so the kernel's average launch duration over the timed region is region / launches.  The duration of a
        # launch bracketed by its own events (no overlap with its neighbours) is reported beside it.
        chained = (fused and rate == 16000 and not mixed and os.environ.get("CVAD_CHAIN", "1") != "0"
                   and dev["launches"] == args.steps)
        flop_frame = FLOP_V5 if model == "v5" else FLOP_V4
        flop_fe = FLOP_V5_FE if model == "v5" else FLOP_V4 - 2 * 65_600
        flop_rec = FLOP_V5_REC if model == "v5" else 2 * 65_600
        if rate != 16000:
            rs = (FLOP_RESAMPLE[24000] + FLOP_RESAMPLE[48000]) // 2 if mixed else FLOP_RESAMPLE[rate]
            flop_fe += rs
            flop_frame += rs
        fe_s, rec_s = dev["fe_ms"] * 1e-3, dev["rec_ms"] * 1e-3
        isolated_ms = dev["fe_ms"]
        if fused:
            flop_fe = flop_frame            # one kernel does the whole step
            if chained:
                fe_s = step_ms * 1e-3
        fe_tflops = frames_per_step * flop_fe / fe_s / 1e12 if fe_s > 0 else 0.0
        rec_tflops = frames_per_step * flop_rec / rec_s / 1e12 if rec_s > 0 else 0.0
        step_tflops = frames_per_step * flop_frame / (step_ms * 1e-3) / 1e12
        fe_kernel = (("v4_stft_fft_kernel+v4tc_stft_kernel<CORR>+v4_frontend_kernel" if math == "fft" else
                      "v4tc_stft_kernel+v4_frontend_kernel" if model == "v4" else
                      "v5tc_frontend_kernel<FUSED,H16>" if h16 else
                      "v5tc_frontend_kernel<FUSED>" if fused else "v5tc_frontend_kernel") if (tc or math == "fft")
                     else f"{model}_frontend_kernel") + ("+resample_fft_kernel" if rate != 16000 else "")
        # (prefixes: the kernel's trailing template argument PROF is 0 in the build that runs unless a profile was asked for)
        variant = ("v5tc_frontend_kernel<0, 1, 1" if h16 else "v5tc_frontend_kernel<0, 1, 0" if fused else
                   "v5tc_frontend_kernel<0, 0" if tc else "v5_frontend_kernel")
        traffic = ncu_traffic_bytes(variant) if (n == 4096 and F == 1 and model == "v5" and rate == 16000) else None
        fe_weight_bytes = ((622_592 + 524_288) if h16 else (933_888 + (786_432 if fused else 0))) if tc else 156032 * 4
        peak = peak_bf16 if tc else peak_fp32
        roofline = {
            # tc: every algorithmic MAC is executed as 6 BF16 tensor-core products (3-way operand split) -- 3 FP16
            # products (2-way split, per-stream scaling) in the tc16 build of the fused kernel -- so the executed
            # rate is 6x / 3x `achieved` (DESIGN.md section 3)
            "bound": "tensor" if tc else "fp32_ffma", "kernel": fe_kernel,
            "achieved": fe_tflops, "peak": peak, "unit": "TFLOP/s", "frac": fe_tflops / peak,
            "traffic": (traffic or {}).get("bytes"), "traffic_source": (traffic or {}).get("source"),
            "algorithmic_bytes_per_launch": frames_per_step * 2048 + fe_weight_bytes +
            frames_per_step * ((2 * 1024 + 5) if fused else 768 if tc else 512),
            "peak_source": peak_bf16_src if tc else peak_fp32_src,
            "algorithmic_flop_per_frame": flop_fe, "frames_per_launch": frames_per_step,
            "avg_launch_ms": fe_s * 1e3, "isolated_launch_ms": isolated_ms,
            "kernel_timing": ("avg_launch_ms = timed region (CUDA events on the engine's stream) / launches: the region holds "
                              "nothing but this kernel's K launches, chained by programmatic dependent launch; "
                              "isolated_launch_ms = separate pass with events around every launch (no overlap)" if chained else
                              "separate pass over the same K steps with a CUDA event between the kernels"),
            "recurrent_kernel": ({"kernel": "(fused into the kernel above for one-frame steps)", "avg_launch_ms": 0.0,
                                  "achieved": 0.0, "algorithmic_flop_per_frame": 0} if fused else
                                 {"kernel": "v5tc_recurrent_kernel" if tc else f"{model}_recurrent_kernel",
                                  "avg_launch_ms": rec_s * 1e3, "achieved": rec_tflops, "algorithmic_flop_per_frame": flop_rec}),
            "whole_step": {"achieved": step_tflops, "frac": step_tflops / peak, "algorithmic_flop_per_frame": flop_frame},
            "vs_fp32_ffma_peak": {"peak": peak_fp32, "kernel_frac": fe_tflops / peak_fp32, "whole_step_frac": step_tflops / peak_fp32},
            "hbm": {"algorithmic_bytes_per_frame": 2048 + 2 * 1024 + 4 + 1,
                    "achieved_gbs": frames_per_step * (2048 + 2048 + 5) / (step_ms * 1e-3) / 1e9, "peak_gbs": peaks.get("hbm_gbs")},
        }
        if tc:
            products = 3 if h16 else 6
            roofline["tensor_products_per_mac"] = products
            roofline["executed_bf16_tflops"] = products * fe_tflops
            roofline["executed_frac"] = products * fe_tflops / peak_bf16
        cpu = None if args.skip_cpu else cpu_baseline_sample(n)
        e2e["f32"] = {k: e2e_f32[k] for k in ("value", "h2d_bytes_per_step", "ms_per_step")}
        e2e["pinned_h2d_gbs"] = h2d_gbs
        e2e["transfer_bound_value"] = transfer_bound(n, F, rate, mixed, world, h2d_gbs)
        e2e["numa"] = numa
        e2e["api"] = ("StreamEngine.submit/collect -> cvad_step_submit/cvad_step_collect, four steps in flight (every lane of the engine), pinned host "
                      "buffers; p50/p99_call_ms = one blocking StreamEngine.step at a time")
        line = {
            "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("f16x2 operands with per-stream scaling, f32 accumulate (FP32-equivalent)" if h16 else
                      "bf16x3 operands, f32 accumulate (FP32-equivalent)" if tc else
                      "f64 FFT + bf16 basis correction (STFT), f32 elsewhere" if math == "fft" else "f32"),
            "data": "synthetic", "config": workload_config(model, n, F, rate, mixed),
            "math": math,
            "l2": f"inputs cycle through a pool of distinct step buffers totalling {round(dev_pool_mb(n, F, rate, mixed))} MB (> 126 MB L2)",
            "timing": f"value = K steps / one timed region of exactly K = {args.steps} steps after {dev['warmup']} untimed ones "
                      "(W, and at least one pass over the input pool; barrier + synchronize around the region, max over ranks)",
            "p99_step_ms": dev["p99_step_ms"], "p50_step_ms": dev["p50_step_ms"],
            "frames_per_s": value / 0.032,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "value_fp32": value_fp32,
            "extra": extras,
            "gpu_launches": dev["launches"],
            "clocks": clocks,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def _protect_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line there.
    Send fd 1 to stderr for the duration of the run and keep the real stdout for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def host_threads() -> int:
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm ignores it)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--streams", type=int, default=4096, help="concurrent streams per GPU")
    ap.add_argument("--frames-per-step", type=int, default=1, help="512-sample frames per stream per step")
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-extras", action="store_true", help="headline configuration only (no value_fp32 / extra records)")
    ap.add_argument("--mixed-rates", action="store_true",
                    help="BASELINE.json configs[3] per-GPU share: 24 / 48 kHz streams by parity, resampled in one step")
    ap.add_argument("--math", choices=["tc16", "tc", "fp32", "fft"], default=None,
                    help="arithmetic: tc16 (v5 default) = tcgen05 tensor cores, FP16 2-way split with per-stream scaling; tc = BF16 "
                         "3-way split; fp32 = packed FP32 FMA; fft (v4 default) = FP64 FFT STFT + tensor-core basis correction")
    ap.add_argument("--model", choices=["v5", "v4"], default="v5", help="v5 = headline (configs[1]); v4 = configs[2]")
    ap.add_argument("--src-rate", type=int, default=16000, choices=[8000, 16000, 24000, 48000],
                    help="source rate of the synthetic streams; != 16000 adds the GPU resampler (configs[2..3])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline configuration returned (rank 0's streams) as "
                         "DIR/<name>.npy; the inputs depend only on the arguments, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed: not with --impl reference")
    if args.math is None:
        args.math = "tc16" if args.model == "v5" else "fft"
    args.warmup = max(args.warmup, 3)
    _protect_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
