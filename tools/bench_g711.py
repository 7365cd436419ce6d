#!/usr/bin/env python
"""bench_g711.py -- what G.711 input costs against int16 PCM on the same audio.

4,096 streams at 8 kHz (telephony), one-frame steps (256 source samples = 32 ms per stream and step), v5 in its default
math mode.  The same seeded audio is stepped as mu-law codes (CVAD_PCM_ULAW, 1 byte per sample, decoded by the input stage
before the resampler) and as int16 (CVAD_PCM_S16_32768 of the same linear values, 2 bytes per sample, converted inside
the resampler's loader).  The two legs alternate, `--rounds` times each; the median is reported.

  device   cvad_step_device over a pool of device-resident input steps larger than the B200's 126 MB L2 (every step reads
           its audio from HBM).  int16 one-frame steps run chained (kernel after kernel, no memset or event record);
           G.711 steps run unchained: memsets, the decode kernel, the resampler and the model kernel.
  e2e      StreamEngine.submit / collect from pinned host buffers, four steps in flight (H2D + kernels + D2H).
  decode   the decode kernel's own time (downmix_kernel with one channel), from a separate torch.profiler run.

Prints one JSON line, with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "cutter-vad_b200"))
sys.path.insert(0, str(ROOT / "tests"))

N, RATE, W = 4096, 8000, 256
L2_BYTES = 126 << 20


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return out[0].strip(), float(out[1])


def make_audio(pool_steps):
    """[pool_steps][N][W] mu-law codes and the int16 linear values they decode to (voice-like, seeded)."""
    from conftest import synth_streams
    from real_time_vad.utils.audio import G711_LINEAR
    from scipy import signal
    base = synth_streams(64, 2 * W * pool_steps + 64, seed=3)
    x = signal.resample_poly(base, 1, 2, axis=1)[:, :W * pool_steps].astype(np.float32)
    t = G711_LINEAR["ulaw"].astype(np.int64)
    order = np.argsort(t, kind="stable")
    codes64 = order[np.clip(np.searchsorted(t[order], np.round(x * 32767.0)), 0, 255)].astype(np.uint8)
    codes = np.empty((pool_steps, N, W), np.uint8)
    rng = np.random.default_rng(0)
    for j in range(pool_steps):
        codes[j] = codes64[rng.integers(0, 64, N), j * W:(j + 1) * W]
    return codes, G711_LINEAR["ulaw"][codes]


def device_leg(eng, pool, fmt, steps):
    import torch
    from real_time_vad.engine import capi
    cu = "cuda:0"
    probs = torch.empty((N, 1), dtype=torch.float32, device=cu)
    flags = torch.empty((N, 1), dtype=torch.uint8, device=cu)
    events = torch.empty((2 * N * 24,), dtype=torch.uint8, device=cu)
    nev = torch.zeros((1,), dtype=torch.int32, device=cu)
    args = []
    for j in range(pool.shape[0]):
        a = capi.StepArgs()
        a.n_streams = N
        a.audio = pool[j].data_ptr()
        a.pcm_format = fmt
        a.stream_stride = W
        a.max_frames = 1
        a.frame_len = a.hop = W
        a.src_rate = RATE
        a.probs_out = probs.data_ptr()
        a.flags_out = flags.data_ptr()
        a.events_out = events.data_ptr()
        a.max_events = 2 * N
        a.n_events_out = nev.data_ptr()
        args.append(a)
    eng.reset()
    for j in range(len(args)):                      # warm-up: every pool entry once
        eng.step_device(args[j])
    eng.sync()
    t0 = time.perf_counter()
    for j in range(steps):
        eng.step_device(args[j % len(args)])
    eng.sync()
    return 1e3 * (time.perf_counter() - t0) / steps


def e2e_leg(eng, pinned, fmt, steps):
    eng.reset()
    P = len(pinned)
    inflight = []

    def run(k):
        for j in range(k):
            if len(inflight) == 4:
                inflight.pop(0).collect()
            inflight.append(eng.submit(pinned[j % P], pcm_format=fmt, src_rate=RATE, max_frames=1))
        while inflight:
            inflight.pop(0).collect()

    run(min(P, 32))
    t0 = time.perf_counter()
    run(steps)
    return 1e3 * (time.perf_counter() - t0) / steps


def decode_kernel_us(eng, pool, steps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        device_leg(eng, pool, 3, steps)
        torch.cuda.synchronize()
    times = [e for e in prof.key_averages() if "downmix_kernel" in e.key]
    if not times:
        raise RuntimeError("the profiler recorded no downmix_kernel")
    ev = times[0]
    total_us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total")
    return total_us / ev.count, ev.count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000, help="timed steps per leg and round")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    from real_time_vad.engine import capi
    from real_time_vad.engine.stream_engine import StreamEngine
    name, power = card()
    pool_steps = -(-L2_BYTES * 5 // 4 // (N * W))      # the mu-law pool alone is 1.25 x L2
    codes, lin = make_audio(pool_steps)
    cu = "cuda:0"
    dev_pool = {capi.PCM_ULAW: torch.from_numpy(codes).to(cu),
                capi.PCM_S16_32768: torch.from_numpy(lin.astype(np.int16)).to(cu)}
    e2e_n = 64
    pinned = {capi.PCM_ULAW: [torch.from_numpy(codes[j]).pin_memory().numpy() for j in range(e2e_n)],
              capi.PCM_S16_32768: [torch.from_numpy(lin[j].astype(np.int16)).pin_memory().numpy() for j in range(e2e_n)]}
    eng = StreamEngine("v5", max_streams=N)
    legs = {"device": {}, "e2e": {}}
    for r in range(args.rounds):
        order = (capi.PCM_ULAW, capi.PCM_S16_32768) if r % 2 == 0 else (capi.PCM_S16_32768, capi.PCM_ULAW)
        for fmt in order:
            legs["device"].setdefault(fmt, []).append(device_leg(eng, dev_pool[fmt], fmt, args.steps))
            legs["e2e"].setdefault(fmt, []).append(e2e_leg(eng, pinned[fmt], fmt, args.steps // 4))
    dec_us, dec_n = decode_kernel_us(eng, dev_pool[capi.PCM_ULAW], 200)
    out = {"bench": "g711", "card": name, "power_limit_w": power, "streams": N, "src_rate": RATE,
           "frames_per_step": 1, "math": eng.math, "rounds": args.rounds,
           "device_pool_mb": {"ulaw": round(dev_pool[capi.PCM_ULAW].numel() / 2 ** 20, 1),
                              "s16": round(dev_pool[capi.PCM_S16_32768].numel() * 2 / 2 ** 20, 1)}}
    for leg, res in legs.items():
        u, s = statistics.median(res[capi.PCM_ULAW]), statistics.median(res[capi.PCM_S16_32768])
        out[leg] = {"ulaw_ms_per_step": round(u, 4), "s16_ms_per_step": round(s, 4),
                    "ulaw_over_s16": round(u / s, 3),
                    "ulaw_audio_s_per_s": round(N * W / RATE / (u / 1e3)), "s16_audio_s_per_s": round(N * W / RATE / (s / 1e3)),
                    "ulaw_runs": [round(x, 4) for x in res[capi.PCM_ULAW]],
                    "s16_runs": [round(x, 4) for x in res[capi.PCM_S16_32768]]}
    out["decode_kernel_us"] = round(dec_us, 2)
    out["decode_kernel_launches"] = dec_n
    out["decode_bytes_per_step"] = N * W * (1 + 4)        # codes in, float32 out
    out["decode_gbs"] = round(N * W * 5 / (dec_us * 1e-6) / 1e9, 1)
    eng.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
