"""GPU parity at BASELINE.json's full size: configs[1] = 4,096 concurrent 16 kHz streams, one frame per step.

At this size the oracle still finishes in seconds (the C restatement runs its streams on every host thread), so
every probability of every stream is checked against it; on top of that the size-independent properties the path
offers: replicated streams give bit-identical results wherever they sit in the batch, the one-frame-per-step form
(fused kernel) and the many-frames-per-call form (two kernels) agree, and the event list equals the oracle's state
machine run on the oracle's probabilities."""
import numpy as np
import pytest

from conftest import synth_streams

pytestmark = pytest.mark.gpu
TOL = 1e-4
N, DISTINCT, T = 4096, 256, 24


@pytest.fixture(scope="module")
def workload(ref_v5):
    base = synth_streams(DISTINCT, 512 * T, seed=91)
    audio = np.tile(base, (N // DISTINCT, 1))              # stream s carries base[s % DISTINCT]
    want, _, _ = ref_v5.run(base, T, denoise=True)
    return base, audio, want


@pytest.mark.parametrize("math", ["tc", "fp32", "tc16"])
def test_4096_streams_one_frame_per_step(engine_factory, ref_lib, workload, math):
    from vad_oracle import sm_run_c
    base, audio, want = workload
    eng = engine_factory(N, math=math)
    eng.configure(enable_denoising=True, vad_start_probability=0.5, vad_end_probability=0.35,
                  voice_start_frame_count=3, voice_end_frame_count=4)
    got = np.zeros((N, T), np.float32)
    flags = np.zeros((N, T), np.uint8)
    events = []
    for j in range(T):
        r = eng.step(audio[:, j * 512:(j + 1) * 512])
        assert r.status.sum() == 0
        got[:, j] = r.probs[:, 0]
        flags[:, j] = r.flags[:, 0]
        events += [(k, j, kind) for (k, slot, f, kind, sf) in r.events]
    # every stream against the oracle
    err = np.abs(got.reshape(N // DISTINCT, DISTINCT, T) - want[None]).max()
    assert err <= TOL, err
    # replicas are bit-identical wherever they sit in the batch (tile, lane, SM)
    rep = got.reshape(N // DISTINCT, DISTINCT, T)
    assert np.array_equal(rep, np.broadcast_to(rep[0], rep.shape))
    # events == the oracle's state machine on the oracle's probabilities
    n_ev = 0
    for s in range(DISTINCT):
        fl, _ = sm_run_c(ref_lib, want[s], 0.5, 0.35, 0.8, 0.95, 3, 4)
        assert np.array_equal(fl & 7, flags[s] & 7), s
        n_ev += int(((fl & 1) != 0).sum() + ((fl & 2) != 0).sum())
    assert n_ev > 50 and len(events) == n_ev * (N // DISTINCT)
    assert eng.get_state(N - 1)[3] == T


def test_4096_streams_one_call_equals_one_frame_steps(engine_factory, workload):
    """The two-kernel form (all frames in one call) against the oracle, and against the fused one-frame form."""
    base, audio, want = workload
    eng = engine_factory(N, math="tc")
    eng.configure(enable_denoising=True)
    r = eng.step(audio)
    assert r.probs.shape == (N, T)
    assert np.abs(r.probs.reshape(N // DISTINCT, DISTINCT, T) - want[None]).max() <= TOL
    eng.reset()
    steps = np.stack([eng.step(audio[:, j * 512:(j + 1) * 512]).probs[:, 0] for j in range(T)], axis=1)
    assert np.abs(steps - r.probs).max() <= 2e-5            # same arithmetic, different accumulation grouping of the gates


# ---------------------------------------------------------------------------------------------------------------
# Parity at the sizes bench.py measures, and over time
# ---------------------------------------------------------------------------------------------------------------

def _flags_match_up_to_ties(ref_lib, want, flags, cfg, tie):
    """flags [n][T] of the engine vs the oracle's state machine on the oracle's probabilities `want`; a stream that has
    a frame within `tie` of a threshold may legitimately differ and is skipped.  -> (compared, skipped, events)"""
    from vad_oracle import sm_run_c
    sp, ep, ns, ne = cfg
    compared = skipped = n_ev = 0
    for s in range(want.shape[0]):
        if (np.abs(want[s] - sp) <= tie).any() or (np.abs(want[s] - ep) <= tie).any():
            skipped += 1
            continue
        fl, _ = sm_run_c(ref_lib, want[s], sp, ep, 0.8, 0.95, ns, ne)
        assert np.array_equal(fl & 7, flags[s] & 7), s
        n_ev += int(((fl & 3) != 0).sum())
        compared += 1
    return compared, skipped, n_ev


def test_4096_streams_2000_chained_steps_no_drift(engine_factory, ref_v5, ref_lib):
    """BASELINE.json configs[1] exactly as bench.py's `value` leg runs it -- 4,096 streams, one frame per step, FP16-split
    default build, cvad_step_device, steps chained kernel to kernel -- for 2,000 consecutive steps (64 s of audio per
    stream, 512,000 distinct stateful frames), every probability of every step checked against the float64 evaluation
    (oracle/torch_reference.py in float64, itself pinned against the interpreter).

    Why float64 and not the FP32 oracle: over this many stateful frames the LSTM passes through a few moments that
    amplify float32 rounding ~1000x, and there NO float32 executor holds 1e-4: the C oracle is up to 3.7e-4 from
    float64 and PyTorch's float32 kernels 3.1e-4, both on ~10 frames, and the two are 6.8e-4 apart.  The deviations do
    not persist and do not grow.  Measured on B200 (tools/dev/drift_dump.py): the engine's FP32-FMA build behaves like
    the CPU executors (12 frames > 1e-4, max 5.3e-4); the tensor-core builds are ~3x noisier at those moments (28
    frames, max 7.1e-4) because tcgen05 accumulates in TMEM with truncation, a bias of half an ulp per MMA.

    Asserted, with "ill-conditioned" = a float32 CPU executor is >= 1e-5 from float64 on that frame (0.07 % of the frames):
      * every well-conditioned frame within 1e-4 -- LSTM-state drift of the 22-bit operand split would show here;
      * ill-conditioned frames within 3x the worst float32-CPU deviation (and 1e-3), and the number of frames over 1e-4
        at most 5x what the float32 CPU executors need themselves;
      * no growth over time (last 500 steps vs the bar, 99.9th percentile);
      * replicas bit-identical for 2,000 steps; flags identical to the state machine on the float64 probabilities for every
        stream without a frame within its tolerance of a threshold, and to the state machine on the device's own
        probabilities for ALL streams; the device's event count equals its flags."""
    import torch
    from real_time_vad.engine import capi
    from torch_reference import TorchV5
    from vad_oracle import sm_flags, v5_named_weights
    from conftest import V5_ONNX
    n, distinct, T = 4096, 256, 2000
    base = synth_streams(distinct, 512 * T, seed=123)
    want, _, _ = ref_v5.run(base, T, denoise=True)
    named = v5_named_weights(str(V5_ONNX))
    t64 = TorchV5(named, torch.float64).run(base, T, denoise=True).astype(np.float64)
    t32 = TorchV5(named, torch.float32).run(base, T, denoise=True).astype(np.float64)
    dev_c, dev_t = np.abs(want - t64), np.abs(t32 - t64)
    fp32_dev = np.maximum(dev_c, dev_t)                                  # what float32 rounding does on this frame
    ill = fp32_dev >= 1e-5
    assert ill.mean() < 2e-3, f"{ill.sum()} ill-conditioned frames"
    cfg = (0.5, 0.35, 3, 4)
    eng = engine_factory(n, math="tc16")
    eng.reset()
    eng.configure(enable_denoising=True, vad_start_probability=cfg[0], vad_end_probability=cfg[1],
                  voice_start_frame_count=cfg[2], voice_end_frame_count=cfg[3])
    cu = "cuda:0"
    base_d = torch.from_numpy(base).to(cu)
    probs_d = torch.full((T, n), -1.0, dtype=torch.float32, device=cu)
    flags_d = torch.full((T, n), 255, dtype=torch.uint8, device=cu)
    nev_d = torch.zeros((T,), dtype=torch.int32, device=cu)
    ev_d = torch.zeros((T, n * 24), dtype=torch.uint8, device=cu)
    # the engine and the per-step gather of the 16 replicas share one torch stream, so that they are ordered.  Not torch's
    # default stream: its handle is 0, which set_stream takes as "the engine's own stream", unordered with the gather.
    stream = torch.cuda.Stream(device=cu)
    stream.wait_stream(torch.cuda.current_stream())
    eng.set_stream(stream.cuda_stream)
    try:
        with torch.cuda.stream(stream):
            bufs = [torch.empty((n, 512), dtype=torch.float32, device=cu) for _ in range(4)]
            for j in range(T):
                x = bufs[j % 4]
                x.view(n // distinct, distinct, 512).copy_(base_d[:, j * 512:(j + 1) * 512].unsqueeze(0).expand(n // distinct, -1, -1))
                a = capi.StepArgs()
                a.n_streams = n
                a.audio = x.data_ptr()
                a.pcm_format = capi.PCM_F32
                a.stream_stride = 512
                a.max_frames = 1
                a.frame_len = a.hop = 512
                a.src_rate = 16000
                a.probs_out = probs_d[j].data_ptr()
                a.flags_out = flags_d[j].data_ptr()
                a.events_out = ev_d[j].data_ptr()
                a.max_events = n
                a.n_events_out = nev_d[j:j + 1].data_ptr()
                eng.step_device(a)
        eng.sync()
        torch.cuda.synchronize()
    finally:
        eng.set_stream(0)
    got = probs_d.cpu().numpy().T.reshape(n // distinct, distinct, T)          # stream s carries base[s % distinct]
    flags = flags_d.cpu().numpy().T.reshape(n // distinct, distinct, T)
    assert np.array_equal(got, np.broadcast_to(got[0], got.shape))            # replicas: bit-identical for 2,000 steps
    assert np.array_equal(flags, np.broadcast_to(flags[0], flags.shape))
    err = np.abs(got[0].astype(np.float64) - t64)
    n_over = {"engine": int((err > TOL).sum()), "C oracle": int((dev_c > TOL).sum()), "torch f32": int((dev_t > TOL).sum())}
    print(f"\n512,000 stateful frames vs float64: frames over 1e-4 {n_over}; max |dp| engine {err.max():.2e}, C oracle {dev_c.max():.2e}, "
          f"torch f32 {dev_t.max():.2e}; well-conditioned frames ({100 * (1 - ill.mean()):.2f} %): engine max {err[~ill].max():.2e}; "
          f"engine 99.99th percentile {np.percentile(err, 99.99):.2e}, median {np.median(err):.1e}; by 500-step quarter "
          f"{[float(f'{err[:, q * 500:(q + 1) * 500][~ill[:, q * 500:(q + 1) * 500]].max():.2e}') for q in range(4)]}")
    assert err[~ill].max() <= TOL, f"well-conditioned frame off by {err[~ill].max():.2e}"
    assert err.max() <= min(1e-3, 3.0 * fp32_dev.max()), err.max()
    assert n_over["engine"] <= 5 * max(n_over["C oracle"], n_over["torch f32"], 4), n_over
    # no growth over time: the last 500 steps are no worse than the run as a whole
    last = err[:, -500:][~ill[:, -500:]]
    assert last.max() <= TOL and np.percentile(last, 99.9) <= 2e-5
    # flags against the state machine on the float64 probabilities
    tol = np.where(ill, np.maximum(TOL, 3.0 * fp32_dev.max()), TOL)
    compared = 0
    for s in range(distinct):
        near = (np.abs(t64[s] - cfg[0]) <= tol[s]) | (np.abs(t64[s] - cfg[1]) <= tol[s])
        if near.any():
            continue
        assert np.array_equal(sm_flags(t64[s], *cfg) & 7, flags[0, s] & 7), s
        compared += 1
    assert compared >= distinct * 0.6, compared
    # the device's state machine on its OWN probabilities, every stream (the reference's rule applied to what it computed)
    for s in range(distinct):
        assert np.array_equal(sm_flags(got[0, s], *cfg) & 7, flags[0, s] & 7), s
    nev = nev_d.cpu().numpy()
    assert int(nev.sum()) == int(((flags & 1) != 0).sum() + ((flags & 2) != 0).sum())


def test_8192_mixed_rate_streams_per_gpu_share_of_configs3(engine_factory, ref_v5, ref_lib):
    """BASELINE.json configs[3]'s per-GPU share as bench.py runs it: 8,192 streams, 24 / 48 kHz by stream parity, resampled
    on the GPU and stepped one frame per call, 24 steps: every probability against [scipy.signal.resample per chunk ->
    FP32 oracle] (1e-4), events against the oracle's state machine."""
    n, distinct, T = 8192, 128, 24
    rates = np.where(np.arange(n) & 1, 48000, 24000).astype(np.int32)
    from scipy import signal
    from vad_oracle import resample_chunks
    base16 = synth_streams(2 * distinct, 512 * T, seed=321)
    src, y = {}, {}
    for k, rate in enumerate((24000, 48000)):
        n_in = rate * 512 // 16000
        b = base16[k * distinct:(k + 1) * distinct]
        up = signal.resample(b, n_in * T, axis=1).astype(np.float32)
        up += (0.003 * np.random.default_rng(rate).standard_normal(up.shape)).astype(np.float32)
        src[rate] = up
        y[rate] = resample_chunks(up, rate)
    want = {rate: ref_v5.run(y[rate], T, denoise=True)[0] for rate in (24000, 48000)}
    cfg = (0.5, 0.35, 3, 4)
    eng = engine_factory(n, math="tc16")
    eng.reset()
    eng.configure(enable_denoising=True, vad_start_probability=cfg[0], vad_end_probability=cfg[1],
                  voice_start_frame_count=cfg[2], voice_end_frame_count=cfg[3])
    got = np.zeros((n, T), np.float32)
    flags = np.zeros((n, T), np.uint8)
    audio = np.zeros((n, 1536), np.float32)
    idx24, idx48 = np.nonzero(rates == 24000)[0], np.nonzero(rates == 48000)[0]
    for j in range(T):
        audio[idx24, :768] = np.tile(src[24000][:, j * 768:(j + 1) * 768], (len(idx24) // distinct, 1))
        audio[idx48, :] = np.tile(src[48000][:, j * 1536:(j + 1) * 1536], (len(idx48) // distinct, 1))
        r = eng.step(audio, src_rates=rates, max_frames=1)
        assert r.status.sum() == 0
        got[:, j] = r.probs[:, 0]
        flags[:, j] = r.flags[:, 0]
    for rate, idx in ((24000, idx24), (48000, idx48)):
        g = got[idx].reshape(-1, distinct, T)
        assert np.array_equal(g, np.broadcast_to(g[0], g.shape))
        assert np.abs(g[0] - want[rate]).max() <= TOL, rate
        compared, skipped, n_ev = _flags_match_up_to_ties(ref_lib, want[rate], flags[idx].reshape(-1, distinct, T)[0], cfg, tie=1e-4)
        assert compared >= distinct * 0.8 and n_ev > 20, (rate, compared, skipped, n_ev)


def test_16384_streams_v4_behind_the_8k_resampler_configs2(engine_factory, ref_v4):
    """BASELINE.json configs[2] at its size: the v4 model, 16,384 streams of 8 kHz input resampled on the GPU, one frame per
    step, 24 steps.  Anchor = the float64 evaluation (tests/test_gpu_resample.py explains why no FP32 executor can be):
    every probability within 1e-4, events identical on every stream without a threshold tie."""
    from conftest import V4_ONNX
    from scipy import signal
    from vad_oracle import Truth64, resample_chunks, sm_flags
    n, distinct, T = 16384, 128, 24
    base16 = synth_streams(distinct, 512 * T, seed=654)
    up = signal.resample(base16, 256 * T, axis=1).astype(np.float32)
    up += (0.003 * np.random.default_rng(2).standard_normal(up.shape)).astype(np.float32)
    truth = Truth64(V4_ONNX, "v4").run(resample_chunks(up, 8000, exact=True), T)
    cfg = (0.5, 0.35, 2, 3)
    eng = engine_factory(n, model_version="v4")
    assert eng.math == "fft"
    eng.reset()
    eng.configure(enable_denoising=False, vad_start_probability=cfg[0], vad_end_probability=cfg[1],
                  voice_start_frame_count=cfg[2], voice_end_frame_count=cfg[3])
    got = np.zeros((n, T), np.float32)
    flags = np.zeros((n, T), np.uint8)
    for j in range(T):
        r = eng.step(np.tile(up[:, j * 256:(j + 1) * 256], (n // distinct, 1)), src_rate=8000)
        got[:, j] = r.probs[:, 0]
        flags[:, j] = r.flags[:, 0]
    g = got.reshape(-1, distinct, T)
    assert np.array_equal(g, np.broadcast_to(g[0], g.shape))
    err = np.abs(g[0].astype(np.float64) - truth)
    assert err.max() <= TOL, err.max()
    fl = flags.reshape(-1, distinct, T)[0]
    compared = 0
    for s in range(distinct):
        if (np.abs(truth[s] - cfg[0]) <= 2e-6).any() or (np.abs(truth[s] - cfg[1]) <= 2e-6).any():
            continue
        assert np.array_equal(sm_flags(truth[s], *cfg) & 7, fl[s] & 7), s
        compared += 1
    assert compared >= distinct - 2
