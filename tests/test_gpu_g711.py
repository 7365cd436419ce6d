"""GPU: G.711 mu-law / A-law input (CVAD_PCM_ULAW / CVAD_PCM_ALAW), decoded by the input stage (downmix_kernel) before the
resamplers and the model kernels.  Everything after the decode sees float32, so every result is held bit for bit against
the same step on the decoded float32 audio and on PCM_S16_32768 of the linear values: the decode stage's own output
(debug_input), probabilities, flags, events and engine records of every model and math mode, host, pipelined and device
steps, and two BatchedVADManagers fed the same calls as 160-byte packets and as decoded float32."""
import zlib

import numpy as np
import pytest
from scipy import signal

from conftest import synth_streams

pytestmark = pytest.mark.gpu

LAWS = {"ulaw": 3, "alaw": 4}
RATES = (8000, 16000, 24000, 48000)


def _table(law):
    from real_time_vad.utils.audio import G711_LINEAR
    return G711_LINEAR[law]


def _encode(x, law):
    """float32 audio -> the G.711 codes whose linear value is nearest above (any code mapping is fine: the tests compare
    formats on the decoded values)."""
    t = _table(law).astype(np.int64)
    order = np.argsort(t, kind="stable")
    idx = np.clip(np.searchsorted(t[order], np.round(np.asarray(x) * 32767.0)), 0, 255)
    return order[idx].astype(np.uint8)


def _formats(codes, law):
    """(G.711 codes, decoded float32, linear int16) of the same audio, with their pcm_format codes."""
    from real_time_vad.engine import capi
    lin = _table(law)[codes]
    return [(codes, LAWS[law]), ((lin.astype(np.float32) / np.float32(32768.0)), capi.PCM_F32),
            (lin.astype(np.int16), capi.PCM_S16_32768)]


def _voice(n, rate, n_samples, seed):
    """synth_streams' voice-like audio at `rate` (made at 16 kHz and resampled polyphase)."""
    if rate == 16000:
        return synth_streams(n, n_samples, seed=seed)
    base = synth_streams(n, n_samples * 16000 // rate + 64, seed=seed)
    g = np.gcd(rate, 16000)
    return signal.resample_poly(base, rate // g, 16000 // g, axis=1)[:, :n_samples].astype(np.float32)


@pytest.fixture(scope="module")
def engines():
    from real_time_vad.engine.stream_engine import StreamEngine
    made = {}

    def get(model):
        if model not in made:
            made[model] = [StreamEngine(model, max_streams=512) for _ in range(3)]
        return made[model]

    yield get
    for trio in made.values():
        for e in trio:
            e.close()


# --------------------------------------------------------------------------------------------------- the decode stage
def _u32(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


@pytest.mark.parametrize("law", ["ulaw", "alaw"])
def test_decode_of_every_code_at_every_position_is_the_table(engine_factory, law):
    eng = engine_factory(256)
    codes = ((np.arange(256)[:, None] + np.arange(1536)[None, :]) % 256).astype(np.uint8)    # every code in every column
    want = _table(law)[codes].astype(np.float32) / np.float32(32768.0)
    for frame_len, hop in ((512, 512), (480, 480), (512, 256)):
        got = eng.debug_input(codes, pcm_format=LAWS[law], frame_len=frame_len, hop=hop)
        span = got.shape[1]
        assert span == ((1536 - frame_len) // hop) * hop + frame_len
        assert np.array_equal(_u32(got), _u32(want[:, :span])), (frame_len, hop)


@pytest.mark.parametrize("channels", [1, 2, 3, 8])
@pytest.mark.parametrize("rate", [8000, 16000, 24000, 48000, "mixed"])
def test_decode_then_downmix_and_resample_equals_the_float32_input(engine_factory, channels, rate):
    """G.711 through every input stage equals the decoded float32 through the same stages, bit for bit; frames beyond a
    stream's n_frames stay NaN in resampled and mixed-rate output."""
    law = "ulaw" if channels % 2 else "alaw"
    eng = engine_factory(96)
    rng = np.random.default_rng(channels * 7 + (0 if rate == "mixed" else rate))
    n, T = 70, 3
    kw = {}
    if rate == "mixed":
        rates = np.array([RATES[k % 4] for k in range(n)], np.int32)
        W = T * 1536
        kw = dict(src_rates=rates, max_frames=T)
    else:
        W = T * rate * 512 // 16000
        kw = dict(src_rate=rate)
    resampled = rate != 16000
    if resampled:
        kw["n_frames"] = rng.integers(0, T + 1, n).astype(np.int32)
        kw["max_frames"] = T
    codes = rng.integers(0, 256, (n, W, channels) if channels > 1 else (n, W), dtype=np.uint8)
    # (16 kHz mono float32 has no input stage: there the decode alone is held against the table)
    todo = _formats(codes, law)[:1 if channels == 1 and rate == 16000 else 2]
    outs = [eng.debug_input(x, pcm_format=fmt, **kw) for x, fmt in todo]
    assert np.array_equal(_u32(outs[0]), _u32(outs[-1]))
    if resampled:
        for i in range(n):
            assert np.isnan(outs[0][i, kw["n_frames"][i] * 512:]).all()
            assert not np.isnan(outs[0][i, :kw["n_frames"][i] * 512]).any()
    if channels == 1 and rate == 16000:
        assert np.array_equal(_u32(outs[0]), _u32(_table(law)[codes].astype(np.float32) / np.float32(32768.0)))


# --------------------------------------------------------------------------------------------------- engine steps
def _step_args(rate, T, n):
    """-> (samples per stream and step, advance per step, step kwargs)"""
    kw = {}
    if rate == "mixed":
        kw["src_rates"] = np.array([RATES[k % 4] for k in range(n)], np.int32)
        kw["max_frames"] = T
        return T * 1536, None, kw
    if rate != 16000:
        kw["src_rate"] = rate
        kw["max_frames"] = T
        W = T * rate * 512 // 16000
        return W, W, kw
    hop = 256 if T > 2 else 512
    kw.update(frame_len=512, hop=hop, max_frames=T)
    return (T - 1) * hop + 512, T * hop, kw


CASES = [("v5", "tc16", "ulaw", 16000, 1, "step"), ("v5", "tc16", "alaw", 16000, 6, "submit"),
         ("v5", "tc16", "ulaw", 8000, 1, "submit"), ("v5", "tc16", "alaw", 24000, 3, "step"),
         ("v5", "tc16", "ulaw", 48000, 2, "step"), ("v5", "tc16", "alaw", "mixed", 3, "submit"),
         ("v5", "tc", "ulaw", 16000, 4, "step"), ("v5", "tc", "alaw", "mixed", 1, "step"),
         ("v5", "fp32", "alaw", 8000, 4, "step"), ("v5", "fp32", "ulaw", 16000, 1, "submit"),
         ("v4", "fft", "ulaw", 16000, 3, "step"), ("v4", "fft", "alaw", 8000, 1, "submit"),
         ("v4", "tc", "alaw", 8000, 2, "submit"), ("v4", "fp32", "ulaw", "mixed", 2, "step"),
         ("v4_8k", None, "alaw", 16000, 4, "step"), ("v4_8k", None, "ulaw", 16000, 1, "submit")]


@pytest.mark.parametrize("model,math,law,rate,T,mode", CASES)
def test_g711_steps_equal_float32_and_int16_steps(engines, model, math, law, rate, T, mode):
    """The same streams stepped from G.711 codes, from the decoded float32 and from the linear int16 on three engines:
    probabilities, flags, events and the engines' records are identical.  Ragged n_frames and a slot list throughout."""
    trio = engines(model)
    rng = np.random.default_rng(zlib.crc32(repr((model, math, law, rate, T)).encode()))
    n = 300
    slots = rng.permutation(512)[:n].astype(np.int32)
    W, adv, kw = _step_args(rate, T, n)
    steps = max(10, 48 // T)
    if adv is None:
        # mixed rates: stream k advances by T chunks of its own rate per step
        per = [T * r * 512 // 16000 for r in kw["src_rates"]]
        src = [_voice(1, int(r), per[k] * steps, seed=k)[0] for k, r in enumerate(kw["src_rates"])]
    else:
        src = _voice(n, rate if rate != "mixed" else 16000, adv * (steps - 1) + W, seed=5)
    for e in trio:
        if math is not None:
            e.set_math(math)
        e.reset()
        e.configure(vad_start_probability=0.5, vad_end_probability=0.35, voice_start_frame_count=2,
                    voice_end_frame_count=3, enable_denoising=True)
    n_events = 0
    pending = []

    def check(results):
        nonlocal n_events
        (g, f, s) = results
        for other in (f, s):
            assert g.probs.tobytes() == other.probs.tobytes()
            assert np.array_equal(g.flags, other.flags) and np.array_equal(g.status, other.status)
            assert g.events == other.events
        assert not g.status.any()
        n_events += len(g.events)

    for j in range(steps):
        if adv is None:
            x = np.zeros((n, W), np.float32)
            for k in range(n):
                x[k, :per[k]] = src[k][j * per[k]:(j + 1) * per[k]]
        else:
            x = np.ascontiguousarray(src[:, j * adv:j * adv + W])
        codes = _encode(x, law)
        nfr = rng.integers(0, T + 1, n).astype(np.int32) if j % 3 == 1 else None      # ragged every third step
        calls = [(e, fmt_x, fmt) for e, (fmt_x, fmt) in zip(trio, _formats(codes, law))]
        if mode == "submit":
            pending.append([e.submit(fx, slots=slots, n_frames=nfr, pcm_format=fmt, **kw) for e, fx, fmt in calls])
            if len(pending) == 4 or j == steps - 1:
                while pending:
                    check([p.collect() for p in pending.pop(0)])
        else:
            check([e.step(fx, slots=slots, n_frames=nfr, pcm_format=fmt, **kw) for e, fx, fmt in calls])
    recs = [e.export_states(slots) for e in trio]
    assert recs[0].tobytes() == recs[1].tobytes() == recs[2].tobytes()
    assert recs[0]["frames_done"].max() > 0
    assert n_events > 0


@pytest.mark.parametrize("n,rate,math,law", [(4096, 8000, "tc16", "ulaw"), (300, 16000, "tc16", "alaw"),
                                             (300, 16000, "tc", "ulaw"), (257, "mixed", "tc16", "alaw"),
                                             (300, 8000, "fp32", "alaw")])
def test_device_steps_equal_host_steps_on_the_decoded_audio(engine_factory, n, rate, math, law):
    """cvad_step_device on G.711 device buffers (one-frame steps, unchained: the decode stage runs first) equals
    cvad_step on the decoded float32 on a second engine, step by step."""
    import torch
    from real_time_vad.engine import capi
    T = 16
    dev, host = engine_factory(n, math=math), engine_factory(n, math=math)
    for e in (dev, host):
        e.reset()
        e.configure(vad_start_probability=0.5, vad_end_probability=0.35, voice_start_frame_count=2,
                    voice_end_frame_count=3, enable_denoising=True)
    if rate == "mixed":
        rates = np.array([RATES[k % 4] for k in range(n)], np.int32)
        W = 1536
        src = np.zeros((n, W * T), np.float32)
        for r in RATES:
            idx = np.flatnonzero(rates == r)
            w = r * 512 // 16000
            v = _voice(idx.size, r, w * T, seed=r)
            for q, k in enumerate(idx):
                for j in range(T):
                    src[k, j * W:j * W + w] = v[q, j * w:(j + 1) * w]
        rate_kw = dict(src_rates=rates)
    else:
        W = rate * 512 // 16000
        src = _voice(n, rate, W * T, seed=9)
        rate_kw = dict(src_rate=rate)
    codes = _encode(src, law)
    decoded = _table(law)[codes].astype(np.float32) / np.float32(32768.0)
    cu = "cuda:0"
    frames = [torch.from_numpy(np.ascontiguousarray(codes[:, W * j:W * (j + 1)])).to(cu) for j in range(T)]
    rates_d = torch.from_numpy(rate_kw["src_rates"]).to(cu) if rate == "mixed" else None
    probs_d = [torch.full((n, 1), -1.0, dtype=torch.float32, device=cu) for _ in range(T)]
    flags_d = [torch.full((n, 1), 255, dtype=torch.uint8, device=cu) for _ in range(T)]
    events_d = [torch.zeros((2 * n * 24,), dtype=torch.uint8, device=cu) for _ in range(T)]
    nev_d = [torch.full((1,), 12345, dtype=torch.int32, device=cu) for _ in range(T)]
    torch.cuda.synchronize()
    for j in range(T):
        a = capi.StepArgs()
        a.n_streams = n
        a.audio = frames[j].data_ptr()
        a.pcm_format = LAWS[law]
        a.stream_stride = W
        a.max_frames = 1
        a.frame_len = a.hop = 512 if rate == "mixed" else W
        a.src_rate = 16000 if rate == "mixed" else rate
        if rates_d is not None:
            a.src_rates = rates_d.data_ptr()
        a.probs_out = probs_d[j].data_ptr()
        a.flags_out = flags_d[j].data_ptr()
        a.events_out = events_d[j].data_ptr()
        a.max_events = 2 * n
        a.n_events_out = nev_d[j].data_ptr()
        dev.step_device(a)
    dev.sync()
    n_events = 0
    for j in range(T):
        r = host.step(np.ascontiguousarray(decoded[:, W * j:W * (j + 1)]), max_frames=1, **rate_kw)
        assert probs_d[j].cpu().numpy().tobytes() == r.probs.tobytes(), j
        assert np.array_equal(flags_d[j].cpu().numpy(), r.flags), j
        k = int(nev_d[j].cpu()[0])
        assert k == len(r.events), j
        rec = events_d[j].cpu().numpy().view(np.int64)[:3 * k]
        got = sorted((int(q[0]), int(q[1]), int(q[2]), int(q[3]), int(f))
                     for q, f in zip(rec.view(np.int32).reshape(k, 6), rec.reshape(k, 3)[:, 2]))
        assert got == sorted(r.events), j
        n_events += k
    assert dev.export_states(None).tobytes() == host.export_states(None).tobytes()
    assert n_events > 0


def test_a_wrong_dtype_is_refused_and_changes_nothing(engine_factory):
    from real_time_vad.core.exceptions import AudioProcessingError
    from real_time_vad.engine import capi
    from real_time_vad.engine.stream_engine import EngineError
    from real_time_vad import BatchedVADManager
    eng = engine_factory(8)
    eng.reset()
    codes = _encode(synth_streams(4, 1024, seed=1), "ulaw")
    eng.step(codes, slots=[0, 1, 2, 3], pcm_format=capi.PCM_ULAW)
    before = eng.export_states(None)
    for bad in (codes.astype(np.float32), codes.astype(np.int16), codes.astype(np.float32) / 255.0):
        for fmt in (capi.PCM_ULAW, capi.PCM_ALAW):
            with pytest.raises(EngineError) as ei:
                eng.step(bad, slots=[0, 1, 2, 3], pcm_format=fmt)
            assert ei.value.code == capi.E_INVALID
            with pytest.raises(EngineError):
                eng.debug_input(bad, pcm_format=fmt)
    assert eng.export_states(None).tobytes() == before.tobytes()
    mgr = BatchedVADManager(max_streams=4, source_rate=8000, pcm_format=capi.PCM_ALAW)
    sid = mgr.open_stream(_cfg(8000))
    with pytest.raises(AudioProcessingError):
        mgr.push(sid, np.zeros((160, 2), np.uint8))
    with pytest.raises(AudioProcessingError):
        mgr.push(sid, np.zeros(160, np.float32))
    with pytest.raises(AudioProcessingError):
        mgr.push_bytes(sid, b"")
    assert mgr.pending(sid) == 0
    mgr.push(sid, bytes(160))
    mgr.push(sid, np.zeros(160, np.uint8))
    assert mgr.pending(sid) == 320
    mgr.close()


# --------------------------------------------------------------------------------------------------- the manager
def _cfg(rate):
    from real_time_vad import VADConfig
    from real_time_vad.core.config import SampleRate
    return VADConfig(sample_rate=SampleRate(int(rate)), vad_start_probability=0.5, vad_end_probability=0.35,
                     voice_start_frame_count=2, voice_end_frame_count=3)


def _recorder():
    log = {"start": 0, "wav": [], "cont": []}
    return log, dict(on_voice_start=lambda: log.__setitem__("start", log["start"] + 1), on_voice_end=log["wav"].append,
                     on_voice_continue=log["cont"].append)


def _callbacks(k, cbs):
    # three payload modes: events only, segments, segments + continue frames
    return [dict(on_voice_start=cbs["on_voice_start"]),
            dict(on_voice_start=cbs["on_voice_start"], on_voice_end=cbs["on_voice_end"]), cbs][k % 3]


def _telephony_audio(n, ticks, rates, law):
    codes = np.zeros((n, 160 * ticks), np.uint8)
    for r in set(rates):
        idx = [k for k in range(n) if rates[k] == r]
        codes[idx] = _encode(_voice(len(idx), r, 160 * ticks, seed=r), law)
    return codes, _table(law)[codes].astype(np.float32) / np.float32(32768.0)


@pytest.mark.parametrize("source_rate,law", [(8000, "ulaw"), (16000, "alaw"), (None, "ulaw")])
def test_g711_manager_equals_a_float32_manager_fed_the_decoded_audio(source_rate, law):
    from real_time_vad import BatchedVADManager
    from real_time_vad.engine import capi
    n, ticks = 1000, 200
    rates = [source_rate or RATES[k % 4] for k in range(n)]
    codes, decoded = _telephony_audio(n, ticks, rates, law)
    mg = BatchedVADManager(max_streams=1024, source_rate=source_rate, pcm_format=LAWS[law])
    mf = BatchedVADManager(max_streams=1024, source_rate=source_rate, pcm_format=capi.PCM_F32)
    logs = {}
    ids = {}
    for name, m in (("g", mg), ("f", mf)):
        logs[name] = [_recorder() for _ in range(n)]
        ids[name] = [m.open_stream(_cfg(rates[k]), **_callbacks(k, logs[name][k][1])) for k in range(n)]
    n_frames = 0
    for t in range(ticks):
        for k in range(n):
            mg.push_bytes(ids["g"][k], codes[k, 160 * t:160 * (t + 1)].tobytes())
            mf.push_bytes(ids["f"][k], decoded[k, 160 * t:160 * (t + 1)].tobytes())
        og, of = mg.step(), mf.step()
        assert og.events == of.events, t
        assert np.array_equal(og.stream_ids, of.stream_ids) and np.array_equal(og.counts, of.counts)
        assert og.probs.tobytes() == of.probs.tobytes() and np.array_equal(og.flags, of.flags)
        n_frames += og.frames
    mg.close()
    mf.close()
    for k in range(n):
        a, b = logs["g"][k][0], logs["f"][k][0]
        assert a == b, k
    tot = {key: sum(len(logs["g"][k][0][key]) for k in range(n)) for key in ("wav", "cont")}
    assert n_frames > n * 50 and tot["wav"] > 20 and tot["cont"] > 200, (n_frames, tot)


@pytest.mark.parametrize("source_rate,law", [(8000, "alaw"), (16000, "ulaw")])
def test_g711_streams_move_mid_voice_and_continue_bit_for_bit(source_rate, law):
    from real_time_vad import BatchedVADManager, StreamSnapshot
    n, ticks = 48, 240
    rates = [source_rate] * n
    codes, _ = _telephony_audio(n, ticks, rates, law)
    fmt = LAWS[law]

    def run(mgr, ids, t0, t1, active=None):
        for t in range(t0, t1):
            for k in range(n):
                mgr.push_bytes(ids[k], codes[k, 160 * t:160 * (t + 1)].tobytes())
            mgr.step()
            if active is not None:
                active.append(sum(mgr.is_voice_active(ids[k]) for k in range(n)))

    ref = BatchedVADManager(max_streams=n, source_rate=source_rate, pcm_format=fmt)
    ref_logs = [_recorder() for _ in range(n)]
    rid = [ref.open_stream(_cfg(source_rate), **ref_logs[k][1]) for k in range(n)]
    active = []
    run(ref, rid, 0, ticks, active)
    ref.close()
    cut = next(t for t in range(20, ticks - 20) if active[t] >= 3)

    src = BatchedVADManager(max_streams=n, source_rate=source_rate, pcm_format=fmt)
    logs = [_recorder() for _ in range(n)]
    sid = [src.open_stream(_cfg(source_rate), **logs[k][1]) for k in range(n)]
    run(src, sid, 0, cut + 1)
    for k in range(n):                                     # half a packet pending at the cut
        src.push_bytes(sid[k], codes[k, 160 * (cut + 1):160 * (cut + 1) + 80].tobytes())
    assert sum(src.is_voice_active(s) for s in sid) >= 3
    snap = StreamSnapshot.from_bytes(src.snapshot_streams().to_bytes())
    src.close()
    dst = BatchedVADManager(max_streams=2 * n, source_rate=source_rate, pcm_format=fmt)
    dst.open_stream(_cfg(source_rate))                      # ids move
    moved = dst.restore_streams(snap, callbacks={sid[k]: logs[k][1] for k in range(n)})
    did = [moved[s] for s in sid]
    for k in range(n):
        dst.push_bytes(did[k], codes[k, 160 * (cut + 1) + 80:160 * (cut + 2)].tobytes())
    dst.step()
    run(dst, did, cut + 2, ticks)
    dst.close()
    for k in range(n):
        assert logs[k][0] == ref_logs[k][0], k
    assert sum(len(lg["cont"]) for lg, _ in ref_logs) > 100
