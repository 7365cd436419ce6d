"""GPU: stream snapshots.  A stream exported from one engine (cvad_export_states) and imported into another
(cvad_import_states) -- other capacity, other slot, other device -- continues bit for bit as if it had never moved; the
same holds for a BatchedVADManager stream taken through snapshot_streams -> to_bytes -> from_bytes -> restore_streams
in a new manager, callbacks and their payloads included.  Refused imports and restores change nothing."""
import hashlib

import numpy as np
import pytest

from conftest import GOLDEN, synth_streams

pytestmark = pytest.mark.gpu

RATES = (8000, 16000, 24000, 48000)


def _engine(version, math, max_streams, device=0):
    from real_time_vad.engine.stream_engine import StreamEngine
    return StreamEngine(version, max_streams=max_streams, device=device, math=math)


def _configure_per_stream(eng, slots):
    """Per-stream thresholds: eight threshold sets spread over the streams."""
    slots = np.asarray(slots)
    for g in range(8):
        eng.configure(slots[g::8], vad_start_probability=0.35 + 0.03 * g, vad_end_probability=0.2 + 0.02 * g,
                      voice_start_frame_count=1 + g % 3, voice_end_frame_count=2 + g % 4, enable_denoising=g % 2 == 0)


def _run(eng, audio, kind, frame0, n_frames, slots=None):
    """n_frames frames of `audio` from frame0 on, as one-frame steps, 8-frame steps or 8-frame mixed-rate steps.
    -> probs [n, n_frames], flags [n, n_frames], events [(stream, frame since frame0, kind, stream_frame, slot)]."""
    n = audio.shape[0]
    probs, flags, events = [], [], []
    step = 1 if kind == "one" else 8
    t = 0
    while t < n_frames:
        m = min(step, n_frames - t)
        f0 = frame0 + t
        if kind == "mixed":
            rates = np.array([RATES[i % 4] for i in range(n)], np.int32)
            x = np.zeros((n, 1536 * m), np.float32)
            for i in range(n):
                w = rates[i] * 512 // 16000
                x[i, :w * m] = audio[i, w * f0:w * (f0 + m)]
            r = eng.step(x, slots=slots, src_rates=rates, max_frames=m)
        else:
            r = eng.step(np.ascontiguousarray(audio[:, 512 * f0:512 * (f0 + m)]), slots=slots)
        probs.append(r.probs.copy())
        flags.append(r.flags.copy())
        events += [(s, t + j, k, sf, sl) for (s, sl, j, k, sf) in r.events]
        t += m
    return np.concatenate(probs, axis=1), np.concatenate(flags, axis=1), events


def _streams_audio(kind, n, frames, seed):
    """Rows long enough for `frames` frames at the highest rate a step of this kind reads (48 kHz when mixed)."""
    return synth_streams(n, (1536 if kind == "mixed" else 512) * frames, seed=seed)


@pytest.mark.parametrize("kind", ["one", "eight", "mixed"])
@pytest.mark.parametrize("version,math", [("v5", "tc16"), ("v5", "tc"), ("v5", "fp32"), ("v4", "fft"), ("v4", "fp32"),
                                          ("v4_8k", "fft")])
def test_continuation_after_export_import_is_bit_identical(version, math, kind):
    N, K, M = 2048, 30, 30
    audio = _streams_audio(kind, N, K + M, seed=31)
    A = _engine(version, math, N)
    B = _engine(version, math, 3000)
    assert A.fingerprint == B.fingerprint
    A.reset()
    _configure_per_stream(A, np.arange(N))
    B.configure(vad_start_probability=0.9, vad_end_probability=0.9, voice_start_frame_count=7, voice_end_frame_count=9)
    _run(A, audio, kind, 0, K)
    perm = np.random.default_rng(5).permutation(3000)[:N].astype(np.int32)
    rec = A.export_states(np.arange(N))
    assert (rec["frames_done"] == K).all()
    B.import_states(perm, rec)
    pa, fa, ea = _run(A, audio, kind, K, M)
    pb, fb, eb = _run(B, audio, kind, K, M, slots=perm)
    assert np.array_equal(pa, pb), f"probabilities differ: max {np.abs(pa - pb).max()}"
    assert np.array_equal(fa, fb)
    assert [e[:4] for e in ea] == [e[:4] for e in eb]
    assert all(perm[e[0]] == e[4] for e in eb) and all(e[0] == e[4] for e in ea)
    assert len(ea) > 50 and min(e[3] for e in ea) >= K          # events continue the stream's frame count
    for s in range(0, N, 7):
        ga, gb = A.get_state(s), B.get_state(int(perm[s]))
        assert all(np.array_equal(x, y) for x, y in zip(ga[:3], gb[:3])) and ga[3] == gb[3] == K + M
    A.close()
    B.close()


# ------------------------------------------------------------------------------------------------ chained device steps

def _dev_args(capi, n, audio_d, probs_d, flags_d, events_d, nev_d, slots_d=None):
    a = capi.StepArgs()
    a.n_streams = n
    a.audio = audio_d.data_ptr()
    a.pcm_format = capi.PCM_F32
    a.stream_stride = audio_d.shape[1]
    a.max_frames = 1
    a.frame_len = a.hop = 512
    a.src_rate = 16000
    if slots_d is not None:
        a.slots = slots_d.data_ptr()
    a.probs_out = probs_d.data_ptr()
    a.flags_out = flags_d.data_ptr()
    a.events_out = events_d.data_ptr()
    a.max_events = 2 * n
    a.n_events_out = nev_d.data_ptr()
    return a


def _chain(eng, torch, capi, audio, j0, j1, dev, slots_d=None, in_flight=None):
    """One-frame cvad_step_device steps j0..j1-1, enqueued back to back (then `in_flight()` is called while they may
    still run); -> [(probs, flags, sorted events)]."""
    n = audio.shape[0]
    bufs = []
    for j in range(j0, j1):
        x = torch.from_numpy(np.ascontiguousarray(audio[:, 512 * j:512 * (j + 1)])).to(dev)
        b = (x, torch.full((n, 1), -1.0, device=dev), torch.full((n, 1), 255, dtype=torch.uint8, device=dev),
             torch.zeros(2 * n * 24, dtype=torch.uint8, device=dev), torch.zeros(1, dtype=torch.int32, device=dev))
        bufs.append(b)
    torch.cuda.synchronize(dev)
    for b in bufs:
        eng.step_device(_dev_args(capi, n, *b, slots_d=slots_d))
    if in_flight is not None:
        in_flight()
    eng.sync()
    out = []
    for x, p, f, ev, nev in bufs:
        k = min(int(nev.cpu()[0]), 2 * n)
        rec = ev.cpu().numpy().view(np.int64)[:3 * k]
        r32 = rec.view(np.int32).reshape(k, 6)
        sf = rec.reshape(k, 3)[:, 2]
        out.append((p.cpu().numpy(), f.cpu().numpy(), sorted((int(r[0]), int(r[2]), int(r[3]), int(s)) for r, s in zip(r32, sf))))
    return out


def _chained_move(device_b):
    import torch
    from real_time_vad.engine import capi
    N, K, M = 4096, 10, 20
    audio = synth_streams(N, 512 * (K + M), seed=8)
    A = _engine("v5", "tc16", N)
    B = _engine("v5", "tc16", 5000, device=device_b)
    for e in (A, B):
        e.reset()
        _configure_per_stream(e, np.arange(N))
    recs = torch.zeros(N * 1072, dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    # exported while A's chain may still run: the export waits for it, and A's chain continues afterwards
    _chain(A, torch, capi, audio, 0, K, "cuda:0",
           in_flight=lambda: A.export_states(np.arange(N), device_ptr=recs.data_ptr()))
    assert np.array_equal(recs.cpu().numpy().view(capi.STATE_DTYPE), A.export_states(np.arange(N)))
    devb = f"cuda:{device_b}"
    recs_b = recs.to(devb)
    torch.cuda.synchronize(devb)
    perm = np.random.default_rng(9).permutation(5000)[:N].astype(np.int32)
    B.import_states(perm, recs_b.data_ptr())
    slots_d = torch.from_numpy(perm).to(devb)
    got_a = _chain(A, torch, capi, audio, K, K + M, "cuda:0")
    got_b = _chain(B, torch, capi, audio, K, K + M, devb, slots_d=slots_d)
    n_ev = 0
    for j, (a, b) in enumerate(zip(got_a, got_b)):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), f"step {K + j} differs"
        assert a[2] == b[2]
        n_ev += len(a[2])
    assert n_ev > 50
    for s in (0, 1, 777, N - 1):
        ga, gb = A.get_state(s), B.get_state(int(perm[s]))
        assert all(np.array_equal(x, y) for x, y in zip(ga[:3], gb[:3])) and ga[3] == gb[3] == K + M
    A.close()
    B.close()


def test_chained_device_steps_continue_after_a_device_memory_move():
    _chained_move(0)


def test_chained_device_steps_continue_on_another_gpu():
    from real_time_vad.engine import capi
    if capi.lib().cvad_device_count() < 2:
        pytest.skip("one sm_100 device visible")
    _chained_move(1)


def test_a_tc16_stream_continues_in_fp32_math_within_the_parity_bar():
    N, K, M = 64, 30, 30
    audio = synth_streams(N, 512 * (K + M), seed=12)
    A = _engine("v5", "tc16", N)
    C = _engine("v5", "fp32", N)
    A.reset()
    _configure_per_stream(A, np.arange(N))
    _run(A, audio, "one", 0, K)
    C.import_states(None, A.export_states(None))
    pa, _, _ = _run(A, audio, "one", K, M)
    pc, _, _ = _run(C, audio, "one", K, M)
    err = float(np.abs(pa - pc).max())
    assert 0 < err <= 1e-4, err
    A.close()
    C.close()


# --------------------------------------------------------------------------------------------------- refused imports

def _bad_records():
    yield "h NaN", lambda r: r["h"].__setitem__(5, np.nan)
    yield "c Inf", lambda r: r["c"].__setitem__(127, np.inf)
    yield "|h| > 2", lambda r: r["h"].__setitem__(64, np.nextafter(np.float32(-2), np.float32(-3)))
    yield "active 2", lambda r: r.__setitem__("is_voice_active", 2)
    yield "start count < 0", lambda r: r.__setitem__("voice_start_frame_count", -1)
    yield "end count < 0", lambda r: r.__setitem__("voice_end_frame_count", -3)
    yield "frames_done < 0", lambda r: r.__setitem__("frames_done", -1)
    yield "start p > 1", lambda r: r.__setitem__("vad_start_probability", 1.5)
    yield "end p < 0", lambda r: r.__setitem__("vad_end_probability", -0.1)
    yield "start p NaN", lambda r: r.__setitem__("vad_start_probability", np.nan)
    yield "n_start 0", lambda r: r.__setitem__("n_start", 0)
    yield "n_end 0", lambda r: r.__setitem__("n_end", 0)
    yield "denoise 2", lambda r: r.__setitem__("enable_denoising", 2)


def test_refused_imports_change_no_slot():
    import torch
    from real_time_vad.engine import capi
    from real_time_vad.engine.stream_engine import EngineError
    eng = _engine("v5", "tc16", 256)
    eng.reset()
    _configure_per_stream(eng, np.arange(256))
    _run(eng, synth_streams(256, 512 * 12, seed=3), "eight", 0, 12)
    targets = np.random.default_rng(1).permutation(256)[:100].astype(np.int32)
    good = eng.export_states(np.arange(100, 200))           # valid records, not the targets' own
    before = [eng.get_state(int(s)) for s in targets]

    def unchanged():
        for s, b in zip(targets, before):
            g = eng.get_state(int(s))
            assert all(np.array_equal(x, y) for x, y in zip(g[:3], b[:3])) and g[3] == b[3]

    for i, (name, spoil) in enumerate(_bad_records()):
        bad_at = (17 * i + 3) % 100
        rec = good.copy()
        spoil(rec[bad_at])
        for where in ("host", "device"):
            with pytest.raises(EngineError) as ei:
                if where == "host":
                    eng.import_states(targets, rec)
                else:
                    d = torch.from_numpy(rec.view(np.uint8).copy()).to("cuda:0")
                    torch.cuda.synchronize()
                    eng.import_states(targets, d.data_ptr())
            assert ei.value.code == capi.E_INVALID, name
            assert f"record {bad_at} " in ei.value.message, (name, ei.value.message)
        unchanged()
    d = torch.from_numpy(good.view(np.uint8).copy()).to("cuda:0")
    pad = torch.zeros(good.nbytes + 4, dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    for rec_ptr in (pad.data_ptr() + 4,):                  # device records must be 8-byte aligned
        with pytest.raises(EngineError) as ei:
            eng.import_states(targets, rec_ptr)
        assert ei.value.code == capi.E_INVALID and "aligned" in ei.value.message
        with pytest.raises(EngineError) as ei:
            eng.export_states(targets, device_ptr=rec_ptr)
        assert ei.value.code == capi.E_INVALID and "aligned" in ei.value.message
    with pytest.raises(EngineError) as ei:
        eng.import_states(np.r_[targets[:99], 256], good)
    assert ei.value.code == capi.E_CAPACITY
    with pytest.raises(EngineError) as ei:
        eng.import_states(np.r_[targets[:99], targets[0]], good)
    assert ei.value.code == capi.E_INVALID and "twice" in ei.value.message
    unchanged()
    eng.import_states(targets, good)                       # and the valid set goes through
    assert eng.get_state(int(targets[4]))[3] == 12
    eng.close()


# ------------------------------------------------------------------------------------- the manager: snapshot / restore

def _golden_manager():
    from real_time_vad import BatchedVADManager
    from real_time_vad.engine import capi
    return BatchedVADManager(max_streams=8, frame_len=480, pcm_format=capi.PCM_S16_32767)


def _golden_cfg():
    from real_time_vad import SampleRate, VADConfig
    return VADConfig(sample_rate=SampleRate.SAMPLERATE_16, buffer_size=480, vad_start_probability=0.4,
                     vad_end_probability=0.3, voice_start_frame_count=6, voice_end_frame_count=12)


def _recorder():
    log = {"ev": [], "wav": [], "cont": [], "start": 0}
    cbs = dict(on_voice_start=lambda: log.__setitem__("start", log["start"] + 1), on_voice_end=log["wav"].append,
               on_voice_continue=log["cont"].append)
    return log, cbs


def _step_events(mgr, log):
    out = mgr.step()
    log["ev"] += [(e.frame_index, 1 if e.kind == "start" else 2) for e in out.events]


@pytest.mark.parametrize("cut", [180, 154, 250])
def test_known_answer_continues_across_a_restore(cut):
    """tests/golden/sample_voice.npz, mode A (480-sample int16 messages, one frame each), cut after frame `cut` with 200
    samples of the next message already pushed: inside segment 2 (START 157, END 207), in its pre-roll (frames 152-154
    are at or above 0.4) and between segments.  Events, WAV bytes and continue frames equal an uninterrupted run and
    the reference's known answer."""
    from real_time_vad import StreamSnapshot
    g = np.load(GOLDEN / "sample_voice.npz")
    q = g["q16k"]
    msgs = [np.ascontiguousarray(q[i * 480:(i + 1) * 480]) for i in range(len(q) // 480)]
    assert g["A_probs"][152:155].min() >= 0.4 and g["A_events"][2].tolist() == [157, 1]

    ref, (ref_log, ref_cbs) = _golden_manager(), _recorder()
    sid = ref.open_stream(_golden_cfg(), **ref_cbs)
    for m in msgs:
        ref.push(sid, m)
        _step_events(ref, ref_log)
    ref.close()
    assert ref_log["ev"] == [tuple(e) for e in g["A_events"].tolist()]
    assert [hashlib.sha256(b).hexdigest() for b in ref_log["wav"]] == g["A_wav_sha"].tolist()

    src, (log, cbs) = _golden_manager(), _recorder()
    sid = src.open_stream(_golden_cfg(), **cbs)
    for m in msgs[:cut + 1]:
        src.push(sid, m)
        _step_events(src, log)
    src.push(sid, msgs[cut + 1][:200])
    data = src.snapshot_streams().to_bytes()
    src.close_stream(sid)
    src.close()

    dst = _golden_manager()
    other = dst.open_stream(_golden_cfg())                   # the target already serves someone
    ids = dst.restore_streams(StreamSnapshot.from_bytes(data), callbacks={sid: cbs})
    new = ids[sid]
    assert new != other and dst.pending(new) == 200
    dst.push(new, msgs[cut + 1][200:])
    _step_events(dst, log)
    for m in msgs[cut + 2:]:
        dst.push(new, m)
        _step_events(dst, log)
    dst.close()
    assert log["ev"] == ref_log["ev"]
    assert [hashlib.sha256(b).hexdigest() for b in log["wav"]] == g["A_wav_sha"].tolist()
    assert log["cont"] == ref_log["cont"] and log["start"] == ref_log["start"] == 4


def test_mixed_rate_streams_continue_with_every_callback_payload():
    """source_rate=None: 8 / 16 / 24 / 48 kHz streams with all three callbacks, cut in the middle of a segment of a
    resampled stream (whose pre-roll and segment the manager keeps in Python): every payload equals the
    uninterrupted run's."""
    from real_time_vad import BatchedVADManager, SampleRate, StreamSnapshot, VADConfig
    from scipy import signal
    sr = {8000: SampleRate.SAMPLERATE_8, 16000: SampleRate.SAMPLERATE_16, 24000: SampleRate.SAMPLERATE_24,
          48000: SampleRate.SAMPLERATE_48}
    plan = [8000, 16000, 24000, 48000] * 3
    n, T, per = len(plan), 96, 4
    base = synth_streams(n, 512 * T, seed=21)
    audio = [signal.resample(base[k], plan[k] * 512 // 16000 * T).astype(np.float32) for k in range(n)]

    def cfg(rate):
        return VADConfig(sample_rate=sr[rate], vad_start_probability=0.5, vad_end_probability=0.35,
                         voice_start_frame_count=2, voice_end_frame_count=3)

    def piece(k, step, lo=0.0, hi=1.0):
        w = plan[k] * 512 // 16000 * per
        a = step * w
        return audio[k][a + int(lo * w):a + int(hi * w)]

    def open_all(mgr):
        logs = [_recorder() for _ in range(n)]
        return [mgr.open_stream(cfg(plan[k]), **logs[k][1]) for k in range(n)], [lg for lg, _ in logs], [c for _, c in logs]

    ref = BatchedVADManager(max_streams=16, source_rate=None)
    ids, ref_logs, _ = open_all(ref)
    active = []
    for step in range(T // per):
        for k in range(n):
            ref.push(ids[k], piece(k, step))
        ref.step()
        active.append([ref.is_voice_active(ids[k]) for k in range(n)])
    ref.close()
    # cut after the first step at which a resampled stream is in the middle of a segment
    cut = next(s for s in range(3, T // per - 3) if any(active[s][k] and plan[k] != 16000 for k in range(n)))

    src = BatchedVADManager(max_streams=16, source_rate=None)
    ids, logs, cbs = open_all(src)
    for step in range(cut + 1):
        for k in range(n):
            src.push(ids[k], piece(k, step))
        src.step()
    for k in range(n):
        src.push(ids[k], piece(k, cut + 1, 0.0, 0.4))
    snap = StreamSnapshot.from_bytes(src.snapshot_streams().to_bytes())
    src.close()
    dst = BatchedVADManager(max_streams=32, source_rate=None)
    moved = dst.restore_streams(snap, callbacks={ids[k]: cbs[k] for k in range(n)})
    for step in range(cut + 1, T // per):
        for k in range(n):
            dst.push(moved[ids[k]], piece(k, step, 0.4 if step == cut + 1 else 0.0, 1.0))
        dst.step()
    dst.close()
    for k in range(n):
        assert logs[k]["start"] == ref_logs[k]["start"], k
        assert logs[k]["wav"] == ref_logs[k]["wav"], k
        assert logs[k]["cont"] == ref_logs[k]["cont"], k
    assert sum(len(lg["cont"]) for lg in ref_logs) > 100


def test_refused_restores_open_nothing():
    from real_time_vad import BatchedVADManager, ConfigurationError, SileroModelVersion, StreamSnapshot, VADConfig
    from real_time_vad.engine import capi
    v5 = BatchedVADManager(max_streams=8)
    keep = v5.open_stream(VADConfig())
    v4 = BatchedVADManager(max_streams=8, model_version=SileroModelVersion.V4)
    s4 = v4.open_stream(VADConfig(model_version=SileroModelVersion.V4))
    v4.push(s4, np.zeros(700, np.float32))
    snap4 = v4.snapshot_streams()
    v4.close()
    other = BatchedVADManager(max_streams=8, frame_len=480)
    s = other.open_stream(VADConfig())
    other.push(s, np.zeros(300, np.float32))
    snap_framing = other.snapshot_streams()
    other.close()
    pcm = BatchedVADManager(max_streams=8, pcm_format=capi.PCM_S16_32768)
    pcm.open_stream(VADConfig())
    snap_pcm = pcm.snapshot_streams()
    pcm.close()
    same = BatchedVADManager(max_streams=8)
    same.open_stream(VADConfig())
    snap_fp = StreamSnapshot.from_bytes(same.snapshot_streams().to_bytes())
    snap_fp.fingerprint ^= 1
    for bad in (snap4, snap_framing, snap_pcm, snap_fp):
        with pytest.raises(ConfigurationError):
            v5.restore_streams(bad)
        assert v5.open_streams == [keep]
    # a stream in the middle of voice whose snapshot carries no audio cannot get audio callbacks
    g = np.load(GOLDEN / "sample_voice.npz")
    mid = _golden_manager()
    sid = mid.open_stream(_golden_cfg(), on_voice_start=lambda: None)
    q = g["q16k"]
    for i in range(181):
        mid.push(sid, np.ascontiguousarray(q[i * 480:(i + 1) * 480]))
        mid.step()
    assert mid.is_voice_active(sid)
    snap_mid = mid.snapshot_streams()
    target = _golden_manager()
    t0 = target.open_stream(_golden_cfg())
    with pytest.raises(ConfigurationError):
        target.restore_streams(snap_mid, callbacks={sid: dict(on_voice_end=lambda b: None)})
    assert target.open_streams == [t0]
    ids = target.restore_streams(snap_mid, callbacks={sid: dict(on_voice_start=lambda: None)})   # what it carried: fine
    assert target.is_voice_active(ids[sid]) and target.open_streams == sorted([t0, ids[sid]])
    # ... nor can one in its pre-roll: frames 152-154 reach the start threshold, the start is at 157, and a snapshot
    # taken with voice_start only carries none of those frames for the voice_end WAV
    pre = _golden_manager()
    sid = pre.open_stream(_golden_cfg(), on_voice_start=lambda: None)
    for i in range(155):
        pre.push(sid, np.ascontiguousarray(q[i * 480:(i + 1) * 480]))
        pre.step()
    assert not pre.is_voice_active(sid)
    snap_pre = pre.snapshot_streams()
    assert snap_pre.states[0]["voice_start_frame_count"] == 3
    before = target.open_streams
    for cb in (dict(on_voice_end=lambda b: None), dict(on_voice_continue=lambda b: None)):
        with pytest.raises(ConfigurationError):
            target.restore_streams(snap_pre, callbacks={sid: cb})
        assert target.open_streams == before
    ids = target.restore_streams(snap_pre, callbacks={sid: dict(on_voice_start=lambda: None)})
    assert not target.is_voice_active(ids[sid])
    pre.close()
    # not enough free slots
    small = BatchedVADManager(max_streams=2, frame_len=480, pcm_format=capi.PCM_S16_32767)
    small.open_stream(_golden_cfg())
    small.open_stream(_golden_cfg())
    with pytest.raises(ConfigurationError):
        small.restore_streams(snap_mid)
    for m in (v5, same, mid, target, small):
        m.close()
