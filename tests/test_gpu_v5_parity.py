"""GPU parity: CUDA v5 path (through the C ABI) vs the CPU oracle.

Bars (BASELINE.json north_star): per-frame speech probability within 1e-4 absolute
of the FP32 oracle; voice start/end events at identical frame indices.
"""
import numpy as np
import pytest

from conftest import GOLDEN, synth_streams

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["tc", "fp32", "tc16"])
def math_mode(request, monkeypatch):
    """Every test runs on every arithmetic path of the v5 engine: tcgen05 tensor cores with the BF16 3-way split,
    packed FP32 FMA, and the FP16 2-way split with per-stream scaling that one-frame steps take under "tc16" (its
    multi-frame steps run as "tc").  cvad_create reads CVAD_MATH; engines are created inside the tests."""
    monkeypatch.setenv("CVAD_MATH", request.param)
    return request.param

TOL = 1e-4


def _oracle_dbg(ref_v5, frames):
    """frames [n,512] (already gated) -> dict of per-layer arrays shaped like the GPU dump."""
    n = frames.shape[0]
    out = {"mag": np.zeros((129, 3, n), np.float32), "e0": np.zeros((128, 3, n), np.float32),
           "e1": np.zeros((64, 2, n), np.float32), "e2": np.zeros((64, n), np.float32),
           "feat": np.zeros((128, n), np.float32)}
    for s in range(n):
        h = np.zeros(128, np.float32)
        c = np.zeros(128, np.float32)
        _, d = ref_v5.frame(frames[s], h, c, want_dbg=True)
        out["mag"][:, :, s] = d[0:387].reshape(129, 3)
        out["e0"][:, :, s] = d[387:771].reshape(128, 3)
        out["e1"][:, :, s] = d[771:899].reshape(64, 2)
        out["e2"][:, s] = d[899:963]
        out["feat"][:, s] = d[963:1091]
    return out


def test_frontend_layers_match_oracle(engine_factory, ref_v5):
    eng = engine_factory(64)
    eng.configure(enable_denoising=False)
    x = synth_streams(32, 16000 + 512, seed=3)[:, 16000:16000 + 512].copy()
    got = eng.debug_dump(x)
    want = _oracle_dbg(ref_v5, x)
    for name in ("mag", "e0", "e1", "e2", "feat"):
        w = want[name]
        g = got[name][..., :w.shape[-1]]
        scale = max(1.0, float(np.abs(w).max()))
        err = float(np.abs(g - w).max())
        assert err <= 2e-5 * scale, f"{name}: max abs err {err} (scale {scale})"


@pytest.mark.parametrize("n_streams", [1, 31, 32, 70])
def test_probs_one_frame_per_step_carries_state(engine_factory, ref_v5, n_streams):
    eng = engine_factory(128)
    eng.reset()
    eng.configure(enable_denoising=True)
    n_steps = 12
    audio = synth_streams(n_streams, 512 * n_steps, seed=5)
    want, h_ref, c_ref = ref_v5.run(audio, n_steps, hop=512, frame_len=512, denoise=True)
    got = np.zeros_like(want)
    for j in range(n_steps):
        r = eng.step(audio[:, j * 512:(j + 1) * 512])
        assert r.status.sum() == 0
        got[:, j] = r.probs[:, 0]
    assert np.abs(got - want).max() <= TOL
    h, c, sm, fd = eng.get_state(n_streams - 1)
    assert fd == n_steps
    assert np.abs(h - h_ref[n_streams - 1]).max() <= 1e-4
    assert np.abs(c - c_ref[n_streams - 1]).max() <= 1e-3


def test_probs_many_frames_one_call_hop256(engine_factory, ref_v5):
    eng = engine_factory(128)
    eng.reset()
    eng.configure(enable_denoising=True)
    n, T = 45, 37
    audio = synth_streams(n, 256 * (T - 1) + 512, seed=7)
    want, _, _ = ref_v5.run(audio, T, hop=256, frame_len=512, denoise=True)
    r = eng.step(audio, hop=256)
    assert r.probs.shape == (n, T)
    assert np.abs(r.probs - want).max() <= TOL


def test_ragged_frames_and_slot_indirection(engine_factory, ref_v5):
    eng = engine_factory(128)
    eng.reset()
    eng.configure(enable_denoising=False)
    n, T = 40, 9
    rng = np.random.default_rng(11)
    audio = synth_streams(n, 512 * T, seed=9)
    nfr = rng.integers(0, T + 1, size=n).astype(np.int32)
    nfr[0], nfr[1] = T, 0
    slots = rng.permutation(128)[:n].astype(np.int32)
    r = eng.step(audio, slots=slots, n_frames=nfr)
    for s in range(n):
        if nfr[s] == 0:
            assert not r.probs[s].any() and not r.flags[s].any()
            continue
        want, h_ref, c_ref = ref_v5.run(audio[s:s + 1], int(nfr[s]), denoise=False)
        assert np.abs(r.probs[s, :nfr[s]] - want[0]).max() <= TOL
        assert not r.probs[s, nfr[s]:].any()
        h, c, sm, fd = eng.get_state(int(slots[s]))
        assert fd == nfr[s]
        assert np.abs(h - h_ref[0]).max() <= 1e-4
    # a slot that was never stepped is still zero
    unused = [k for k in range(128) if k not in set(slots.tolist())][0]
    h, c, sm, fd = eng.get_state(unused)
    assert not h.any() and not c.any() and fd == 0


def test_events_identical_to_oracle_state_machine(engine_factory, ref_v5, ref_lib):
    from vad_oracle import sm_run_c
    eng = engine_factory(128)
    n, T = 48, 140
    audio = synth_streams(n, 512 * T, seed=13)
    eng.reset()
    cfgs = {}
    for s in range(n):
        cfg = dict(vad_start_probability=(0.4, 0.5, 0.7)[s % 3], vad_end_probability=(0.3, 0.35, 0.7)[s % 3],
                   voice_start_frame_count=(3, 6, 10)[s % 3], voice_end_frame_count=(5, 12, 20)[(s // 3) % 3])
        cfgs[s] = cfg
        eng.configure([s], enable_denoising=True, **cfg)
    # two calls, so state-machine counters have to survive between steps
    r1 = eng.step(audio[:, :512 * 60])
    r2 = eng.step(audio[:, 512 * 60:])
    probs = np.concatenate([r1.probs, r2.probs], axis=1)
    flags = np.concatenate([r1.flags, r2.flags], axis=1)
    want_p, _, _ = ref_v5.run(audio, T, denoise=True)
    assert np.abs(probs - want_p).max() <= TOL
    n_events = 0
    for s in range(n):
        c = cfgs[s]
        # (1) the device state machine is bit-exact on the device's own probabilities
        f_dev, _ = sm_run_c(ref_lib, probs[s], c["vad_start_probability"], c["vad_end_probability"], 0.8, 0.95,
                            c["voice_start_frame_count"], c["voice_end_frame_count"])
        assert np.array_equal(f_dev, flags[s]), f"stream {s}"
        # (2) and the events equal those of the oracle's own probabilities
        f_ref, _ = sm_run_c(ref_lib, want_p[s], c["vad_start_probability"], c["vad_end_probability"], 0.8, 0.95,
                            c["voice_start_frame_count"], c["voice_end_frame_count"])
        assert np.array_equal(f_ref & 3, flags[s] & 3), f"stream {s}"
        n_events += int(((flags[s] & 1) != 0).sum() + ((flags[s] & 2) != 0).sum())
    assert n_events > 20, "signal recipe should make the state machine fire"
    # event records: same content as the flags, stream-then-frame order
    ev = [(e[0], e[2], e[3]) for e in r1.events]
    want_ev = []
    for s in range(n):
        for j in range(60):
            if r1.flags[s, j] & 1:
                want_ev.append((s, j, 1))
            if r1.flags[s, j] & 2:
                want_ev.append((s, j, 2))
    assert ev == want_ev
    assert all(e[4] == e[2] for e in r1.events)            # stream_frame counts from the reset
    assert all(e[4] == e[2] + 60 for e in r2.events)


def test_pcm16_short_frames_match_reference_scaling(engine_factory, ref_v5):
    from real_time_vad.engine import capi
    eng = engine_factory(128)
    n, T = 33, 20
    x = synth_streams(n, 480 * T, seed=17)
    q = np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16)
    for fmt, div in ((capi.PCM_S16_32767, 32767.0), (capi.PCM_S16_32768, 32768.0)):
        eng.reset()
        eng.configure(enable_denoising=True)
        xf = (q.astype(np.float32) / np.float32(div)).astype(np.float32)
        want, _, _ = ref_v5.run(xf, T, hop=480, frame_len=480, denoise=True)
        r = eng.step(q, frame_len=480, hop=480, pcm_format=fmt)
        assert np.abs(r.probs - want).max() <= TOL


def test_unaligned_hop_takes_scalar_loader(engine_factory, ref_v5):
    eng = engine_factory(128)
    eng.reset()
    eng.configure(enable_denoising=True)
    n, T, hop, flen = 5, 7, 301, 509
    audio = synth_streams(n, hop * (T - 1) + flen, seed=19)
    want, _, _ = ref_v5.run(audio, T, hop=hop, frame_len=flen, denoise=True)
    r = eng.step(audio, hop=hop, frame_len=flen)
    assert np.abs(r.probs - want).max() <= TOL


def test_nonfinite_stream_is_rejected_without_state_change(engine_factory, ref_v5):
    eng = engine_factory(128)
    eng.reset()
    eng.configure(enable_denoising=True)
    n, T = 34, 4
    audio = synth_streams(n, 512 * T, seed=23)
    r0 = eng.step(audio[:, :512])
    h_before = eng.get_state(7)[0]
    bad = audio[:, 512:].copy()
    bad[7, 512 * 2 + 5] = np.nan
    bad[20, 3] = np.inf
    r = eng.step(bad)
    assert r.status[7] == 1 and r.status[20] == 1 and r.status.sum() == 2
    assert not r.probs[7].any() and not r.flags[7].any()
    h_after, _, _, fd = eng.get_state(7)
    assert np.array_equal(h_before, h_after) and fd == 1
    ok = [s for s in range(n) if s not in (7, 20)]
    want, _, _ = ref_v5.run(audio[ok], T, denoise=True)
    got = np.concatenate([r0.probs[ok], r.probs[ok]], axis=1)
    assert np.abs(got - want).max() <= TOL


def test_set_state_within_the_h_bound_reset_and_errors(engine_factory):
    """cvad_set_state writes any h within [-2, 2] (both ends included) and any c exactly; an h beyond the bound, or a
    NaN, is refused before anything is written (the FP16-split kernels cannot hold it)."""
    from real_time_vad.engine import capi
    from real_time_vad.engine.stream_engine import EngineError
    eng = engine_factory(128)
    eng.reset()
    rng = np.random.default_rng(1)
    h = np.clip(rng.standard_normal(128), -2, 2).astype(np.float32)
    h[:2] = 2.0, -2.0
    c = rng.standard_normal(128).astype(np.float32)
    eng.set_state(100, h, c, np.array([1, 2, 3, 0], np.int32))
    h2, c2, sm, _ = eng.get_state(100)
    assert np.array_equal(h, h2) and np.array_equal(c, c2) and sm[:3].tolist() == [1, 2, 3]
    for bad in (np.nextafter(np.float32(2), np.float32(3)), -4.0, np.nan):
        hb = h.copy()
        hb[77] = bad
        with pytest.raises(EngineError) as ei:
            eng.set_state(100, hb, np.zeros(128, np.float32), np.zeros(4, np.int32))
        assert ei.value.code == capi.E_INVALID and "h[77]" in ei.value.message
        h2, c2, sm, _ = eng.get_state(100)
        assert np.array_equal(h, h2) and np.array_equal(c, c2) and sm[:3].tolist() == [1, 2, 3]
    eng.reset([100])
    h2, c2, sm, _ = eng.get_state(100)
    assert not h2.any() and not c2.any() and not sm.any()
    with pytest.raises(EngineError):
        eng.get_state(128)
    with pytest.raises(EngineError):
        eng.step(np.zeros((200, 512), np.float32))          # more streams than slots
    with pytest.raises(EngineError):
        eng.configure(voice_start_frame_count=0)
    r = eng.step(np.zeros((3, 100), np.float32))              # shorter than one frame: zero frames
    assert r.probs.shape == (3, 0)


def test_sample_voice_known_answer_four_segments(engine_factory, ref_v5):
    """websocket_service/README.md:290 / examples/test_python_vad_client.py:201-204:
    SampleVoiceMono.wav at 16 kHz, 30 ms frames, 0.4/0.3/6/12 -> exactly 4 segments."""
    from scipy.io import wavfile
    from vad_oracle import resample
    from real_time_vad.engine import capi
    sr, x = wavfile.read(str(GOLDEN / "SampleVoiceMono.wav"))
    y = resample(x.astype(np.float32) / 32768.0, sr, 16000)
    q = np.clip(np.round(y * 32767.0), -32768, 32767).astype(np.int16)
    T = len(q) // 480
    eng = engine_factory(128)
    eng.reset()
    eng.configure(vad_start_probability=0.4, vad_end_probability=0.3, voice_start_frame_count=6,
                  voice_end_frame_count=12, enable_denoising=True)
    r = eng.step(q[None, :T * 480], frame_len=480, hop=480, pcm_format=capi.PCM_S16_32767)
    kinds = [e[3] for e in r.events]
    assert kinds == [1, 2] * 4
    xf = (q[:T * 480].astype(np.float32) / np.float32(32767.0))[None]
    want, _, _ = ref_v5.run(xf, T, hop=480, frame_len=480, denoise=True)
    assert np.abs(r.probs - want).max() <= TOL


def test_pipelined_submit_collect_equals_blocking_steps(engine_factory, ref_v5):
    """Up to four steps in flight (cvad_step_submit/collect) must give what blocking cvad_step gives,
    in submission order, with state carried from step to step."""
    from real_time_vad.engine.stream_engine import EngineError
    eng = engine_factory(128)
    eng.reset()
    eng.configure(enable_denoising=True, vad_start_probability=0.5, vad_end_probability=0.35,
                  voice_start_frame_count=3, voice_end_frame_count=4)
    n, steps, F = 70, 14, 3
    audio = synth_streams(n, 512 * F * steps, seed=29)
    want, _, _ = ref_v5.run(audio, F * steps, denoise=True)
    chunks = [np.ascontiguousarray(audio[:, k * 512 * F:(k + 1) * 512 * F]) for k in range(steps)]
    got, flags = [], []
    from collections import deque
    inflight = deque()
    refused = False
    for k in range(steps):
        inflight.append(eng.submit(chunks[k]))
        if len(inflight) == 4:
            if not refused:
                with pytest.raises(EngineError):
                    eng.submit(chunks[k])                  # a fifth step in flight is refused
                refused = True
            r = inflight.popleft().collect()
            got.append(r.probs.copy())
            flags.append(r.flags.copy())
    while inflight:
        r = inflight.popleft().collect()
        got.append(r.probs.copy())
        flags.append(r.flags.copy())
    assert refused
    got = np.concatenate(got, axis=1)
    assert np.abs(got - want).max() <= TOL
    # same run with blocking calls: bit-identical
    eng.reset()
    again = np.concatenate([eng.step(c).probs for c in chunks], axis=1)
    assert np.array_equal(got, again)
    assert eng.get_state(0)[3] == F * steps


@pytest.mark.parametrize("case", ["zeros", "tiny", "denormal", "loud_x30", "int16_scale", "huge_1e8", "square", "dc", "impulses"])
def test_extreme_inputs_stay_finite_and_on_the_oracle(engine_factory, ref_v5, case):
    """The reference accepts any finite float32 audio (audio.py:211-231 only rejects NaN/Inf): un-normalised
    int16-scale floats, silence, denormals, clipping square waves.  Both arithmetic paths must stay finite and on
    the oracle there too (the BF16 operand parts keep FP32's exponent range), one call and one frame per step."""
    T = 20
    rng = np.random.default_rng(3)
    base = synth_streams(4, 512 * T, seed=9)
    t = np.arange(512 * T)
    x = {"zeros": np.zeros((4, 512 * T), np.float32),
         "tiny": (1e-6 * rng.standard_normal((4, 512 * T))).astype(np.float32),
         "denormal": np.full((4, 512 * T), 1e-40, np.float32),
         "loud_x30": (30 * base).astype(np.float32),
         "int16_scale": (32768 * base).astype(np.float32),
         "huge_1e8": (1e8 * base).astype(np.float32),
         "square": np.sign(np.sin(2 * np.pi * 200 * t / 16000))[None, :].repeat(4, 0).astype(np.float32),
         "dc": np.full((4, 512 * T), 0.5, np.float32),
         "impulses": (rng.random((4, 512 * T)) > 0.999).astype(np.float32)}[case]
    eng = engine_factory(8)
    eng.reset()
    eng.configure(enable_denoising=False)
    want, _, _ = ref_v5.run(x, T, denoise=False)
    one = eng.step(x).probs
    eng.reset()
    steps = np.stack([eng.step(x[:, j * 512:(j + 1) * 512]).probs[:, 0] for j in range(T)], axis=1)
    assert np.isfinite(one).all() and np.isfinite(steps).all()
    assert np.abs(one - want).max() <= TOL and np.abs(steps - want).max() <= TOL


def test_wide_rows_only_the_samples_read_are_copied(engine_factory):
    """stream_stride much larger than what the step reads (the feeder stepping the first frame of longer rows): the
    host path copies a dense block (2-D copy for pinned input, row-wise staging for pageable input); results are
    those of a tight block, bit for bit, for float32 and int16, one and several frames."""
    import ctypes as C
    from real_time_vad.engine import capi
    n, wide = 70, 4096
    audio = synth_streams(n, wide, seed=97)
    eng = engine_factory(128)
    eng.configure(enable_denoising=True)
    L = capi.lib()
    for dtype, fmt in ((np.float32, capi.PCM_F32), (np.int16, capi.PCM_S16_32767)):
        block = audio if dtype is np.float32 else np.clip(np.round(audio * 32767.0), -32768, 32767).astype(np.int16)
        ptr = L.cvad_alloc_pinned(block.nbytes)
        pinned = np.frombuffer((C.c_char * block.nbytes).from_address(ptr), dtype).reshape(block.shape)
        pinned[:] = block
        for T in (1, 3):
            tight = np.ascontiguousarray(block[:, :512 * T])
            eng.reset()
            want = eng.step(tight, pcm_format=fmt, max_frames=T).probs
            for src in (block, pinned):                                  # pageable, pinned
                eng.reset()
                got = eng.step(src, pcm_format=fmt, max_frames=T).probs
                assert np.array_equal(got, want), (dtype, T)
        L.cvad_free_pinned(ptr)
