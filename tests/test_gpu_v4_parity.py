"""GPU parity: CUDA v4 path (silero_vad.onnx, 16 kHz branch) vs the CPU oracle.

v4 feeds log(1 + 2^20 |STFT|) into the network, which amplifies FP32 rounding of
near-zero bins (a pure tone moves the probability by 7e-4 between FP32 and FP64
evaluation of the SAME graph -- DESIGN.md section 5).  Parity is therefore asserted on
signals with a noise floor, as real audio has; the 1e-4 bar is kept."""
import numpy as np
import pytest

from conftest import GOLDEN, synth_streams

pytestmark = pytest.mark.gpu
TOL = 1e-4
# the FFT-mode STFT's per-bin bar in units of 2^-24 max(|re|, |im|) (test_v4_frontend_layers_match_oracle); the worst
# ratio measured on a B200 (6.6) with 2x headroom
K_V4_FFT = 14.0


@pytest.fixture(autouse=True, params=["fft", "tc", "fp32"])
def math_mode(request, monkeypatch):
    """The three builds of v4's STFT: double-precision FFT + tensor-core basis-rounding correction (the default),
    tcgen05 tensor cores with the BF16 3-way split, FP32 FMA."""
    monkeypatch.setenv("CVAD_MATH", request.param)
    from real_time_vad.engine import pool
    for (version, _dev, _path), engines in pool._ENGINES.items():
        if version.startswith("v4"):
            for pe in engines:
                pe.engine.set_math(request.param)
    return request.param


def test_v4_frontend_layers_match_oracle(engine_factory, ref_v4, math_mode):
    eng = engine_factory(64, model_version="v4")
    eng.configure(enable_denoising=False)
    x = synth_streams(16, 16000 + 512, seed=3)[:, 16000:16000 + 512].copy()
    got = eng.debug_dump(x)
    want = {k: [] for k in ("mag", "norm", "r3", "r15", "r27", "r39", "feat")}
    for s in range(16):
        h = np.zeros((2, 64), np.float32)
        c = np.zeros((2, 64), np.float32)
        _, d = ref_v4.frame(x[s], h, c, want_dbg=True)
        o = 0
        for name, shape in (("mag", (129, 8)), ("norm", (129, 8)), ("r3", (16, 8)), ("r7", (16, 4)), ("r15", (32, 4)),
                            ("r19", (32, 2)), ("r27", (32, 2)), ("r31", (32,)), ("r39", (64,)), ("feat", (64,))):
            n = int(np.prod(shape))
            if name in want:
                want[name].append(d[o:o + n].reshape(shape))
            o += n
    mag_ref = np.stack(want["mag"], axis=-1)
    for name in ("mag", "norm", "r3", "r15", "r27", "r39", "feat"):
        w = np.stack(want[name], axis=-1)
        g = got[name]
        scale = max(1.0, float(np.abs(w).max()))
        if name == "norm":
            # norm = log(1 + 2^20 |STFT|) - mean: a weak bin turns an absolute spectrogram difference d into up to
            # 2^20 d.  The FP32 build accumulates in the oracle's own order and lands on it (|d| <= 2e-6 here); the
            # tensor cores accumulate 16 partial dot products with truncation (|d| <= 1.5e-5 = 6e-7 of full scale),
            # so the bound carries the derivative of the log at d = 2e-6 for the bin's own magnitude
            allowed = 5e-5 * scale + 2.0 ** 20 * 2e-6 / (1.0 + 2.0 ** 20 * mag_ref)
            assert np.all(np.abs(g - w) <= allowed), f"norm: max abs err {np.abs(g - w).max()}"
            continue
        if name == "mag" and math_mode == "fft":
            # v4_stft_fft_kernel: the transform in float64, plus a correction of at most 7.7e-8 per basis entry for the
            # file basis' float32 rounding, so every bin is held to |B_file @ x| evaluated in float64
            from conftest import V4_ONNX
            from real_time_vad.engine.onnx_weights import canonical_blob_v4
            B = canonical_blob_v4(V4_ONNX)[:258 * 256].reshape(258, 256).astype(np.float64)
            xp = np.pad(x.astype(np.float64), ((0, 0), (96, 96)), mode="reflect")
            win = np.stack([xp[:, 64 * t:64 * t + 256] for t in range(8)], axis=1)        # [item, column, 256]
            re64 = np.einsum("kn,itn->kti", B[:129], win)
            im64 = np.einsum("kn,itn->kti", B[129:], win)
            unit = 2.0 ** -24 * np.maximum(np.abs(re64), np.abs(im64))
            ratio = np.abs(g.astype(np.float64) - np.hypot(re64, im64)) / np.maximum(unit, 1e-300)
            print(f"v4 FFT-mode STFT: worst |mag - mag64| / (2^-24 max(|re64|, |im64|)) = {ratio.max():.3f}")
            assert ratio.max() <= K_V4_FFT, f"mag: {ratio.max():.3g} x 2^-24 max(|re|, |im|) (bar {K_V4_FFT})"
        err = float(np.abs(g - w).max())
        assert err <= 5e-5 * scale, f"{name}: max abs err {err} (scale {scale})"


@pytest.mark.parametrize("n_streams", [1, 17, 70])
def test_v4_probs_and_state_carry(engine_factory, ref_v4, n_streams):
    eng = engine_factory(128, model_version="v4")
    eng.reset()
    eng.configure(enable_denoising=True)
    steps, F = 5, 4
    audio = synth_streams(n_streams, 512 * F * steps, seed=5)
    want, h_ref, c_ref = ref_v4.run(audio, F * steps, denoise=True)
    got = np.concatenate([eng.step(audio[:, k * 512 * F:(k + 1) * 512 * F]).probs for k in range(steps)], axis=1)
    assert np.abs(got - want).max() <= TOL
    h, c, sm, fd = eng.get_state(n_streams - 1)
    assert fd == F * steps
    assert np.abs(h - h_ref[n_streams - 1].reshape(128)).max() <= 1e-4
    assert np.abs(c - c_ref[n_streams - 1].reshape(128)).max() <= 1e-3


def test_v4_hop256_ragged_pcm16_and_events(engine_factory, ref_v4, ref_lib):
    from real_time_vad.engine import capi
    from vad_oracle import sm_run_c
    eng = engine_factory(128, model_version="v4")
    eng.reset()
    eng.configure(vad_start_probability=0.5, vad_end_probability=0.35, voice_start_frame_count=3,
                  voice_end_frame_count=5, enable_denoising=True)
    n, T = 40, 61
    x = synth_streams(n, 256 * (T - 1) + 512, seed=7)
    q = np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16)
    xf = (q.astype(np.float32) / np.float32(32768.0)).astype(np.float32)
    nfr = np.full(n, T, np.int32)
    nfr[3], nfr[9] = 0, 20
    r = eng.step(q, hop=256, n_frames=nfr, pcm_format=capi.PCM_S16_32768)
    n_ev = 0
    for s in range(n):
        k = int(nfr[s])
        if k == 0:
            assert not r.probs[s].any()
            continue
        want, _, _ = ref_v4.run(xf[s:s + 1], k, hop=256, denoise=True)
        assert np.abs(r.probs[s, :k] - want[0]).max() <= TOL, s
        fl, _ = sm_run_c(ref_lib, want[0], 0.5, 0.35, 0.8, 0.95, 3, 5)
        assert np.array_equal(fl & 3, r.flags[s, :k] & 3), s
        n_ev += int((fl & 3 != 0).sum())
    assert n_ev > 10


def test_v4_wrapper_and_compat_session(ref_v4):
    """VADWrapper with model_version=V4: fast path == per-frame compat path == oracle."""
    from real_time_vad import SileroModelVersion, VADConfig, VADWrapper
    x = synth_streams(1, 512 * 40, seed=11)[0]
    cfg = VADConfig(model_version=SileroModelVersion.V4, vad_start_probability=0.5, vad_end_probability=0.35,
                    voice_start_frame_count=3, voice_end_frame_count=4)
    a, b = VADWrapper(cfg), VADWrapper(cfg)
    assert a.processor.supports_batched() is True
    assert a.processor.model.model_state.hidden_state.shape == (2, 1, 64)
    ev_a, ev_b = [], []
    a.set_callbacks(voice_start_callback=lambda: ev_a.append(("S", a._state.total_frames_processed)),
                    voice_end_callback=lambda w: ev_a.append(("E", a._state.total_frames_processed, len(w))))
    b.set_callbacks(voice_start_callback=lambda: ev_b.append(("S", b._state.total_frames_processed)),
                    voice_end_callback=lambda w: ev_b.append(("E", b._state.total_frames_processed, len(w))))
    a.process_audio_data(x)
    T = (len(x) - 512) // 256 + 1
    for j in range(T):                                       # compat path, one frame per call
        r = b.processor.process_frame(x[j * 256:j * 256 + 512].copy())
        b._handle_callbacks(r)
        b._state.total_frames_processed += 1
    assert ev_a == ev_b
    pa, pb = np.array(a.processor.voice_probabilities), np.array(b.processor.voice_probabilities)
    assert np.abs(pa - pb).max() <= 2e-6
    want, _, _ = ref_v4.run(x[None], T, hop=256, denoise=True)
    assert np.abs(pa - want[0, -len(pa):]).max() <= TOL


def _interp_v4(audio, sr, dtype=np.float32):
    """Frames of 512 samples through the reference's silero_vad.onnx, op by op (oracle/onnx_interp.py)."""
    from conftest import V4_ONNX
    from onnx_interp import OnnxInterpreter
    it = OnnxInterpreter(str(V4_ONNX), dtype=dtype)
    n, L = audio.shape
    T = L // 512
    probs = np.zeros((n, T), np.float32)
    hs, cs = [], []
    for s in range(n):
        h = np.zeros((2, 1, 64), np.float32)
        c = np.zeros((2, 1, 64), np.float32)
        for j in range(T):
            out, h, c = it.run({"input": audio[s:s + 1, j * 512:(j + 1) * 512], "h": h, "c": c,
                                "sr": np.array(sr, np.int64)})
            probs[s, j] = out.reshape(-1)[0]
        hs.append(np.asarray(h).reshape(128))
        cs.append(np.asarray(c).reshape(128))
    return probs, np.stack(hs), np.stack(cs)


def test_v4_8k_submodel_matches_onnx_graph(engine_factory):
    """SURVEY.md 8(f) item 4: v4's 8 kHz sub-model (the graph's else-branch, what the reference runs for v4 with
    sample_rate 8000): two LSTM time steps per 512-sample frame, the two sigmoid outputs averaged."""
    n, T = 6, 9
    audio = synth_streams(n, 512 * T, seed=61)           # interpreted as 8 kHz samples; a noise floor keeps v4 well conditioned
    want, h_ref, c_ref = _interp_v4(audio, 8000)
    want16, _, _ = _interp_v4(audio[:2], 16000)
    assert np.abs(want[:2] - want16).max() > 1e-3          # it really is a different model
    eng = engine_factory(32, model_version="v4_8k")
    eng.configure(enable_denoising=False)
    got = np.concatenate([eng.step(audio[:, :512 * 4]).probs, eng.step(audio[:, 512 * 4:]).probs], axis=1)
    assert got.shape == (n, T)
    assert np.abs(got - want).max() <= TOL
    h, c, _, fd = eng.get_state(n - 1)
    assert fd == T
    assert np.abs(h - h_ref[n - 1]).max() <= 1e-4 and np.abs(c - c_ref[n - 1]).max() <= 1e-3


def test_v4_8k_through_the_reference_facing_session():
    """The `ort` seam: a v4 InferenceSession fed sr = 8000 runs the 8 kHz sub-model (state in, state out), as
    onnxruntime does for the reference (silero_model.py:433, :476-499); a v5 session refuses, as the graph does."""
    from conftest import V4_ONNX, V5_ONNX
    from real_time_vad.engine import ort_compat as ort
    audio = synth_streams(1, 512 * 5, seed=63)
    want, _, _ = _interp_v4(audio, 8000)
    sess = ort.InferenceSession(str(V4_ONNX))
    h = np.zeros((2, 1, 64), np.float32)
    c = np.zeros((2, 1, 64), np.float32)
    got = []
    for j in range(5):
        out, h, c = sess.run(None, {"input": audio[:, j * 512:(j + 1) * 512], "h": h, "c": c,
                                    "sr": np.array([8000], np.int64)})
        got.append(float(out[0, 0]))
    assert np.abs(np.array(got) - want[0]).max() <= TOL
    sess.close()
    s5 = ort.InferenceSession(str(V5_ONNX))
    with pytest.raises(ValueError):
        s5.run(None, {"input": audio[:, :512], "state": np.zeros((2, 1, 128), np.float32), "sr": np.array([8000], np.int64)})
    s5.close()


@pytest.mark.parametrize("sr,version", [(16000, "v4"), (8000, "v4_8k")])
def test_v4_engine_against_opencv_dnn_on_the_reference_graph(engine_factory, sr, version):
    """v4's CUDA path against a third-party ONNX runtime executing the reference's own graph (oracle/onnx_flatten.py:
    silero_vad.onnx's 16 kHz branch / 8 kHz sub-model inside OpenCV's DNN module, h / c fed back per frame)."""
    from conftest import V4_ONNX, require_cv2
    require_cv2()
    from onnx_flatten import OpenCVSession
    n, T = 4, 10
    audio = synth_streams(n, 512 * T, seed=71) + 0.02 * np.random.default_rng(2).standard_normal((n, 512 * T)).astype(np.float32)
    z = {"input": np.zeros((1, 512), np.float32), "h": np.zeros((2, 1, 64), np.float32), "c": np.zeros((2, 1, 64), np.float32),
         "sr": np.array([sr], np.int64)}
    sess = OpenCVSession(str(V4_ONNX), z, ["input", "h", "c"])
    want = np.zeros((n, T))
    for s in range(n):
        h = c = np.zeros((2, 1, 64), np.float32)
        for j in range(T):
            out, h, c = sess.run({"input": audio[s:s + 1, j * 512:(j + 1) * 512].astype(np.float32), "h": h, "c": c})
            want[s, j] = float(out.reshape(-1)[0])
    eng = engine_factory(32, model_version=version)
    eng.reset()
    eng.configure(enable_denoising=False)
    got = eng.step(audio.astype(np.float32)).probs
    assert np.abs(got - want).max() <= TOL
