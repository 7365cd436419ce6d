"""GPU: the input stages' own output, sample by sample, against float64 references (StreamEngine.debug_input).

Stage -1 (downmix_kernel) and stage 0 (resample_fft_kernel<1|3|6>, resample_tc_kernel<false|true>, resample_kernel,
passthrough_kernel) produce the float32 16 kHz samples the model kernels read.  test_gpu_resample.py sees them only
through the model's probability, where a wrong rounding, a wrong int16 scale or a scale that leaks between streams
stays far under its 1e-4 bar.  Here every sample is compared with a reference of the same operation in float64.

FFT resampler (the default, DESIGN.md section 3c: scipy.signal.resample per chunk in float64, rounded once):
    y64 = scipy.signal.resample(x.astype(float64), 512) per chunk, x the float32 input the kernel sees;
    |y - y64| <= 0.5 ulp(float32(y64)) (1 + 1e-6) + 2e-15 max|x_chunk|.
The second term is the float64 noise of the two transforms (kernel and scipy) around outputs near zero.  It scales with
the chunk, so subnormal outputs (1e-40 input, no -ftz in the build) must be correctly rounded too.

Dense operator (resampler "gemm" under math fp32 / tc / tc16):
    y64 = R64 @ x,  R64 = scipy.signal.resample(eye(n_in), 512, axis=0);
    |y - y64| <= k 2^-24 ((|R64| + |R32 - R64|) @ |x|) + |R32 - R64| @ |x| + n_in 2^-149 + floor.
The second term is the operator's own float32 rounding (the engine's R32, pinned to scipy by test_capi_boundary.py);
the third is float32's absolute rounding unit below 2^-126, once per accumulated product (the subnormal inputs).
`k` is one constant per build, from its arithmetic, set from the worst ratio measured on a B200 with 2x headroom
(printed by every check):
  - fp32: one serial FFMA chain of n_in products per output, so k <= n_in in the worst case; measured 86 (48 kHz,
    the target's Nyquist tone), about 2.2 sqrt(1536): k = 176;
  - tc:   x and R each as three BF16 parts, the six leading cross products in FP32 tensor-core accumulators (16
    products per issue), then the main and correction accumulators added; measured 55: k = 112;
  - tc16: R (scaled by a power of two) and x (scaled per stream from its chunk maximum) each as two FP16 parts, three
    cross products in FP32 accumulators, the sum scaled back; measured 55: k = 112.
`floor` is zero for fp32.  The tensor cores take no subnormal operands, so under tc an input below 2^-126 may be lost:
floor = 2^-126 rowsum|R|.  Under tc16 each operand is resolved to FP16's 2^-24 of its scaled range: R's maximum lies
at 2^14 and so does x's, except that the per-stream scale is capped at 2^125 (DESIGN.md section 3a), which leaves a
subnormal-only chunk below FP16's range (the 1e-40 input): floor = 2^-38 max|R| sum|x| + 2^-24 max(2^-14 max|x|,
2^-125) rowsum|R|.  Both floors are far below float32's rounding of any normal chunk's largest term.
"""
import numpy as np
import pytest

from conftest import synth_streams

pytestmark = pytest.mark.gpu

RATES = (8000, 24000, 48000)
CONFIGS = [("fft", "tc16"), ("gemm", "fp32"), ("gemm", "tc"), ("gemm", "tc16")]
CONFIG_IDS = ["fft", "gemm-fp32", "gemm-tc", "gemm-tc16"]
# k of the dense bar per build (module docstring); measured worst ratios on a B200 are printed by every test
K_DENSE = {"fp32": 176.0, "tc": 112.0, "tc16": 112.0}
PCMS = ("f32", "s16_32767", "s16_32768")
CAP = 2048
_WORST = {}


@pytest.fixture(scope="module")
def engines(engine_factory):
    made = {}

    def get(resampler, math):
        if (resampler, math) not in made:
            made[(resampler, math)] = engine_factory(CAP, math=math, resampler=resampler)
        return made[(resampler, math)]

    yield get
    if _WORST:
        print("\nworst ratio |y - y64| / (2^-24 |R64| @ |x|) of the dense builds:",
              {m: f"{v:.3f}" for m, v in _WORST.items()})


def _pcm_code(pcm):
    from real_time_vad.engine import capi
    return {"f32": capi.PCM_F32, "s16_32767": capi.PCM_S16_32767, "s16_32768": capi.PCM_S16_32768}[pcm]


def _wire(x, pcm):
    """Float test signal -> what the caller passes (float32, or int16 full scale 32767)."""
    if pcm == "f32":
        return np.asarray(x, np.float32)
    return np.clip(np.round(np.asarray(x, np.float64) * 32767.0), -32768, 32767).astype(np.int16)


def _unit(w, pcm):
    """The float32 samples the kernels see: int16 as float32(q) / 32767 (correctly rounded) or q * 2^-15."""
    if pcm == "f32":
        return np.asarray(w, np.float32)
    q = np.asarray(w).astype(np.float32)
    return q / np.float32(32767.0) if pcm == "s16_32767" else q * np.float32(1.0 / 32768.0)


def _signals(rate, T, pcm, seed=0):
    """One kind of input per stream (float, before the wire format), each T chunks of n_in samples."""
    from scipy import signal
    n_in = rate * 512 // 16000
    L = n_in * T
    rng = np.random.default_rng(seed + rate)
    k = np.arange(L)
    rows = [0.3 * rng.standard_normal(L),
            # test_gpu_resample.py's band-limited source: the 16 kHz recipe resampled to the source rate, plus noise
            signal.resample(synth_streams(1, 512 * T, seed=seed)[0], L) + 0.003 * rng.standard_normal(L),
            np.cos(np.pi * k),                                     # the source's Nyquist tone
            np.cos(np.pi * k * 512 / n_in),                        # the target's Nyquist tone
            np.full(L, 0.5), np.zeros(L),                          # DC and zeros
            np.where(k % 2 == 0, 32767.0, -32768.0) / 32767.0]     # full-scale int16, alternating
    if pcm == "f32":
        rows += [1e-40 * rng.standard_normal(L), 1e30 * rng.standard_normal(L)]   # subnormal, and huge
    for m in range(n_in):                                          # an impulse at every phase of the chunk
        e = np.zeros(L)
        e[m::n_in] = 1.0
        rows.append(e)
    return np.stack(rows), n_in


def _operator(n_in):
    from scipy import signal
    from real_time_vad.engine.stream_engine import StreamEngine
    R64 = signal.resample(np.eye(n_in), 512, axis=0)
    R32 = StreamEngine.resample_matrix(n_in * 16000 // 512).T.astype(np.float64)
    return R64, np.abs(R64), np.abs(R32 - R64)


def _check_chunks(y, x, n_in, resampler, math, live=None, label=""):
    """y [n, T*512] engine output, x [n, T*n_in] float32 input it saw; frames where `live` [n, T] is False must be
    NaN (the hook's fill).  -> worst dense ratio (0 for the FFT resampler)."""
    from scipy import signal
    n = x.shape[0]
    T = x.shape[1] // n_in
    assert y.shape == (n, T * 512), label
    yc = y.reshape(n * T, 512)
    xc = x.reshape(n * T, n_in).astype(np.float64)
    lv = np.ones(n * T, bool) if live is None else np.asarray(live, bool).reshape(n * T)
    if (~lv).any():
        dead = yc[~lv].view(np.uint32)
        assert np.all(dead == 0xFFFFFFFF), f"{label}: a frame that is not live was written"
    yc, xc = yc[lv].astype(np.float64), xc[lv]
    if not len(xc):
        return 0.0
    assert np.all(np.isfinite(yc)), f"{label}: non-finite output in a live frame"
    if resampler == "fft":
        y64 = signal.resample(xc, 512, axis=1)
        half = 0.5 * np.spacing(np.abs(y64).astype(np.float32)).astype(np.float64)
        bar = half * (1 + 1e-6) + 2e-15 * np.abs(xc).max(axis=1, keepdims=True)
        err = np.abs(yc - y64)
        bad = err > bar
        assert not bad.any(), (f"{label}: {int(bad.sum())} samples not correctly rounded; worst "
                               f"{float((err / np.maximum(bar, 1e-300)).max()):.3g} x the bar, at chunk "
                               f"{int((err / np.maximum(bar, 1e-300)).max(axis=1).argmax())}")
        return 0.0
    R64, Ra, Rd = _operator(n_in)
    y64 = xc @ R64.T
    ax = np.abs(xc)
    mag = (ax @ (Ra + Rd).T) * 2.0 ** -24
    fixed = ax @ Rd.T + n_in * 2.0 ** -149
    rowsum = Ra.sum(axis=1)[None, :]
    if math == "tc":
        fixed = fixed + 2.0 ** -126 * rowsum
    elif math == "tc16":
        xmax = ax.max(axis=1, keepdims=True)
        fixed = fixed + 2.0 ** -38 * Ra.max() * ax.sum(axis=1, keepdims=True) + \
            2.0 ** -24 * np.maximum(2.0 ** -14 * xmax, 2.0 ** -125) * rowsum
    err = np.abs(yc - y64)
    excess = np.maximum(err - fixed, 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(excess > 0, excess / mag, 0.0)
    worst = float(ratio.max())
    _WORST[math] = max(_WORST.get(math, 0.0), worst)
    print(f"{label} [gemm/{math}]: worst ratio {worst:.3f} (chunk {int(ratio.max(axis=1).argmax())})")
    k = K_DENSE[math]
    bad = excess > k * mag
    assert not bad.any(), f"{label}: {int(bad.sum())} samples over the {math} bar (k = {k}); worst ratio {worst:.3g}"
    return worst


def _run(eng, wire, pcm, **kw):
    return eng.debug_input(wire, pcm_format=_pcm_code(pcm), **kw)


def _osplit(n, T, num_sms, n_rates=1):
    """launch_step's share of a 64-stream tile's four output blocks (resample_tc_kernel)."""
    rs_tiles = T * ((n + 63) // 64)
    share = (rs_tiles + n_rates - 1) // n_rates
    return 4 if 4 * share <= num_sms else (2 if 2 * share <= num_sms else 1)


def _num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("resampler,math", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("pcm", PCMS)
@pytest.mark.parametrize("rate", RATES)
def test_every_rate_and_pcm_format(engines, resampler, math, pcm, rate):
    eng = engines(resampler, math)
    xf, n_in = _signals(rate, 2, pcm)
    wire = _wire(xf, pcm)
    y = _run(eng, wire, pcm, src_rate=rate)
    worst = _check_chunks(y, _unit(wire, pcm), n_in, resampler, math, label=f"{rate} Hz {pcm}")
    print(f"{resampler}/{math} {rate} Hz {pcm}: {wire.shape[0]} streams, worst ratio {worst:.3f}")


@pytest.mark.parametrize("resampler,math", CONFIGS, ids=CONFIG_IDS)
def test_batch_shapes(engines, resampler, math):
    """Odd batches leave the FFT kernel's warp pair half empty, 64 / 65 is a dense tile edge; the large sizes give each
    osplit regime of resample_tc_kernel (1, 40 and 80 tiles of 64 streams on 148 SMs) and wrap the FFT kernel's
    grid-stride loop (more units than one pass of its grid)."""
    eng = engines(resampler, math)
    rng = np.random.default_rng(5)
    num_sms = _num_sms()
    for i, n in enumerate((1, 2, 3, 33, 63, 64, 65)):
        rate = RATES[i % 3]
        n_in = rate * 512 // 16000
        x = (0.3 * rng.standard_normal((n, 3 * n_in))).astype(np.float32)
        _check_chunks(_run(eng, x, "f32", src_rate=rate), x, n_in, resampler, math, label=f"n={n}")
    T, n_in = 8, 1536
    s2 = num_sms // 2 // T                               # the most 64-stream tiles per frame that still give osplit 2
    seen = set()
    for n in (61, 64 * s2 - 5, 64 * (s2 + 1)):
        x = (0.3 * rng.standard_normal((n, T * n_in))).astype(np.float32)
        _check_chunks(_run(eng, x, "f32", src_rate=48000), x, n_in, resampler, math, label=f"n={n} T={T}")
        seen.add(_osplit(n, T, num_sms))
        if n > 256:
            assert T * ((n + 1) // 2) > num_sms * 8       # the FFT kernel's grid (8 warps per CTA at 48 kHz) wraps
    assert seen == {1, 2, 4}


@pytest.mark.parametrize("resampler,math", CONFIGS, ids=CONFIG_IDS)
def test_ragged_frames(engines, resampler, math):
    """n_frames with 0 and with neighbours of different liveness: live frames meet the bar, the others stay NaN."""
    eng = engines(resampler, math)
    rng = np.random.default_rng(9)
    n, T = 131, 4
    nfr = rng.integers(0, T + 1, n).astype(np.int32)
    nfr[:8] = [0, T, T, 0, 1, 3, 2, 0]
    nfr[64:70] = 0                                           # a dead stretch at a tile edge
    for rate in (8000, 48000):
        n_in = rate * 512 // 16000
        x = (0.3 * rng.standard_normal((n, T * n_in))).astype(np.float32)
        y = _run(eng, x, "f32", src_rate=rate, n_frames=nfr)
        live = np.arange(T)[None, :] < nfr[:, None]
        _check_chunks(y, x, n_in, resampler, math, live=live, label=f"ragged {rate} Hz")


@pytest.mark.parametrize("resampler,math", CONFIGS, ids=CONFIG_IDS)
def test_load_paths(engines, resampler, math):
    """An odd stream_stride (rows too narrow for the 2-D staging): the kernels' scalar loaders; rows 4x wider than
    read: the dense 2-D copy, which must give the tight block's output bit for bit."""
    eng = engines(resampler, math)
    rng = np.random.default_rng(13)
    n, T = 70, 3
    for rate in RATES:
        n_in = rate * 512 // 16000
        for pcm in ("f32", "s16_32767"):
            tight = _wire(0.3 * rng.standard_normal((n, T * n_in)), pcm)
            odd = np.zeros((n, T * n_in + 3), tight.dtype)
            odd[:, :T * n_in] = tight
            wide = np.zeros((n, 4 * T * n_in), tight.dtype)
            wide[:, :T * n_in] = tight
            y0 = _run(eng, tight, pcm, src_rate=rate, max_frames=T)
            y1 = _run(eng, odd, pcm, src_rate=rate, max_frames=T)
            y2 = _run(eng, wide, pcm, src_rate=rate, max_frames=T)
            _check_chunks(y1, _unit(tight, pcm), n_in, resampler, math, label=f"odd stride {rate} {pcm}")
            assert np.array_equal(y0.view(np.uint32), y2.view(np.uint32)), f"dense 2-D staging {rate} {pcm}"
            _check_chunks(y0, _unit(tight, pcm), n_in, resampler, math, label=f"tight {rate} {pcm}")


def _mixed_batch(rng, T, pcm, rates_present=(8000, 48000, 16000)):
    """Rate groups of size 1 (8 kHz), > 64 (48 kHz) and 5 (16 kHz); 24 kHz is absent (a group of size 0)."""
    rates = np.array([8000] + [48000] * 70 + [16000] * 5, np.int32)
    rates = rates[rng.permutation(len(rates))]
    W = T * 1536
    xf = np.zeros((len(rates), W))
    for i, r in enumerate(rates):
        L = T * (r * 512 // 16000)
        xf[i, :L] = 0.3 * rng.standard_normal(L)
    return rates, _wire(xf, pcm)


def _check_mixed(y, wire, rates, pcm, T, resampler, math, label):
    xu = _unit(wire, pcm)
    for r in (8000, 24000, 48000, 16000):
        idx = np.flatnonzero(rates == r)
        if not len(idx):
            continue
        n_in = r * 512 // 16000
        if r == 16000:     # passthrough_kernel: the float32 conversion, bit for bit
            assert np.array_equal(y[idx].view(np.uint32), xu[idx, :T * 512].view(np.uint32)), f"{label}: 16 kHz"
        else:
            _check_chunks(y[idx], xu[idx, :T * n_in], n_in, resampler, math, label=f"{label}: {r} Hz")


@pytest.mark.parametrize("resampler,math", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("pcm", PCMS)
def test_mixed_rates(engines, resampler, math, pcm):
    eng = engines(resampler, math)
    rng = np.random.default_rng(17)
    T = 3
    rates, wire = _mixed_batch(rng, T, pcm)
    y = _run(eng, wire, pcm, src_rates=rates, max_frames=T)
    _check_mixed(y, wire, rates, pcm, T, resampler, math, f"mixed {pcm}")
    # ragged: frames that are not live stay NaN in the pass-through too
    nfr = rng.integers(0, T + 1, len(rates)).astype(np.int32)
    y = _run(eng, wire, pcm, src_rates=rates, max_frames=T, n_frames=nfr)
    dead = (np.arange(T * 512)[None, :] >> 9) >= nfr[:, None]
    assert np.all(y.view(np.uint32)[dead] == 0xFFFFFFFF)
    y = np.where(dead, 0.0, y).astype(np.float32)
    xu = _unit(wire, pcm)
    for i in np.flatnonzero(rates == 16000):
        k = nfr[i] * 512
        assert np.array_equal(y[i, :k].view(np.uint32), xu[i, :k].view(np.uint32))


@pytest.mark.parametrize("resampler,math", CONFIGS, ids=CONFIG_IDS)
def test_output_does_not_depend_on_the_batch(engines, resampler, math):
    """The resampler's copy of test_tc16_result_does_not_depend_on_the_neighbours: fixed probe streams give the same
    output bits alone, among streams 1e6 louder, 1e-5 quieter and all-zero, at other positions, under each osplit."""
    eng = engines(resampler, math)
    rng = np.random.default_rng(21)
    T, n_in = 8, 1536
    probes = np.concatenate([(0.3 * rng.standard_normal((3, T * n_in))),
                             signal_band_limited(T, n_in)]).astype(np.float32)
    P = len(probes)
    ref = _run(eng, probes, "f32", src_rate=48000)
    _check_chunks(ref, probes, n_in, resampler, math, label="probes alone")
    num_sms = _num_sms()
    seen = set()
    s2 = num_sms // 2 // T
    for n, scale in ((70, 1e6), (70, 1e-5), (70, 0.0), (64 * s2 - 5, 1e6), (64 * (s2 + 1), 1e-5)):
        batch = (scale * rng.standard_normal((n, T * n_in))).astype(np.float32)
        pos = rng.choice(np.setdiff1d(np.arange(n), [63]), P, replace=False)
        pos[0] = 63                                           # one probe at the last row of a tile
        batch[pos] = probes
        y = _run(eng, batch, "f32", src_rate=48000)
        seen.add(_osplit(n, T, num_sms))
        assert np.array_equal(y[pos].view(np.uint32), ref.view(np.uint32)), f"n={n} neighbours x{scale}"
    assert seen == {1, 2, 4}


def signal_band_limited(T, n_in):
    from scipy import signal
    return signal.resample(synth_streams(2, 512 * T, seed=4), T * n_in, axis=1)


def _downmix_ref(wire, pcm, C):
    """downmix_kernel's documented arithmetic: the channels converted, added in order in float32, the sum divided by C
    (correctly rounded)."""
    u = _unit(wire, pcm)
    acc = u[..., 0].copy()
    for c in range(1, C):
        acc = (acc + u[..., c]).astype(np.float32)
    return (acc / np.float32(C)).astype(np.float32)


@pytest.mark.parametrize("C", [2, 3, 6])
@pytest.mark.parametrize("pcm", PCMS)
def test_downmix(engines, C, pcm):
    eng = engines("fft", "tc16")
    rng = np.random.default_rng(C * 7 + len(pcm))
    n, T = 37, 3
    # 16 kHz: down-mix only, bit for bit
    wire = _wire(0.4 * rng.standard_normal((n, 512 * T, C)), pcm)
    y = _run(eng, wire, pcm)
    assert y.shape == (n, 512 * T)
    assert np.array_equal(y.view(np.uint32), _downmix_ref(wire, pcm, C).view(np.uint32))
    # hop < frame_len: the d_mono layout (max_frames - 1) * hop + frame_len
    y = _run(eng, wire, pcm, hop=256, max_frames=4)
    assert np.array_equal(y.view(np.uint32), _downmix_ref(wire, pcm, C)[:, :3 * 256 + 512].view(np.uint32))
    # 48 kHz: down-mix, then the FFT bar
    wire = _wire(0.4 * rng.standard_normal((n, 1536 * T, C)), pcm)
    y = _run(eng, wire, pcm, src_rate=48000)
    _check_chunks(y, _downmix_ref(wire, pcm, C), 1536, "fft", "tc16", label=f"downmix C={C} 48 kHz")
    # mixed rates
    rates, _ = _mixed_batch(rng, T, pcm)
    wire = np.zeros((len(rates), T * 1536, C), np.float32 if pcm == "f32" else np.int16)
    for i, r in enumerate(rates):
        L = T * (r * 512 // 16000)
        wire[i, :L] = _wire(0.4 * rng.standard_normal((L, C)), pcm)
    y = _run(eng, wire, pcm, src_rates=rates, max_frames=T)
    mono = _downmix_ref(wire, pcm, C)
    for r in (8000, 48000, 16000):
        idx = np.flatnonzero(rates == r)
        n_in = r * 512 // 16000
        if r == 16000:
            assert np.array_equal(y[idx].view(np.uint32), mono[idx, :T * 512].view(np.uint32))
        else:
            _check_chunks(y[idx], mono[idx, :T * n_in], n_in, "fft", "tc16", label=f"downmix C={C} mixed {r}")


@pytest.mark.parametrize("resampler,math", [("fft", "tc16"), ("gemm", "tc16"), ("gemm", "fp32")])
def test_the_hook_changes_nothing(engine_factory, resampler, math):
    """After debug_input the touched slots' records are unchanged, and the next real step gives the probabilities of a
    fresh engine fed the same audio, bit for bit."""
    n, T = 40, 4
    rng = np.random.default_rng(31)
    a1 = signal_band_limited(T, 1536).astype(np.float32)
    a1 = np.concatenate([a1] * (n // 2)) + (0.01 * rng.standard_normal((n, T * 1536))).astype(np.float32)
    a2 = np.roll(a1, 777, axis=1)
    probe = (0.5 * rng.standard_normal((n, 2 * 1536))).astype(np.float32)
    kw = dict(vad_start_probability=0.5, vad_end_probability=0.35, voice_start_frame_count=2, voice_end_frame_count=3)
    eng_a = engine_factory(64, math=math, resampler=resampler)
    eng_b = engine_factory(64, math=math, resampler=resampler)
    for e in (eng_a, eng_b):
        e.reset()
        e.configure(**kw)
        e.step(a1, src_rate=48000)
    before = eng_a.export_states(list(range(n)))
    eng_a.debug_input(probe, src_rate=48000)
    eng_a.debug_input(probe[:, :1024 * 3].reshape(n, 1024, 3), src_rate=16000)        # down-mix only
    assert before.tobytes() == eng_a.export_states(list(range(n))).tobytes()
    ra, rb = eng_a.step(a2, src_rate=48000), eng_b.step(a2, src_rate=48000)
    assert np.array_equal(ra.probs.view(np.uint32), rb.probs.view(np.uint32))
    assert np.array_equal(ra.flags, rb.flags) and ra.events == rb.events


def test_hook_refuses_what_it_cannot_do(engines):
    from real_time_vad.engine import capi
    from real_time_vad.engine.stream_engine import EngineError
    eng = engines("fft", "tc16")
    with pytest.raises(EngineError) as ei:
        eng.debug_input(np.zeros((2, 1024), np.float32))                 # 16 kHz mono: no input stage
    assert ei.value.code == capi.E_INVALID
    import ctypes as C
    x = np.zeros((2, 1536), np.float32)
    a, keep = eng._args(x, None, None, 1, 1536, 1536, capi.PCM_F32, 48000)
    out = np.zeros(2 * 512 - 1, np.float32)
    assert eng._L.cvad_debug_input(eng.handle, C.byref(a), out.ctypes.data, out.size) == capi.E_CAPACITY
    out = np.zeros(2 * 512, np.float32)
    assert eng._L.cvad_debug_input(eng.handle, C.byref(a), out.ctypes.data, out.size) == 2 * 512


@pytest.mark.parametrize("pcm", ["f32", "s16_32767"])
@pytest.mark.parametrize("rate", [48000, 16000])
def test_misaligned_device_input_equals_the_host_step(engine_factory, pcm, rate):
    """cvad_step_device with the audio one element past an aligned address (float32: 4 bytes, int16: 2 bytes): only
    this path reaches the pointer-alignment half of the `vec` tests of resample_fft_kernel and of the model's loader.
    Probabilities, flags and events equal the host step's bit for bit (the _run_pair pattern of
    test_gpu_device_steps.py, one-frame steps)."""
    import torch
    from real_time_vad.engine import capi
    n, T = 70, 40
    W = rate * 512 // 16000
    audio = _wire(synth_streams(n, W * T, seed=41) * 0.9, pcm)
    cfg = dict(vad_start_probability=0.5, vad_end_probability=0.35, voice_start_frame_count=2, voice_end_frame_count=3,
               enable_denoising=True)
    dev = engine_factory(128)
    host = engine_factory(128)
    for e in (dev, host):
        e.reset()
        e.configure(**cfg)
    cu = "cuda:0"
    dt = torch.float32 if pcm == "f32" else torch.int16
    bufs, outs = [], []
    for j in range(T):
        buf = torch.zeros(n * W + 1, dtype=dt, device=cu)
        frame = torch.from_numpy(np.ascontiguousarray(audio[:, W * j:W * (j + 1)])).to(cu)
        buf[1:] = frame.reshape(-1)
        bufs.append(buf)
        outs.append((torch.full((n,), -1.0, device=cu), torch.full((n,), 255, dtype=torch.uint8, device=cu),
                     torch.zeros(2 * n * 24, dtype=torch.uint8, device=cu), torch.full((1,), 12345, dtype=torch.int32, device=cu)))
    torch.cuda.synchronize()
    for j in range(T):
        a = capi.StepArgs()
        a.n_streams = n
        a.audio = bufs[j].data_ptr() + bufs[j].element_size()
        assert a.audio % 16 != 0
        a.pcm_format = _pcm_code(pcm)
        a.stream_stride = W
        a.max_frames = 1
        a.frame_len = a.hop = W
        a.src_rate = rate
        p, f, ev, nev = outs[j]
        a.probs_out, a.flags_out, a.events_out, a.n_events_out = p.data_ptr(), f.data_ptr(), ev.data_ptr(), nev.data_ptr()
        a.max_events = 2 * n
        dev.step_device(a)
    dev.sync()
    n_events = 0
    for j in range(T):
        r = host.step(np.ascontiguousarray(audio[:, W * j:W * (j + 1)]), max_frames=1, src_rate=rate,
                      pcm_format=_pcm_code(pcm))
        p, f, ev, nev = outs[j]
        assert np.array_equal(p.cpu().numpy().view(np.uint32), r.probs[:, 0].view(np.uint32)), j
        assert np.array_equal(f.cpu().numpy(), r.flags[:, 0]), j
        k = int(nev.cpu()[0])
        assert k == len(r.events), j
        rec = ev.cpu().numpy().view(np.int64)[:3 * k]
        got = sorted((int(q[0]), int(q[1]), int(q[2]), int(q[3]), int(s))
                     for q, s in zip(rec.view(np.int32).reshape(k, 6), rec.reshape(k, 3)[:, 2]))
        assert got == sorted(r.events), j
        n_events += k
    assert n_events > 0
