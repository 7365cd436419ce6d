"""One step's LSTM state transition, unit by unit, against float64, in every build and every step form.

The suite otherwise sees the model kernels through the speech probability (one sigmoid of a dot product over relu(h'),
which barely moves when a unit with a negative h' or a small decoder weight is wrong) and through one stream's h / c
after several steps.  Here cvad_import_states sets each slot's h, c, counters, thresholds and frames_done, one step
runs, and cvad_export_states reads all 128 h' and 128 c' back, so every unit of every stream is held to its own bar.

The float64 references are the reference's own .onnx files interpreted op by op (oracle/onnx_interp.py).  A subclass
records the inputs of every LSTM node it runs (input x, W, R, biases, initial h / c), so the bar of each unit is
derived from the float64 values of that very step:
    da = 2^-24 (|W| |x| + |R| |h| + |b_W| + |b_R|) + |W| dx + |R| dh
is carried through the cell's derivatives (sigmoid' = s (1 - s), tanh' = 1 - t^2) to c' = f c + i g and
h' = o tanh(c'), with one activation error eps added at each sigmoid / tanh, then through the decoder to the
probability.  The bar is K * (that bound) + float32's subnormal unit, K per build measured on a B200.  Layer 1 of v4
takes layer 0's h' and its bound; v4's 8 kHz sub-model runs two time steps per frame and averages two sigmoids.

Part (e) holds the engine's one state rule: |h| <= 2.  The FP16-split kernels of the tc16 build store h in FP16 parts
(scaled by 2^14 in the fused kernel), which overflow from |h| ~ 4 on; such a record is refused, and h = +-2 is computed
on the bar.
"""

import numpy as np
import pytest
from scipy.special import expit

from conftest import V4_ONNX, V5_ONNX, synth_streams

U = 2.0 ** -24
FLOOR = 2.0 ** -149                     # float32's subnormal unit
SFU_EPS = 4e-7                          # ex2.approx + rcp.approx sigmoid / tanh of the v5 tensor-core builds (DESIGN 3e)
LIBM_EPS = 2.0 ** -23                   # expf / tanhf of the FP32 kernels (and v4's recurrent kernel in every math)

BUILDS = [("v5", "tc16"), ("v5", "tc"), ("v5", "fp32"), ("v4", "fft"), ("v4", "tc"), ("v4", "fp32"),
          ("v4_8k", "fft"), ("v4_8k", "tc"), ("v4_8k", "fp32")]
FORMS = ["one", "nofuse", "chained", "three"]

# K: per-unit bar of part (a), in units of the propagated bound: twice the worst ratio measured on one NVIDIA B200
# (1,000 W power limit) over h', c' and the probability, every step form.  The worst is on c' in all of them.  The v4
# builds share one recurrent kernel, and its tanhf / expf error is what reaches 4.9.  The bound of v4's 8 kHz
# sub-model is loose: its two chained time steps double-count the first step's rounding, so its ratio stays below 1.
K_CELL = {("v5", "tc16"): 7.0,       # 3.44
          ("v5", "tc"): 7.5,         # 3.69
          ("v5", "fp32"): 7.0,       # 3.46
          ("v4", "fft"): 10.0,       # 4.91
          ("v4", "tc"): 10.0,        # 4.91
          ("v4", "fp32"): 10.0,      # 4.91
          ("v4_8k", "fft"): 0.7,     # 0.326
          ("v4_8k", "tc"): 0.7,      # 0.326
          ("v4_8k", "fp32"): 0.7}    # 0.326
# kappa: per-stream bar of part (b), in units of the float32 oracle's own deviation from float64, for one-frame forms
# (T = 1) and the 3-frame step (T = 3): twice the worst ratio measured on the same B200 beside each.  One-frame worsts
# are on the probability, a scalar for which the oracle's deviation is a single sample of float32 rounding (the split
# tensor-core builds of v5 are the loosest).  The 3-frame worsts of v5 are on c' of a gated 3e4-gain stream: its gate
# pre-activations are sums of terms near 1e4 whose cancellation error the oracle happens to hit less often.
KAPPA = {("v5", "tc16", 1): 135.0, ("v5", "tc16", 3): 224.0,       # 67.5 (p), 112 (c')
         ("v5", "tc", 1): 109.0, ("v5", "tc", 3): 128.0,           # 54.5 (p), 63.6 (c')
         ("v5", "fp32", 1): 15.0, ("v5", "fp32", 3): 304.0,        # 7.18 (p), 152 (c')
         ("v4", "fft", 1): 13.0, ("v4", "fft", 3): 9.2,            # 6.51 (p), 4.58 (p)
         ("v4", "tc", 1): 11.0, ("v4", "tc", 3): 9.2,              # 5.47 (p), 4.58 (p)
         ("v4", "fp32", 1): 13.0, ("v4", "fp32", 3): 9.2,          # 6.51 (p), 4.58 (p)
         ("v4_8k", "fft", 1): 35.0, ("v4_8k", "fft", 3): 29.0,     # 17.5 (p), 14.5 (p)
         ("v4_8k", "tc", 1): 31.0, ("v4_8k", "tc", 3): 31.0,       # 15.5 (p), 15.4 (p)
         ("v4_8k", "fp32", 1): 30.0, ("v4_8k", "fp32", 3): 27.0}   # 14.8 (p), 13.2 (p)


def _eps(version, math):
    return SFU_EPS if version == "v5" and math in ("tc", "tc16") else LIBM_EPS


# ------------------------------------------------------------------------------------------------ float64 references

def _onnx(version):
    return str(V5_ONNX if version == "v5" else V4_ONNX)


class _Recorder:
    """OnnxInterpreter that keeps the inputs and outputs of every LSTM node it runs."""

    def __new__(cls, path, dtype):
        from onnx_interp import OnnxInterpreter

        class Rec(OnnxInterpreter):
            def _op_LSTM(self, node, ins, scope):
                out = super()._op_LSTM(node, ins, scope)
                self.calls.append(([None if a is None else np.asarray(a, np.float64) for a in ins],
                                   [np.asarray(o, np.float64) for o in out]))
                return out

        it = Rec(path, dtype)
        it.calls = []
        return it


_INTERP = {}


def _interp(version, dtype):
    key = (version, np.dtype(dtype).str)
    if key not in _INTERP:
        _INTERP[key] = _Recorder(_onnx(version), dtype)
    return _INTERP[key]


def _decoder(version):
    """(w, b) of the decoder the probability is made of (the tail of the engine's canonical blob)."""
    from real_time_vad.engine.onnx_weights import canonical_blob_v4, canonical_blob_v5
    if version == "v5":
        blob = canonical_blob_v5(V5_ONNX)
        return blob[-129:-1].astype(np.float64), float(blob[-1])
    blob = canonical_blob_v4(V4_ONNX, branch="8k" if version == "v4_8k" else "16k")
    return blob[-65:-1].astype(np.float64), float(blob[-1])


def _feeds(version, x, h, c, dtype):
    """x [n, 512] f32 (gated), h / c [n, 128] engine rows -> interpreter feeds."""
    n = x.shape[0]
    sr = np.array(8000 if version == "v4_8k" else 16000, np.int64)
    if version == "v5":
        return {"input": x.astype(dtype), "sr": sr, "state": np.stack([h, c]).astype(dtype).reshape(2, n, 128)}
    return {"input": x.astype(dtype), "sr": sr, "h": h.reshape(n, 2, 64).transpose(1, 0, 2).astype(dtype),
            "c": c.reshape(n, 2, 64).transpose(1, 0, 2).astype(dtype)}


def _rows(version, out):
    """interpreter outputs -> probs [n], h [n, 128], c [n, 128] in the engine's row order"""
    p = np.asarray(out[0], np.float64).reshape(-1)
    if version == "v5":
        st = np.asarray(out[1], np.float64)
        return p, st[0], st[1]
    h, c = (np.asarray(o, np.float64) for o in out[1:3])
    return p, h.transpose(1, 0, 2).reshape(-1, 128), c.transpose(1, 0, 2).reshape(-1, 128)


def _gate(x, denoise):
    return np.where(np.abs(x) > 0.01, x, 0.0).astype(np.float32) if denoise else x.astype(np.float32)


def _cell_bound(ins, dx, dh, dc):
    """Propagated error bound of one LSTM node (ONNX gate order i, o, f, c), time step by time step.

    Every error is a pair (m, s): m in units of K 2^-24, s in units of K eps, so the bar is K (2^-24 m + eps s).
    dx: pair of [T, n, in] (None: exact input), dh / dc: pairs of [n, H] -> (pairs of Y [T, n, H], h', c')."""
    X, W, R, B = ins[0], ins[1][0], ins[2][0], ins[3][0]
    H = R.shape[1]
    h, c = ins[5][0], ins[6][0]
    aW, aR, ab = np.abs(W), np.abs(R), np.abs(B[:4 * H]) + np.abs(B[4 * H:])
    ys_m, ys_s = [], []
    for t in range(X.shape[0]):
        x = X[t]
        a = x @ W.T + h @ R.T + B[:4 * H] + B[4 * H:]
        da_m = np.abs(x) @ aW.T + np.abs(h) @ aR.T + ab + dh[0] @ aR.T
        da_s = dh[1] @ aR.T
        if dx is not None:
            da_m = da_m + dx[0][t] @ aW.T
            da_s = da_s + dx[1][t] @ aW.T
        sg = expit(a)
        th = np.tanh(a)
        gi, go, gf, gg = sg[:, :H], sg[:, H:2 * H], sg[:, 2 * H:3 * H], th[:, 3 * H:]
        d = lambda k: (da_m[:, k * H:(k + 1) * H], da_s[:, k * H:(k + 1) * H])   # noqa: E731
        di = (gi * (1 - gi) * d(0)[0], gi * (1 - gi) * d(0)[1] + 1)
        do = (go * (1 - go) * d(1)[0], go * (1 - go) * d(1)[1] + 1)
        df = (gf * (1 - gf) * d(2)[0], gf * (1 - gf) * d(2)[1] + 1)
        dg = ((1 - gg ** 2) * d(3)[0], (1 - gg ** 2) * d(3)[1] + 1)
        cn = gf * c + gi * gg
        dcn = tuple(np.abs(c) * df[k] + gf * dc[k] + np.abs(gg) * di[k] + gi * dg[k] for k in range(2))
        dcn = (dcn[0] + np.abs(gf * c) + np.abs(gi * gg) + np.abs(cn), dcn[1])
        tc = np.tanh(cn)
        dt = ((1 - tc ** 2) * dcn[0], (1 - tc ** 2) * dcn[1] + 1)
        hn = go * tc
        dh = (np.abs(tc) * do[0] + go * dt[0] + np.abs(hn), np.abs(tc) * do[1] + go * dt[1])
        dc = dcn
        h, c = hn, cn
        ys_m.append(dh[0])
        ys_s.append(dh[1])
    return (np.stack(ys_m), np.stack(ys_s)), dh, dc


def reference_frame(version, x, h, c, dh=None, dc=None):
    """One frame in float64 from state (h, c) [n, 128] and its error pairs (None: exact).  x [n, 512] float32, gated.
    -> dict p, h, c (float64) and their bounds dp, dh, dc (pairs, see _cell_bound)."""
    it = _interp(version, np.float64)
    it.calls = []
    p, h1, c1 = _rows(version, it.run(_feeds(version, x, h, c, np.float64)))
    n = x.shape[0]
    layers = len(it.calls)
    H = 128 // layers
    z = np.zeros((n, 128))
    dh = dh or (z, z)
    dc = dc or (z, z)
    out_h, out_c, dx, Y = [], [], None, None
    for L, (ins, outs) in enumerate(it.calls):
        sl = slice(L * H, (L + 1) * H)
        ys, dhL, dcL = _cell_bound(ins, dx if L else None, (dh[0][:, sl], dh[1][:, sl]), (dc[0][:, sl], dc[1][:, sl]))
        dx, Y = ys, outs[0][:, 0]                      # [T, n, H]: the next layer's input
        out_h.append(dhL)
        out_c.append(dcL)
    bh = tuple(np.concatenate([o[k] for o in out_h], axis=1) for k in range(2))
    bc = tuple(np.concatenate([o[k] for o in out_c], axis=1) for k in range(2))
    # the probability: sigmoid(w . relu(y) + b) per time step, averaged over the time steps
    w, b = _decoder(version)
    zz = np.maximum(Y, 0) @ w + b                       # [T, n]
    pt = expit(zz)
    dz_m = dx[0] @ np.abs(w) + np.maximum(Y, 0) @ np.abs(w) + abs(b)
    dz_s = dx[1] @ np.abs(w)
    dp = ((pt * (1 - pt) * dz_m).mean(0) + np.abs(p), (pt * (1 - pt) * dz_s + 1).mean(0))
    return dict(p=p, h=h1, c=c1, dp=dp, dh=bh, dc=bc, p_dec=pt.mean(0))


def reference_run(version, audio, h, c, denoise, frames):
    """`frames` frames from (h, c) in float64 with the bound carried from frame to frame -> probs [n, T], bounds [n, T]
    (pairs), final state and its bounds."""
    dh = dc = None
    ps, dps = [], []
    for j in range(frames):
        r = reference_frame(version, _gate(audio[:, 512 * j:512 * (j + 1)], denoise), h, c, dh, dc)
        h, c, dh, dc = r["h"], r["c"], r["dh"], r["dc"]
        ps.append(r["p"])
        dps.append(r["dp"])
    return (np.stack(ps, 1), tuple(np.stack([d[k] for d in dps], 1) for k in range(2)), h, c, dh, dc)


def fp32_oracle_run(version, audio, h, c, denoise, frames, ref_v5, ref_v4):
    """The float32 oracle from (h, c): the C restatement (RefV5 / RefV4 .frame) or, for v4's 8 kHz sub-model, the
    interpreter in float32."""
    n = audio.shape[0]
    h, c = h.astype(np.float32).copy(), c.astype(np.float32).copy()
    probs = np.zeros((n, frames))
    for j in range(frames):
        x = _gate(audio[:, 512 * j:512 * (j + 1)], denoise)
        if version == "v4_8k":
            probs[:, j], h, c = _rows(version, _interp(version, np.float32).run(_feeds(version, x, h, c, np.float32)))
            h, c = h.astype(np.float32), c.astype(np.float32)
            continue
        for s in range(n):
            if version == "v5":
                hs, cs = h[s].copy(), c[s].copy()
                probs[s, j], _ = ref_v5.frame(x[s], hs, cs)
            else:
                hs, cs = h[s].reshape(2, 64).copy(), c[s].reshape(2, 64).copy()
                probs[s, j], _ = ref_v4.frame(x[s], hs, cs)
            h[s], c[s] = hs.reshape(128), cs.reshape(128)
    return probs, h.astype(np.float64), c.astype(np.float64)


# ---------------------------------------------------------------------------------------------------- engine helpers

def _engine(version, math, max_streams, form, monkeypatch):
    from real_time_vad.engine.stream_engine import StreamEngine
    if form == "nofuse":
        monkeypatch.setenv("CVAD_FUSE", "0")
    else:
        monkeypatch.delenv("CVAD_FUSE", raising=False)
    eng = StreamEngine(version, max_streams=max_streams, math=math)
    monkeypatch.delenv("CVAD_FUSE", raising=False)
    return eng


def _records(h, c, *, denoise=False, start_p=1.0, end_p=0.0, active=0, scount=0, ecount=0, n_start=1000,
             n_end=1000, frames_done=0):
    from real_time_vad.engine import capi
    n = h.shape[0]
    r = np.zeros(n, capi.STATE_DTYPE)
    r["h"], r["c"] = h, c
    r["frames_done"] = frames_done
    r["vad_start_probability"], r["vad_end_probability"] = start_p, end_p
    r["is_voice_active"], r["voice_start_frame_count"], r["voice_end_frame_count"] = active, scount, ecount
    r["n_start"], r["n_end"] = n_start, n_end
    r["enable_denoising"] = int(denoise)
    return r


def _step(eng, form, audio, slots, n_frames=None):
    """One step of `form` over audio [n, T * 512] -> (probs [n, T], flags [n, T], events (stream, frame, kind,
    stream_frame))."""
    if form == "chained":
        import torch
        from real_time_vad.engine import capi
        n = audio.shape[0]
        dev = f"cuda:{eng.device}"
        x = torch.from_numpy(np.ascontiguousarray(audio[:, :512])).to(dev)
        p = torch.full((n, 1), -1.0, device=dev)
        f = torch.full((n, 1), 255, dtype=torch.uint8, device=dev)
        ev = torch.zeros(2 * n * 24, dtype=torch.uint8, device=dev)
        nev = torch.zeros(1, dtype=torch.int32, device=dev)
        sd = torch.from_numpy(np.ascontiguousarray(slots, np.int32)).to(dev)
        a = capi.StepArgs()
        a.n_streams, a.audio, a.pcm_format, a.stream_stride = n, x.data_ptr(), capi.PCM_F32, 512
        a.max_frames, a.frame_len, a.hop, a.src_rate = 1, 512, 512, 16000
        a.slots, a.probs_out, a.flags_out = sd.data_ptr(), p.data_ptr(), f.data_ptr()
        a.events_out, a.max_events, a.n_events_out = ev.data_ptr(), 2 * n, nev.data_ptr()
        torch.cuda.synchronize(dev)
        eng.step_device(a)
        eng.sync()
        k = min(int(nev.cpu()[0]), 2 * n)
        rec = ev.cpu().numpy().view(np.int64)[:3 * k]
        r32 = rec.view(np.int32).reshape(k, 6)
        sf = rec.reshape(k, 3)[:, 2]
        events = sorted((int(r[0]), int(r[2]), int(r[3]), int(s)) for r, s in zip(r32, sf))
        return p.cpu().numpy().astype(np.float64), f.cpu().numpy(), events
    T = audio.shape[1] // 512
    r = eng.step(np.ascontiguousarray(audio), slots=np.asarray(slots, np.int32), n_frames=n_frames, max_frames=T)
    events = sorted((s, j, k, sf) for (s, _, j, k, sf) in r.events)
    return r.probs.astype(np.float64), r.flags, events


def _frames(form):
    return 3 if form == "three" else 1


# ---------------------------------------------------------------------------------------------------- imported states

def _cell_states(n_rep=4, seed=0):
    """h / c rows covering the cases of part (a): h ~ U(-1, 1), h = +-1 and +-2 exactly, h = 0, h at 1e-30 and at the
    subnormal 1e-40, one unit at 1 with the rest at 1e-6; c at 0, 1e-3 N(0, 1), N(0, 1), 30 N(0, 1) and subnormal."""
    rng = np.random.default_rng(seed)
    hs = [rng.uniform(-1, 1, 128), np.ones(128), -np.ones(128), np.where(rng.random(128) < 0.5, 1.0, -1.0),
          np.zeros(128), np.full(128, 1e-30), np.full(128, 1e-40) * np.where(rng.random(128) < 0.5, 1, -1),
          np.where(np.arange(128) == 37, 1.0, 1e-6), np.full(128, 2.0), np.where(rng.random(128) < 0.5, 2.0, -2.0)]
    cs = [np.zeros(128), 1e-3 * rng.standard_normal(128), rng.standard_normal(128), 30 * rng.standard_normal(128),
          np.full(128, 1e-40) * np.where(rng.random(128) < 0.5, 1, -1)]
    H, Cc = [], []
    for _ in range(n_rep):
        for hv in hs:
            for cv in cs:
                H.append(hv)
                Cc.append(cv)
    H = np.array(H, np.float32)
    Cc = np.array(Cc, np.float32)
    return H, Cc


def _bar(K, eps, pair):
    return K * (U * pair[0] + eps * pair[1]) + FLOOR


def _worst(name, err, pair, K, eps):
    """print and return the worst ratio of err to the bound with K = 1"""
    ratio = err / (U * pair[0] + eps * pair[1] + FLOOR / K)
    w = float(ratio.max())
    print(f"{name}: worst ratio {w:.3g} (K {K:g})")
    return w


# --------------------------------------------------------------------------------------------------- (a) the cell

@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("version,math", BUILDS)
def test_cell_in_isolation_per_unit(version, math, form, monkeypatch):
    """Zero audio (and, with the gate on, audio whose samples are all within 0.01): the cell's input is the front end's
    constant, and every unit's c' and h', and the probability, stay within K times the propagated float64 bound."""
    H, Cc = _cell_states()
    n = H.shape[0]
    T = _frames(form)
    rng = np.random.default_rng(3)
    denoise = np.arange(n) % 2 == 1
    audio = np.where(denoise[:, None], rng.uniform(-0.0099, 0.0099, (n, 512 * T)), 0.0).astype(np.float32)
    eng = _engine(version, math, n + 5, form, monkeypatch)
    slots = np.arange(n, dtype=np.int32)[::-1].copy()
    rec = _records(H, Cc)
    rec["enable_denoising"] = denoise
    eng.import_states(slots, rec)
    probs, _, _ = _step(eng, form, audio, slots)
    out = eng.export_states(slots)
    eng.close()
    p64, dp, h64, c64, dh, dc = reference_run(version, audio, H.astype(np.float64), Cc.astype(np.float64), True, T)
    K, eps = K_CELL[(version, math)], _eps(version, math)
    eh = np.abs(out["h"] - h64)
    ec = np.abs(out["c"] - c64)
    ep = np.abs(probs - p64)
    tag = f"{version}/{math}/{form}"
    w = max(_worst(tag + " h'", eh, dh, K, eps), _worst(tag + " c'", ec, dc, K, eps), _worst(tag + " p", ep, dp, K, eps))
    assert np.isfinite(out["h"]).all() and np.isfinite(out["c"]).all() and np.isfinite(probs).all()
    bad = np.argwhere(eh > _bar(K, eps, dh))
    assert not bad.size, f"h' off the bar at (stream, unit) {bad[:5].tolist()}: worst ratio {w:.3g}"
    bad = np.argwhere(ec > _bar(K, eps, dc))
    assert not bad.size, f"c' off the bar at (stream, unit) {bad[:5].tolist()}: worst ratio {w:.3g}"
    bad = np.argwhere(ep > _bar(K, eps, dp))
    assert not bad.size, f"p off the bar at (stream, frame) {bad[:5].tolist()}: worst ratio {w:.3g}"
    assert (out["frames_done"] == T).all()


# ---------------------------------------------------------------------------------------- (b) front end through cell

@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("version,math", BUILDS)
def test_front_end_through_the_cell_per_stream(version, math, form, monkeypatch, ref_v5, ref_v4):
    """synth_streams audio at gains 1e-4 ... 3e4 from random imported states: per stream, the engine's deviation from
    float64 on h', c' and the probability is at most kappa times the float32 oracle's own (or 2^-24 of the value)."""
    gains = np.array([1e-4, 1e-2, 1.0, 30.0, 3e4])
    n = 40
    T = _frames(form)
    rng = np.random.default_rng(11)
    audio = synth_streams(n, 512 * (T + 4), seed=5)[:, 512 * 4:] * np.repeat(gains, n // len(gains))[:, None]
    audio = audio.astype(np.float32)
    H = rng.uniform(-1, 1, (n, 128)).astype(np.float32)
    Cc = (rng.standard_normal((n, 128)) * 3).astype(np.float32)
    denoise = np.arange(n) % 3 == 0
    eng = _engine(version, math, 64, form, monkeypatch)
    slots = rng.permutation(64)[:n].astype(np.int32)
    rec = _records(H, Cc)
    rec["enable_denoising"] = denoise
    eng.import_states(slots, rec)
    probs, _, _ = _step(eng, form, audio, slots)
    out = eng.export_states(slots)
    eng.close()
    kappa = KAPPA[(version, math, T)]
    stream_gain = np.repeat(gains, n // len(gains))
    worst, fails = {}, []
    for dn in (False, True):
        sel = denoise == dn
        a = audio[sel]
        p64, _, h64, c64, _, _ = reference_run(version, a, H[sel].astype(np.float64), Cc[sel].astype(np.float64), dn, T)
        p32, h32, c32 = fp32_oracle_run(version, a, H[sel], Cc[sel], dn, T, ref_v5, ref_v4)
        for name, eng_v, v64, v32 in (("h'", out["h"][sel], h64, h32), ("c'", out["c"][sel], c64, c32),
                                      ("p", probs[sel], p64, p32)):
            assert np.isfinite(eng_v).all(), name
            e = np.abs(eng_v - v64).reshape(len(a), -1).max(1)
            ref = np.maximum(np.abs(v32 - v64).reshape(len(a), -1).max(1),
                             U * np.abs(v64).reshape(len(a), -1).max(1))
            ratio = e / np.maximum(ref, FLOOR)
            k = int(ratio.argmax())
            if ratio[k] > worst.get(name, (0.0,))[0]:
                worst[name] = (float(ratio[k]), float(stream_gain[sel][k]), dn)
            fails += [(name, float(stream_gain[sel][i]), dn, float(ratio[i])) for i in np.flatnonzero(ratio > kappa)]
    for name, (r, g, dn) in worst.items():
        print(f"{version}/{math}/{form} {name}: worst kappa ratio {r:.3g} at gain {g:g}, gate {dn} (kappa {kappa:g})")
    assert not fails, fails[:5]


# ----------------------------------------------------------------------------------- (c) layout and store of state

def _slot_lists(n_slots, rng):
    g = (n_slots - 8) // 8
    aligned = np.concatenate([8 * k + np.arange(8) for k in rng.permutation(g)[:38]])
    yield "one", np.array([n_slots - 1], np.int32)
    yield "aligned", aligned[:32]
    yield "shifted", (aligned[:33] + 1)
    yield "reversed", np.concatenate([a[::-1] for a in aligned[:32].reshape(4, 8)])[:31]
    mix = np.concatenate([aligned[:16], rng.choice(np.setdiff1d(np.arange(n_slots), aligned[:16]), 17, replace=False)])
    yield "aligned+scattered", mix
    yield "permutation", rng.permutation(n_slots)[:300]


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["one", "nofuse", "three"])
@pytest.mark.parametrize("version,math", BUILDS)
def test_state_layout_and_store_paths(version, math, form, monkeypatch):
    """max_streams = 1003 (state_at's last row of 8 is partial), 1 ... 300 streams over aligned, shifted, reversed,
    mixed and permuted slot lists, with a dead stream (n_frames = 0) and a NaN stream inside aligned groups.  Every slot
    not stepped, and the dead and NaN streams, keep their whole record bit for bit; the others are on the cell's bar."""
    N = 1003
    T = _frames(form)
    rng = np.random.default_rng(7)
    eng = _engine(version, math, N, form, monkeypatch)
    H0 = rng.uniform(-1, 1, (N, 128)).astype(np.float32)
    C0 = (2 * rng.standard_normal((N, 128))).astype(np.float32)
    K, eps = K_CELL[(version, math)], _eps(version, math)
    for name, slots in _slot_lists(N, rng):
        slots = np.asarray(slots, np.int32)
        n = slots.size
        rec0 = _records(H0, C0, frames_done=5)
        eng.import_states(None, rec0)
        before = eng.export_states(None)
        audio = np.zeros((n, 512 * T), np.float32)
        n_frames = np.full(n, T, np.int32)
        dead = nan = -1
        if n >= 16:
            dead, nan = 3, 12                              # inside the first and second group of an aligned list
            n_frames[dead] = 0
            audio[nan, 100] = np.nan
        _step(eng, form, audio, slots, n_frames=n_frames)
        after = eng.export_states(None)
        keep = np.ones(N, bool)
        keep[slots] = False
        for k in (dead, nan):
            if k >= 0:
                keep[slots[k]] = True
        changed = [int(i) for i in np.flatnonzero(keep) if after[i].tobytes() != before[i].tobytes()]
        assert not changed, (name, changed[:5])
        live = np.array([k for k in range(n) if k not in (dead, nan)])
        ls = slots[live]
        _, _, h64, c64, dh, dc = reference_run(version, audio[live], H0[ls].astype(np.float64),
                                               C0[ls].astype(np.float64), False, T)
        assert (np.abs(after["h"][ls] - h64) <= _bar(K, eps, dh)).all(), name
        assert (np.abs(after["c"][ls] - c64) <= _bar(K, eps, dc)).all(), name
        assert (after["frames_done"][ls] == 5 + T).all(), name
    eng.close()


# ---------------------------------------------------------------------------- (d) the state machine from imports

def _oracle_sm(p_rows, start_p, end_p, active, scount, ecount, n_start, n_end):
    """vad_oracle.StateMachine with its deques pre-filled to match imported counters: `scount` consecutive frames at
    or above the start threshold (`ecount` below the end threshold) end the deque; what came before them cannot reach
    a window of n_start (n_end) frames that the counter does not already fill."""
    from vad_oracle import StateMachine
    sm = StateMachine(start_p, end_p, 0.8, 0.95, n_start, n_end)
    sm.active = bool(active)
    sm.scount, sm.ecount = scount, ecount
    sm.recent_start.extend([True] * scount)
    sm.recent_end.extend([True] * ecount)
    flags = [sm.step(float(np.float32(p))) for p in p_rows]
    return flags, sm


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("version,math", BUILDS)
def test_state_machine_from_imported_counters(version, math, form, monkeypatch):
    """Thresholds at the engine's own probability p (fires: start p >= thr, end p < thr) and one double ulp beside it
    (does not), counters one short of n_start in {20, 21} / n_end in {100, 101} (the deque caps: 21 and 101 never
    fire), frames_done = 2^40 + 7: events, flags, counters and frames_done against the oracle's state machine."""
    T = _frames(form)
    fd0 = (1 << 40) + 7
    cases = []
    for n_start in (20, 21):
        for thr in ("eq", "up", "down"):
            cases.append(dict(active=0, n_start=n_start, n_end=100, thr=thr))
    for n_end in (100, 101):
        for thr in ("eq", "up", "down"):
            cases.append(dict(active=1, n_start=20, n_end=n_end, thr=thr))
    reps = 6
    n = len(cases) * reps
    rng = np.random.default_rng(17)
    H = rng.uniform(-1, 1, (n, 128)).astype(np.float32)
    Cc = rng.standard_normal((n, 128)).astype(np.float32)
    audio = synth_streams(n, 512 * T, seed=23)
    eng = _engine(version, math, n + 8, form, monkeypatch)
    slots = rng.permutation(n + 8)[:n].astype(np.int32)
    eng.import_states(slots, _records(H, Cc, frames_done=fd0))
    p_probe, _, _ = _step(eng, form, audio, slots)
    act = np.array([cases[i // reps]["active"] for i in range(n)])
    ns = np.array([cases[i // reps]["n_start"] for i in range(n)])
    ne = np.array([cases[i // reps]["n_end"] for i in range(n)])
    thr = [cases[i // reps]["thr"] for i in range(n)]
    p0 = p_probe[:, 0]
    pick = {"eq": lambda p: p, "up": lambda p: np.nextafter(p, 1.0), "down": lambda p: np.nextafter(p, 0.0)}
    tp = np.array([pick[thr[i]](float(p0[i])) for i in range(n)])
    start_p = np.where(act == 0, tp, 0.5)
    end_p = np.where(act == 1, tp, 0.5)
    rec = _records(H, Cc, start_p=start_p, end_p=end_p, active=act, scount=np.where(act == 0, ns - 1, 0),
                   ecount=np.where(act == 1, ne - 1, 0), n_start=ns, n_end=ne, frames_done=fd0)
    eng.import_states(slots, rec)
    probs, flags, events = _step(eng, form, audio, slots)
    out = eng.export_states(slots)
    eng.close()
    assert np.array_equal(probs, p_probe), "the kernels are not deterministic"
    want_events = []
    fired = 0
    for i in range(n):
        fl, sm = _oracle_sm(probs[i], start_p[i], end_p[i], act[i], rec["voice_start_frame_count"][i],
                            rec["voice_end_frame_count"][i], ns[i], ne[i])
        assert [int(f) & 7 for f in flags[i]] == fl, (i, cases[i // reps], flags[i].tolist(), fl)
        for j, f in enumerate(fl):
            for kind, bit in ((1, 1), (2, 2)):
                if f & bit:
                    want_events.append((i, j, kind, fd0 + j))
        fired += bool(fl[0] & 3)
        assert (out["is_voice_active"][i], out["voice_start_frame_count"][i], out["voice_end_frame_count"][i]) == \
            (int(sm.active), sm.scount, sm.ecount), (i, cases[i // reps])
    assert sorted(events) == sorted(want_events)
    assert (out["frames_done"] == fd0 + T).all()
    # fired on frame 0: n_start 20 with the threshold at p or below it, n_end 100 with the threshold above p
    assert fired == 3 * reps, fired


# ------------------------------------------------------------------------------------------------ (e) the |h| bound

@pytest.mark.gpu
@pytest.mark.parametrize("version,math", BUILDS)
def test_states_beyond_the_h_bound_are_refused(version, math, monkeypatch):
    """|h| > 2 is refused by cvad_import_states (all or nothing, the index named) and cvad_set_state, host and device
    records alike; h = +-2 is accepted.  After real runs the engine never exports |h| > 1 + 2^-20."""
    import torch
    from real_time_vad.engine import capi
    from real_time_vad.engine.stream_engine import EngineError
    n = 64
    eng = _engine(version, math, n, "one", monkeypatch)
    eng.reset()
    audio = synth_streams(n, 512 * 24, seed=29) * np.repeat([1.0, 30.0, 3e4, 1e-3], n // 4)[:, None].astype(np.float32)
    for j in range(0, 24, 8):
        eng.step(audio[:, 512 * j:512 * (j + 8)])
    for j in range(3):
        eng.step(audio[:, 512 * j:512 * (j + 1)])          # one-frame steps: the fused kernel under tc / tc16
    before = eng.export_states(None)
    assert np.abs(before["h"]).max() <= 1 + 2.0 ** -20, float(np.abs(before["h"]).max())
    assert np.isfinite(before["c"]).all()
    for bad_h in (4.0, -4.0, float(np.nextafter(np.float32(2), np.float32(3))), np.inf):
        rec = before[10:20].copy()
        rec["h"][6, 77] = bad_h
        for where in ("host", "device"):
            with pytest.raises(EngineError) as ei:
                if where == "host":
                    eng.import_states(np.arange(10, 20), rec)
                else:
                    d = torch.from_numpy(rec.view(np.uint8).copy()).to("cuda:0")
                    torch.cuda.synchronize()
                    eng.import_states(np.arange(10, 20), d.data_ptr())
            assert ei.value.code == capi.E_INVALID and "record 6 " in ei.value.message and "[-2, 2]" in ei.value.message
        h = before["h"][3].copy()
        h[0] = bad_h
        with pytest.raises(EngineError) as ei:
            eng.set_state(3, h, before["c"][3])
        assert ei.value.code == capi.E_INVALID
        assert eng.export_states(None).tobytes() == before.tobytes()
    ok = before[:2].copy()
    ok["h"][0] = 2.0
    ok["h"][1] = -2.0
    eng.import_states([0, 1], ok)
    eng.set_state(2, np.full(128, -2.0, np.float32), before["c"][2])
    assert np.array_equal(eng.export_states([0, 1])["h"], ok["h"])
    eng.close()


@pytest.mark.gpu
def test_ort_seam_and_wrapper_refuse_h_beyond_the_bound():
    from real_time_vad import SileroModelVersion, VADConfig
    from real_time_vad.core.exceptions import ConfigurationError
    from real_time_vad.core.silero_model import VADProcessor
    from real_time_vad.engine import ort_compat
    s5 = ort_compat.InferenceSession(str(V5_ONNX))
    x = np.zeros((1, 512), np.float32)
    state = np.zeros((2, 1, 128), np.float32)
    state[0, 0, 5] = 2.0
    s5.run(None, {"input": x, "state": state, "sr": np.array(16000, np.int64)})       # at the bound: fine
    for v in (2.5, -4.0, np.nan):
        state[0, 0, 5] = v
        with pytest.raises(ValueError):
            s5.run(None, {"input": x, "state": state, "sr": np.array(16000, np.int64)})
    s5.close()
    s4 = ort_compat.InferenceSession(str(V4_ONNX))
    h = np.zeros((2, 1, 64), np.float32)
    h[1, 0, 3] = -3.0
    for sr in (16000, 8000):
        with pytest.raises(ValueError):
            s4.run(None, {"input": x, "h": h, "c": np.zeros((2, 1, 64), np.float32), "sr": np.array(sr, np.int64)})
    s4.close()
    proc = VADProcessor(VADConfig(model_version=SileroModelVersion.V5))
    assert proc.supports_batched()
    ms = proc.model.model_state
    st = np.zeros((2, 1, 128), np.float32)
    st[0, 0, 9] = 3.0
    ms.__dict__["state"] = st
    with pytest.raises(ConfigurationError):
        list(proc.process_audio_batched(np.zeros(512 * 4, np.float32), 512, 512))


# ------------------------------------------------------------------------------------- CPU pin of the references

def test_float64_references_agree_from_arbitrary_states(ref_v4):
    """The float64 interpreter against PyTorch's LSTMCell (v5, to 1e-12) and against the C oracle's float32 v4 (within
    float32's deviation) from h ~ U(-1, 1), c ~ N(0, 3); the bound machinery's own cell and decoder reproduce the
    interpreter's h', c' and probability to 1e-12 in every model."""
    import torch
    from torch_reference import TorchV5
    from vad_oracle import v5_named_weights
    rng = np.random.default_rng(2)
    n = 16
    x = (0.3 * rng.standard_normal((n, 512))).astype(np.float32)
    x[:4] = 0.0
    h = rng.uniform(-1, 1, (n, 128))
    c = 3 * rng.standard_normal((n, 128))
    t64 = TorchV5(v5_named_weights(str(V5_ONNX)), torch.float64)
    pt, ht, ct = t64.frame(x.astype(np.float64), h, c)
    r = reference_frame("v5", x, h, c)
    assert np.abs(pt - r["p"]).max() <= 1e-12
    assert np.abs(ht - r["h"]).max() <= 1e-12 and np.abs(ct - r["c"]).max() <= 1e-12
    for version in ("v5", "v4", "v4_8k"):
        r = reference_frame(version, x, h, c)
        assert np.abs(r["p_dec"] - r["p"]).max() <= 1e-12, version
        calls = _interp(version, np.float64).calls
        H = 128 // len(calls)
        for L, (_, outs) in enumerate(calls):
            assert np.abs(outs[1][0] - r["h"][:, L * H:(L + 1) * H]).max() <= 1e-12, (version, L)
            assert np.abs(outs[2][0] - r["c"][:, L * H:(L + 1) * H]).max() <= 1e-12, (version, L)
        for name in ("dh", "dc", "dp"):
            assert all(np.isfinite(a).all() and (a >= 0).all() for a in r[name]), (version, name)
    # v4 (16 kHz): the C oracle in float32 from the same states
    r = reference_frame("v4", x, h, c)
    p32 = np.zeros(n)
    h32 = np.zeros((n, 128))
    c32 = np.zeros((n, 128))
    for s in range(n):
        hs = h[s].astype(np.float32).reshape(2, 64).copy()
        cs = c[s].astype(np.float32).reshape(2, 64).copy()
        p32[s], _ = ref_v4.frame(x[s], hs, cs)
        h32[s], c32[s] = hs.reshape(128), cs.reshape(128)
    assert np.abs(p32 - r["p"]).max() <= 1e-5
    assert np.abs(h32 - r["h"]).max() <= 1e-5
    assert (np.abs(c32 - r["c"]) <= 1e-5 * np.maximum(1, np.abs(r["c"]))).all()
