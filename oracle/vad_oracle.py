"""ORACLE (test infrastructure, never shipped): CPU restatement of the hot path.

Python/numpy restatements of the reference's host-side steps (each function cites
the reference file:line it follows) plus ctypes bindings for the plain-C model
restatement in oracle/silero_ref.c.  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs may import this module; the
product (cutter-vad_b200/) never does.

Pinning (tests/test_oracle_pinning.py): the reference pins no probability vectors and its own runtime,
onnxruntime, is absent from this image, so model arithmetic is pinned against the two third-party executors that
ARE here -- OpenCV's DNN module running the reference's own graphs (oracle/onnx_flatten.py) and PyTorch's conv1d /
LSTMCell kernels fed the file's tensors (oracle/torch_reference.py); NOT against onnxruntime itself.  The state machine
is pinned against the reference's own test expectations, framing against tests/test_audio_utils.py, end to end
against SampleVoiceMono.wav -> 4 segments.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys
from collections import deque
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
if _HERE not in sys.path:
    sys.path.insert(0, _HERE)

from onnx_wire import Graph, load_model  # noqa: E402

BUILD_DIR = os.path.join(_HERE, "_build")

# ----------------------------------------------------------------------------
# weights: canonical blob from the reference's .onnx (see silero_ref.c header)
# ----------------------------------------------------------------------------

V5_ORDER = [
    ("stft.forward_basis_buffer", (258, 1, 256)),
    ("encoder.0.reparam_conv.weight", (128, 129, 3)),
    ("encoder.0.reparam_conv.bias", (128,)),
    ("encoder.1.reparam_conv.weight", (64, 128, 3)),
    ("encoder.1.reparam_conv.bias", (64,)),
    ("encoder.2.reparam_conv.weight", (64, 64, 3)),
    ("encoder.2.reparam_conv.bias", (64,)),
    ("encoder.3.reparam_conv.weight", (128, 64, 3)),
    ("encoder.3.reparam_conv.bias", (128,)),
    ("decoder.rnn.weight_ih", (512, 128)),
    ("decoder.rnn.weight_hh", (512, 128)),
    ("decoder.rnn.bias_ih", (512,)),
    ("decoder.rnn.bias_hh", (512,)),
    ("decoder.decoder.2.weight", (1, 128, 1)),
    ("decoder.decoder.2.bias", (1,)),
]


def v5_named_weights(onnx_path: str, branch: str = "then_branch") -> Dict[str, np.ndarray]:
    """v5.onnx keeps its weights as Constant nodes inside the If(sr==16000) branches,
    named `If_0_<branch>__Inline_0__<torch name>` (SURVEY.md section 2 row 10)."""
    m = load_model(onnx_path)
    if_node = [n for n in m.graph.nodes if n.op == "If"][0]
    g: Graph = if_node.attrs[branch]
    out: Dict[str, np.ndarray] = {}
    for n in g.nodes:
        if n.op == "Constant":
            v = n.attrs.get("value")
            if isinstance(v, np.ndarray) and v.dtype == np.float32 and "__Inline_0__" in n.outputs[0]:
                out[n.outputs[0].split("__Inline_0__", 1)[1]] = v
    return out


def v5_blob(onnx_path: str) -> np.ndarray:
    named = v5_named_weights(onnx_path)
    parts = []
    for name, shape in V5_ORDER:
        a = named[name]
        assert tuple(a.shape) == shape, (name, a.shape, shape)
        parts.append(np.ascontiguousarray(a, dtype=np.float32).reshape(-1))
    blob = np.concatenate(parts)
    assert blob.size == 309633
    return blob


V4_ORDER = [
    ("model.feature_extractor.forward_basis_buffer", 258 * 256), ("model.adaptive_normalization.filter_", 7),
    ("model.first_layer.0.dw_conv.0.weight", 258 * 5), ("model.first_layer.0.dw_conv.0.bias", 258),
    ("model.first_layer.0.pw_conv.0.weight", 16 * 258), ("model.first_layer.0.pw_conv.0.bias", 16),
    ("model.first_layer.0.proj.weight", 16 * 258), ("model.first_layer.0.proj.bias", 16),
    ("1110", 256), ("1111", 16),
    ("model.encoder.3.0.dw_conv.0.weight", 80), ("model.encoder.3.0.dw_conv.0.bias", 16),
    ("model.encoder.3.0.pw_conv.0.weight", 512), ("model.encoder.3.0.pw_conv.0.bias", 32),
    ("model.encoder.3.0.proj.weight", 512), ("model.encoder.3.0.proj.bias", 32),
    ("1113", 1024), ("1114", 32),
    ("model.encoder.7.0.dw_conv.0.weight", 160), ("model.encoder.7.0.dw_conv.0.bias", 32),
    ("model.encoder.7.0.pw_conv.0.weight", 1024), ("model.encoder.7.0.pw_conv.0.bias", 32),
    ("1116", 1024), ("1117", 32),
    ("model.encoder.11.0.dw_conv.0.weight", 160), ("model.encoder.11.0.dw_conv.0.bias", 32),
    ("model.encoder.11.0.pw_conv.0.weight", 2048), ("model.encoder.11.0.pw_conv.0.bias", 64),
    ("model.encoder.11.0.proj.weight", 2048), ("model.encoder.11.0.proj.bias", 64),
    ("1119", 4096), ("1120", 64),
    ("343", 16384), ("345", 16384), ("347", 512), ("415", 16384), ("417", 16384), ("419", 512),
    ("model.decoder.decoder.1.weight", 64), ("model.decoder.decoder.1.bias", 1),
]


def _all_float_tensors(g: Graph, out: Dict[str, np.ndarray]) -> None:
    for k, v in g.initializers.items():
        if v.dtype == np.float32:
            out.setdefault(k, v)
    for n in g.nodes:
        for a in n.attrs.values():
            if isinstance(a, Graph):
                _all_float_tensors(a, out)


def v4_blob(onnx_path: str) -> np.ndarray:
    """v4 keeps conv weights as top-level initializers (`model.*`, anonymous 1110..1120) and the
    LSTM weights as anonymous initializers inside the nested If subgraphs of the 16 kHz branch
    (343,345,347 / 415,417,419) -- SURVEY.md section 2 row 10 and section 8a S4 row 13."""
    m = load_model(onnx_path)
    named: Dict[str, np.ndarray] = {}
    _all_float_tensors(m.graph, named)
    parts = []
    for name, size in V4_ORDER:
        a = named[name]
        assert a.size == size, (name, a.shape, size)
        parts.append(np.ascontiguousarray(a, dtype=np.float32).reshape(-1))
    blob = np.concatenate(parts)
    assert blob.size == 155908
    return blob


# ----------------------------------------------------------------------------
# C restatement: build + bind
# ----------------------------------------------------------------------------

def build_ref_lib(native: bool = False, force: bool = False, build_dir: str = BUILD_DIR) -> str:
    """Compile oracle/silero_ref.c into `build_dir`.  `native=True` (bench's CPU-baseline leg, run on
    the GPU box's host) uses -march=native into a separate file; the default is a
    portable AVX2+FMA build that may travel between machines of this image."""
    os.makedirs(build_dir, exist_ok=True)
    tag = "native" if native else "avx2"
    so = os.path.join(build_dir, f"libsilero_ref_{tag}.so")
    src = os.path.join(_HERE, "silero_ref.c")
    if (not force) and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src):
        return so
    arch = ["-march=native"] if native else ["-mavx2", "-mfma"]
    cmd = ["gcc", "-O3", "-fPIC", "-shared", "-fopenmp", "-fno-math-errno", *arch, src, "-o", so, "-lm"]
    subprocess.run(cmd, check=True)
    return so


_f32p = ctypes.POINTER(ctypes.c_float)


def _fp(a: np.ndarray):
    return a.ctypes.data_as(_f32p)


class RefLib:
    def __init__(self, native: bool = False, build_dir: str = BUILD_DIR):
        self.path = build_ref_lib(native=native, build_dir=build_dir)
        L = ctypes.CDLL(self.path)
        L.sref_v5_create.restype = ctypes.c_void_p
        L.sref_v5_create.argtypes = [_f32p]
        L.sref_v5_free.argtypes = [ctypes.c_void_p]
        L.sref_v5_frame.argtypes = [ctypes.c_void_p, _f32p, _f32p, _f32p, _f32p, _f32p]
        L.sref_v5_run.argtypes = [ctypes.c_void_p, _f32p, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_int, ctypes.c_int, _f32p, _f32p, _f32p, ctypes.c_int]
        L.sref_sm_run.argtypes = [_f32p, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                  ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                  ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_ubyte)]
        L.sref_max_threads.restype = ctypes.c_int
        L.sref_v4_create.restype = ctypes.c_void_p
        L.sref_v4_create.argtypes = [_f32p]
        L.sref_v4_free.argtypes = [ctypes.c_void_p]
        L.sref_v4_frame.argtypes = [ctypes.c_void_p, _f32p, _f32p, _f32p, _f32p, _f32p]
        L.sref_v4_run.argtypes = [ctypes.c_void_p, _f32p, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_int, ctypes.c_int, _f32p, _f32p, _f32p, ctypes.c_int]
        self.L = L

    def max_threads(self) -> int:
        return int(self.L.sref_max_threads())


class RefV5:
    """Batched v5/16 kHz model: plain-C restatement (oracle/silero_ref.c)."""

    DBG = 1603

    def __init__(self, blob: np.ndarray, lib: Optional[RefLib] = None):
        self.lib = lib or RefLib()
        self.blob = np.ascontiguousarray(blob, dtype=np.float32)
        self.handle = ctypes.c_void_p(self.lib.L.sref_v5_create(_fp(self.blob)))

    def __del__(self):
        try:
            self.lib.L.sref_v5_free(self.handle)
        except Exception:
            pass

    def frame(self, x512: np.ndarray, h: np.ndarray, c: np.ndarray, want_dbg: bool = False):
        x = np.ascontiguousarray(x512, dtype=np.float32)
        assert x.shape == (512,) and h.shape == (128,) and c.shape == (128,)
        p = np.zeros(1, np.float32)
        dbg = np.zeros(self.DBG, np.float32) if want_dbg else None
        self.lib.L.sref_v5_frame(self.handle, _fp(x), _fp(h), _fp(c), _fp(p), _fp(dbg) if want_dbg else None)
        return float(p[0]), dbg

    def run(self, audio: np.ndarray, n_frames: int, hop: int = 512, frame_len: int = 512,
            denoise: bool = True, h: Optional[np.ndarray] = None, c: Optional[np.ndarray] = None,
            nthreads: int = 0):
        """audio [n_streams, >= (n_frames-1)*hop + frame_len] f32 -> probs [n_streams, n_frames]."""
        audio = np.ascontiguousarray(audio, dtype=np.float32)
        n = audio.shape[0]
        assert audio.shape[1] >= (n_frames - 1) * hop + frame_len
        h = np.zeros((n, 128), np.float32) if h is None else h
        c = np.zeros((n, 128), np.float32) if c is None else c
        probs = np.zeros((n, n_frames), np.float32)
        self.lib.L.sref_v5_run(self.handle, _fp(audio), audio.shape[1], n, n_frames, hop, frame_len,
                               int(denoise), _fp(h), _fp(c), _fp(probs), nthreads)
        return probs, h, c


class RefV4:
    """Batched v4/16 kHz model: plain-C restatement.  State per stream: h[2][64], c[2][64]."""

    DBG = 1032 + 1032 + 128 + 64 + 128 + 64 + 64 + 32 + 64 + 64

    def __init__(self, blob: np.ndarray, lib: Optional[RefLib] = None):
        self.lib = lib or RefLib()
        self.blob = np.ascontiguousarray(blob, dtype=np.float32)
        self.handle = ctypes.c_void_p(self.lib.L.sref_v4_create(_fp(self.blob)))

    def __del__(self):
        try:
            self.lib.L.sref_v4_free(self.handle)
        except Exception:
            pass

    def frame(self, x512: np.ndarray, h: np.ndarray, c: np.ndarray, want_dbg: bool = False):
        x = np.ascontiguousarray(x512, dtype=np.float32)
        assert x.shape == (512,) and h.shape == (2, 64) and c.shape == (2, 64)
        p = np.zeros(1, np.float32)
        dbg = np.zeros(self.DBG, np.float32) if want_dbg else None
        self.lib.L.sref_v4_frame(self.handle, _fp(x), _fp(h), _fp(c), _fp(p), _fp(dbg) if want_dbg else None)
        return float(p[0]), dbg

    def run(self, audio: np.ndarray, n_frames: int, hop: int = 512, frame_len: int = 512, denoise: bool = True,
            h: Optional[np.ndarray] = None, c: Optional[np.ndarray] = None, nthreads: int = 0):
        audio = np.ascontiguousarray(audio, dtype=np.float32)
        n = audio.shape[0]
        assert audio.shape[1] >= (n_frames - 1) * hop + frame_len
        h = np.zeros((n, 2, 64), np.float32) if h is None else h
        c = np.zeros((n, 2, 64), np.float32) if c is None else c
        probs = np.zeros((n, n_frames), np.float32)
        self.lib.L.sref_v4_run(self.handle, _fp(audio), audio.shape[1], n, n_frames, hop, frame_len,
                               int(denoise), _fp(h), _fp(c), _fp(probs), nthreads)
        return probs, h, c


def sm_run_c(lib: RefLib, probs: np.ndarray, start_p=0.7, end_p=0.7, start_ratio=0.8, end_ratio=0.95,
             n_start=10, n_end=50, state: Optional[np.ndarray] = None):
    probs = np.ascontiguousarray(probs, dtype=np.float32)
    state = np.zeros(125, np.int32) if state is None else state
    flags = np.zeros(probs.size, np.uint8)
    lib.L.sref_sm_run(_fp(probs), probs.size, start_p, end_p, start_ratio, end_ratio, n_start, n_end,
                      state.ctypes.data_as(ctypes.POINTER(ctypes.c_int)),
                      flags.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)))
    return flags, state


# ----------------------------------------------------------------------------
# host-side steps, restated in numpy
# ----------------------------------------------------------------------------

def split_into_frames(audio: np.ndarray, frame_size: int, hop_size: Optional[int] = None) -> np.ndarray:
    """AudioUtils.split_into_frames, /root/reference/src/real_time_vad/utils/audio.py:164-190.
    n = (len - frame)//hop + 1; a negative n raises exactly as np.zeros((-1, f)) does."""
    if hop_size is None:
        hop_size = frame_size // 2
    n = (len(audio) - frame_size) // hop_size + 1
    frames = np.zeros((n, frame_size), dtype=audio.dtype)
    for i in range(n):
        frames[i] = audio[i * hop_size:i * hop_size + frame_size]
    return frames


def denoise(audio: np.ndarray, thr: float = 0.01) -> np.ndarray:
    """AudioUtils.denoise_audio, audio.py:104-121 (a gate, not a subtraction)."""
    return np.where(np.abs(audio) > thr, audio, 0.0)


def validate(audio: np.ndarray) -> None:
    """AudioUtils.validate_audio_data, audio.py:211-231."""
    if audio.size == 0:
        raise ValueError("Audio data is empty")
    if not np.isfinite(audio).all():
        raise ValueError("Audio data contains infinite or NaN values")
    if audio.ndim > 2:
        raise ValueError(f"Audio data has too many dimensions: {audio.ndim}")


def to_mono(audio: np.ndarray) -> np.ndarray:
    """AudioUtils.convert_to_mono, audio.py:193-208."""
    return audio if audio.ndim == 1 else np.mean(audio, axis=1)


def prepare_512(chunk: np.ndarray) -> np.ndarray:
    """SileroVADModel._prepare_audio_input, silero_model.py:449-474."""
    if len(chunk) < 512:
        chunk = np.pad(chunk, (0, 512 - len(chunk)))
    elif len(chunk) > 512:
        chunk = chunk[:512]
    return chunk.astype(np.float32)


def resample(audio: np.ndarray, original_rate: int, target_rate: int) -> np.ndarray:
    """AudioUtils.resample_audio, audio.py:19-55: scipy.signal.resample (FFT method)
    to int(len * target/original) samples, cast to float32.  scipy is a dependency
    of the reference (pyproject.toml) and IS present in this image, so the oracle
    calls the same function the reference calls."""
    from scipy import signal
    if original_rate == target_rate:
        return audio
    n = int(len(audio) * (target_rate / original_rate))
    return signal.resample(audio, n).astype(np.float32)


class StateMachine:
    """VADProcessor._process_voice_state and helpers, silero_model.py:790-923, with the
    two deques kept literally (:620-628)."""

    def __init__(self, start_p=0.7, end_p=0.7, start_ratio=0.8, end_ratio=0.95, n_start=10, n_end=50):
        self.start_p, self.end_p = start_p, end_p
        self.start_ratio, self.end_ratio = start_ratio, end_ratio
        self.n_start, self.n_end = n_start, n_end
        self.reset()

    def reset(self):
        self.active = False
        self.scount = 0
        self.ecount = 0
        self.recent_start = deque(maxlen=20)
        self.recent_end = deque(maxlen=100)

    def step(self, probability: float) -> int:
        """-> flags: bit0 started, bit1 ended, bit2 continuing."""
        fl = 0
        if not self.active:
            above = probability >= self.start_p
            self.recent_start.append(above)
            if above:
                self.scount += 1
                if self.scount >= self.n_start and len(self.recent_start) >= self.n_start:
                    win = list(self.recent_start)[-self.n_start:]
                    if sum(win) / len(win) >= self.start_ratio:
                        self.active = True
                        self.scount = 0
                        self.ecount = 0
                        fl |= 1
            else:
                self.scount = 0
        else:
            fl |= 4
            below = probability < self.end_p
            self.recent_end.append(below)
            if below:
                self.ecount += 1
                if self.ecount >= self.n_end and len(self.recent_end) >= self.n_end:
                    win = list(self.recent_end)[-self.n_end:]
                    if sum(win) / len(win) >= self.end_ratio:
                        self.active = False
                        self.ecount = 0
                        fl |= 2
            else:
                self.ecount = 0
        return fl


def events_from_flags(flags: Sequence[int]) -> List[Tuple[int, str]]:
    ev = []
    for i, f in enumerate(flags):
        if f & 1:
            ev.append((i, "S"))
        if f & 2:
            ev.append((i, "E"))
    return ev


class VoiceBuffer:
    """The audio side of VADProcessor, restated literally: `voice_buffer` (pre-roll of above-threshold frames,
    silero_model.py:839, cleared at :874), `current_voice_data` (:867-869 on start, :925-930 while active) and
    `_finalize_voice_segment` (:932-949).  Fed the gated frame, its probability and the state machine's flags of
    that frame; returns (segment handed to voice_end or None, frame handed to voice_continue or None)."""

    def __init__(self, start_p: float):
        self.start_p = start_p
        self.active = False
        self.voice_buffer: List[np.ndarray] = []
        self.current: Optional[np.ndarray] = None

    def step(self, frame: np.ndarray, probability: float, flags: int):
        if not self.active:
            if probability >= self.start_p:
                self.voice_buffer.append(frame.copy())
                if flags & 1:
                    self.active = True
                    if self.voice_buffer:
                        self.current = np.concatenate(self.voice_buffer)
                    self.voice_buffer = []
            else:
                self.voice_buffer = []
            return None, None
        self.current = frame.copy() if self.current is None else np.concatenate([self.current, frame])
        seg = None
        if flags & 2:
            seg, self.current, self.active = self.current, None, False
        return seg, frame


# ----------------------------------------------------------------------------
# float64 "truth": where FP32 executors of the SAME graph disagree by more than the parity bar
# ----------------------------------------------------------------------------

def resample_exact(audio: np.ndarray, original_rate: int, target_rate: int = 16000) -> np.ndarray:
    """AudioUtils.resample_audio (audio.py:19-55) with scipy's FFT evaluated in float64 and the function's final
    `.astype(np.float32)` kept: the correctly rounded value of what the reference computes in float32 (scipy's
    float32 FFT is within 3e-7 of it).  Used as the anchor where a consumer amplifies that 3e-7 (v4 on band-limited
    input, the noise gate's threshold)."""
    from scipy import signal
    if original_rate == target_rate:
        return np.asarray(audio, np.float32)
    n = int(len(audio) * (target_rate / original_rate))
    return signal.resample(np.asarray(audio, np.float64), n).astype(np.float32)


def resample_chunks(x: np.ndarray, rate: int, exact: bool = False) -> np.ndarray:
    """[n, T * n_in] source-rate streams -> [n, T * 512]: every chunk of n_in = 512 * rate / 16000 samples resampled on
    its own (the unit of resampling the engine defines, SURVEY.md section 7)."""
    n_in = rate * 512 // 16000
    n, L = x.shape
    T = L // n_in
    fn = resample_exact if exact else resample
    y = np.zeros((n, 512 * T), np.float32)
    for s in range(n):
        for j in range(T):
            y[s, j * 512:(j + 1) * 512] = fn(x[s, j * n_in:(j + 1) * n_in], rate, 16000)
    return y


class Truth64:
    """The reference's .onnx interpreted op by op in float64 (oracle/onnx_interp.py), batched over streams, LSTM state
    carried in float64: the anchor for cases in which two conforming FP32 executors differ by more than 1e-4."""

    def __init__(self, onnx_path: str, version: str):
        from onnx_interp import OnnxInterpreter
        self.it = OnnxInterpreter(str(onnx_path), np.float64)
        self.version = version

    def run(self, audio: np.ndarray, n_frames: int, hop: int = 512, frame_len: int = 512, denoise: bool = False,
            sr: int = 16000) -> np.ndarray:
        audio = np.asarray(audio, np.float32)
        n = audio.shape[0]
        if self.version == "v5":
            state = {"state": np.zeros((2, n, 128), np.float64)}
        else:
            state = {"h": np.zeros((2, n, 64), np.float64), "c": np.zeros((2, n, 64), np.float64)}
        probs = np.zeros((n, n_frames), np.float64)
        for j in range(n_frames):
            f = audio[:, j * hop:j * hop + frame_len]
            if denoise:
                f = np.where(np.abs(f) > 0.01, f, 0.0).astype(np.float32)        # audio.py:117-118, float32 like the reference
            if f.shape[1] < 512:
                f = np.pad(f, ((0, 0), (0, 512 - f.shape[1])))
            feeds = {"input": f[:, :512].astype(np.float64), "sr": np.array(sr, np.int64), **state}
            out = self.it.run(feeds)
            probs[:, j] = np.asarray(out[0], np.float64).reshape(n)
            if self.version == "v5":
                state = {"state": np.asarray(out[1], np.float64)}
            else:
                state = {"h": np.asarray(out[1], np.float64), "c": np.asarray(out[2], np.float64)}
        return probs


def sm_flags(probs: np.ndarray, start_p=0.7, end_p=0.7, n_start=10, n_end=50) -> np.ndarray:
    """State machine (literal deques, StateMachine above) over one stream's probabilities -> flags per frame."""
    sm = StateMachine(start_p, end_p, 0.8, 0.95, n_start, n_end)
    return np.array([sm.step(float(np.float32(p))) for p in probs], np.uint8)
