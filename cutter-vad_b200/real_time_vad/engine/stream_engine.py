"""StreamEngine: numpy-facing handle on one GPU's VAD engine (thin layer over the C ABI).

One engine owns `max_streams` slots.  Each slot carries the per-stream state the
reference keeps on a `VADProcessor` / `SileroVADModel` pair
(/root/reference/src/real_time_vad/core/silero_model.py:264-267 LSTM state,
:596-628 state-machine fields), resident in HBM.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from pathlib import Path
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import capi
from .onnx_weights import canonical_blob_v4, canonical_blob_v5

MODELS_DIR = Path(__file__).resolve().parents[1] / "models"


class EngineError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[cvad {code}] {message}")
        self.code = code
        self.message = message


@dataclass
class StepResult:
    probs: np.ndarray            # [n_streams, max_frames] float32
    flags: np.ndarray            # [n_streams, max_frames] uint8 (FLAG_* bits)
    status: np.ndarray           # [n_streams] uint8 (STATUS_* bits)
    events: List[Tuple[int, int, int, int, int]]  # (stream, slot, frame, kind, stream_frame), stream-then-frame order


class PendingStep:
    """A step in flight (see StreamEngine.submit)."""

    def __init__(self, engine, ticket, args, keep, probs, flags, status, ev, nev):
        self._engine, self._ticket, self._args, self._keep = engine, ticket, args, keep
        self._probs, self._flags, self._status, self._ev, self._nev = probs, flags, status, ev, nev
        self._result: Optional[StepResult] = None

    def collect(self) -> StepResult:
        if self._result is None:
            eng = self._engine
            eng._check(eng._L.cvad_step_collect(eng._h, self._ticket))
            k = min(int(self._nev[0]), self._args.max_events)
            events = []
            if k:
                rec = self._ev[:3 * k].view(np.int32).reshape(k, 6)
                sf = self._ev[:3 * k].reshape(k, 3)[:, 2]
                events = [(int(r[0]), int(r[1]), int(r[2]), int(r[3]), int(f)) for r, f in zip(rec, sf)]
            self._result = StepResult(self._probs, self._flags, self._status, events)
            self._keep = None
        return self._result


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class StreamEngine:
    def __init__(self, model_version: str = "v5", max_streams: int = 1, device: int = 0,
                 model_path: Optional[Path] = None, math: Optional[str] = None, resampler: Optional[str] = None):
        self._L = capi.lib()
        self._h = C.c_void_p()
        if model_version == "v5":
            path = Path(model_path) if model_path else MODELS_DIR / "silero_vad_v5.onnx"
            self.weights, code = canonical_blob_v5(path), capi.MODEL_V5
        elif model_version == "v4":
            path = Path(model_path) if model_path else MODELS_DIR / "silero_vad.onnx"
            self.weights, code = canonical_blob_v4(path), capi.MODEL_V4
        elif model_version == "v4_8k":
            # v4's 8 kHz sub-model: what the reference's session runs for v4 when sr != 16000
            path = Path(model_path) if model_path else MODELS_DIR / "silero_vad.onnx"
            self.weights, code = canonical_blob_v4(path, branch="8k"), capi.MODEL_V4_8K
        else:
            raise EngineError(capi.E_INVALID, f"unknown model version {model_version!r}")
        rc = self._L.cvad_create(_ptr(self.weights), self.weights.size, code, int(max_streams),
                                 int(device), C.byref(self._h))
        if rc != capi.OK:
            raise EngineError(rc, (self._L.cvad_last_error(None) or b"").decode())
        self.max_streams = int(max_streams)
        self.device = int(device)
        self.model_version = model_version
        if math is not None:
            self.set_math(math)
        if resampler is not None:
            self.set_resampler(resampler)

    # ------------------------------------------------------------------ plumbing
    def set_math(self, math: str) -> None:
        """'fp32' = packed FP32 FMA kernels; 'tc' = tcgen05 tensor cores with the 3-way BF16 split; 'tc16' (v5, its
        default) = tensor cores with the 2-way FP16 split and per-stream scaling (3 products per MAC); 'fft' (v4, its
        default) = the STFT as a double-precision FFT plus a tensor-core correction for the basis' float32 rounding."""
        code = {"fp32": capi.MATH_FP32, "tc": capi.MATH_TC, "tc16": capi.MATH_TC16, "fft": capi.MATH_FFT}.get(math)
        if code is None:
            raise EngineError(capi.E_INVALID, f"unknown math mode {math!r}")
        self._check(self._L.cvad_set_math(self._h, code))

    @property
    def math(self) -> str:
        return {capi.MATH_TC: "tc", capi.MATH_TC16: "tc16", capi.MATH_FFT: "fft"}.get(self._L.cvad_get_math(self._h), "fp32")

    def set_resampler(self, resampler: str) -> None:
        """'fft' (default) = scipy.signal.resample's FFT method in double, rounded once to float32; 'gemm' = the dense
        operator on the arithmetic `math` selects (FP32 FMA or split-precision tensor cores)."""
        code = {"fft": capi.RESAMPLE_FFT, "gemm": capi.RESAMPLE_GEMM}.get(resampler)
        if code is None:
            raise EngineError(capi.E_INVALID, f"unknown resampler {resampler!r}")
        self._check(self._L.cvad_set_resampler(self._h, code))

    @property
    def resampler(self) -> str:
        return "gemm" if self._L.cvad_get_resampler(self._h) == capi.RESAMPLE_GEMM else "fft"

    def _check(self, rc: int) -> None:
        if rc < 0:
            raise EngineError(rc, (self._L.cvad_last_error(self._h) or b"").decode())

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.cvad_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def set_stream(self, cuda_stream: int) -> None:
        self._check(self._L.cvad_set_stream(self._h, C.c_void_p(cuda_stream)))

    @staticmethod
    def resample_matrix(src_rate: int) -> np.ndarray:
        """R^T [n_in][512] of the engine's resampler (== scipy.signal.resample's operator)."""
        n_in = src_rate * 512 // 16000
        rt = np.zeros((n_in, 512), np.float32)
        rc = capi.lib().cvad_resample_matrix(int(src_rate), rt.ctypes.data, rt.size)
        if rc != n_in:
            raise EngineError(rc, f"no resampler for {src_rate} Hz")
        return rt

    def sync(self) -> None:
        self._check(self._L.cvad_sync(self._h))

    def launch_count(self) -> int:
        return int(self._L.cvad_launch_count(self._h))

    def set_timing(self, enabled: bool) -> None:
        self._check(self._L.cvad_set_timing(self._h, int(enabled)))

    def read_timing(self):
        """-> (frontend_ms_total, recurrent_ms_total, n_steps) since the last read."""
        fe, rec, n = C.c_double(0), C.c_double(0), C.c_int(0)
        self._check(self._L.cvad_read_timing(self._h, C.byref(fe), C.byref(rec), C.byref(n)))
        return fe.value, rec.value, n.value

    def step_device(self, args: "capi.StepArgs") -> None:
        """Enqueue one step whose buffers are all device pointers (no sync)."""
        self._check(self._L.cvad_step_device(self._h, C.byref(args)))

    # ------------------------------------------------------------------ per-slot control
    @staticmethod
    def _slots(slots: Optional[Sequence[int]]):
        if slots is None:
            return 0, None
        arr = np.ascontiguousarray(slots, dtype=np.int32)
        return int(arr.size), arr

    def reset(self, slots: Optional[Sequence[int]] = None) -> None:
        n, arr = self._slots(slots)
        self._check(self._L.cvad_reset(self._h, n, _ptr(arr)))

    def configure(self, slots: Optional[Sequence[int]] = None, *, vad_start_probability: float = 0.7,
                  vad_end_probability: float = 0.7, voice_start_frame_count: int = 10,
                  voice_end_frame_count: int = 50, enable_denoising: bool = True) -> None:
        n, arr = self._slots(slots)
        self._check(self._L.cvad_configure(self._h, n, _ptr(arr), float(vad_start_probability),
                                           float(vad_end_probability), int(voice_start_frame_count),
                                           int(voice_end_frame_count), int(bool(enable_denoising))))

    def get_state(self, slot: int):
        h = np.zeros(128, np.float32)
        c = np.zeros(128, np.float32)
        sm = np.zeros(4, np.int32)
        fd = C.c_int64(0)
        self._check(self._L.cvad_get_state(self._h, int(slot), _ptr(h), _ptr(c), _ptr(sm), C.byref(fd)))
        return h, c, sm, int(fd.value)

    def set_state(self, slot: int, h: Optional[np.ndarray] = None, c: Optional[np.ndarray] = None,
                  sm: Optional[np.ndarray] = None) -> None:
        h = None if h is None else np.ascontiguousarray(h, np.float32)
        c = None if c is None else np.ascontiguousarray(c, np.float32)
        sm = None if sm is None else np.ascontiguousarray(sm, np.int32)
        self._check(self._L.cvad_set_state(self._h, int(slot), _ptr(h), _ptr(c), _ptr(sm)))

    # ------------------------------------------------------------------ stream snapshots
    @property
    def fingerprint(self) -> int:
        """Model version + FNV-1a 64 of the weight blob (cvad_model_fingerprint): records move between engines with
        equal fingerprints."""
        v = C.c_uint64(0)
        self._check(self._L.cvad_model_fingerprint(self._h, C.byref(v)))
        return int(v.value)

    def export_states(self, slots: Optional[Sequence[int]], device_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        """The state of `slots` (None = 0..max_streams-1) as capi.STATE_DTYPE records, one per slot in order.  With
        `device_ptr` the records are written to that device address (len(slots) * 1072 bytes on the engine's device)
        and None is returned."""
        n, arr = self._slots(slots)
        if slots is None:
            n = self.max_streams
        if device_ptr is not None:
            self._check(self._L.cvad_export_states(self._h, n, _ptr(arr), C.c_void_p(int(device_ptr))))
            return None
        out = np.zeros(n, capi.STATE_DTYPE)
        self._check(self._L.cvad_export_states(self._h, n, _ptr(arr), _ptr(out)))
        return out

    def import_states(self, slots: Optional[Sequence[int]], records) -> None:
        """Write records into `slots` (None = 0..n-1), all or nothing.  `records`: a STATE_DTYPE array (or bytes of
        one), or an int device address of len(slots) records on the engine's device."""
        n, arr = self._slots(slots)
        if isinstance(records, int):
            if slots is None:
                raise EngineError(capi.E_INVALID, "import_states from a device address needs the slot list")
            self._check(self._L.cvad_import_states(self._h, n, _ptr(arr), C.c_void_p(records)))
            return
        rec = np.frombuffer(records, capi.STATE_DTYPE) if isinstance(records, (bytes, bytearray, memoryview)) \
            else np.ascontiguousarray(records)
        if rec.dtype != capi.STATE_DTYPE:
            raise EngineError(capi.E_INVALID, "records must have capi.STATE_DTYPE")
        if slots is None:
            n = rec.size
        elif rec.size != n:
            raise EngineError(capi.E_INVALID, "len(records) != len(slots)")
        self._check(self._L.cvad_import_states(self._h, n, _ptr(arr), _ptr(rec)))

    # ------------------------------------------------------------------ the hot call
    def _args(self, audio: np.ndarray, slots, n_frames, max_frames, frame_len, hop, pcm_format, src_rate=16000,
              src_rates=None):
        if audio.ndim not in (2, 3):
            raise EngineError(capi.E_INVALID, "audio must be [n_streams, samples] or [n_streams, samples, channels]")
        if pcm_format == capi.PCM_F32:
            audio = np.ascontiguousarray(audio, dtype=np.float32)
        else:
            audio = np.ascontiguousarray(audio, dtype=np.int16)
        n = audio.shape[0]
        keep = [audio]
        a = capi.StepArgs()
        a.n_streams = n
        if slots is not None:
            s = np.ascontiguousarray(slots, dtype=np.int32)
            if s.size != n:
                raise EngineError(capi.E_INVALID, "len(slots) != n_streams")
            keep.append(s)
            a.slots = s.ctypes.data
        if n_frames is not None:
            nf = np.ascontiguousarray(n_frames, dtype=np.int32)
            if nf.size != n:
                raise EngineError(capi.E_INVALID, "len(n_frames) != n_streams")
            keep.append(nf)
            a.n_frames = nf.ctypes.data
        a.audio = audio.ctypes.data
        a.pcm_format = pcm_format
        # [n, samples, channels]: interleaved sample frames, averaged to mono on the GPU (AudioUtils.convert_to_mono)
        a.channels = audio.shape[2] if audio.ndim == 3 else 1
        a.stream_stride = audio.shape[1] * (audio.shape[2] if audio.ndim == 3 else 1)
        a.max_frames = int(max_frames)
        a.frame_len = int(frame_len)
        a.hop = int(hop)
        a.src_rate = int(src_rate)
        if src_rates is not None:
            sr = np.ascontiguousarray(src_rates, dtype=np.int32)
            if sr.size != n:
                raise EngineError(capi.E_INVALID, "len(src_rates) != n_streams")
            keep.append(sr)
            a.src_rates = sr.ctypes.data
        return a, keep

    @staticmethod
    def _framing(audio, max_frames, frame_len, hop, src_rate, src_rates):
        """-> (max_frames, frame_len, hop) of a step over `audio`"""
        if src_rates is not None:
            # per-stream source rates in ONE step: stream i holds max_frames chunks of 512*rate_i/16000 samples
            if max_frames is None:
                raise EngineError(capi.E_INVALID, "max_frames is required with src_rates")
            frame_len = hop = 512
        elif src_rate not in (0, 16000):
            # source-rate input: every chunk of 512*src_rate/16000 samples becomes one model frame
            frame_len = hop = src_rate * 512 // 16000
        if max_frames is None:
            max_frames = 0 if audio.shape[1] < frame_len else (audio.shape[1] - frame_len) // hop + 1
        return max_frames, frame_len, hop

    def submit(self, audio: np.ndarray, *, slots: Optional[Sequence[int]] = None,
               n_frames: Optional[Sequence[int]] = None, max_frames: Optional[int] = None,
               frame_len: int = 512, hop: int = 512, pcm_format: int = capi.PCM_F32,
               max_events: int = 0, src_rate: int = 16000,
               src_rates: Optional[Sequence[int]] = None) -> "PendingStep":
        """Enqueue one step (H2D, kernels, D2H) and return at once; `.collect()` waits for it.
        Up to four steps may be in flight: later copies overlap earlier steps' kernels and result copies.
        `audio` must stay untouched until collect (pinned arrays are DMA'd in place)."""
        audio = np.asarray(audio)
        max_frames, frame_len, hop = self._framing(audio, max_frames, frame_len, hop, src_rate, src_rates)
        a, keep = self._args(audio, slots, n_frames, max_frames, frame_len, hop, pcm_format, src_rate, src_rates)
        n = a.n_streams
        probs = np.empty((n, max_frames), np.float32)
        flags = np.empty((n, max_frames), np.uint8)
        status = np.zeros(n, np.uint8)
        if max_events <= 0:
            max_events = max(16, 2 * n * max(max_frames, 1))
        ev = np.empty(max_events * 3, np.int64)           # 24-byte cvad_event records
        nev = np.zeros(1, np.int32)
        a.probs_out = probs.ctypes.data
        a.flags_out = flags.ctypes.data
        a.status_out = status.ctypes.data
        a.events_out = ev.ctypes.data
        a.max_events = max_events
        a.n_events_out = nev.ctypes.data
        ticket = C.c_int(0)
        self._check(self._L.cvad_step_submit(self._h, C.byref(a), C.byref(ticket)))
        return PendingStep(self, ticket.value, a, keep, probs, flags, status, ev, nev)

    def step(self, audio: np.ndarray, **kw) -> StepResult:
        """Advance every listed stream by its n_frames frames (host buffers in and out)."""
        return self.submit(audio, **kw).collect()

    def debug_dump(self, audio: np.ndarray, *, frame_len: int = 512, hop: int = 512,
                   pcm_format: int = capi.PCM_F32):
        """Front-end intermediates of the first tile, frame 0 (test hook; engine state untouched)."""
        a, keep = self._args(np.asarray(audio), None, None, 1, frame_len, hop, pcm_format)
        if self.model_version == "v5":
            layout = (("mag", (129, 3, 32)), ("e0", (128, 3, 32)), ("e1", (64, 2, 32)), ("e2", (64, 32)),
                      ("feat", (128, 32)))
        else:
            layout = (("mag", (129, 8, 16)), ("norm", (129, 8, 16)), ("r3", (16, 8, 16)), ("r15", (32, 4, 16)),
                      ("r27", (32, 2, 16)), ("r39", (64, 16)), ("feat", (64, 16)))
        n_dbg = sum(int(np.prod(sh)) for _, sh in layout)
        out = np.zeros(n_dbg, np.float32)
        rc = self._L.cvad_debug_dump(self._h, C.byref(a), _ptr(out), out.size)
        self._check(rc)
        o = 0
        res = {}
        for name, shape in layout:
            size = int(np.prod(shape))
            res[name] = out[o:o + size].reshape(shape)
            o += size
        return res

    def debug_input(self, audio: np.ndarray, *, src_rate: int = 16000, src_rates: Optional[Sequence[int]] = None,
                    max_frames: Optional[int] = None, n_frames: Optional[Sequence[int]] = None,
                    pcm_format: int = capi.PCM_F32, frame_len: int = 512, hop: int = 512) -> np.ndarray:
        """The float32 mono 16 kHz samples the model kernels would read for the step `submit` would run on the same
        arguments (cvad_debug_input: input stages only; test hook, engine state untouched).  Resampled and mixed-rate
        steps -> [n_streams, max_frames * 512], frames beyond a stream's n_frames NaN; down-mix only ->
        [n_streams, (max_frames - 1) * hop + frame_len]."""
        audio = np.asarray(audio)
        max_frames, frame_len, hop = self._framing(audio, max_frames, frame_len, hop, src_rate, src_rates)
        a, keep = self._args(audio, None, n_frames, max_frames, frame_len, hop, pcm_format, src_rate, src_rates)
        resampled = src_rates is not None or src_rate not in (0, 16000)
        per = max_frames * 512 if resampled else max(max_frames - 1, 0) * hop + frame_len
        out = np.empty((a.n_streams, per if max_frames else 0), np.float32)
        rc = self._L.cvad_debug_input(self._h, C.byref(a), _ptr(out), out.size)
        self._check(rc)
        return out
