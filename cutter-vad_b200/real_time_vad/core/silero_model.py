"""Model wrapper and per-stream VAD pipeline of the drop-in API, backed by the B200 engine.

Mirrors the public surface of the reference's `src/real_time_vad/core/silero_model.py`
(result/state types :33-232, SileroVADModel :238-566, VADProcessor :569-1033): same
class names, fields, method names, exception classes and message prefixes.  What is
different is where the arithmetic runs:

* `ort` below is `engine.ort_compat`, an onnxruntime-shaped seam over the CUDA engine.
  `SileroVADModel.predict` / `VADProcessor.process_frame` are the one-frame
  COMPATIBILITY path (state in, state out per call, state machine on the host).
* `VADProcessor.process_audio_batched` is the FAST path used by `VADWrapper`: all frames
  of one `process_audio_data` call go to the GPU in ONE `cvad_step` (frame loader, noise
  gate, model, LSTM state and the start/end state machine on the device); the host only
  assembles callback payloads from the flags that come back.
"""
from __future__ import annotations

import logging
import os
from collections import deque
from pathlib import Path
from typing import Any, Dict, Iterator, List, Optional

import numpy as np
from pydantic import BaseModel, ConfigDict, Field, field_validator, model_validator

from ..engine import ort_compat as ort
from ..utils.audio import AudioUtils
from ..utils.wav_writer import WAVWriter
from .config import SampleRate, SileroModelVersion, VADConfig  # noqa: F401
from .exceptions import (AudioProcessingError, CallbackError, ConfigurationError,  # noqa: F401
                         ModelInitializationError, ModelNotFoundError, VADError)

FRAME = 512                    # samples the model consumes per call (silero_model.py:464-471)
START_WINDOW_CAP = 20          # deque(maxlen=20)  (silero_model.py:620-623)
END_WINDOW_CAP = 100           # deque(maxlen=100) (silero_model.py:625-628)

_PYD = dict(arbitrary_types_allowed=True, validate_assignment=True, extra="forbid")


# ============================================================== value types

class ModelState(BaseModel):
    """LSTM state as numpy: `state` (2,1,128) for v5, `hidden_state`/`cell_state` (2,1,64) for v4."""
    model_config = ConfigDict(**_PYD)

    state: Optional[np.ndarray] = Field(default=None)
    hidden_state: Optional[np.ndarray] = Field(default=None)
    cell_state: Optional[np.ndarray] = Field(default=None)

    @field_validator("state", "hidden_state", "cell_state")
    @classmethod
    def _float32_arrays_only(cls, v):
        if v is None:
            return v
        if not isinstance(v, np.ndarray):
            raise ValueError("State must be a numpy array")
        if v.dtype != np.float32:
            raise ValueError("State arrays must be float32")
        return v

    @model_validator(mode="after")
    def _one_representation(self):
        if self.state is not None and (self.hidden_state is not None or self.cell_state is not None):
            raise ValueError("Cannot have both combined state and separate states")
        return self


class ProcessingResult(BaseModel):
    """Outcome of one frame."""
    model_config = ConfigDict(**_PYD)

    voice_started: bool = Field(default=False)
    voice_ended: bool = Field(default=False)
    voice_continuing: bool = Field(default=False)
    probability: float = Field(ge=0.0, le=1.0)
    wav_data: Optional[bytes] = Field(default=None)
    pcm_data: Optional[bytes] = Field(default=None)

    @field_validator("wav_data", "pcm_data")
    @classmethod
    def _bytes_only(cls, v):
        if v is not None and not isinstance(v, bytes):
            raise ValueError("Audio data must be bytes")
        return v


class ProcessingStatistics(BaseModel):
    model_config = ConfigDict(**_PYD)

    is_voice_active: bool
    voice_start_frame_count: int = Field(ge=0)
    voice_end_frame_count: int = Field(ge=0)
    recent_probabilities: List[float] = Field(default_factory=list)
    average_probability: float = Field(ge=0.0, le=1.0)
    voice_buffer_size: int = Field(ge=0)
    current_voice_length: int = Field(ge=0)

    @field_validator("recent_probabilities")
    @classmethod
    def _unit_interval(cls, v: List[float]) -> List[float]:
        for p in v:
            if not (0.0 <= p <= 1.0):
                raise ValueError(f"Probability {p} must be between 0.0 and 1.0")
        return v


class ModelConfiguration(BaseModel):
    model_config = ConfigDict(validate_assignment=True, extra="forbid")

    model_path: str
    model_version: SileroModelVersion

    @field_validator("model_path")
    @classmethod
    def _existing_onnx_file(cls, v: str) -> str:
        if not os.path.exists(v):
            raise ModelNotFoundError(v)
        if not os.path.isfile(v):
            raise ValueError(f"Model path must be a file: {v}")
        if not v.endswith(".onnx"):
            raise ValueError(f"Model file must have .onnx extension: {v}")
        return v


# ============================================================== model wrapper

class SileroVADModel(BaseModel):
    """One model file opened through `ort` plus the stream's LSTM state."""
    model_config = ConfigDict(**_PYD)

    config: ModelConfiguration
    session: Optional[Any] = Field(default=None)
    model_state: ModelState = Field(default_factory=ModelState)
    prediction_count: int = Field(default=0, ge=0)

    def __init__(self, model_path: str, model_version: SileroModelVersion, **data: Any) -> None:
        super().__init__(config=ModelConfiguration(model_path=model_path, model_version=model_version), **data)
        self._load_model()
        self._reset_states()

    # ---- construction
    def _is_v5(self) -> bool:
        return self.config.model_version == SileroModelVersion.V5

    def _load_model(self) -> None:
        try:
            opts = ort.SessionOptions()
            opts.inter_op_num_threads = 1
            opts.intra_op_num_threads = 1
            opts.graph_optimization_level = ort.GraphOptimizationLevel.ORT_ENABLE_ALL
            self.session = ort.InferenceSession(self.config.model_path, sess_options=opts,
                                                providers=self._get_execution_providers())
            self._validate_model_signature()
        except Exception as exc:
            raise ModelInitializationError(self.config.model_version.value,
                                           f"Failed to load model from {self.config.model_path}: {exc}")

    def _get_execution_providers(self) -> List[str]:
        chosen = ["CPUExecutionProvider"]
        available = ort.get_available_providers()
        if available and "CUDAExecutionProvider" in available:
            chosen.insert(0, "CUDAExecutionProvider")
        return chosen

    def _validate_model_signature(self) -> None:
        if self.session is None:
            raise ModelInitializationError(self.config.model_version.value, "Session not initialized")
        try:
            want_in, want_out = (3, 2) if self._is_v5() else (4, 3)
            n_in, n_out = len(self.session.get_inputs()), len(self.session.get_outputs())
            if n_in != want_in:
                raise ValueError(f"Expected {want_in} inputs, got {n_in}")
            if n_out != want_out:
                raise ValueError(f"Expected {want_out} outputs, got {n_out}")
        except Exception as exc:
            raise ModelInitializationError(self.config.model_version.value,
                                           f"Model signature validation failed: {exc}")

    def _reset_states(self) -> None:
        if self._is_v5():
            self.model_state = ModelState(state=np.zeros((2, 1, 128), dtype=np.float32))
        else:
            self.model_state = ModelState(hidden_state=np.zeros((2, 1, 64), dtype=np.float32),
                                          cell_state=np.zeros((2, 1, 64), dtype=np.float32))

    # ---- one frame
    def predict(self, audio_chunk: np.ndarray, sample_rate: int) -> float:
        try:
            if self.session is None:
                raise ModelInitializationError(self.config.model_version.value, "Model not loaded")
            feeds = self._prepare_model_inputs(self._prepare_audio_input(audio_chunk), sample_rate)
            outputs = self.session.run(None, feeds)
            probability = self._extract_probability(outputs)
            self._update_states(outputs)
            self.prediction_count += 1
            return probability
        except (ModelInitializationError, AudioProcessingError):
            raise
        except Exception as exc:
            raise AudioProcessingError(f"Model prediction failed: {exc}")

    def _prepare_audio_input(self, audio_chunk: np.ndarray) -> np.ndarray:
        try:
            n = len(audio_chunk)
            if n < FRAME:
                audio_chunk = np.pad(audio_chunk, (0, FRAME - n))
            elif n > FRAME:
                audio_chunk = audio_chunk[:FRAME]
            return audio_chunk.reshape(1, -1).astype(np.float32)
        except Exception as exc:
            raise AudioProcessingError(f"Audio input preparation failed: {exc}")

    def _prepare_model_inputs(self, audio_input: np.ndarray, sample_rate: int) -> Dict[str, np.ndarray]:
        sr = np.array([sample_rate], dtype=np.int64)
        if self._is_v5():
            return {"input": audio_input, "state": self.model_state.state, "sr": sr}
        return {"input": audio_input, "h": self.model_state.hidden_state, "c": self.model_state.cell_state, "sr": sr}

    def _extract_probability(self, outputs: List[np.ndarray]) -> float:
        try:
            probability = float(outputs[0][0][0])
            if not (0.0 <= probability <= 1.0):
                raise ValueError(f"Invalid probability value: {probability}")
            return probability
        except Exception as exc:
            raise AudioProcessingError(f"Probability extraction failed: {exc}")

    def _update_states(self, outputs: List[np.ndarray]) -> None:
        if self._is_v5():
            self.model_state.state = outputs[1]
        else:
            self.model_state.hidden_state = outputs[1]
            self.model_state.cell_state = outputs[2]

    def reset(self) -> None:
        self._reset_states()

    def get_model_info(self) -> Dict[str, Any]:
        providers = self.session.get_providers() if self.session else None
        ms = self.model_state
        return {
            "model_path": self.config.model_path,
            "model_version": self.config.model_version.value,
            "prediction_count": self.prediction_count,
            "session_providers": providers,
            "has_cuda": "CUDAExecutionProvider" in (providers or []),
            "state_shape": {
                "state": ms.state.shape if ms.state is not None else None,
                "hidden_state": ms.hidden_state.shape if ms.hidden_state is not None else None,
                "cell_state": ms.cell_state.shape if ms.cell_state is not None else None,
            },
        }


# ============================================================== per-stream pipeline

class VADProcessor(BaseModel):
    """validate -> gate -> model -> start/end state machine -> callback payloads, for ONE stream."""
    model_config = ConfigDict(**_PYD)

    config: VADConfig
    model: Optional[Any] = Field(default=None)
    is_voice_active: bool = Field(default=False)
    voice_start_frame_count: int = Field(default=0, ge=0)
    voice_end_frame_count: int = Field(default=0, ge=0)
    voice_probabilities: deque = Field(default_factory=lambda: deque(maxlen=100))
    recent_start_frames: deque = Field(default_factory=lambda: deque(maxlen=START_WINDOW_CAP))
    recent_end_frames: deque = Field(default_factory=lambda: deque(maxlen=END_WINDOW_CAP))
    voice_buffer: deque = Field(default_factory=deque)
    current_voice_data: Optional[np.ndarray] = Field(default=None)
    wav_writer: WAVWriter

    def __init__(self, config: VADConfig, **data: Any) -> None:
        writer = WAVWriter(sample_rate=config.output_wav_sample_rate, bit_depth=config.output_wav_bit_depth,
                           channels=1)
        super().__init__(config=config, wav_writer=writer, **data)
        self._load_model()

    # ---- model lifecycle
    def _load_model(self) -> None:
        try:
            model_path = self._get_model_directory() / self.config.get_model_filename()
            if not model_path.exists():
                raise ModelNotFoundError(str(model_path))
            self.model = SileroVADModel(str(model_path), self.config.model_version)
        except (ModelNotFoundError, ModelInitializationError):
            raise
        except Exception as exc:
            raise ModelInitializationError(self.config.model_version.value,
                                           f"Failed to initialize VAD processor: {exc}")

    def _get_model_directory(self) -> Path:
        if self.config.model_path:
            model_dir = Path(self.config.model_path)
            logging.info(f"Using configured model path: {model_dir}")
        else:
            model_dir = Path(__file__).parent.parent / "models"
            logging.info(f"Using package model path: {model_dir}")
        return model_dir

    # ---- compatibility path: one frame per call
    def process_frame(self, audio_frame: np.ndarray) -> ProcessingResult:
        try:
            if self.model is None:
                raise ModelInitializationError(self.config.model_version.value, "Model not loaded")
            frame = self._preprocess_audio_frame(audio_frame)
            probability = self.model.predict(frame, self.config.sample_rate)
            self.voice_probabilities.append(probability)
            fields = self._process_voice_state(probability, frame)
            fields["probability"] = probability
            return ProcessingResult(**fields)
        except (ModelInitializationError, AudioProcessingError):
            raise
        except Exception as exc:
            raise AudioProcessingError(f"Frame processing failed: {exc}")

    def _preprocess_audio_frame(self, audio_frame: np.ndarray) -> np.ndarray:
        try:
            AudioUtils.validate_audio_data(audio_frame)
            if self.config.enable_denoising:
                audio_frame = AudioUtils.denoise_audio(audio_frame)
            return audio_frame
        except Exception as exc:
            raise AudioProcessingError(f"Audio preprocessing failed: {exc}")

    def _process_voice_state(self, probability: float, audio_frame: np.ndarray) -> Dict[str, Any]:
        out: Dict[str, Any] = {"voice_started": False, "voice_ended": False, "voice_continuing": False,
                               "wav_data": None, "pcm_data": None}
        step = self._handle_ongoing_voice_activity if self.is_voice_active else self._handle_voice_start_detection
        out.update(step(probability, audio_frame))
        return out

    def _handle_voice_start_detection(self, probability: float, audio_frame: np.ndarray) -> Dict[str, Any]:
        out: Dict[str, Any] = {}
        need = self.config.voice_start_frame_count
        hit = probability >= self.config.vad_start_probability
        self.recent_start_frames.append(hit)
        if not hit:
            self._reset_voice_start_detection()
            return out
        self.voice_start_frame_count += 1
        self.voice_buffer.append(audio_frame.copy())
        if self.voice_start_frame_count >= need and len(self.recent_start_frames) >= need:
            window = list(self.recent_start_frames)[-need:]
            if sum(window) / len(window) >= self.config.voice_start_ratio:
                self._confirm_voice_start()
                out["voice_started"] = True
        return out

    def _confirm_voice_start(self) -> None:
        self.is_voice_active = True
        self.voice_start_frame_count = 0
        self.voice_end_frame_count = 0
        if self.voice_buffer:
            self.current_voice_data = np.concatenate(list(self.voice_buffer))
        self.voice_buffer.clear()

    def _reset_voice_start_detection(self) -> None:
        self.voice_start_frame_count = 0
        self.voice_buffer.clear()

    def _handle_ongoing_voice_activity(self, probability: float, audio_frame: np.ndarray) -> Dict[str, Any]:
        out: Dict[str, Any] = {}
        self._accumulate_voice_data(audio_frame)
        out["voice_continuing"] = True
        out["pcm_data"] = audio_frame.tobytes()
        need = self.config.voice_end_frame_count
        quiet = probability < self.config.vad_end_probability
        self.recent_end_frames.append(quiet)
        if not quiet:
            self.voice_end_frame_count = 0
            return out
        self.voice_end_frame_count += 1
        if self.voice_end_frame_count >= need and len(self.recent_end_frames) >= need:
            window = list(self.recent_end_frames)[-need:]
            if sum(window) / len(window) >= self.config.voice_end_ratio:
                out["wav_data"] = self._finalize_voice_segment()
                out["voice_ended"] = True
        return out

    def _accumulate_voice_data(self, audio_frame: np.ndarray) -> None:
        if self.current_voice_data is None:
            self.current_voice_data = audio_frame.copy()
        else:
            self.current_voice_data = np.concatenate([self.current_voice_data, audio_frame])

    def _finalize_voice_segment(self) -> Optional[bytes]:
        wav = None
        if self.current_voice_data is not None:
            wav = self.wav_writer.write_wav_data(self.current_voice_data)
        self.is_voice_active = False
        self.voice_end_frame_count = 0
        self.current_voice_data = None
        return wav

    # ---- fast path: every frame of one call in a single engine step
    def supports_batched(self) -> bool:
        """True when the model is the real engine-backed one (not a test double) on the 16 kHz v5 path."""
        m = self.model
        return (isinstance(m, SileroVADModel) and isinstance(m.session, ort.InferenceSession)
                and m.session.version == self.config.model_version.value
                and int(self.config.sample_rate) == 16000)

    # frames per engine step of one process_audio_data call: bounds the device scratch of an hour-long buffer (the
    # reference streams frame by frame) and the work that is redone when a callback raises
    _BATCH_FRAMES = 512

    def process_audio_batched(self, audio: np.ndarray, frame_size: int, hop_size: int,
                              src_rate: int = 16000) -> Iterator[ProcessingResult]:
        """All frames `audio[j*hop : j*hop+frame_size]` through `cvad_step` on this stream's model session slot, up to
        `_BATCH_FRAMES` frames per step.  Yields one ProcessingResult per frame, in order, equal to what
        `process_frame` would have returned; callbacks run between yields.  If the consumer stops early -- a callback
        raised (vad_wrapper.py:470-476 aborts the call at that frame) -- the stream is put back where the reference
        leaves it: LSTM state and counters after the frame that raised, nothing later.

        `src_rate` 8000 / 24000 / 48000 (opt-in, VADWrapper.process_audio_data(..., input_sample_rate=...)): `audio` is
        at that rate, frame_size == hop_size == 512 * src_rate / 16000 source samples, and every chunk is resampled to
        one 512-sample model frame ON THE GPU (AudioUtils.resample_audio per chunk, utils/audio.py:19-55 -- the step the
        reference's wrapper leaves as a placeholder, vad_wrapper.py:619-624).  Callback payloads are 16 kHz audio made
        from the same chunks with the reference's own resampler, only for frames that reach a payload."""
        if src_rate != 16000:
            if src_rate not in (8000, 24000, 48000):
                raise ValueError("src_rate must be 8000, 16000, 24000 or 48000")
            if frame_size != hop_size or frame_size != 512 * src_rate // 16000:
                raise ValueError("resampled input is framed in chunks of 512 * src_rate / 16000 samples")
        rate_kw = {} if src_rate == 16000 else {"src_rate": src_rate}

        def payload_frame(lo: int) -> np.ndarray:
            f = audio[lo: lo + frame_size]
            if src_rate != 16000:
                f = AudioUtils.resample_audio(f, src_rate, 16000).astype(np.float32)
            return AudioUtils.denoise_audio(f) if gate else (f.copy() if src_rate == 16000 else f)

        sess = self.model.session
        n_frames = (len(audio) - frame_size) // hop_size + 1
        if n_frames < 0:
            raise ValueError("negative dimensions are not allowed")
        if n_frames == 0:
            return
        audio = np.ascontiguousarray(audio, dtype=np.float32)
        cfg = self.config
        ms = self.model.model_state
        pooled, slot = sess._pooled, sess._slot
        d = self.__dict__  # bypass pydantic's per-assignment validation on the per-frame bookkeeping
        start_p = cfg.vad_start_probability
        end_p = cfg.vad_end_probability
        gate = cfg.enable_denoising

        want_cfg = (start_p, end_p, cfg.voice_start_frame_count, cfg.voice_end_frame_count, bool(gate))

        def run(first: int, count: int, h_in, c_in, sm_in):
            """frames [first, first + count) from the given state -> (step result, h, c, sm).  The session's slot keeps
            its thresholds and its state between calls: both are uploaded only when they differ from what the device
            holds (`_dev_cfg`, `_dev_state` on the session; the compat session.run, which uses the same slot without the
            gate and with its caller's state, invalidates them)."""
            with pooled.lock:
                eng = pooled.engine
                if getattr(sess, "_dev_cfg", None) != want_cfg:
                    eng.configure([slot], vad_start_probability=start_p, vad_end_probability=end_p,
                                  voice_start_frame_count=cfg.voice_start_frame_count,
                                  voice_end_frame_count=cfg.voice_end_frame_count, enable_denoising=gate)
                    sess._dev_cfg = want_cfg
                held = getattr(sess, "_dev_state", None)
                if not (held is not None and np.array_equal(held[0], h_in) and np.array_equal(held[1], c_in)
                        and np.array_equal(held[2][:3], sm_in[:3])):
                    eng.set_state(slot, h_in, c_in, sm_in)
                sess._dev_state = None
                lo = first * hop_size
                r = eng.step(audio[None, lo:lo + (count - 1) * hop_size + frame_size], slots=[slot], n_frames=[count],
                             max_frames=count, frame_len=frame_size, hop=hop_size, **rate_kw)
                if r.status[0]:
                    raise AudioProcessingError("Audio data contains infinite or NaN values")
                h, c, sm_out, _ = eng.get_state(slot)
                sess._dev_state = (h.copy(), c.copy(), np.array(sm_out, np.int32))
            return r, h, c, sm_out

        def adopt(h, c, sm_out, segment):
            if ms.state is not None:
                ms.__dict__["state"] = np.stack([h[None, :], c[None, :]], axis=0).astype(np.float32)
            else:
                ms.__dict__["hidden_state"] = h.reshape(2, 1, 64).astype(np.float32)
                ms.__dict__["cell_state"] = c.reshape(2, 1, 64).astype(np.float32)
            d["is_voice_active"] = bool(sm_out[0])
            d["voice_start_frame_count"] = int(sm_out[1])
            d["voice_end_frame_count"] = int(sm_out[2])
            d["current_voice_data"] = (np.concatenate(segment).astype(np.float32, copy=False)
                                       if (segment and bool(sm_out[0])) else None)

        segment: List[np.ndarray] = [] if d["current_voice_data"] is None else [d["current_voice_data"]]
        for first in range(0, n_frames, self._BATCH_FRAMES):
            count = min(self._BATCH_FRAMES, n_frames - first)
            sm_in = np.array([int(d["is_voice_active"]), d["voice_start_frame_count"], d["voice_end_frame_count"], 0], np.int32)
            if ms.state is not None:
                h_in, c_in = ms.state[0, 0].copy(), ms.state[1, 0].copy()
            else:
                h_in, c_in = ms.hidden_state.reshape(128).copy(), ms.cell_state.reshape(128).copy()
            if not (np.abs(h_in) <= ort.H_BOUND).all():
                # a hand-set model_state the engine refuses (cvad_set_state): no LSTM step produces one
                raise ConfigurationError("model_state", "h outside [-2, 2]",
                                         "LSTM state h must lie within [-2, 2] (an LSTM's h stays within [-1, 1])")
            r, h, c, sm_out = run(first, count, h_in, c_in, sm_in)
            probs = r.probs[0]
            flags = r.flags[0]
            active = d["is_voice_active"]
            done = 0                 # frames of this batch whose result the consumer has taken
            try:
                for j in range(count):
                    p = float(probs[j])
                    fl = int(flags[j])
                    lo = (first + j) * hop_size
                    d["voice_probabilities"].append(p)
                    wav = pcm = None
                    if not active:
                        hit = p >= start_p
                        d["recent_start_frames"].append(hit)
                        if hit:
                            d["voice_buffer"].append(payload_frame(lo))
                            if fl & 1:
                                segment = list(d["voice_buffer"])
                                d["voice_buffer"].clear()
                                active = True
                        else:
                            d["voice_buffer"].clear()
                    else:
                        frame = payload_frame(lo)
                        segment.append(frame)
                        pcm = frame.tobytes()
                        d["recent_end_frames"].append(p < end_p)
                        if fl & 2:
                            wav = self.wav_writer.write_wav_data(np.concatenate(segment))
                            segment = []
                            active = False
                    d["is_voice_active"] = active
                    done = j + 1
                    yield ProcessingResult.model_construct(voice_started=bool(fl & 1), voice_ended=bool(fl & 2),
                                                           voice_continuing=bool(fl & 4), probability=p,
                                                           wav_data=wav, pcm_data=pcm)
            finally:
                if done < count:
                    # the consumer stopped after frame `done - 1` (a callback raised): the reference has run exactly
                    # `done` frames of this batch, so run those again from the batch's starting state and adopt that
                    if done > 0:
                        _, h, c, sm_out = run(first, done, h_in, c_in, sm_in)
                    else:
                        h, c, sm_out = h_in, c_in, sm_in
                    self.model.__dict__["prediction_count"] = self.model.prediction_count + done
                else:
                    self.model.__dict__["prediction_count"] = self.model.prediction_count + count
                adopt(h, c, sm_out, segment)

    # ---- housekeeping
    def reset(self) -> None:
        if self.model:
            self.model.reset()
        self.is_voice_active = False
        self.voice_start_frame_count = 0
        self.voice_end_frame_count = 0
        self.voice_probabilities.clear()
        self.voice_buffer.clear()
        self.current_voice_data = None
        self.recent_start_frames.clear()
        self.recent_end_frames.clear()

    def get_statistics(self) -> ProcessingStatistics:
        probs = self.voice_probabilities
        return ProcessingStatistics(
            is_voice_active=self.is_voice_active,
            voice_start_frame_count=self.voice_start_frame_count,
            voice_end_frame_count=self.voice_end_frame_count,
            recent_probabilities=list(probs),
            average_probability=np.mean(probs) if probs else 0.0,
            voice_buffer_size=len(self.voice_buffer),
            current_voice_length=len(self.current_voice_data) if self.current_voice_data is not None else 0,
        )

    def get_model_info(self) -> Dict[str, Any]:
        if self.model:
            return self.model.get_model_info()
        return {"model_path": None, "model_version": self.config.model_version.value, "model_loaded": False}

    def update_config(self, new_config: VADConfig) -> None:
        reload_model = (new_config.model_version != self.config.model_version
                        or new_config.model_path != self.config.model_path)
        self.config = new_config
        self.wav_writer = WAVWriter(sample_rate=new_config.output_wav_sample_rate,
                                    bit_depth=new_config.output_wav_bit_depth, channels=1)
        if reload_model:
            self._load_model()
        self.reset()
