"""BatchedVADManager: thousands of independent audio streams stepped per GPU launch.

New entry point named by the north star (SURVEY.md section 8b "New entry"); the
reference has no equivalent -- it builds one `VADWrapper` + one onnxruntime session per
stream (websocket_service/server/vad_websocket_server.py:248-290) and runs one model
call per frame on the event loop (:369).  Here a stream is a *slot* of resident state
in HBM (LSTM h/c, the state-machine words, thresholds); `step()` advances every stream
that has at least one complete frame buffered, in ONE `cvad_step`:

    mgr = BatchedVADManager(max_streams=10_000)
    sid = mgr.open_stream(VADConfig(...), on_voice_start=..., on_voice_end=..., on_voice_continue=...)
    mgr.push(sid, samples)            # float32 in [-1,1] or int16 PCM, any length
    out = mgr.step()                  # events in stream-then-frame order, callbacks fired

Per stream the results equal what a `VADWrapper` fed the same frames would produce:
same probabilities (FP32, 1e-4), same start/end frame indices, same callback payloads
(`voice_end` WAV of the gated frames buffered since the first above-threshold frame,
`voice_continue` float32 bytes of the gated frame; silero_model.py:839-869, :891-895, :932-949).
Framing is configurable: `frame_len` samples per frame, `hop` between frames
(hop == frame_len for the websocket service's one-frame-per-message mode, frame_len/2 for
the wrapper's overlapped mode); leftovers shorter than a frame are carried to the next step.

The data path is native: pending samples live in the engine library's pinned stream arena
(`cvad_feeder_*`, engine/feeder.py); `push` is one memcpy, `step` gathers, runs the GPU step and
assembles voice segments in C++, and Python only walks the frames a callback is due on.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass, field
from typing import Callable, Dict, List, NamedTuple, Optional, Sequence

import numpy as np

from ..engine import capi
from ..engine.feeder import FeederError, StreamFeeder, set_row_payloads
from ..engine.stream_engine import EngineError, StreamEngine
from ..utils.wav_writer import WAVWriter
from .config import SileroModelVersion, VADConfig
from .exceptions import AudioProcessingError, CallbackError, ConfigurationError, VADError
from .stream_snapshot import SnapshotStream, StreamSnapshot


class StreamEvent(NamedTuple):
    stream_id: int        # slot id returned by open_stream
    kind: str             # "start" | "end"
    frame_index: int      # frame index since the stream was opened / last reset
    step_frame: int       # frame index inside the step that produced it


class StepOutput:
    """Result of one `step()`.  Arrays are per stepped stream (row k <-> stream_ids[k])."""

    def __init__(self, events: List[StreamEvent], stream_ids: np.ndarray, counts: np.ndarray,
                 probs: np.ndarray, flags: np.ndarray):
        self.events = events                 # stream-then-frame order
        self.stream_ids = stream_ids         # [n] slot ids that ran at least one frame
        self.counts = counts                 # [n] frames run per stream
        self.probs = probs                   # [n, max(counts)] float32 (columns >= counts[k] are 0)
        self.flags = flags                   # [n, max(counts)] uint8, FLAG_* bits
        self.frames = int(counts.sum()) if counts.size else 0

    @property
    def probabilities(self) -> Dict[int, np.ndarray]:
        """stream id -> probabilities of the frames run in this step (built on demand)."""
        return {int(s): self.probs[k, :int(c)].copy() for k, (s, c) in enumerate(zip(self.stream_ids, self.counts))}


@dataclass
class _Stream:
    config: VADConfig
    writer: WAVWriter
    on_start: Optional[Callable[[], None]] = None
    on_end: Optional[Callable[[bytes], None]] = None
    on_continue: Optional[Callable[[bytes], None]] = None
    active: bool = False
    pre_roll: List[np.ndarray] = field(default_factory=list)
    segment: List[np.ndarray] = field(default_factory=list)

    @property
    def wants_audio(self) -> bool:
        return self.on_end is not None or self.on_continue is not None


class BatchedVADManager:
    def __init__(self, max_streams: int = 4096, model_version: SileroModelVersion = SileroModelVersion.V5,
                 device: Optional[int] = None, frame_len: int = 512, hop: Optional[int] = None,
                 pcm_format: int = capi.PCM_F32, source_rate: Optional[int] = 16000,
                 frames_per_step: int = 8) -> None:
        """`source_rate` 8000 / 24000 / 48000: streams deliver audio at that rate and every chunk of
        512*rate/16000 samples is resampled to one 16 kHz model frame on the GPU (frame_len and hop
        are then fixed to that chunk size).  `source_rate=None`: every stream has its own rate
        (`VADConfig.sample_rate` at open_stream, any of 8000 / 16000 / 24000 / 48000) and all of them
        advance in ONE engine step (cvad_step_args.src_rates), the way a websocket server meets them.
        `frames_per_step`: frames one stream runs per step at most; a stream that is further behind
        catches up over the following steps."""
        self.mixed = source_rate is None
        if self.mixed:
            source_rate, frame_len, hop = 48000, 1536, 1536        # arena sizing; per-stream values in the feeder
        if source_rate not in (8000, 16000, 24000, 48000):
            raise ConfigurationError("source_rate", str(source_rate))
        self.source_rate = int(source_rate)
        if source_rate != 16000:
            frame_len = hop = source_rate * 512 // 16000
        if not (1 <= frame_len <= 2048):
            raise ConfigurationError("frame_len", str(frame_len))
        self.frame_len = int(frame_len)
        self.hop = int(hop) if hop is not None else int(frame_len)
        if self.hop < 1:
            raise ConfigurationError("hop", str(hop))
        self.pcm_format = pcm_format
        self._dtype = np.float32 if pcm_format == capi.PCM_F32 else np.int16
        from ..engine.pool import default_device
        try:
            self._engine = StreamEngine(model_version.value, max_streams=max_streams,
                                        device=default_device() if device is None else device)
            self._feeder = StreamFeeder(self._engine, pcm_format=pcm_format, frame_len=self.frame_len, hop=self.hop,
                                        src_rate=0 if self.mixed else self.source_rate,
                                        capacity_frames=max(2, int(frames_per_step)))
        except Exception as exc:
            raise VADError(f"Failed to initialize VAD processor: {exc}")
        self.max_streams = max_streams
        self.model_version = model_version.value
        self._free = list(range(max_streams - 1, -1, -1))
        self._streams: Dict[int, _Stream] = {}
        self._lock = threading.Lock()

    # ------------------------------------------------------------------ stream lifecycle
    @property
    def engine(self) -> StreamEngine:
        return self._engine

    @property
    def feeder(self) -> StreamFeeder:
        return self._feeder

    def open_stream(self, config: Optional[VADConfig] = None, on_voice_start: Optional[Callable[[], None]] = None,
                    on_voice_end: Optional[Callable[[bytes], None]] = None,
                    on_voice_continue: Optional[Callable[[bytes], None]] = None) -> int:
        cfg = config if config is not None else VADConfig()
        if self.mixed:
            if int(cfg.sample_rate) not in (8000, 16000, 24000, 48000):
                raise ConfigurationError("sample_rate", str(cfg.sample_rate), "8000, 16000, 24000 or 48000")
        elif int(cfg.sample_rate) != self.source_rate:
            raise ConfigurationError("sample_rate", str(cfg.sample_rate),
                                     f"this manager takes {self.source_rate} Hz streams")
        with self._lock:
            if not self._free:
                raise VADError(f"all {self.max_streams} stream slots are in use")
            sid = self._free.pop()
            st = _Stream(config=cfg, writer=WAVWriter(cfg.output_wav_sample_rate, cfg.output_wav_bit_depth, 1),
                         on_start=on_voice_start, on_end=on_voice_end, on_continue=on_voice_continue)
            self._engine.reset([sid])
            self._apply_config(sid, st)
            self._streams[sid] = st
            return sid

    @staticmethod
    def _payload_mode(st: _Stream) -> int:
        if st.on_continue is not None:
            return capi.PAYLOAD_FRAMES
        if st.on_end is not None:
            return capi.PAYLOAD_SEGMENTS
        return capi.PAYLOAD_EVENTS if st.on_start is not None else capi.PAYLOAD_NONE

    def _apply_config(self, sid: int, st: _Stream) -> None:
        cfg = st.config
        self._engine.configure([sid], vad_start_probability=cfg.vad_start_probability,
                               vad_end_probability=cfg.vad_end_probability,
                               voice_start_frame_count=cfg.voice_start_frame_count,
                               voice_end_frame_count=cfg.voice_end_frame_count,
                               enable_denoising=cfg.enable_denoising)
        # (re)opening the feeder row drops pending samples and any half-built segment
        self._feeder.open(sid, src_rate=int(cfg.sample_rate) if self.mixed else 0, payload=self._payload_mode(st),
                          vad_start_probability=cfg.vad_start_probability, enable_denoising=cfg.enable_denoising)

    def close_stream(self, stream_id: int) -> None:
        with self._lock:
            if self._streams.pop(stream_id, None) is not None:
                self._engine.reset([stream_id])
                self._feeder.close_stream(stream_id)
                self._free.append(stream_id)

    def reset_stream(self, stream_id: int) -> None:
        """VADProcessor.reset (silero_model.py:951-968) for one stream; buffered samples are dropped."""
        with self._lock:
            st = self._stream(stream_id)
            self._engine.reset([stream_id])
            self._feeder.clear(stream_id)
            st.active = False
            st.pre_roll.clear()
            st.segment.clear()

    def update_config(self, stream_id: int, config: VADConfig) -> None:
        with self._lock:
            st = self._stream(stream_id)
            st.config = config
            st.writer = WAVWriter(config.output_wav_sample_rate, config.output_wav_bit_depth, 1)
            self._engine.reset([stream_id])
            self._apply_config(stream_id, st)
            st.active = False
            st.pre_roll.clear()
            st.segment.clear()

    def _stream(self, stream_id: int) -> _Stream:
        try:
            return self._streams[stream_id]
        except KeyError:
            raise VADError(f"stream {stream_id} is not open")

    def is_voice_active(self, stream_id: int) -> bool:
        self._stream(stream_id)
        return self._feeder.is_active(stream_id)

    @property
    def open_streams(self) -> List[int]:
        return sorted(self._streams)

    # ------------------------------------------------------------------ data path
    def _check_samples(self, samples) -> np.ndarray:
        x = np.asarray(samples)
        if x.size == 0:
            raise AudioProcessingError("Audio data is empty")
        return np.ascontiguousarray(x, dtype=self._dtype)

    @staticmethod
    def _raise(exc: FeederError):
        if "infinite or NaN" in exc.message or "empty" in exc.message:
            raise AudioProcessingError(exc.message)
        raise VADError(exc.message)

    def push(self, stream_id: int, samples) -> None:
        """Append audio to a stream's buffer (no GPU work).  NaN/Inf is rejected here, before any
        state changes, as `AudioUtils.validate_audio_data` does (audio.py:227-228)."""
        self._stream(stream_id)
        x = self._check_samples(samples)
        if x.ndim == 2:
            x = np.ascontiguousarray(x.mean(axis=1).astype(self._dtype))
        try:
            self._feeder.push(stream_id, x)
        except FeederError as exc:
            self._raise(exc)

    def pending(self, stream_id: int) -> int:
        """Samples buffered for a stream that no step has consumed yet (callers use it for backpressure)."""
        return self._feeder.pending(stream_id)

    def push_bytes(self, stream_id: int, data: bytes) -> None:
        """A wire message as received (the websocket server's int16 / float32 payload,
        vad_websocket_server.py:334-344) appended without a numpy round trip."""
        if not data:
            raise AudioProcessingError("Audio data is empty")
        try:
            self._feeder.push_bytes(stream_id, data)
        except FeederError as exc:
            self._raise(exc)

    def push_many(self, stream_ids: Sequence[int], block: np.ndarray) -> None:
        """Lock-step producers: `block[k]` is appended to stream `stream_ids[k]` (all rows the same length)."""
        x = self._check_samples(block)
        ids = np.asarray(stream_ids, np.int32)
        if x.ndim != 2 or x.shape[0] != ids.size:
            raise AudioProcessingError("push_many expects block[len(stream_ids), samples]")
        try:
            self._feeder.push_many(ids, x)
        except FeederError as exc:
            self._raise(exc)

    def _gate(self, st: _Stream, frame: np.ndarray) -> np.ndarray:
        f = frame.astype(np.float32)
        if self.pcm_format == capi.PCM_S16_32767:
            f = f / np.float32(32767.0)
        elif self.pcm_format == capi.PCM_S16_32768:
            f = f / np.float32(32768.0)
        rate = int(st.config.sample_rate) if self.mixed else self.source_rate
        if rate != 16000:
            # callback payloads are 16 kHz audio: same operator as the GPU resampler, host side,
            # only for the frames that actually reach a payload
            from ..utils.audio import AudioUtils
            f = AudioUtils.resample_audio(f, rate, 16000)
        if st.config.enable_denoising:
            f = np.where(np.abs(f) > 0.01, f, 0.0).astype(np.float32)
        return f

    def step(self) -> StepOutput:
        """Run every complete buffered frame of every open stream in one GPU step."""
        with self._lock:
            try:
                r = self._feeder.step(borrow=True)
            except FeederError as exc:
                self._raise(exc)
            import time
            t0 = time.perf_counter()
            events = [StreamEvent(slot, "start" if kind == capi.FLAG_STARTED else "end", stream_frame, j)
                      for (k, slot, j, kind, stream_frame) in r.events]
            t1 = time.perf_counter()
            self._deliver(r.records)
            t2 = time.perf_counter()
            out = StepOutput(events, r.slots.astype(np.int64), r.counts.astype(np.int64), r.probs, r.flags)
            out.phase_ms = r.phase_ms          # (framing, GPU step incl. copies, segment assembly) inside the native step
            # where the rest of step() goes: (native call, unpack into numpy, event tuples, callbacks incl. WAV encoding, result object)
            out.host_ms = (r.call_ms[0], r.call_ms[1], 1e3 * (t1 - t0), 1e3 * (t2 - t1), 1e3 * (time.perf_counter() - t2))
            return out

    def _deliver(self, records) -> None:
        """Fire the callbacks the feeder found due, in stream-then-frame order: start, then end with the WAV
        bytes, then continue with the float32 frame bytes (vad_wrapper.py:498-519).  16 kHz streams arrive with
        their payloads assembled; for resampled streams (`raw` records, one per frame) the pre-roll / segment
        bookkeeping of silero_model.py:839-869,:925-949 runs here on host-resampled frames.  `records` are the native
        delivery records as tuples (engine/feeder.py: FeederStep.records); payload bytes are copied out only for the
        callbacks that exist."""
        sa, streams = C.string_at, self._streams
        STARTED, ENDED = capi.FLAG_STARTED, capi.FLAG_ENDED
        for (slot, _row, _j, fl, frame_p, seg_p, seg_len, frame_len, prob, raw_p, raw_len) in records:
            st = streams.get(slot)
            if st is None:
                continue
            if not raw_p:
                if fl & STARTED:
                    self._call(st.on_start, "voice_start")
                if fl & ENDED and st.on_end is not None and seg_p and seg_len > 0:
                    wav = st.writer.write_wav_data(np.frombuffer(sa(seg_p, seg_len * 4), np.float32))
                    if wav:
                        self._call(st.on_end, "voice_end", wav)
                if frame_p and st.on_continue is not None:
                    self._call(st.on_continue, "voice_continue", sa(frame_p, frame_len * 4))
                continue
            d_raw = np.frombuffer(sa(raw_p, raw_len * self._dtype().itemsize), self._dtype)
            frame = self._gate(st, d_raw) if (st.active or prob >= st.config.vad_start_probability) else None
            if not st.active:
                if prob >= st.config.vad_start_probability:
                    st.pre_roll.append(frame)
                    if fl & capi.FLAG_STARTED:
                        st.segment = st.pre_roll
                        st.pre_roll = []
                        st.active = True
                        self._call(st.on_start, "voice_start")
                else:
                    st.pre_roll = []
            else:
                st.segment.append(frame)
                wav = None
                if fl & capi.FLAG_ENDED:
                    if st.on_end is not None and st.segment:
                        wav = st.writer.write_wav_data(np.concatenate(st.segment))
                    st.segment = []
                    st.active = False
                if wav:
                    self._call(st.on_end, "voice_end", wav)
                self._call(st.on_continue, "voice_continue", frame.tobytes())

    @staticmethod
    def _call(cb: Optional[Callable], name: str, *args) -> None:
        if cb is None:
            return
        try:
            cb(*args)
        except Exception as exc:
            raise CallbackError(name, exc)

    # ------------------------------------------------------------------ stream snapshots
    def snapshot_streams(self, stream_ids: Optional[Sequence[int]] = None) -> StreamSnapshot:
        """Freeze open streams (all of them by default) between steps: the engine's records and the feeder's rows are
        taken under the manager lock, so they describe the same instant.  The streams keep running here; audio pushed
        after the snapshot belongs to them only.  A move is snapshot, close_stream, then restore_streams elsewhere."""
        with self._lock:
            ids = sorted(self._streams) if stream_ids is None else [int(s) for s in stream_ids]
            for s in ids:
                self._stream(s)
            if len(set(ids)) != len(ids):
                raise VADError("snapshot_streams: a stream is listed twice")
            try:
                states = self._engine.export_states(ids) if ids else np.zeros(0, capi.STATE_DTYPE)
                rows = self._feeder.export_rows(ids)
            except (EngineError, FeederError) as exc:
                raise VADError(f"snapshot_streams failed: {exc.message}")
            streams = []
            for s in ids:
                st = self._streams[s]
                streams.append(SnapshotStream(s, st.config._to_serializable_dict(), self._payload_mode(st), st.active,
                                              [f.copy() for f in st.pre_roll], [f.copy() for f in st.segment]))
            return StreamSnapshot(self.model_version, self._engine.fingerprint, int(self.pcm_format), self.frame_len,
                                  self.hop, None if self.mixed else self.source_rate, streams, states, rows)

    def restore_streams(self, snapshot: StreamSnapshot,
                        callbacks: Optional[Dict[int, Dict[str, Callable]]] = None) -> Dict[int, int]:
        """Open the snapshot's streams here, each continuing exactly where it was: same LSTM state, state machine,
        frame count (event frame indices continue), pending samples, pre-roll and half-built segment.  `callbacks` maps
        a stream's id in the snapshot to dict(on_voice_start=..., on_voice_end=..., on_voice_continue=...).  All or
        nothing; -> {id in the snapshot: id here}.

        ConfigurationError, with nothing opened: another model version or weights (fingerprint), PCM format, framing or
        source-rate mode; fewer free slots than streams; or a stream in the middle of voice (active, or with a pre-roll)
        whose new callbacks want audio its snapshot did not carry (it was taken with callbacks that wanted less).
        The math mode may differ: the state is FP32 in every mode."""
        snap = snapshot
        callbacks = callbacks or {}
        if snap.model_version != self.model_version:
            raise ConfigurationError("model_version", snap.model_version, f"this manager runs {self.model_version}")
        if int(snap.fingerprint) != self._engine.fingerprint:
            raise ConfigurationError("fingerprint", f"{int(snap.fingerprint):016x}",
                                     "the snapshot was taken with other model weights")
        if int(snap.pcm_format) != int(self.pcm_format):
            raise ConfigurationError("pcm_format", str(snap.pcm_format), f"this manager takes pcm_format {self.pcm_format}")
        if (snap.frame_len, snap.hop) != (self.frame_len, self.hop):
            raise ConfigurationError("frame_len/hop", f"{snap.frame_len}/{snap.hop}",
                                     f"this manager frames {self.frame_len}/{self.hop}")
        if snap.source_rate != (None if self.mixed else self.source_rate):
            raise ConfigurationError("source_rate", str(snap.source_rate),
                                     f"this manager takes {'mixed-rate' if self.mixed else self.source_rate} streams")
        n = len(snap.streams)
        if len(snap.states) != n:
            raise VADError("invalid stream snapshot: engine records do not match the stream list")
        if len(set(snap.stream_ids)) != n:
            raise VADError("invalid stream snapshot: a stream id appears twice")
        new_streams: List[_Stream] = []
        for k, ss in enumerate(snap.streams):
            try:
                cfg = VADConfig.from_dict(dict(ss.config))
            except Exception as exc:
                raise VADError(f"invalid stream snapshot: stream {ss.stream_id}: bad config ({exc})")
            cb = callbacks.get(ss.stream_id, {})
            unknown = set(cb) - {"on_voice_start", "on_voice_end", "on_voice_continue"}
            if unknown:
                raise ConfigurationError("callbacks", ", ".join(sorted(unknown)))
            st = _Stream(config=cfg, writer=WAVWriter(cfg.output_wav_sample_rate, cfg.output_wav_bit_depth, 1),
                         on_start=cb.get("on_voice_start"), on_end=cb.get("on_voice_end"),
                         on_continue=cb.get("on_voice_continue"))
            carried = ss.payload >= capi.PAYLOAD_SEGMENTS
            # in the middle of voice: active, or in the pre-roll -- frames at or above the start threshold since the
            # last one below it, which is exactly when the engine's start counter is above 0 (the feeder's pre-roll
            # follows the same rule, but only streams that carried audio kept one)
            rec = snap.states[k]
            mid_voice = bool(rec["is_voice_active"]) or int(rec["voice_start_frame_count"]) > 0 or ss.active or \
                bool(ss.pre_roll)
            if st.wants_audio and not carried and mid_voice:
                raise ConfigurationError("callbacks", f"stream {ss.stream_id}",
                                         "the stream is in the middle of voice and its snapshot carries no audio for "
                                         "the voice_end / voice_continue callbacks")
            if st.wants_audio:
                st.active, st.pre_roll, st.segment = ss.active, list(ss.pre_roll), list(ss.segment)
            new_streams.append(st)
        try:
            rows = set_row_payloads(snap.feeder_rows, [self._payload_mode(st) for st in new_streams])
        except ValueError as exc:
            raise VADError(f"invalid stream snapshot: {exc}")
        with self._lock:
            if len(self._free) < n:
                raise ConfigurationError("max_streams", str(self.max_streams),
                                         f"{n} streams to restore, {len(self._free)} slots free")
            ids = [self._free.pop() for _ in range(n)]
            try:
                if n:
                    self._engine.import_states(ids, snap.states)
                self._feeder.import_rows(ids, rows)
            except (EngineError, FeederError) as exc:
                self._free.extend(reversed(ids))
                if n:
                    self._engine.reset(ids)
                raise VADError(f"invalid stream snapshot: {exc.message}")
            for sid, st in zip(ids, new_streams):
                self._streams[sid] = st
            return {ss.stream_id: sid for ss, sid in zip(snap.streams, ids)}

    # ------------------------------------------------------------------ lock-step block API
    def step_block(self, audio: np.ndarray, stream_ids: Optional[Sequence[int]] = None):
        """Lock-step fast path: `audio[k]` holds whole frames for stream `stream_ids[k]` (no buffering,
        no callbacks).  -> engine StepResult (probs, flags, status, events)."""
        ids = list(self.open_streams) if stream_ids is None else list(stream_ids)
        if self.mixed:
            raise ConfigurationError("source_rate", "None", "step_block needs one source rate for all streams")
        with self._lock:
            return self._engine.step(audio, slots=ids, frame_len=self.frame_len, hop=self.hop,
                                     pcm_format=self.pcm_format, src_rate=self.source_rate)

    def close(self) -> None:
        with self._lock:
            self._streams.clear()
            self._feeder.close()
            self._engine.close()

    def __enter__(self) -> "BatchedVADManager":
        return self

    def __exit__(self, *exc) -> None:
        self.close()
