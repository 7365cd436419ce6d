"""StreamFeeder: numpy-facing handle on the native stream feeder (cvad_feeder_* in include/cutter_vad_b200.h).

The feeder is the host half of the service mode: every stream's pending samples sit in one pinned arena, `push`
appends a message, `step` frames whatever is complete, runs ONE `cvad_step` over those streams and replays the callback
side of the reference's `VADProcessor` (pre-roll, voice segment, continue frames;
/root/reference/src/real_time_vad/core/silero_model.py:839-869, :891-895, :925-949) from the device's per-frame flags --
all in native code, so that Python only sees the frames something happened on.
"""
from __future__ import annotations

import ctypes as C
import struct
from typing import List, NamedTuple, Optional, Sequence

import numpy as np

from . import capi


class FeederError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[cvad feeder {code}] {message}")
        self.code = code
        self.message = message


class Delivery(NamedTuple):
    slot: int
    stream: int                     # row in the step's arrays
    step_frame: int
    flags: int                      # capi.FLAG_* bits of the frame
    prob: float
    frame: Optional[np.ndarray]     # gated float32 frame for voice_continue (PAYLOAD_FRAMES)
    segment: Optional[np.ndarray]   # gated float32 samples of the finished segment (on FLAG_ENDED)
    raw: Optional[np.ndarray]       # source-rate samples of the frame (streams the host resamples payloads for)


class FeederStep:
    """One step's results; arrays are copies, safe to keep."""

    __slots__ = ("slots", "counts", "probs", "flags", "events", "deliveries", "records", "frames", "raw", "raw_stride", "phase_ms",
                 "call_ms")

    def __init__(self, slots, counts, probs, flags, events, deliveries, frames, raw=None, raw_stride=0, phase_ms=(0.0, 0.0, 0.0),
                 records=None):
        self.slots, self.counts, self.probs, self.flags = slots, counts, probs, flags
        self.events, self.deliveries, self.frames = events, deliveries, frames
        # `step(borrow=True)`: the native delivery records as plain tuples (slot, stream, step_frame, flags, frame_ptr,
        # segment_ptr, segment_len, frame_len, prob, raw_ptr, raw_len) whose pointers are valid until the feeder's next
        # step -- for a consumer that walks them at once (BatchedVADManager); `deliveries` is then None
        self.records = records
        self.raw, self.raw_stride = raw, raw_stride
        self.phase_ms = phase_ms            # (gather, cvad_step, deliver) wall milliseconds inside the native step
        self.call_ms = (0.0, 0.0)


_EVENT_DT = np.dtype([("stream", "<i4"), ("slot", "<i4"), ("frame", "<i4"), ("kind", "<i4"), ("stream_frame", "<i8")])
_DELIV_DT = np.dtype([("slot", "<i4"), ("stream", "<i4"), ("step_frame", "<i4"), ("flags", "<i4"), ("frame", "<u8"),
                      ("segment", "<u8"), ("segment_len", "<i8"), ("frame_len", "<i4"), ("prob", "<f4"),
                      ("raw", "<u8"), ("raw_len", "<i8")])
assert _EVENT_DT.itemsize == C.sizeof(capi.Event) and _DELIV_DT.itemsize == C.sizeof(capi.Delivery)


def set_row_payloads(blob: bytes, payloads: Sequence[int]) -> bytes:
    """A copy of an export_rows blob with row i's payload mode set to payloads[i] (CVAD_PAYLOAD_*): the payload mode
    follows the callbacks a restored stream gets, not the ones it had.  Raises ValueError for a malformed blob."""
    b = bytearray(blob)
    try:
        magic, version, pcm, _fl, _hop, _sr, n, _z = struct.unpack_from("<IIiiiiii", b, 0)
        if magic != capi.FEEDER_SNAPSHOT_MAGIC or version != capi.FEEDER_SNAPSHOT_VERSION or n != len(payloads):
            raise ValueError("not a feeder snapshot with one row per stream")
        es = capi.pcm_dtype(pcm).itemsize
        pos = 32
        for i in range(n):
            struct.pack_into("<i", b, pos + 8, int(payloads[i]))
            n_pending, n_pre, n_seg = struct.unpack_from("<qqq", b, pos + 40)
            pos += 64 + n_pending * es + (n_pre + n_seg) * 4
    except struct.error as exc:
        raise ValueError(f"truncated feeder snapshot: {exc}")
    return bytes(b)


def _view(ptr: int, dtype, count: int) -> np.ndarray:
    """Borrowed view of `count` items at address `ptr` (caller copies what it keeps)."""
    if not ptr or count <= 0:
        return np.zeros(0, dtype)
    dt = np.dtype(dtype)
    buf = (C.c_char * (count * dt.itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dt, count=count)


class StreamFeeder:
    def __init__(self, engine=None, *, max_streams: Optional[int] = None, pcm_format: int = capi.PCM_F32,
                 frame_len: int = 512, hop: int = 512, src_rate: int = 16000, capacity_frames: int = 8):
        """`engine` is a StreamEngine, or None for the host-only test hooks (`gather_only` / `deliver_only`)."""
        self._L = capi.lib()
        self._h = C.c_void_p()
        self._engine = engine
        eh = engine.handle if engine is not None else None
        n = int(max_streams if max_streams is not None else (engine.max_streams if engine is not None else 0))
        rc = self._L.cvad_feeder_create(eh, n, int(pcm_format), int(frame_len), int(hop), int(src_rate),
                                        int(capacity_frames), C.byref(self._h))
        if rc != capi.OK:
            msg = (self._L.cvad_last_error(eh) or b"").decode() if eh is not None else "bad feeder arguments"
            raise FeederError(rc, msg)
        self.pcm_format = int(pcm_format)
        self.dtype = capi.pcm_dtype(pcm_format).type
        self.max_streams = n
        self._res = capi.FeederResult()

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int) -> int:
        if rc < 0:
            raise FeederError(rc, (self._L.cvad_feeder_last_error(self._h) or b"").decode())
        return rc

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.cvad_feeder_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ streams
    def open(self, slot: int, *, src_rate: int = 0, payload: int = capi.PAYLOAD_NONE,
             vad_start_probability: float = 0.7, enable_denoising: bool = True) -> None:
        self._check(self._L.cvad_feeder_open(self._h, int(slot), int(src_rate), int(payload),
                                             float(vad_start_probability), int(bool(enable_denoising))))

    def close_stream(self, slot: int) -> None:
        self._check(self._L.cvad_feeder_close(self._h, int(slot)))

    def clear(self, slot: int) -> None:
        self._check(self._L.cvad_feeder_clear(self._h, int(slot)))

    def is_active(self, slot: int) -> bool:
        return self._check(self._L.cvad_feeder_is_active(self._h, int(slot))) == 1

    def pending(self, slot: int) -> int:
        return int(self._check(self._L.cvad_feeder_pending(self._h, int(slot))))

    # ------------------------------------------------------------------ row snapshots
    def export_rows(self, slots: Sequence[int]) -> bytes:
        """Pending samples, pre-roll and half-built segment of open `slots` as one persistable blob (cvad_feeder_export;
        layout in include/cutter_vad_b200.h)."""
        ids = np.ascontiguousarray(slots, dtype=np.int32)
        need = C.c_size_t(0)
        self._check(self._L.cvad_feeder_export(self._h, int(ids.size), ids.ctypes.data, None, 0, C.byref(need)))
        while True:
            # pushes from other threads may grow the rows between sizing and copying: the call then reports the new
            # size (CVAD_E_CAPACITY, nothing written) and is repeated with room to spare
            cap = int(need.value) + int(need.value) // 8 + 4096
            buf = C.create_string_buffer(cap)
            rc = self._L.cvad_feeder_export(self._h, int(ids.size), ids.ctypes.data, buf, cap, C.byref(need))
            if rc != capi.E_CAPACITY or int(need.value) <= cap:
                self._check(rc)
                return buf.raw[:int(need.value)]

    def import_rows(self, slots: Sequence[int], blob: bytes) -> None:
        """(Re)open `slots` with the rows of an export_rows blob, in order; the whole blob is checked first."""
        ids = np.ascontiguousarray(slots, dtype=np.int32)
        blob = bytes(blob)
        self._check(self._L.cvad_feeder_import(self._h, int(ids.size), ids.ctypes.data, blob, len(blob)))

    # ------------------------------------------------------------------ data path
    def push(self, slot: int, samples: np.ndarray) -> None:
        """`samples`: 1-D contiguous array of the feeder's dtype (uint8 codes for G.711)."""
        self._check(self._L.cvad_feeder_push(self._h, int(slot), samples.ctypes.data, samples.size))

    def push_bytes(self, slot: int, data: bytes) -> None:
        """A wire message as it arrived (little-endian samples of the feeder's dtype), no numpy in between."""
        self._check(self._L.cvad_feeder_push(self._h, int(slot), data, len(data) // self.dtype().itemsize))

    def push_many(self, slots: Sequence[int], block: np.ndarray) -> None:
        ids = np.ascontiguousarray(slots, dtype=np.int32)
        if block.ndim != 2 or block.shape[0] != ids.size or block.dtype != self.dtype or block.strides[1] != block.itemsize:
            raise FeederError(capi.E_INVALID, "push_many expects block[len(slots), samples] of the feeder's dtype")
        self._check(self._L.cvad_feeder_push_many(self._h, int(ids.size), ids.ctypes.data, block.ctypes.data,
                                                  block.strides[0] // block.itemsize, block.shape[1]))

    def _unpack(self, want_raw: bool = False, borrow: bool = False) -> FeederStep:
        r = self._res
        n, T = int(r.n_streams), int(r.max_frames)
        slots = _view(r.slots, np.int32, n).copy()
        counts = _view(r.counts, np.int32, n).copy()
        probs = _view(r.probs, np.float32, n * T).reshape(n, T).copy()
        flags = _view(r.flags, np.uint8, n * T).reshape(n, T).copy()
        ev = _view(r.events, _EVENT_DT, int(r.n_events))
        events = ev.tolist()                      # [(stream, slot, frame, kind, stream_frame)] as Python ints
        # records as plain tuples (one C loop), payloads as one memcpy each: at 10,000 streams field access on numpy void
        # scalars and view -> copy pairs were most of this function
        records = _view(r.deliveries, _DELIV_DT, int(r.n_deliveries)).tolist()
        if borrow:
            return FeederStep(slots, counts, probs, flags, events, None, int(r.n_frames_total), None, int(r.raw_stride),
                              (float(r.gather_ms), float(r.gpu_ms), float(r.deliver_ms)), records)
        deliveries: List[Delivery] = []
        sa, fb, isz = C.string_at, np.frombuffer, self.dtype().itemsize
        for (slot, stream, step_frame, fl, frame_p, seg_p, seg_len, frame_len, prob, raw_p, raw_len) in records:
            frame = fb(sa(frame_p, frame_len * 4), np.float32) if frame_p else None
            seg = fb(sa(seg_p, seg_len * 4), np.float32) if seg_p and seg_len > 0 else (np.zeros(0, np.float32) if seg_p else None)
            raw = fb(sa(raw_p, raw_len * isz), self.dtype) if raw_p else None
            if fl & capi.FLAG_ENDED and seg is None and not raw_p:
                seg = np.zeros(0, np.float32)
            deliveries.append(Delivery(slot, stream, step_frame, fl, prob, frame, seg, raw))
        raw_block = None
        if want_raw and n:
            raw_block = _view(r.raw, self.dtype, n * int(r.raw_stride)).reshape(n, int(r.raw_stride)).copy()
        return FeederStep(slots, counts, probs, flags, events, deliveries, int(r.n_frames_total), raw_block,
                          int(r.raw_stride), (float(r.gather_ms), float(r.gpu_ms), float(r.deliver_ms)))

    def step(self, borrow: bool = False) -> FeederStep:
        import time
        t0 = time.perf_counter()
        self._check(self._L.cvad_feeder_step(self._h, C.byref(self._res)))
        t1 = time.perf_counter()
        out = self._unpack(borrow=borrow)
        out.call_ms = (1e3 * (t1 - t0), 1e3 * (time.perf_counter() - t1))     # (native call, unpacking into numpy / tuples)
        return out

    # ------------------------------------------------------------------ host-only test hooks
    def gather_only(self) -> FeederStep:
        self._check(self._L.cvad_feeder_gather_only(self._h, C.byref(self._res)))
        return self._unpack(want_raw=True)

    def deliver_only(self, probs: np.ndarray, flags: np.ndarray) -> FeederStep:
        p = np.ascontiguousarray(probs, np.float32)
        f = np.ascontiguousarray(flags, np.uint8)
        self._check(self._L.cvad_feeder_deliver_only(self._h, p.ctypes.data, f.ctypes.data, C.byref(self._res)))
        return self._unpack()
