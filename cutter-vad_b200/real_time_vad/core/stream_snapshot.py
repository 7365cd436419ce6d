"""StreamSnapshot: live streams of a BatchedVADManager, frozen so that another manager -- in this process, in a new
process after a restart, or on another GPU -- can continue them where they were (BatchedVADManager.snapshot_streams /
restore_streams).

What a stream is made of, and where each part comes from:
  - the engine's per-slot state (LSTM h/c, the state-machine words, frames_done, the thresholds): one
    capi.STATE_DTYPE record per stream (cvad_export_states);
  - the feeder's row (pending samples, pre-roll, half-built segment): one blob for all streams (cvad_feeder_export);
  - for streams whose source rate is not 16 kHz and that want audio, the pre-roll / segment frames the manager keeps in
    Python (16 kHz float32, already gated) and its voice-active flag;
  - the stream's VADConfig.

`to_bytes()` is a versioned container that never unpickles: the 8-byte magic b"CVADSNAP", a little-endian uint32
version, a uint64 length and a UTF-8 JSON header, then the raw sections the header lists (the engine records, the feeder
blob, the Python-side frames as float32).  Snapshots may cross machines, so `from_bytes` treats its input as untrusted:
anything truncated, inconsistent or unknown raises VADError("invalid stream snapshot: ...").
"""
from __future__ import annotations

import json
import struct
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional

import numpy as np

from ..engine import capi
from .exceptions import VADError

MAGIC = b"CVADSNAP"
VERSION = 1


def _invalid(why: str) -> VADError:
    return VADError(f"invalid stream snapshot: {why}")


@dataclass
class SnapshotStream:
    """One stream of a snapshot."""
    stream_id: int                         # its id in the manager it was taken from
    config: Dict[str, Any]                 # VADConfig, JSON-ready (VADConfig.from_dict reads it back)
    payload: int                           # capi.PAYLOAD_* it had: what audio the snapshot carries for it
    active: bool = False                   # manager-side voice-active flag (resampled streams with audio)
    pre_roll: List[np.ndarray] = field(default_factory=list)   # manager-side 16 kHz frames (resampled streams with audio)
    segment: List[np.ndarray] = field(default_factory=list)


@dataclass
class StreamSnapshot:
    model_version: str                     # "v5" / "v4"
    fingerprint: int                       # cvad_model_fingerprint of the engine
    pcm_format: int
    frame_len: int
    hop: int
    source_rate: Optional[int]             # None: a mixed-rate manager (every stream has its own rate)
    streams: List[SnapshotStream]
    states: np.ndarray                     # [len(streams)] capi.STATE_DTYPE
    feeder_rows: bytes                     # cvad_feeder_export blob, rows in stream order

    @property
    def stream_ids(self) -> List[int]:
        return [s.stream_id for s in self.streams]

    # ------------------------------------------------------------------ container
    def to_bytes(self) -> bytes:
        frames: List[np.ndarray] = []
        streams = []
        for s in self.streams:
            pre = [np.ascontiguousarray(f, np.float32).ravel() for f in s.pre_roll]
            seg = [np.ascontiguousarray(f, np.float32).ravel() for f in s.segment]
            frames += pre + seg
            streams.append({"id": int(s.stream_id), "config": s.config, "payload": int(s.payload),
                            "active": bool(s.active), "pre_roll": [int(f.size) for f in pre],
                            "segment": [int(f.size) for f in seg]})
        states = np.ascontiguousarray(self.states, capi.STATE_DTYPE).tobytes()
        audio = np.concatenate(frames).tobytes() if frames else b""
        header = {"model_version": self.model_version, "fingerprint": f"{self.fingerprint:016x}",
                  "pcm_format": int(self.pcm_format), "frame_len": int(self.frame_len), "hop": int(self.hop),
                  "source_rate": None if self.source_rate is None else int(self.source_rate), "streams": streams,
                  "sections": {"states": len(states), "feeder_rows": len(self.feeder_rows), "frames": len(audio)}}
        hb = json.dumps(header, separators=(",", ":")).encode("utf-8")
        return b"".join([MAGIC, struct.pack("<IQ", VERSION, len(hb)), hb, states, bytes(self.feeder_rows), audio])

    @classmethod
    def from_bytes(cls, data: bytes) -> "StreamSnapshot":
        data = bytes(data)
        if len(data) < 20 or data[:8] != MAGIC:
            raise _invalid("bad magic")
        version, hlen = struct.unpack_from("<IQ", data, 8)
        if version != VERSION:
            raise _invalid(f"version {version} is not supported (this build reads {VERSION})")
        if hlen > len(data) - 20:
            raise _invalid("truncated header")
        try:
            h = json.loads(data[20:20 + hlen].decode("utf-8"))
            sec = h["sections"]
            n_states, n_rows, n_audio = int(sec["states"]), int(sec["feeder_rows"]), int(sec["frames"])
            streams_in = h["streams"]
            if not isinstance(streams_in, list) or not all(isinstance(x, dict) for x in streams_in):
                raise TypeError("streams is not a list of mappings")
            fingerprint = int(h["fingerprint"], 16)
            model_version, pcm_format = str(h["model_version"]), int(h["pcm_format"])
            frame_len, hop = int(h["frame_len"]), int(h["hop"])
            source_rate = None if h["source_rate"] is None else int(h["source_rate"])
        except (ValueError, KeyError, TypeError, UnicodeDecodeError) as exc:
            raise _invalid(f"unreadable header ({exc})")
        if min(n_states, n_rows, n_audio) < 0 or n_audio % 4:
            raise _invalid("bad section lengths")
        at = 20 + hlen
        if len(data) != at + n_states + n_rows + n_audio:
            raise _invalid(f"{len(data)} bytes, the header describes {at + n_states + n_rows + n_audio}")
        if n_states != len(streams_in) * capi.STATE_DTYPE.itemsize:
            raise _invalid("the engine records do not match the stream list")
        states = np.frombuffer(data, capi.STATE_DTYPE, len(streams_in), at).copy()
        rows = data[at + n_states:at + n_states + n_rows]
        audio = np.frombuffer(data, np.float32, n_audio // 4, at + n_states + n_rows)
        streams: List[SnapshotStream] = []
        o = 0
        try:
            for s in streams_in:
                parts = []
                for key in ("pre_roll", "segment"):
                    lens = [int(x) for x in s[key]]
                    if any(x < 0 for x in lens) or o + sum(lens) > audio.size:
                        raise _invalid("frame lengths exceed the frames section")
                    part = []
                    for x in lens:
                        part.append(audio[o:o + x].copy())
                        o += x
                    parts.append(part)
                if not isinstance(s["config"], dict):
                    raise _invalid("a stream's config is not a mapping")
                streams.append(SnapshotStream(int(s["id"]), s["config"], int(s["payload"]), bool(s["active"]),
                                              parts[0], parts[1]))
        except (KeyError, TypeError, ValueError) as exc:
            if isinstance(exc, VADError):
                raise
            raise _invalid(f"unreadable stream list ({exc})")
        if o != audio.size:
            raise _invalid("the frames section holds more than the stream list describes")
        if len({s.stream_id for s in streams}) != len(streams):
            raise _invalid("a stream id appears twice")
        return cls(model_version, fingerprint, pcm_format, frame_len, hop, source_rate, streams, states, rows)
