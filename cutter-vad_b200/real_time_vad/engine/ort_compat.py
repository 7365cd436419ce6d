"""`ort`: the onnxruntime-shaped seam of the reference, backed by the B200 engine.

`real_time_vad.core.silero_model` binds this module to the name `ort`, exactly where
the reference binds `onnxruntime` (/root/reference/src/real_time_vad/core/silero_model.py:13),
and uses the same five names: `InferenceSession` (:321), `SessionOptions` (:315),
`GraphOptimizationLevel.ORT_ENABLE_ALL` (:318), `get_available_providers` (:345) and
`session.get_inputs/get_outputs/get_providers/run` (:365-366, :433, :559).  The
reference's tests patch `...silero_model.ort.InferenceSession`; that keeps working.

`InferenceSession.run` is the batch-1 COMPATIBILITY path (state in, state out, like the
stateless ORT call).  The fast path never goes through it: VADProcessor and
BatchedVADManager step slots with resident state through `StreamEngine.step`.
There is no CPU execution provider: without the CUDA library or a B200 this raises.
"""
from __future__ import annotations

from pathlib import Path
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import capi, pool
from .onnx_weights import read_float_tensors

__version__ = "cvad-b200"


class GraphOptimizationLevel:
    ORT_DISABLE_ALL = 0
    ORT_ENABLE_BASIC = 1
    ORT_ENABLE_EXTENDED = 2
    ORT_ENABLE_ALL = 99


class SessionOptions:
    def __init__(self) -> None:
        self.inter_op_num_threads = 0
        self.intra_op_num_threads = 0
        self.graph_optimization_level = GraphOptimizationLevel.ORT_ENABLE_ALL


class NodeArg:
    def __init__(self, name: str, shape: Sequence, type_: str) -> None:
        self.name, self.shape, self.type = name, list(shape), type_


def get_available_providers() -> List[str]:
    try:
        return ["CUDAExecutionProvider"] if capi.lib().cvad_device_count() > 0 else []
    except capi.EngineLibraryMissing:
        return []


def get_device() -> str:
    return "GPU"


# the largest |h| cvad_set_state / cvad_import_states accept (include/cutter_vad_b200.h)
H_BOUND = 2.0

_V5_MARK = "If_0_then_branch__Inline_0__stft.forward_basis_buffer"
_V4_MARK = "model.feature_extractor.forward_basis_buffer"


class InferenceSession:
    """One model file opened on the engine; holds a private scratch slot for `run`."""

    def __init__(self, path_or_bytes, sess_options: Optional[SessionOptions] = None,
                 providers: Optional[Sequence[str]] = None, **kwargs) -> None:
        path = Path(str(path_or_bytes))
        names = read_float_tensors(path)
        if _V5_MARK in names:
            self.version = "v5"
        elif _V4_MARK in names:
            self.version = "v4"
        else:
            raise ValueError(f"{path}: not a Silero VAD v4/v5 model")
        self._path = path
        self._pooled8, self._slot8 = None, -1          # v4 only: slot on the 8 kHz sub-model's engine, leased on first use
        self._pooled, self._slot = pool.lease_slot(self.version, model_path=None if _is_packaged(path) else path)
        with self._pooled.lock:
            self._pooled.engine.configure([self._slot], enable_denoising=False)
        if self.version == "v5":
            self._inputs = [NodeArg("input", [None, None], "tensor(float)"),
                            NodeArg("state", [2, None, 128], "tensor(float)"),
                            NodeArg("sr", [], "tensor(int64)")]
            self._outputs = [NodeArg("output", [None, 1], "tensor(float)"),
                             NodeArg("stateN", [None, None, None], "tensor(float)")]
        else:
            self._inputs = [NodeArg("input", [None, None], "tensor(float)"), NodeArg("sr", [], "tensor(int64)"),
                            NodeArg("h", [2, None, 64], "tensor(float)"), NodeArg("c", [2, None, 64], "tensor(float)")]
            self._outputs = [NodeArg("output", [None, 1], "tensor(float)"),
                             NodeArg("hn", [2, None, 64], "tensor(float)"), NodeArg("cn", [2, None, 64], "tensor(float)")]

    # -- introspection used by SileroVADModel._validate_model_signature / get_model_info
    def get_inputs(self) -> List[NodeArg]:
        return list(self._inputs)

    def get_outputs(self) -> List[NodeArg]:
        return list(self._outputs)

    def get_providers(self) -> List[str]:
        return ["CUDAExecutionProvider"]

    @property
    def engine(self):
        return self._pooled.engine

    def close(self) -> None:
        if getattr(self, "_pooled", None) is not None:
            try:
                self._pooled.release(self._slot)
                if getattr(self, "_pooled8", None) is not None:
                    self._pooled8.release(self._slot8)
            finally:
                self._pooled = None
                self._pooled8 = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- the stateless batch-1 call
    def run(self, output_names, input_feed: Dict[str, np.ndarray], run_options=None) -> List[np.ndarray]:
        x = np.asarray(input_feed["input"], dtype=np.float32)
        if x.ndim != 2 or x.shape[0] != 1:
            raise ValueError("compat session.run handles one stream per call; use BatchedVADManager for batches")
        sr = int(np.asarray(input_feed["sr"]).reshape(-1)[0])
        pooled, slot = self._pooled, self._slot
        if sr != 16000:
            # both graphs are `If(sr == 16000) 16 kHz model else 8 kHz model`.  v4's 8 kHz sub-model takes the same
            # 512-sample frames and runs on its own engine; v5's cannot run a 512-sample frame (the LSTM input
            # becomes 5-D, SURVEY.md 8a) and fails in onnxruntime as it does here
            if self.version != "v4":
                raise ValueError(f"sr={sr}: the v5 graph's 8 kHz branch cannot run 512-sample frames "
                                 "(invalid LSTM input in the reference as well)")
            if self._pooled8 is None:
                self._pooled8, self._slot8 = pool.lease_slot(
                    "v4_8k", model_path=None if _is_packaged(self._path) else self._path)
                with self._pooled8.lock:
                    self._pooled8.engine.configure([self._slot8], enable_denoising=False)
            pooled, slot = self._pooled8, self._slot8
        if self.version == "v5":
            state = np.asarray(input_feed["state"], dtype=np.float32)
            if state.shape != (2, 1, 128):
                raise ValueError(f"state must have shape (2, 1, 128), got {state.shape}")
            h_in, c_in = state[0, 0], state[1, 0]
        else:
            h_in = np.asarray(input_feed["h"], dtype=np.float32)
            c_in = np.asarray(input_feed["c"], dtype=np.float32)
            if h_in.shape != (2, 1, 64) or c_in.shape != (2, 1, 64):
                raise ValueError(f"h and c must have shape (2, 1, 64), got {h_in.shape} / {c_in.shape}")
            h_in, c_in = h_in.reshape(128), c_in.reshape(128)      # engine rows: layer-major [2][64]
        if not (np.abs(h_in) <= H_BOUND).all():
            raise ValueError(f"h must lie within [-{H_BOUND:g}, {H_BOUND:g}] (an LSTM's h = o * tanh(c) stays within "
                             "[-1, 1]; the engine's FP16-split kernels cannot hold more)")
        eng = pooled.engine
        with pooled.lock:
            if pooled is self._pooled:
                # the wrapper's fast path (core/silero_model.py: process_audio_batched) leaves its thresholds, gate and state
                # on this slot; this call runs without the gate and from its caller's state
                if getattr(self, "_dev_cfg", None) is not None:
                    eng.configure([slot], enable_denoising=False)
                    self._dev_cfg = None
                self._dev_state = None
            eng.set_state(slot, h_in, c_in, np.zeros(4, np.int32))
            frame_len = min(x.shape[1], 512)
            r = eng.step(x, slots=[slot], max_frames=1, frame_len=frame_len, hop=max(frame_len, 1))
            if r.status[0]:
                raise ValueError("Audio data contains infinite or NaN values")
            h, c, _, _ = eng.get_state(slot)
        out = r.probs.reshape(1, 1).astype(np.float32)
        if self.version == "v5":
            return [out, np.stack([h[None, :], c[None, :]], axis=0).astype(np.float32)]
        return [out, h.reshape(2, 1, 64).astype(np.float32), c.reshape(2, 1, 64).astype(np.float32)]


def _is_packaged(path: Path) -> bool:
    from .stream_engine import MODELS_DIR
    try:
        return path.resolve().parent == MODELS_DIR.resolve()
    except OSError:
        return False
