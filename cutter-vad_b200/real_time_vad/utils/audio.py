"""AudioUtils: the static helpers of the drop-in API.

Hot-path members (SURVEY.md section 8a rows F, V, M, D, R) keep the reference's exact
semantics because the GPU frame loader is defined against them:
  split_into_frames   audio.py:164-190   n = (len - frame)//hop + 1, no partial frame
  validate_audio_data audio.py:211-231   empty / NaN / Inf / ndim > 2
  convert_to_mono     audio.py:193-208   mean over axis 1
  denoise_audio       audio.py:104-121   a gate: x if |x| > thr else 0
  resample_audio      audio.py:19-55     scipy.signal.resample to int(len * ratio)
On the batched engine path the first four run inside `v5_frontend_kernel`; these host
versions serve the compatibility path and callers that use them directly.
"""
from __future__ import annotations

import io
from typing import Optional, Tuple

import numpy as np
from scipy import signal
from scipy.io import wavfile

from ..core.config import SampleRate  # noqa: F401  (re-exported like the reference module)
from ..core.exceptions import AudioProcessingError

_WINDOWS = {"hanning": np.hanning, "hamming": np.hamming, "blackman": np.blackman}


def _g711_tables():
    """ITU-T G.711 expansion of all 256 codes to 16-bit linear values (audioop.ulaw2lin / alaw2lin, width 2), the
    same integer arithmetic as the engine's decode stage."""
    c = np.arange(256, dtype=np.int32)
    u = ~c & 0xFF
    t = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4)
    ulaw = np.where(u & 0x80, 0x84 - t, t - 0x84)
    a = c ^ 0x55
    seg = (a & 0x70) >> 4
    t = (a & 0x0F) << 4
    m = np.where(seg == 0, t + 8, (t + 0x108) << np.maximum(seg - 1, 0))
    alaw = np.where(a & 0x80, m, -m)
    return {"ulaw": ulaw.astype(np.int16), "alaw": alaw.astype(np.int16)}


G711_LINEAR = _g711_tables()


class AudioUtils:
    # ------------------------------------------------------------------ hot-path helpers
    @staticmethod
    def split_into_frames(audio_data: np.ndarray, frame_size: int, hop_size: Optional[int] = None) -> np.ndarray:
        hop = frame_size // 2 if hop_size is None else hop_size
        count = (len(audio_data) - frame_size) // hop + 1
        frames = np.zeros((count, frame_size), dtype=audio_data.dtype)  # count < 0 raises, as in the reference
        for idx in range(count):
            frames[idx] = audio_data[idx * hop: idx * hop + frame_size]
        return frames

    @staticmethod
    def validate_audio_data(audio_data: np.ndarray) -> None:
        if not isinstance(audio_data, np.ndarray):
            raise AudioProcessingError("Audio data must be a numpy array")
        if audio_data.size == 0:
            raise AudioProcessingError("Audio data is empty")
        if not np.isfinite(audio_data).all():
            raise AudioProcessingError("Audio data contains infinite or NaN values")
        if audio_data.ndim > 2:
            raise AudioProcessingError(f"Audio data has too many dimensions: {audio_data.ndim}")

    @staticmethod
    def convert_to_mono(audio_data: np.ndarray) -> np.ndarray:
        if audio_data.ndim == 1:
            return audio_data
        if audio_data.ndim == 2:
            return np.mean(audio_data, axis=1)
        raise AudioProcessingError(f"Unsupported audio shape: {audio_data.shape}")

    @staticmethod
    def denoise_audio(audio_data: np.ndarray, noise_threshold: float = 0.01) -> np.ndarray:
        try:
            return np.where(np.abs(audio_data) > noise_threshold, audio_data, 0.0)
        except Exception as exc:
            raise AudioProcessingError(f"Failed to denoise audio: {exc}")

    @staticmethod
    def resample_audio(audio_data: np.ndarray, original_rate: int, target_rate: int) -> np.ndarray:
        try:
            if original_rate == target_rate:
                return audio_data
            out_len = int(len(audio_data) * (target_rate / original_rate))
            return signal.resample(audio_data, out_len).astype(np.float32)
        except Exception as exc:
            raise AudioProcessingError(
                f"Failed to resample audio from {original_rate}Hz to {target_rate}Hz: {exc}",
                f"Input shape: {audio_data.shape}, dtype: {audio_data.dtype}")

    # ------------------------------------------------------------------ everything else (host only)
    @staticmethod
    def normalize_audio(audio_data: np.ndarray, target_level: float = 0.9) -> np.ndarray:
        try:
            peak = np.max(np.abs(audio_data))
            return audio_data * (target_level / peak) if peak > 0 else audio_data
        except Exception as exc:
            raise AudioProcessingError(f"Failed to normalize audio: {exc}")

    @staticmethod
    def apply_window(audio_data: np.ndarray, window_type: str = "hanning") -> np.ndarray:
        try:
            if window_type not in _WINDOWS:
                raise ValueError(f"Unsupported window type: {window_type}")
            return audio_data * _WINDOWS[window_type](len(audio_data))
        except Exception as exc:
            raise AudioProcessingError(f"Failed to apply window: {exc}")

    @staticmethod
    def detect_clipping(audio_data: np.ndarray, threshold: float = 0.95) -> bool:
        return np.any(np.abs(audio_data) >= threshold)

    @staticmethod
    def calculate_rms(audio_data: np.ndarray) -> float:
        return np.sqrt(np.mean(audio_data ** 2))

    @staticmethod
    def calculate_energy(audio_data: np.ndarray) -> float:
        return np.sum(audio_data ** 2)

    @staticmethod
    def load_audio_file(file_path: str) -> Tuple[np.ndarray, int]:
        try:
            rate, data = wavfile.read(file_path)
            if data.dtype == np.int16:
                data = data.astype(np.float32) / 32768.0
            elif data.dtype == np.int32:
                data = data.astype(np.float32) / 2147483648.0
            elif data.dtype != np.float32:
                data = data.astype(np.float32)
            return AudioUtils.convert_to_mono(data), rate
        except Exception as exc:
            raise AudioProcessingError(f"Failed to load audio file {file_path}: {exc}")

    @staticmethod
    def _to_int(audio_data: np.ndarray, bit_depth: int) -> np.ndarray:
        if bit_depth == 16:
            return (audio_data * 32767).astype(np.int16)
        if bit_depth == 32:
            return (audio_data * 2147483647).astype(np.int32)
        raise ValueError(f"Unsupported bit depth: {bit_depth}")

    @staticmethod
    def save_audio_file(file_path: str, audio_data: np.ndarray, sample_rate: int, bit_depth: int = 16) -> None:
        try:
            wavfile.write(file_path, sample_rate, AudioUtils._to_int(audio_data, bit_depth))
        except Exception as exc:
            raise AudioProcessingError(f"Failed to save audio file {file_path}: {exc}")

    @staticmethod
    def g711_to_float32(codes, law: str) -> np.ndarray:
        """G.711 codes (uint8 array or bytes) -> float32 samples linear / 32768, with `law` "ulaw" or "alaw": exactly
        pcm_to_float32 of the linear PCM, and exactly what the engine's decode stage produces."""
        if law not in G711_LINEAR:
            raise AudioProcessingError(f"unknown G.711 law {law!r}")
        x = np.frombuffer(codes, np.uint8) if isinstance(codes, (bytes, bytearray, memoryview)) else np.asarray(codes)
        if x.dtype != np.uint8:
            raise AudioProcessingError(f"G.711 codes must be uint8, not {x.dtype}")
        return G711_LINEAR[law][x].astype(np.float32) / np.float32(32768.0)

    @staticmethod
    def pcm_to_float32(pcm_data: bytes, bit_depth: int = 16) -> np.ndarray:
        try:
            if bit_depth == 16:
                return np.frombuffer(pcm_data, dtype=np.int16).astype(np.float32) / 32768.0
            if bit_depth == 32:
                return np.frombuffer(pcm_data, dtype=np.int32).astype(np.float32) / 2147483648.0
            raise ValueError(f"Unsupported bit depth: {bit_depth}")
        except Exception as exc:
            raise AudioProcessingError(f"Failed to convert PCM to float32: {exc}")

    @staticmethod
    def float32_to_pcm(audio_data: np.ndarray, bit_depth: int = 16) -> bytes:
        try:
            return AudioUtils._to_int(audio_data, bit_depth).tobytes()
        except Exception as exc:
            raise AudioProcessingError(f"Failed to convert float32 to PCM: {exc}")
