"""real_time_vad -- drop-in for Picurit/cutter-vad's package, running on a B200-native engine.

Same import surface as the reference's `src/real_time_vad/__init__.py` (VADWrapper,
AsyncVADWrapper, VADConfig, SampleRate, SileroModelVersion, the exception family,
AudioUtils, WAVWriter) plus `BatchedVADManager`, the multi-stream entry the north star adds.
The Silero arithmetic runs in hand-written sm_100a CUDA kernels behind the C ABI in
`include/cutter_vad_b200.h`; there is no onnxruntime and no CPU fallback.
"""
from .core.async_vad_wrapper import AsyncVADWrapper
from .core.batched_manager import BatchedVADManager, StreamEvent
from .core.sharded_manager import ShardedVADManager
from .core.stream_snapshot import StreamSnapshot
from .core.config import SampleRate, SileroModelVersion, VADConfig
from .core.exceptions import ConfigurationError, ModelNotFoundError, VADError
from .core.vad_wrapper import VADWrapper
from .utils.audio import AudioUtils
from .utils.wav_writer import WAVWriter

__version__ = "1.0.0+b200"

__all__ = ["VADWrapper", "AsyncVADWrapper", "BatchedVADManager", "ShardedVADManager", "StreamEvent", "StreamSnapshot", "VADConfig", "SampleRate",
           "SileroModelVersion", "VADError", "ModelNotFoundError", "ConfigurationError", "AudioUtils",
           "WAVWriter", "__version__"]
