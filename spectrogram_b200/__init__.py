"""spectrogram_b200: B200-native engine for the frame-producing hot path of amilajack/spectrogram
(window -> real FFT -> magnitude -> dB -> byte/colour with AnalyserNode smoothing).

Python host layer over the C ABI (include/sgcore.h, libsgcore.so); the JavaScript facade and
Node-API shim for the same ABI live in spectrogram_b200/js.  No CPU fallback.
"""
from ._lib import (ALIGN_ANALYSER, ALIGN_VALID, OUT_F32_DB, OUT_F32_MAG, OUT_RGBA8, OUT_U8, WINDOW_BLACKMAN,
                   WINDOW_CUSTOM, WINDOW_HANN, WINDOW_RECT, EngineError, IndexSizeError, InvalidStateError)
from .analyser import AnalyserNode
from .biquad import AudioParam, BiquadFilterNode, biquad_coefficients
from .api import (AudioBuffer, Engine, Options, PinnedArray, SonogramRing, StreamBank, colormap_reference, default_engine, device_count,
                  resample_num_frames, shard_bounds, spectrogram, spectrogram_multi, wav_info)

__all__ = [
    "AnalyserNode", "AudioParam", "BiquadFilterNode", "biquad_coefficients", "AudioBuffer", "wav_info", "resample_num_frames", "Engine", "Options", "PinnedArray", "StreamBank", "SonogramRing", "spectrogram", "spectrogram_multi", "colormap_reference",
    "default_engine", "device_count", "shard_bounds", "IndexSizeError", "EngineError", "InvalidStateError",
    "WINDOW_BLACKMAN", "WINDOW_HANN", "WINDOW_RECT", "WINDOW_CUSTOM",
    "OUT_U8", "OUT_F32_DB", "OUT_RGBA8", "OUT_F32_MAG", "ALIGN_VALID", "ALIGN_ANALYSER",
]
