"""ctypes binding of libsgcore.so (C ABI: include/sgcore.h).

This is the Python stand-in for the Node-API shim a JavaScript host would load (js/ holds that
shim and facade; INTEGRATION.md shows the binding).  There is no CPU fallback: if the CUDA
library is missing, or no B200 is visible, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SG_LIBSGCORE selects another build of the same library (the SG_DEBUG build of tests/test_debug_build.py)
LIB_PATH = os.environ.get("SG_LIBSGCORE") or os.path.join(_HERE, "libsgcore.so")

SG_OK = 0
SG_ERR_INVALID_ARG = -1
SG_ERR_INDEX_SIZE = -2
SG_ERR_CUDA = -3
SG_ERR_OOM = -4
SG_ERR_NO_DEVICE = -5
SG_ERR_STATE = -6

WINDOW_BLACKMAN, WINDOW_HANN, WINDOW_RECT, WINDOW_CUSTOM = 0, 1, 2, 3
OUT_U8, OUT_F32_DB, OUT_RGBA8, OUT_F32_MAG = 0, 1, 2, 3
ALIGN_VALID, ALIGN_ANALYSER = 0, 1
PCM_U8, PCM_S16, PCM_S24, PCM_S32, PCM_F32 = 0, 1, 2, 3, 4
PCM_MONO_MIX, PCM_PLANAR = 0, 1


class IndexSizeError(ValueError):
    """Web Audio ``IndexSizeError`` DOMException (invalid fftSize / dB range / smoothing)."""

    name = "IndexSizeError"


class EngineError(RuntimeError):
    """CUDA failure, out of memory, or no device (the engine has no CPU path)."""


class InvalidStateError(RuntimeError):
    """Web platform ``InvalidStateError`` DOMException: the call is not valid in the object's current state
    (``SG_ERR_STATE``, e.g. a sonogram view of a stream bank without a history)."""

    name = "InvalidStateError"


class StftConfig(C.Structure):
    """``sg_stft_config``."""

    _fields_ = [
        ("n_fft", C.c_int32), ("hop", C.c_int32), ("window", C.c_int32),
        ("output", C.c_int32), ("align", C.c_int32),
        ("min_db", C.c_float), ("max_db", C.c_float), ("smoothing", C.c_float),
        ("custom_window", C.POINTER(C.c_float)), ("colormap", C.POINTER(C.c_uint32)),
    ]


class PcmInfo(C.Structure):
    """``sg_pcm_info``."""

    _fields_ = [("format", C.c_int32), ("channels", C.c_int32), ("sample_rate", C.c_int32),
                ("frames", C.c_int64), ("data_offset", C.c_int64)]


class BiquadParams(C.Structure):
    """``sg_biquad_params``."""

    _fields_ = [("type", C.c_int32), ("sample_rate", C.c_double), ("frequency", C.c_double), ("q", C.c_double),
                ("gain", C.c_double), ("detune", C.c_double)]


BIQUAD_TYPES = ("lowpass", "highpass", "bandpass", "lowshelf", "highshelf", "peaking", "notch", "allpass")

# name -> (restype, argtypes); every symbol include/sgcore.h declares
SIGNATURES = {
    "sg_last_error": (C.c_char_p, []),
    "sg_version": (C.c_int, []),
    "sg_device_count": (C.c_int, []),
    "sg_stft_config_default": (C.c_int, [C.POINTER(StftConfig)]),
    "sg_engine_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "sg_engine_destroy": (C.c_int, [C.c_void_p]),
    "sg_engine_device": (C.c_int, [C.c_void_p]),
    "sg_engine_launch_count": (C.c_int64, [C.c_void_p]),
    "sg_engine_last_kernel": (C.c_char_p, [C.c_void_p]),
    "sg_engine_set_kernel_variant": (C.c_int, [C.c_void_p, C.c_int]),
    "sg_engine_synchronize": (C.c_int, [C.c_void_p]),
    "sg_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "sg_host_free": (C.c_int, [C.c_void_p]),
    "sg_stft_num_bins": (C.c_int, [C.POINTER(StftConfig)]),
    "sg_stft_num_frames": (C.c_int64, [C.POINTER(StftConfig), C.c_int64]),
    "sg_stft_elem_bytes": (C.c_int, [C.POINTER(StftConfig)]),
    "sg_stft_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(StftConfig), C.c_void_p]),
    "sg_stft_batch_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(StftConfig),
                                      C.c_void_p]),
    "sg_stft_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                       C.POINTER(StftConfig), C.c_void_p, C.c_void_p]),
    "sg_colormap_reference": (C.c_int, [C.c_void_p]),
    "sg_analyser_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "sg_analyser_destroy": (C.c_int, [C.c_void_p]),
    "sg_analyser_set_fft_size": (C.c_int, [C.c_void_p, C.c_int]),
    "sg_analyser_get_fft_size": (C.c_int, [C.c_void_p]),
    "sg_analyser_get_frequency_bin_count": (C.c_int, [C.c_void_p]),
    "sg_analyser_set_min_decibels": (C.c_int, [C.c_void_p, C.c_double]),
    "sg_analyser_set_max_decibels": (C.c_int, [C.c_void_p, C.c_double]),
    "sg_analyser_get_min_decibels": (C.c_double, [C.c_void_p]),
    "sg_analyser_get_max_decibels": (C.c_double, [C.c_void_p]),
    "sg_analyser_set_smoothing_time_constant": (C.c_int, [C.c_void_p, C.c_double]),
    "sg_analyser_get_smoothing_time_constant": (C.c_double, [C.c_void_p]),
    "sg_analyser_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "sg_analyser_get_byte_frequency_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "sg_analyser_get_float_frequency_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "sg_analyser_get_byte_time_domain_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "sg_analyser_get_float_time_domain_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "sg_stream_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(StftConfig), C.c_int, C.POINTER(C.c_void_p)]),
    "sg_stream_destroy": (C.c_int, [C.c_void_p]),
    "sg_stream_reset": (C.c_int, [C.c_void_p]),
    "sg_stream_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "sg_stream_frames_emitted": (C.c_int64, [C.c_void_p]),
    "sg_stream_info": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_int)] * 5),
    "sg_stream_set_history": (C.c_int, [C.c_void_p, C.c_int]),
    "sg_stream_history_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sg_stream_history_read": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "sg_stream_view": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "sg_biquad_coefficients": (C.c_int, [C.POINTER(BiquadParams), C.c_void_p]),
    "sg_biquad_filter": (C.c_int, [C.c_void_p, C.POINTER(BiquadParams), C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                   C.c_void_p]),
    "sg_biquad_filter_device": (C.c_int, [C.c_void_p, C.POINTER(BiquadParams), C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "sg_stream_set_filter": (C.c_int, [C.c_void_p, C.POINTER(BiquadParams)]),
    "sg_pcm_sample_bytes": (C.c_int, [C.c_int]),
    "sg_pcm_num_planes": (C.c_int, [C.POINTER(PcmInfo), C.c_int]),
    "sg_wav_parse": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(PcmInfo)]),
    "sg_pcm_ingest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PcmInfo), C.c_int, C.c_void_p]),
    "sg_pcm_ingest_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PcmInfo), C.c_int, C.c_void_p,
                                       C.c_int64, C.c_void_p]),
    "sg_stft_pcm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PcmInfo), C.c_int, C.POINTER(StftConfig),
                              C.c_void_p]),
    "sg_resample_num_frames": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "sg_pcm_ingest_resampled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PcmInfo), C.c_int, C.c_int32,
                                          C.c_void_p]),
    "sg_pcm_ingest_resampled_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PcmInfo), C.c_int,
                                                 C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "sg_stft_pcm_resampled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PcmInfo), C.c_int, C.c_int32,
                                        C.POINTER(StftConfig), C.c_void_p]),
    "sg_ring_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "sg_ring_destroy": (C.c_int, [C.c_void_p]),
    "sg_ring_reset": (C.c_int, [C.c_void_p]),
    "sg_ring_append": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "sg_ring_yoffset": (C.c_int, [C.c_void_p]),
    "sg_ring_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sg_ring_read": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sg_ring_view": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Loads libsgcore.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EngineError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C spectrogram_b200/csrc` (there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    return load().sg_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Maps sg_status to the exception a Web Audio host would see."""
    if rc == SG_OK:
        return
    msg = last_error()
    if rc == SG_ERR_INDEX_SIZE:
        raise IndexSizeError(msg)
    if rc == SG_ERR_INVALID_ARG:
        raise TypeError(msg)
    if rc == SG_ERR_OOM:
        raise MemoryError(msg)
    if rc == SG_ERR_STATE:
        raise InvalidStateError(msg)
    raise EngineError(f"sg_status {rc}: {msg}")
