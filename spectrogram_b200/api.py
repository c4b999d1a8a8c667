"""Host-side mirror of the reference's analyser interface for the frame path.

The reference's frame loop is ``analyser.getByteFrequencyData(freqByteData)`` once per
``requestAnimationFrame`` (src/javascripts/3D/visualizer.js:346-368, UI/spectrogram.js:153-161)
with the analyser configured at UI/player.js:7-11.  ``spectrogram()`` is the batched form of
that loop (fixed hop instead of rAF cadence); ``AnalyserNode`` (analyser.py) is the object form.
Everything computes in libsgcore.so's CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass

import numpy as np

from . import _lib as L

_OUT_NAMES = {"u8": L.OUT_U8, "byte": L.OUT_U8, "db": L.OUT_F32_DB, "float": L.OUT_F32_DB,
              "rgba": L.OUT_RGBA8, "rgba8": L.OUT_RGBA8, "mag": L.OUT_F32_MAG}
_WIN_NAMES = {"blackman": L.WINDOW_BLACKMAN, "hann": L.WINDOW_HANN, "rect": L.WINDOW_RECT}
_ALIGN_NAMES = {"valid": L.ALIGN_VALID, "analyser": L.ALIGN_ANALYSER}


@dataclass
class Options:
    """The options object of the JS facade: {fftSize, hop, window, minDecibels, maxDecibels,
    smoothingTimeConstant, output, align}.  Defaults are the reference's operating point
    (UI/player.js:10-11; AnalyserNode default dB range)."""

    fftSize: int = 2048
    hop: int = 512
    window: object = "blackman"      # name, or an array of fftSize floats
    minDecibels: float = -100.0
    maxDecibels: float = -30.0
    smoothingTimeConstant: float = 0.0
    output: str = "u8"
    align: str = "valid"
    colormap: object = None          # optional 256 x uint32 RGBA8 table

    def to_c(self):
        cfg = L.StftConfig()
        keep = []
        cfg.n_fft, cfg.hop = int(self.fftSize), int(self.hop)
        if isinstance(self.window, str):
            if self.window not in _WIN_NAMES:
                raise TypeError(f"unknown window {self.window!r}")
            cfg.window = _WIN_NAMES[self.window]
        else:
            w = np.ascontiguousarray(self.window, dtype=np.float32)
            if w.shape != (cfg.n_fft,):
                raise TypeError("custom window must have fftSize entries")
            keep.append(w)
            cfg.window = L.WINDOW_CUSTOM
            cfg.custom_window = w.ctypes.data_as(C.POINTER(C.c_float))
        if self.output not in _OUT_NAMES:
            raise TypeError(f"unknown output {self.output!r}")
        if self.align not in _ALIGN_NAMES:
            raise TypeError(f"unknown align {self.align!r}")
        cfg.output, cfg.align = _OUT_NAMES[self.output], _ALIGN_NAMES[self.align]
        cfg.min_db, cfg.max_db = float(self.minDecibels), float(self.maxDecibels)
        cfg.smoothing = float(self.smoothingTimeConstant)
        if self.colormap is not None:
            lut = np.ascontiguousarray(self.colormap, dtype=np.uint32)
            if lut.shape != (256,):
                raise TypeError("colormap must have 256 uint32 entries")
            keep.append(lut)
            cfg.colormap = lut.ctypes.data_as(C.POINTER(C.c_uint32))
        return cfg, keep


_PCM_FMT = {"u8": L.PCM_U8, "s16": L.PCM_S16, "s24": L.PCM_S24, "s32": L.PCM_S32, "f32": L.PCM_F32}
_PCM_FMT_OF = {v: k for k, v in _PCM_FMT.items()}
_PCM_BYTES = {L.PCM_U8: 1, L.PCM_S16: 2, L.PCM_S24: 3, L.PCM_S32: 4, L.PCM_F32: 4}


def _pcm_args(data, fmt, channels, sample_rate, n_clips):
    if fmt not in _PCM_FMT:
        raise TypeError(f"unknown PCM format {fmt!r}")
    raw = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else \
        np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    bpf = int(channels) * _PCM_BYTES[_PCM_FMT[fmt]]
    if channels < 1 or n_clips < 1 or raw.size % (bpf * n_clips):
        raise TypeError("PCM byte count is not clips x frames x channels x sample size")
    info = L.PcmInfo(_PCM_FMT[fmt], int(channels), int(sample_rate), raw.size // (bpf * n_clips), 0)
    return raw, info


def wav_info(file_bytes) -> "L.PcmInfo":
    """RIFF/WAVE header walk (host only, no GPU): format, channels, sample rate, frames, data offset."""
    buf = np.frombuffer(file_bytes, dtype=np.uint8) if not isinstance(file_bytes, np.ndarray) else file_bytes
    info = L.PcmInfo()
    L.check(L.load().sg_wav_parse(buf.ctypes.data, buf.size, C.byref(info)))
    return info


def resample_num_frames(frames: int, in_rate: int, out_rate: int) -> int:
    """Length after resampling ``frames`` sample frames from ``in_rate`` to ``out_rate`` Hz: ceil(frames*up/down)
    (``sg_resample_num_frames``; host only).  IndexSizeError for rates the resampler does not take."""
    n = int(L.load().sg_resample_num_frames(int(frames), int(in_rate), int(out_rate)))
    if n < 0:
        L.check(n)
    return n


class AudioBuffer:
    """What ``decodeAudioData`` hands the reference (util/util.js:10-12): planar float32 channels."""

    def __init__(self, planes: np.ndarray, sample_rate: int):
        self._planes = planes
        self.sampleRate = int(sample_rate)
        self.numberOfChannels = int(planes.shape[-2])
        self.length = int(planes.shape[-1])
        self.duration = self.length / self.sampleRate if self.sampleRate else 0.0

    def getChannelData(self, channel: int) -> np.ndarray:
        if not 0 <= channel < self.numberOfChannels:
            raise L.IndexSizeError("channel index out of range")
        return self._planes[..., channel, :]

    @property
    def planes(self) -> np.ndarray:
        return self._planes


def out_dtype_shape(output: int, n_clips: int, frames: int, bins: int):
    if output == L.OUT_U8:
        return np.uint8, (n_clips, frames, bins)
    if output == L.OUT_RGBA8:
        return np.uint8, (n_clips, frames, bins, 4)
    return np.float32, (n_clips, frames, bins)


class Engine:
    """One per GPU (``sg_engine``)."""

    def __init__(self, device: int = 0):
        self._lib = L.load()
        h = C.c_void_p()
        L.check(self._lib.sg_engine_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.sg_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        if not self._h:
            raise L.EngineError("engine is closed")
        return self._h

    @property
    def launch_count(self) -> int:
        return int(self._lib.sg_engine_launch_count(self.handle))

    @property
    def last_kernel(self) -> str:
        return self._lib.sg_engine_last_kernel(self.handle).decode()

    def set_kernel_variant(self, variant: int) -> None:
        L.check(self._lib.sg_engine_set_kernel_variant(self.handle, int(variant)))

    def synchronize(self) -> None:
        L.check(self._lib.sg_engine_synchronize(self.handle))

    # -- batched path on host arrays ------------------------------------------------------
    def num_frames(self, opts: Options, clip_len: int) -> int:
        cfg, _keep = opts.to_c()
        n = int(self._lib.sg_stft_num_frames(C.byref(cfg), int(clip_len)))
        if n < 0:
            L.check(L.SG_ERR_INDEX_SIZE if "must" in L.last_error() else L.SG_ERR_INVALID_ARG)
        return n

    def spectrogram(self, pcm, opts: Options | None = None, out: np.ndarray | None = None, **kw) -> np.ndarray:
        """pcm: [clips, samples] (or [samples]) float32 -> [clips, frames, bins(,4)]."""
        opts = opts or Options(**kw)
        x = np.asarray(pcm)
        if x.dtype != np.float32:
            x = x.astype(np.float32)
        squeeze = x.ndim == 1
        x = np.ascontiguousarray(np.atleast_2d(x))
        if x.ndim != 2:
            raise TypeError("pcm must be [samples] or [clips, samples]")
        cfg, _keep = opts.to_c()
        n_clips, clip_len = x.shape
        frames = int(self._lib.sg_stft_num_frames(C.byref(cfg), clip_len))
        if frames < 0:
            L.check(L.SG_ERR_INDEX_SIZE)
        dt, shape = out_dtype_shape(cfg.output, n_clips, frames, cfg.n_fft // 2)
        if out is None:
            out = np.empty(shape, dtype=dt)
        elif out.dtype != dt or out.shape != shape or not out.flags.c_contiguous:
            raise TypeError(f"out must be C-contiguous {dt} {shape}")
        L.check(self._lib.sg_stft_batch(self.handle, x.ctypes.data, n_clips, clip_len, C.byref(cfg), out.ctypes.data))
        return out[0] if squeeze else out

    # -- PCM ingestion in front of the path (decodeAudioData for uncompressed PCM) -------------
    def decode_pcm(self, data, fmt: str = "s16", channels: int = 1, sample_rate: int = 48000, n_clips: int = 1,
                   mix: bool = False, context_rate: int | None = None) -> "AudioBuffer":
        """Interleaved samples (bytes-like or array) -> float32 planes on the GPU.  ``mix=True`` applies the
        AnalyserNode's speakers down-mix to mono; otherwise every channel is a plane (AudioBuffer.getChannelData).
        ``context_rate``: resample from ``sample_rate`` to this rate on the GPU, as decodeAudioData does for a
        context running at that rate (``sg_pcm_ingest_resampled``)."""
        raw, info = _pcm_args(data, fmt, channels, sample_rate, n_clips)
        layout = L.PCM_MONO_MIX if mix else L.PCM_PLANAR
        planes = 1 if mix else channels
        if context_rate is None:
            out = np.empty((n_clips, planes, info.frames), dtype=np.float32)
            L.check(self._lib.sg_pcm_ingest(self.handle, raw.ctypes.data, n_clips, C.byref(info), layout, out.ctypes.data))
            return AudioBuffer(out[0] if n_clips == 1 else out, sample_rate)
        length = resample_num_frames(info.frames, sample_rate, context_rate)
        out = np.empty((n_clips, planes, length), dtype=np.float32)
        L.check(self._lib.sg_pcm_ingest_resampled(self.handle, raw.ctypes.data, n_clips, C.byref(info), layout,
                                                  int(context_rate), out.ctypes.data))
        return AudioBuffer(out[0] if n_clips == 1 else out, context_rate)

    def decode_audio_data(self, file_bytes, mix: bool = False, context_rate: int | None = None) -> "AudioBuffer":
        """``context.decodeAudioData(arrayBuffer)`` (util/util.js:9) for RIFF/WAVE files holding uncompressed PCM.
        ``context_rate``: the context's sample rate; the file's samples are resampled to it on the GPU."""
        buf = np.frombuffer(bytes(file_bytes) if not isinstance(file_bytes, (bytes, bytearray, memoryview)) else file_bytes,
                            dtype=np.uint8)
        info = wav_info(buf)
        body = buf[info.data_offset:info.data_offset + info.frames * info.channels * _PCM_BYTES[info.format]]
        return self.decode_pcm(body, _PCM_FMT_OF[info.format], info.channels, info.sample_rate, 1, mix, context_rate)

    def spectrogram_pcm(self, data, fmt: str = "s16", channels: int = 1, n_clips: int = 1, mix: bool = True,
                        opts: Options | None = None, sample_rate: int | None = None, context_rate: int | None = None,
                        **kw) -> np.ndarray:
        """Interleaved PCM bytes -> [clips, planes, frames, bins(,4)]: ingest fused in front of the batched path
        (the raw bytes are what crosses PCIe).  ``context_rate``: resample from ``sample_rate`` (then required)
        to this rate before framing, so bin k is k*context_rate/fftSize Hz whatever the source rate."""
        opts = opts or Options(**kw)
        if context_rate is not None and sample_rate is None:
            raise TypeError("context_rate needs the source sample_rate")
        raw, info = _pcm_args(data, fmt, channels, sample_rate or 0, n_clips)
        cfg, _keep = opts.to_c()
        length = info.frames if context_rate is None else resample_num_frames(info.frames, sample_rate, context_rate)
        frames = int(self._lib.sg_stft_num_frames(C.byref(cfg), length))
        if frames < 0:
            L.check(L.SG_ERR_INDEX_SIZE)
        planes = 1 if mix else channels
        dt, shape = out_dtype_shape(cfg.output, n_clips * planes, frames, cfg.n_fft // 2)
        out = np.empty((n_clips, planes) + shape[1:], dtype=dt)
        layout = L.PCM_MONO_MIX if mix else L.PCM_PLANAR
        if context_rate is None:
            L.check(self._lib.sg_stft_pcm(self.handle, raw.ctypes.data, n_clips, C.byref(info), layout, C.byref(cfg),
                                          out.ctypes.data))
        else:
            L.check(self._lib.sg_stft_pcm_resampled(self.handle, raw.ctypes.data, n_clips, C.byref(info), layout,
                                                    int(context_rate), C.byref(cfg), out.ctypes.data))
        return out

    # -- batched path on device memory (pointers + a CUDA stream handle) ---------------------
    def spectrogram_device(self, pcm_ptr: int, n_clips: int, clip_len: int, clip_stride: int, opts: Options,
                           out_ptr: int, stream: int = 0) -> None:
        cfg, _keep = opts.to_c()
        L.check(self._lib.sg_stft_batch_device(self.handle, C.c_void_p(pcm_ptr), n_clips, clip_len, clip_stride,
                                               C.byref(cfg), C.c_void_p(out_ptr), C.c_void_p(stream)))

    def biquad_device(self, node, in_ptr: int, n_channels: int, length: int, in_stride: int, out_ptr: int,
                      out_stride: int, state_ptr: int = 0, stream: int = 0) -> None:
        """``sg_biquad_filter_device`` with ``node``'s parameters (a BiquadFilterNode; its own state is not used):
        float32 channels at ``in_ptr + c*in_stride`` -> ``out_ptr + c*out_stride``, in place when the pointers and
        strides are equal.  ``state_ptr``: device [n_channels][4] float64 carried state, or 0.  Asynchronous."""
        p = node.params()
        L.check(self._lib.sg_biquad_filter_device(self.handle, C.byref(p), C.c_void_p(in_ptr), n_channels, length,
                                                  in_stride, C.c_void_p(out_ptr), out_stride,
                                                  C.c_void_p(state_ptr or None), C.c_void_p(stream)))


_default_engines: dict[int, Engine] = {}
_default_lock = threading.Lock()


def default_engine(device: int = 0) -> Engine:
    with _default_lock:
        if device not in _default_engines:
            _default_engines[device] = Engine(device)
        return _default_engines[device]


def device_count() -> int:
    return int(L.load().sg_device_count())


def shard_bounds(n_units: int, n_shards: int) -> list[tuple[int, int]]:
    """Contiguous block partition: unit i -> shard floor(i*G/n) (SURVEY 8(e))."""
    return [(n_units * s // n_shards, n_units * (s + 1) // n_shards) for s in range(n_shards)]


def spectrogram(pcm, devices=None, **kw) -> np.ndarray:
    """Batched frame path.  ``devices``: None/int -> one GPU; list -> clips sharded in contiguous
    blocks over one engine per GPU by ``sg_stft_batch_multi`` (a host thread per engine inside the
    library), results gathered by host copy into one array (no collective; shards are independent)."""
    opts = kw.pop("opts", None) or Options(**kw)
    if devices is None or isinstance(devices, int):
        return default_engine(devices or 0).spectrogram(pcm, opts)
    x = np.ascontiguousarray(np.atleast_2d(np.asarray(pcm, dtype=np.float32)))
    devs = list(devices)
    if len(set(devs)) != len(devs):
        raise TypeError("a device may be listed only once")
    return spectrogram_multi([default_engine(d) for d in devs], x, opts)


def spectrogram_multi(engines, pcm, opts: Options) -> np.ndarray:
    """``sg_stft_batch_multi`` on explicit engines (normally one per GPU; several engines on one GPU also work)."""
    x = np.ascontiguousarray(np.atleast_2d(np.asarray(pcm, dtype=np.float32)))
    engs = list(engines)
    cfg, _keep = opts.to_c()
    frames = engs[0].num_frames(opts, x.shape[1])
    dt, shape = out_dtype_shape(cfg.output, x.shape[0], frames, cfg.n_fft // 2)
    out = np.empty(shape, dtype=dt)
    # sg_stft_batch_multi: contiguous clip blocks, one host thread per engine inside the library, disjoint output slices
    handles = (C.c_void_p * len(engs))(*[e.handle for e in engs])
    L.check(L.load().sg_stft_batch_multi(handles, len(engs), x.ctypes.data, x.shape[0], x.shape[1], C.byref(cfg),
                                         out.ctypes.data))
    return out


def colormap_reference() -> np.ndarray:
    lut = np.empty(256, dtype=np.uint32)
    L.check(L.load().sg_colormap_reference(lut.ctypes.data))
    return lut


class PinnedArray:
    """numpy view over page-locked host memory (sg_host_alloc), for DMA without staging."""

    def __init__(self, shape, dtype):
        self._lib = L.load()
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        L.check(self._lib.sg_host_alloc(max(nbytes, 1), C.byref(p)))
        self._p = p
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if getattr(self, "_p", None):
            self.array = None
            self._lib.sg_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _param_key(p: L.BiquadParams) -> tuple:
    return (p.type, p.sample_rate, p.frequency, p.q, p.gain, p.detune)


class StreamBank:
    """``sg_stream``: n_channels analysers advanced in lock step (BASELINE config 5).

    ``history_rows``: keep a sonogram history per channel on the device (``sg_stream_set_history``) -- what a
    ``SonogramRing(bins, history_rows)`` fed every push's byte rows would hold -- so ``view()`` renders every channel's
    picture in one launch without the rows crossing PCIe twice.  Needs ``output="u8"``.

    ``filter``: a BiquadFilterNode in front of every channel's analyser (``sg_stream_set_filter``; the reference's draw
    mode).  The bank keeps the filter state on the device and re-sends the node's parameters before a push when they
    changed since the last one; the node's own ``process`` state is not used."""

    def __init__(self, n_channels: int, opts: Options, max_chunk: int | None = None, engine: Engine | None = None,
                 history_rows: int | None = None, filter=None):
        self.engine = engine or default_engine(0)
        self._lib = L.load()
        self.opts = opts
        self.n_channels = int(n_channels)
        self.max_chunk = int(max_chunk or opts.hop)
        cfg, self._keep = opts.to_c()
        self._cfg = cfg
        h = C.c_void_p()
        L.check(self._lib.sg_stream_create(self.engine.handle, self.n_channels, C.byref(cfg), self.max_chunk, C.byref(h)))
        self._h = h
        self._filter = None
        self._filter_sent = None
        if history_rows is not None:
            self.set_history(history_rows)
        if filter is not None:
            self.set_filter(filter)

    # -- biquad filter in front of the analysers ---------------------------------------------------
    def set_filter(self, node) -> None:
        """Attach ``node`` (a BiquadFilterNode) or detach with None.  The first attach starts from zero state; a new
        node or new parameters while attached keep it; detaching drops it."""
        if node is None:
            L.check(self._lib.sg_stream_set_filter(self._h, None))
            self._filter = self._filter_sent = None
            return
        p = node.params()
        L.check(self._lib.sg_stream_set_filter(self._h, C.byref(p)))
        self._filter, self._filter_sent = node, _param_key(p)

    @property
    def filter(self):
        return self._filter

    def _sync_filter(self) -> None:
        if self._filter is not None:
            p = self._filter.params()
            if _param_key(p) != self._filter_sent:
                L.check(self._lib.sg_stream_set_filter(self._h, C.byref(p)))
                self._filter_sent = _param_key(p)

    def push(self, chunk, out=None, out_rgba=None, want_rgba: bool = False):
        x = np.ascontiguousarray(chunk, dtype=np.float32)
        if x.ndim != 2 or x.shape[0] != self.n_channels:
            raise TypeError("chunk must be [n_channels, chunk_len]")
        chunk_len = x.shape[1]
        frames = chunk_len // self.opts.hop
        dt, shape = out_dtype_shape(self._cfg.output, self.n_channels, frames, self._cfg.n_fft // 2)
        if out is None:
            out = np.empty(shape, dtype=dt)
        if want_rgba and out_rgba is None:
            out_rgba = np.empty((self.n_channels, frames, self._cfg.n_fft // 2, 4), dtype=np.uint8)
        self._sync_filter()
        L.check(self._lib.sg_stream_push(self._h, x.ctypes.data, chunk_len, out.ctypes.data,
                                         out_rgba.ctypes.data if out_rgba is not None else None))
        return (out, out_rgba) if out_rgba is not None else out

    def advance(self, chunk) -> None:
        """``push`` whose byte rows only go to the sonogram history: nothing is copied back to the host."""
        x = np.ascontiguousarray(chunk, dtype=np.float32)
        if x.ndim != 2 or x.shape[0] != self.n_channels:
            raise TypeError("chunk must be [n_channels, chunk_len]")
        self._sync_filter()
        L.check(self._lib.sg_stream_push(self._h, x.ctypes.data, x.shape[1], None, None))

    def reset(self):
        L.check(self._lib.sg_stream_reset(self._h))

    # -- sonogram history ----------------------------------------------------------------------
    def set_history(self, rows: int) -> None:
        """Attach an empty history of ``rows`` rows per channel ([2, 65536]); 0 detaches it."""
        L.check(self._lib.sg_stream_set_history(self._h, int(rows)))

    def _history_info(self):
        rows, y = C.c_int(), C.c_int()
        L.check(self._lib.sg_stream_history_info(self._h, C.byref(rows), C.byref(y)))
        return rows.value, y.value

    @property
    def history_rows(self) -> int:
        return self._history_info()[0]

    @property
    def history_yoffset(self) -> int:
        return self._history_info()[1]

    def _range(self, first, count):
        first = int(first)
        return first, (self.n_channels - first if count is None else int(count))

    def history(self, first: int = 0, count: int | None = None) -> np.ndarray:
        """Textures of channels [first, first+count): uint8 [count, rows, bins] in texture row order."""
        first, count = self._range(first, count)
        rows = self.history_rows
        out = np.empty((max(count, 0), rows, self._cfg.n_fft // 2), dtype=np.uint8)
        L.check(self._lib.sg_stream_history_read(self._h, first, count, out.ctypes.data))
        return out

    def view(self, width: int, height: int, first: int = 0, count: int | None = None,
             out: np.ndarray | None = None) -> np.ndarray:
        """Sonogram pictures of channels [first, first+count), one launch: RGBA8 [count, height, width, 4], each equal
        to ``SonogramRing.view`` of that channel's ring."""
        first, count = self._range(first, count)
        shape = (max(count, 0), max(int(height), 0), max(int(width), 0), 4)
        if out is None:
            out = np.empty(shape, dtype=np.uint8)
        elif out.dtype != np.uint8 or out.shape != shape or not out.flags.c_contiguous:
            raise TypeError(f"out must be C-contiguous uint8 {shape}")
        L.check(self._lib.sg_stream_view(self._h, first, count, int(width), int(height), out.ctypes.data))
        return out

    @property
    def frames_emitted(self) -> int:
        return int(self._lib.sg_stream_frames_emitted(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sg_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SonogramRing:
    """``sg_ring``: the reference's spectrogram history -- a ``bins x rows`` byte texture written one row per frame at
    ``yoffset`` (3D/visualizer.js:60, 301-329, 399-416) -- kept on the device, plus its headless sonogram view
    (bin/shaders/sonogram-fragment.shader:14-27, sonogram-vertex.shader:19-58)."""

    def __init__(self, bins: int, rows: int = 256, engine: Engine | None = None):
        self.engine = engine or default_engine(0)
        self._lib = L.load()
        self.bins, self.rows = int(bins), int(rows)
        h = C.c_void_p()
        L.check(self._lib.sg_ring_create(self.engine.handle, self.bins, self.rows, C.byref(h)))
        self._h = h

    def append(self, frames) -> None:
        """texSubImage2D of one or more byte rows ([bins] or [n, bins] uint8) at yoffset, then advance yoffset."""
        f = np.ascontiguousarray(frames, dtype=np.uint8)
        if f.ndim == 1:
            f = f[None, :]
        if f.ndim != 2 or f.shape[1] != self.bins:
            raise TypeError("frames must be [n, bins] uint8")
        L.check(self._lib.sg_ring_append(self._h, f.ctypes.data, f.shape[0]))

    @property
    def yoffset(self) -> int:
        return int(self._lib.sg_ring_yoffset(self._h))

    def texture(self) -> np.ndarray:
        out = np.empty((self.rows, self.bins), dtype=np.uint8)
        L.check(self._lib.sg_ring_read(self._h, out.ctypes.data))
        return out

    def view(self, width: int, height: int, out: np.ndarray | None = None) -> np.ndarray:
        """RGBA8 image [height, width, 4] of the sonogram view (log-frequency x axis, time along y, edge fade)."""
        if out is None:
            out = np.empty((int(height), int(width), 4), dtype=np.uint8)
        L.check(self._lib.sg_ring_view(self._h, int(width), int(height), out.ctypes.data))
        return out

    def reset(self) -> None:
        L.check(self._lib.sg_ring_reset(self._h))

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.sg_ring_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
