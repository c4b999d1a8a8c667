"""``BiquadFilterNode`` (W3C Web Audio) on the GPU.

The reference's draw mode (``Player.setBandpassFrequency``, UI/player.js) routes the mix through
``bandpass.type = 'bandpass'; bandpass.Q.value = 10; bandpass.frequency.value = f`` into the analyser, so the
sonogram shows only the band under the pointer.  ``analyser.push(node.process(x))`` reproduces that chain, and
``StreamBank(..., filter=node)`` does it inside the bank.  Coefficients follow the spec's table (``sgcore.h``,
"biquad filter"); the float64 recurrence runs in libsgcore.so's kernels.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib as L


class AudioParam:
    """The ``.value`` of an AudioParam (no automation).  Non-finite values are a TypeError, as WebIDL's ``float``."""

    def __init__(self, default: float):
        self.defaultValue = float(default)
        self._value = float(default)

    @property
    def value(self) -> float:
        return self._value

    @value.setter
    def value(self, v) -> None:
        v = float(v)
        if not math.isfinite(v):
            raise TypeError("AudioParam value must be finite")
        self._value = v


def biquad_params(type: str = "lowpass", frequency: float = 350.0, Q: float = 1.0, gain: float = 0.0,
                  detune: float = 0.0, sample_rate: float = 48000) -> L.BiquadParams:
    """``sg_biquad_params`` from the node's attribute names."""
    if type not in L.BIQUAD_TYPES:
        raise TypeError(f"unknown biquad type {type!r}")
    return L.BiquadParams(L.BIQUAD_TYPES.index(type), float(sample_rate), float(frequency), float(Q), float(gain),
                          float(detune))


def biquad_coefficients(type: str = "lowpass", frequency: float = 350.0, Q: float = 1.0, gain: float = 0.0,
                        detune: float = 0.0, sample_rate: float = 48000) -> np.ndarray:
    """Normalised ``[b0, b1, b2, a1, a2]`` (float64) of a BiquadFilterNode with these parameters."""
    p = biquad_params(type, frequency, Q, gain, detune, sample_rate)
    c = np.empty(5, np.float64)
    L.check(L.load().sg_biquad_coefficients(C.byref(p), c.ctypes.data))
    return c


class BiquadFilterNode:
    """``context.createBiquadFilter()`` for ``channels`` channels at the context's ``sample_rate``.

    ``process(x)`` filters [channels, n] (or [n] for one channel) float32 samples on the GPU and carries the
    per-channel state ``{x1, x2, y1, y2}`` to the next call; ``reset()`` zeroes it.  A parameter change between
    calls keeps the state, as an AudioParam change between render quanta does."""

    def __init__(self, engine=None, sample_rate: float = 48000, channels: int = 1):
        if int(channels) < 1:
            raise TypeError("channels must be >= 1")
        self._engine = engine
        self.sample_rate = sample_rate
        self.channels = int(channels)
        self._type = "lowpass"
        self.frequency = AudioParam(350.0)
        self.Q = AudioParam(1.0)
        self.gain = AudioParam(0.0)
        self.detune = AudioParam(0.0)
        self._state = np.zeros((self.channels, 4), np.float64)

    @property
    def type(self) -> str:
        return self._type

    @type.setter
    def type(self, value: str) -> None:
        if value not in L.BIQUAD_TYPES:
            raise TypeError(f"unknown biquad type {value!r}")
        self._type = value

    @property
    def engine(self):
        if self._engine is None:
            from .api import default_engine
            self._engine = default_engine(0)
        return self._engine

    def params(self) -> L.BiquadParams:
        return biquad_params(self._type, self.frequency.value, self.Q.value, self.gain.value, self.detune.value,
                             self.sample_rate)

    def coefficients(self) -> np.ndarray:
        return biquad_coefficients(self._type, self.frequency.value, self.Q.value, self.gain.value, self.detune.value,
                                   self.sample_rate)

    @property
    def state(self) -> np.ndarray:
        """[channels, 4] float64 ``{x1, x2, y1, y2}`` (a copy)."""
        return self._state.copy()

    def process(self, x) -> np.ndarray:
        a = np.ascontiguousarray(x, dtype=np.float32)
        squeeze = a.ndim == 1 and self.channels == 1
        if squeeze:
            a = a[None]
        if a.ndim != 2 or a.shape[0] != self.channels:
            raise TypeError(f"samples must be [{self.channels}, n]" + (" or [n]" if self.channels == 1 else ""))
        out = np.empty_like(a)
        p = self.params()
        L.check(L.load().sg_biquad_filter(self.engine.handle, C.byref(p), a.ctypes.data, a.shape[0], a.shape[1],
                                          self._state.ctypes.data, out.ctypes.data))
        return out[0] if squeeze else out

    def reset(self) -> None:
        self._state[:] = 0.0
