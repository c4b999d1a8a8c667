"""Float64 oracle for the sample-rate conversion in front of the path (decodeAudioData resamples decoded audio to
its context's rate).  TEST INFRASTRUCTURE ONLY: nothing under ``spectrogram_b200/`` imports it.

The contract is rational polyphase resampling equal to ``scipy.signal.resample_poly(x, up, down)`` with scipy's
default filter.  Restated here independently of scipy (numpy's sinc and Kaiser window, a direct sum instead of
``upfirdn``), so that scipy stays a second, independent check (tests/test_pcm_resample.py).
"""
from __future__ import annotations

import math

import numpy as np


def resample_ratio(in_rate: int, out_rate: int) -> tuple[int, int]:
    """(up, down) = out_rate/in_rate in lowest terms."""
    g = math.gcd(int(in_rate), int(out_rate))
    return int(out_rate) // g, int(in_rate) // g


def resample_filter(up: int, down: int) -> np.ndarray:
    """The polyphase filter, float64, designed from its closed form with numpy only: h[m] = c sinc(c (m - half))
    kaiser_5(m), m = 0 .. 2 half, half = 10 max(up, down), c = 1/max(up, down), scaled to sum 1, then times up
    (what scipy.signal.resample_poly builds with firwin(2 half + 1, c, window=('kaiser', 5.0)) * up)."""
    mx = max(up, down)
    half = 10 * mx
    m = np.arange(2 * half + 1, dtype=np.float64)
    c = 1.0 / mx
    h = c * np.sinc(c * (m - half)) * np.kaiser(2 * half + 1, 5.0)
    return h / h.sum() * up


def resample(x, in_rate: int, out_rate: int, absolute: bool = False) -> np.ndarray:
    """Rational resampling of a 1-D signal by the direct float64 sum y[k] = sum_n x[n] h[k down + half - n up]
    over the n with 0 <= k down + half - n up <= 2 half (x is 0 outside [0, len(x))), len(y) = ceil(len(x) up/down).
    ``absolute=True`` returns sum_n |x[n] h[...]| instead (the scale of a float32 evaluation's rounding error)."""
    x = np.asarray(x, dtype=np.float64)
    up, down = resample_ratio(in_rate, out_rate)
    if up == down:
        return np.abs(x) if absolute else x.copy()
    h = resample_filter(up, down)
    half = (h.size - 1) // 2
    n_out = -(-x.size * up // down)
    k = np.arange(n_out, dtype=np.int64)
    t = k * down + half
    n_max, r = t // up, t % up
    y = np.zeros(n_out)
    for j in range(-(-h.size // up)):
        idx = r + j * up
        n = n_max - j
        ok = (idx < h.size) & (n >= 0) & (n < x.size)
        term = h[np.where(ok, idx, 0)] * x[np.clip(n, 0, max(x.size - 1, 0))] if x.size else np.zeros(n_out)
        y += np.where(ok, np.abs(term) if absolute else term, 0.0)
    return y
