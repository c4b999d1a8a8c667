"""Float64 oracle of the W3C BiquadFilterNode: the coefficient table of include/sgcore.h ("biquad filter") restated,
and the direct-form-I recurrence (scipy.signal.lfilter with the carried state turned into zi by lfiltic, checked
against a plain loop in tests/test_biquad.py)."""
import math

import numpy as np
from scipy import signal

TYPES = ("lowpass", "highpass", "bandpass", "lowshelf", "highshelf", "peaking", "notch", "allpass")


def coefficients(type="lowpass", frequency=350.0, Q=1.0, gain=0.0, detune=0.0, sample_rate=48000):
    """Normalised [b0, b1, b2, a1, a2]; raises ValueError where the library returns SG_ERR_INVALID_ARG."""
    fs = float(sample_rate)
    if type not in TYPES:
        raise ValueError("type")
    if not all(math.isfinite(v) for v in (fs, frequency, Q, gain, detune)):
        raise ValueError("non-finite")
    if not (3000 <= fs <= 768000) or fs != math.floor(fs):
        raise ValueError("sample_rate")
    nyq = fs / 2.0
    f0 = 0.0 if frequency == 0.0 else frequency * 2.0 ** (detune / 1200.0)
    f0 = min(max(f0, 0.0), nyq)
    A = 10.0 ** (gain / 40.0)
    if f0 == 0.0:
        k = {"lowpass": 0.0, "bandpass": 0.0, "highshelf": A * A}.get(type, 1.0)
        return np.array([k, 0, 0, 0, 0], np.float64)
    if f0 == nyq:
        k = {"highpass": 0.0, "bandpass": 0.0, "lowshelf": A * A}.get(type, 1.0)
        return np.array([k, 0, 0, 0, 0], np.float64)
    if Q <= 0 and type in ("bandpass", "notch", "allpass", "peaking"):
        k = {"bandpass": 1.0, "notch": 0.0, "allpass": -1.0, "peaking": A * A}[type]
        return np.array([k, 0, 0, 0, 0], np.float64)
    w0 = 2.0 * math.pi * f0 / fs
    c, s = math.cos(w0), math.sin(w0)
    aq = s / (2.0 * Q) if Q > 0 else 0.0
    aqdb = s / (2.0 * 10.0 ** (Q / 20.0))
    k = 2.0 * (s / math.sqrt(2.0)) * math.sqrt(A)
    b0, b1, b2, a0, a1, a2 = {
        "lowpass": ((1 - c) / 2, 1 - c, (1 - c) / 2, 1 + aqdb, -2 * c, 1 - aqdb),
        "highpass": ((1 + c) / 2, -(1 + c), (1 + c) / 2, 1 + aqdb, -2 * c, 1 - aqdb),
        "bandpass": (aq, 0.0, -aq, 1 + aq, -2 * c, 1 - aq),
        "lowshelf": (A * ((A + 1) - (A - 1) * c + k), 2 * A * ((A - 1) - (A + 1) * c), A * ((A + 1) - (A - 1) * c - k),
                     (A + 1) + (A - 1) * c + k, -2 * ((A - 1) + (A + 1) * c), (A + 1) + (A - 1) * c - k),
        "highshelf": (A * ((A + 1) + (A - 1) * c + k), -2 * A * ((A - 1) + (A + 1) * c), A * ((A + 1) + (A - 1) * c - k),
                      (A + 1) - (A - 1) * c + k, 2 * ((A - 1) - (A + 1) * c), (A + 1) - (A - 1) * c - k),
        "peaking": (1 + aq * A, -2 * c, 1 - aq * A, 1 + aq / A, -2 * c, 1 - aq / A),
        "notch": (1.0, -2 * c, 1.0, 1 + aq, -2 * c, 1 - aq),
        "allpass": (1 - aq, -2 * c, 1 + aq, 1 + aq, -2 * c, 1 - aq),
    }[type]
    return np.array([b0 / a0, b1 / a0, b2 / a0, a1 / a0, a2 / a0], np.float64)


def filter_df1(coef, x, state=None):
    """y (float64) of x [channels, n] and the final state [channels, 4] {x1, x2, y1, y2}."""
    x = np.atleast_2d(np.asarray(x, np.float64))
    st = np.zeros((x.shape[0], 4)) if state is None else np.asarray(state, np.float64)
    b, a = coef[:3], np.array([1.0, coef[3], coef[4]])
    y = np.empty_like(x)
    out = np.empty((x.shape[0], 4))
    for ch in range(x.shape[0]):
        zi = signal.lfiltic(b, a, y=st[ch, 2:], x=st[ch, :2])
        y[ch], _ = signal.lfilter(b, a, x[ch], zi=zi)
        xs = np.concatenate([st[ch, 1::-1], x[ch]])          # ..., x2, x1, x[0], ...
        ys = np.concatenate([st[ch, 3:1:-1], y[ch]])
        out[ch] = (xs[-1], xs[-2], ys[-1], ys[-2])
    return y, out


def filter_loop(coef, x, state=(0.0, 0.0, 0.0, 0.0)):
    """The recurrence as written, one channel."""
    b0, b1, b2, a1, a2 = coef
    x1, x2, y1, y2 = state
    y = np.empty(len(x))
    for n, v in enumerate(np.asarray(x, np.float64)):
        y[n] = b0 * v + b1 * x1 + b2 * x2 - a1 * y1 - a2 * y2
        x2, x1, y2, y1 = x1, v, y1, y[n]
    return y, np.array([x1, x2, y1, y2])


def bound_violations(got, want64, x):
    """Samples outside max(1 float32 ulp of the rounded oracle, 2^-30 max|x| of the channel)."""
    got = np.atleast_2d(got)
    want = np.atleast_2d(want64).astype(np.float32)
    x = np.atleast_2d(x)
    tol = np.maximum(np.spacing(np.abs(want)), np.abs(x).max(axis=1, keepdims=True).astype(np.float32) * 2.0 ** -30)
    diff = np.abs(got.astype(np.float64) - want.astype(np.float64))
    return int(np.count_nonzero(~(diff <= tol) & ~(np.isnan(got) & np.isnan(want))))
