"""The streaming bank (``StreamBank`` / ``sg_stream_*``) against the float64 oracle, on every kernel family and smoothing
path a push can reach.

A push runs no kernel of its own.  ``sg_stream_push`` hands the batch dispatcher every channel as a clip that starts
``hop`` samples into its ``[history | chunk]`` row.  The rows are ``n_fft + max_chunk`` samples apart (rounded up to 4),
each clip has one to a few frames, and with tau > 0 the smoothing state is carried from one push to the next.  Which
kernel takes the push then depends on the channel count, the SM count and the frames per push.  Every case below names
the family it expects (``last_kernel``) and the launches per push, so that a dispatcher change that moves a case to
another family fails instead of quietly testing something else.

The reference: a bank fed chunks c_1 .. c_k of a signal x returns, concatenated along frames, what
``O.spectrogram(x, Config(align=ALIGN_ANALYSER, smoothing=tau))`` returns.  Push i owns rows F_{i-1} .. F_i - 1, where
F_i is the number of samples pushed up to and including push i, over hop.  After a reset the reference starts again
from the samples pushed after it.  ``test_push_rows_are_the_oracle_run_push_by_push`` checks that statement on the
oracle alone, without a GPU.

The expected families are the dispatcher's choices on a 148-SM B200.  "Many" channels is twice the SM count (296 there):
at or above every fused family's chain threshold.  "Few" is 4.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable

import numpy as np
import pytest

from oracle import analyser_oracle as O
from _tol import assert_bytes_close, assert_db_close, assert_mag_close

gpu = pytest.mark.gpu
FEW = 4
MANY = -1          # stands for 2 x the SM count


# ----------------------------------------------------------------------------- the reference
def cut_rows(rows, push_lens, hop):
    """Rows [clips, frames, ...] of one oracle call on the concatenated pushes -> the rows of each push."""
    bounds = np.cumsum([0] + [int(n) for n in push_lens]) // hop
    return [rows[:, bounds[i]:bounds[i + 1]] for i in range(len(push_lens))]


def reference_rows(pushes, cfg: O.Config):
    """What the bank must return for each push: one oracle call on the samples pushed since the last reset, cut at the
    push boundaries.  ``pushes``: [channels, samples] chunks in order, ``None`` for a reset."""
    out, run = [], []

    def flush():
        if run:
            with np.errstate(invalid="ignore", over="ignore"):
                rows = O.spectrogram(np.concatenate(run, axis=1), cfg)
            out.extend(cut_rows(rows, [c.shape[1] for c in run], cfg.hop))
            run.clear()

    for c in pushes:
        if c is None:
            flush()
        else:
            run.append(c)
    flush()
    return out


def oracle_push_by_push(pushes, cfg: O.Config):
    """The oracle run the way the bank runs: every push frames ``[history | chunk]`` with the last n_fft samples of the
    previous row as history (zeros at the start and after a reset), and smooths from the state the previous push
    left."""
    n, hop = cfg.n_fft, cfg.hop
    w = O.make_window(cfg.window, n, cfg.custom_window)
    hist = state = None
    out = []
    for c in pushes:
        if c is None:
            hist = state = None
            continue
        x = np.asarray(c, np.float64)
        if hist is None:
            hist = np.zeros((x.shape[0], n))
            state = np.zeros((x.shape[0], n // 2))
        row = np.concatenate([hist, x], axis=1)
        frames = x.shape[1] // hop
        idx = (np.arange(frames)[:, None] + 1) * hop + np.arange(n)[None, :]     # frame t ends at chunk sample (t+1)*hop
        mags = []
        for ch in range(x.shape[0]):
            with np.errstate(invalid="ignore", over="ignore"):
                m = O.magnitudes(row[ch][idx], w)
            if cfg.smoothing > 0.0:
                m, state[ch] = O.smooth(m, cfg.smoothing, state[ch])
            else:
                m = np.where(np.isfinite(m), m, 0.0)
            mags.append(m)
        hist = row[:, -n:]
        out.append(O.finish(np.stack(mags), cfg))
    return out


def make_signal(channels, n, seed, bursts=()):
    """Noise plus a chirp, a different gain per channel; ``bursts``: sample ranges made 20x louder."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((channels, n), dtype=np.float32)
    x *= np.float32(0.05)
    x += O.chirp(n, 44100.0, 100.0, 15000.0, 0.3)[None, :]
    x *= rng.uniform(0.3, 1.0, (channels, 1)).astype(np.float32)
    for a, b in bursts:
        x[:, a:b] *= np.float32(20.0)
    return x


def asymmetric_window(n):
    return (np.kaiser(n, 8) * np.linspace(0.3, 1.0, n)).astype(np.float32)


def custom_colormap(seed=11):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 1 << 24, 256, dtype=np.uint32) | np.uint32(0xFF000000)


def lut_bytes(lut_u32):
    """A 256 x uint32 RGBA8 table (R | G<<8 | B<<16 | A<<24) as the [256, 4] bytes the bank writes."""
    return np.stack([(lut_u32 >> (8 * i)) & 0xFF for i in range(4)], axis=-1).astype(np.uint8)


# ----------------------------------------------------------------------------- the reference on the CPU
@pytest.mark.parametrize("n_fft,hop,tau", [(64, 16, 0.0), (64, 16, 0.8), (48, 60, 0.5), (30, 6, 0.8), (100, 100, 0.3)])
def test_push_rows_are_the_oracle_run_push_by_push(n_fft, hop, tau):
    """Cutting one oracle call at the push boundaries is the oracle run push by push (carried history, carried state):
    ragged pushes, hop > n_fft, a non-finite sample in each of two channels, a reset."""
    frames = [3, 1, 7, 2, None, 2, 5, 1, 4, 1]
    x = make_signal(3, sum(f for f in frames if f) * hop, seed=n_fft + hop, bursts=[(4 * hop, 6 * hop)])
    x[1, 6 * hop - 1] = np.nan           # sample k*hop - 1 is in frame k - 1 even when hop > n_fft
    x[2, 17 * hop - 1] = -np.inf
    pushes, i = [], 0
    for f in frames:
        if f is None:
            pushes.append(None)
            continue
        pushes.append(x[:, i:i + f * hop])
        i += f * hop
    cfg = O.Config(n_fft=n_fft, hop=hop, align=O.ALIGN_ANALYSER, smoothing=tau, output=O.OUT_F32_MAG)
    cut = reference_rows(pushes, cfg)
    step = oracle_push_by_push(pushes, cfg)
    assert len(cut) == len(step) == len([f for f in frames if f])
    for f, a, b in zip([f for f in frames if f], cut, step):
        assert a.shape == b.shape == (3, f, n_fft // 2)
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=0.0)
    rows = np.concatenate(cut, axis=1)
    assert (rows == 0).all(axis=-1).any(axis=-1)[1:].all()      # the bad samples zero whole frames ...
    assert not (rows[0] == 0).all(axis=-1).any()                 # ... of their own channel only
    # the rows after the reset do not depend on what came before it
    later = reference_rows([p for p in pushes[frames.index(None) + 1:]], cfg)
    assert all(np.array_equal(a, b) for a, b in zip(later, cut[frames.index(None):]))


# ----------------------------------------------------------------------------- the GPU runs
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def one(name):
    """A frame kernel (tau 0) or a fused smoothing kernel: one launch per push."""
    return lambda out, frames: (name, 1)


def two(name):
    """tau > 0 on the two-kernel path: a kernel flags the frames that hold a non-finite sample, the frame kernel
    (``name``) writes magnitudes, a recurrence kernel emits."""
    return lambda out, frames: (name, 3)


def by_frames(many_frames, one_frame, min_frames=4):
    """The pair kernels take a push from 4 frames per channel on; a shorter push stays on the per-frame kernel."""
    return lambda out, frames: (many_frames if frames >= min_frames else one_frame, 1)


@dataclass
class Case:
    n_fft: int
    hop: int
    channels: int                 # FEW, MANY or a count
    frames: list                  # frames per push; None: reset
    tau: float
    family: Callable              # (output kind, frames of the push) -> (last_kernel, launches without the LUT kernel)
    outs: tuple = ("u8", "db", "mag")     # "rgba" (a bank whose output is colour) must come after "u8"
    custom: bool = False          # asymmetric window, dB range (-90, -20), a colour map of the caller's
    bursts: tuple = ()            # pushes (counted without the resets) made 20x louder
    batch: bool = False           # also compare with engine.spectrogram(align="analyser") on the same samples


def pick(channels, seed):
    """All channels when few; else the first, middle and last and a seeded random 16."""
    if channels <= 8:
        return np.arange(channels)
    rng = np.random.default_rng(seed)
    return np.unique(np.r_[0, channels // 2, channels - 1, rng.choice(channels, 16, replace=False)])


def run_case(engine, sms, c: Case):
    channels = 2 * sms if c.channels == MANY else c.channels
    starts = np.cumsum([0] + [f * c.hop for f in c.frames if f is not None])
    x = make_signal(channels, int(starts[-1]), 7 * c.n_fft + c.hop, [(starts[k], starts[k + 1]) for k in c.bursts])
    run_signal(engine, c, x, channels)


def run_signal(engine, c: Case, x, channels, keep_all=False, also=()):
    """Pushes ``x`` through a bank once per output kind of the case and checks every push on the channels ``pick``
    chooses and those in ``also``.  Returns the rows of each push per output kind: the compared channels, or all of
    them with ``keep_all``."""
    import spectrogram_b200 as sg

    n, hop = c.n_fft, c.hop
    sel = np.union1d(pick(channels, n + hop), np.asarray(also, int))
    win = asymmetric_window(n) if c.custom else None
    lut = custom_colormap() if c.custom else None
    min_db, max_db = (-90.0, -20.0) if c.custom else (-100.0, -30.0)
    cfg = O.Config(n_fft=n, hop=hop, window=O.WINDOW_CUSTOM if c.custom else O.WINDOW_BLACKMAN,
                   custom_window=None if win is None else win.astype(np.float64), align=O.ALIGN_ANALYSER,
                   smoothing=c.tau, output=O.OUT_F32_MAG, min_db=min_db, max_db=max_db)
    u8cfg = O.Config(**{**cfg.__dict__, "output": O.OUT_U8})
    chunks, i = [], 0
    for f in c.frames:
        if f is None:
            chunks.append(None)
        else:
            chunks.append(x[:, i:i + f * hop])
            i += f * hop
    ref = reference_rows([None if ch is None else ch[sel] for ch in chunks], cfg)
    lut_rgba = O.colormap_lut() if lut is None else lut_bytes(lut)
    max_chunk = max(ch.shape[1] for ch in chunks if ch is not None)
    results = {}
    for out in c.outs:
        opts = sg.Options(fftSize=n, hop=hop, window="blackman" if win is None else win, minDecibels=min_db,
                          maxDecibels=max_db, smoothingTimeConstant=c.tau, output=out, colormap=lut)
        bank = sg.StreamBank(channels, opts, max_chunk=max_chunk, engine=engine)
        rows, k = [], 0
        try:
            for p, ch in enumerate(chunks):
                if ch is None:
                    bank.reset()
                    continue
                frames = ch.shape[1] // hop
                before = engine.launch_count
                res = bank.push(ch, want_rgba=out == "u8")
                name, launches = c.family(out, frames)
                where = f"{out} push {p} ({frames} frames)"
                assert engine.last_kernel == name, f"{where}: ran {engine.last_kernel}, expected {name}"
                assert engine.launch_count - before == launches + (out == "u8"), where
                got = res[0] if out == "u8" else res
                assert got.shape == (channels, frames, n // 2) + ((4,) if out == "rgba" else ()), where
                if out == "rgba":
                    # the colour rows of an RGBA bank: the table applied to the bytes of the same push in a byte bank
                    u8 = results["u8"][k]
                    assert np.array_equal(got if keep_all else got[sel], lut_rgba[u8]), f"{where}: not the LUT of the bytes"
                elif out == "mag":
                    assert_mag_close(got[sel], ref[k])
                elif out == "db":
                    assert_db_close(got[sel], ref[k])
                else:
                    # one level at most on every push; the 0.2 % rate is a rate, taken over the whole stream below
                    # (a one-frame push of few channels at a small n_fft holds a few hundred bytes)
                    assert_bytes_close(got[sel], O.finish(ref[k], u8cfg), max_mismatch_frac=1.0)
                    assert np.array_equal(res[1], lut_rgba[got]), f"{where}: RGBA is not the LUT of the bytes"
                rows.append(got if keep_all else got[sel])
                k += 1
        finally:
            bank.close()
        if out == "u8":
            assert_bytes_close(np.concatenate([r[sel] if keep_all else r for r in rows], axis=1),
                               np.concatenate([O.finish(r, u8cfg) for r in ref], axis=1))
        results[out] = rows
    if c.batch and "mag" in c.outs and None not in c.frames:
        # The same samples as one batch call, forced onto the same fused kernel (as a batch of a few clips it would
        # take the two-kernel path, whose frame kernel may be another FFT): there the state crosses segments inside one
        # launch, in the bank it crosses launches.  The rows agree to rounding of the carried state.
        engine.set_kernel_variant(7)
        try:
            b = engine.spectrogram(x[sel], sg.Options(fftSize=n, hop=hop, window="blackman" if win is None else win,
                                                      smoothingTimeConstant=c.tau, output="mag", align="analyser"))
        finally:
            engine.set_kernel_variant(0)
        assert engine.last_kernel == c.family("mag", 1)[0]
        a = np.concatenate(results["mag"], axis=1)
        a = a[sel] if keep_all else a
        assert a.shape == b.shape
        assert np.all(np.abs(a - b) <= 2e-5 * np.abs(b) + 1e-7 * b.max(axis=-1, keepdims=True))
    return results


def case_id(c: Case):
    who = {FEW: "few", MANY: "many"}.get(c.channels, f"{c.channels}ch")
    return f"{c.n_fft}-{c.hop}-{who}-tau{c.tau}" + ("-custom" if c.custom else "")


def params(cases):
    return [pytest.param(c, id=case_id(c)) for c in cases]


WITH_RGBA = ("u8", "rgba", "db", "mag")
ONE_HOP = [1] * 12
SMALL = [1, 3, 2, 1, 3, 1, 2, 1, 1, 2]
RAGGED = [4, 7, 16, 5, 1, 9]
# one-frame pushes, then ragged multi-frame ones: 151 frames per channel
LONG = [1] * 40 + [4, 7, 16, 5, 1, 9, 13, 33, 2, 21]

# A: tau 0, one hop per push (the per-frame kernels; smem for the shapes without a dedicated kernel)
CASES_A = [
    # u8 rows at hop 512 take the register-pipelined pair kernel; dB and magnitude rows the TMA-staged one
    Case(2048, 512, MANY, [1] * 40, 0.0, lambda out, f: ("warp32x32x2p" if out == "u8" else "warp32x32x2", 1)),
    Case(2048, 441, MANY, ONE_HOP, 0.0, one("warp32x32x2"), custom=True, outs=WITH_RGBA),
    Case(2048, 1536, MANY, ONE_HOP, 0.0, one("warp32x32")),
    Case(4096, 1024, MANY, ONE_HOP, 0.0, one("eo4096"), custom=True, outs=WITH_RGBA),
    Case(4096, 441, MANY, ONE_HOP, 0.0, one("wreg")),
    Case(8192, 2048, MANY, ONE_HOP, 0.0, one("wreg")),
    Case(512, 128, MANY, ONE_HOP, 0.0, one("w16")),
    Case(256, 64, MANY, ONE_HOP, 0.0, one("w16")),
    Case(400, 160, MANY, ONE_HOP, 0.0, one("r400"), custom=True, outs=WITH_RGBA),
    Case(32768, 8192, FEW, SMALL, 0.0, one("smem")),
    Case(32, 8, FEW, SMALL * 3, 0.0, one("smem")),
    Case(600, 700, FEW, SMALL, 0.0, one("smem")),          # hop > n_fft
    Case(1200, 300, FEW, SMALL, 0.0, one("smem"), custom=True, outs=WITH_RGBA),
    Case(6, 2, FEW, SMALL * 3, 0.0, one("smem")),
]

# B: tau 0, ragged pushes: the pair kernels from 4 frames per channel, at the stream's stride
CASES_B = [
    Case(1024, 128, MANY, RAGGED, 0.0, by_frames("p16", "wreg")),
    Case(1024, 160, MANY, RAGGED, 0.0, by_frames("p16", "wreg")),
    Case(512, 128, MANY, RAGGED, 0.0, by_frames("p8", "w16")),
    Case(512, 160, MANY, RAGGED, 0.0, by_frames("p8", "w16"), custom=True, outs=WITH_RGBA),
    # n_fft 256: the pair kernel serves bytes only; float rows stay on the 16 x 8 kernel
    Case(256, 32, MANY, RAGGED, 0.0, lambda out, f: ("p4" if out == "u8" and f >= 4 else "w16", 1)),
]

# C: tau > 0 at twice the SM count in channels: every push is one chain per channel on a fused kernel, starting from
# the state the previous push left.  Loud pushes put a large state in front of quieter ones.
CASES_C = [
    Case(2048, 512, MANY, LONG, 0.8, one("warp32x32x2s"), bursts=(5, 42), batch=True),
    Case(2048, 441, MANY, LONG, 0.8, one("warp32x32x2s"), bursts=(5, 42), batch=True),
    Case(1024, 128, MANY, LONG, 0.8, one("p16s"), bursts=(5, 42), batch=True, custom=True, outs=WITH_RGBA),
    Case(1024, 200, MANY, LONG, 0.3, one("p16s"), bursts=(5, 42), batch=True),
    Case(512, 128, MANY, LONG, 0.8, one("p8s"), bursts=(5, 42), batch=True),
    Case(256, 64, MANY, LONG, 0.8, one("p4s"), bursts=(5, 42), batch=True),
    Case(4096, 1024, MANY, LONG, 0.8, one("eo4096s"), bursts=(5, 42), batch=True),
    Case(4096, 441, MANY, LONG, 0.8, one("wregs"), bursts=(5, 42), batch=True, custom=True, outs=WITH_RGBA),
    Case(8192, 2048, MANY, LONG, 0.8, one("wregs"), bursts=(5, 42), batch=True),
]

# D, F: tau > 0 with few channels: the frame kernel writes magnitudes, the recurrence kernel continues the carried state
CASES_D = [
    Case(1024, 256, FEW, [1] * 30, 0.8, two("wreg"), bursts=(4, 17)),
    Case(512, 128, FEW, [1] * 30, 0.8, two("w16"), bursts=(4, 17)),
    # 300 frames of 8 channels: the cooperative chunked scan (smooth_scan_kernel) from the state of a loud short push.
    # launch_smooth_t takes the scan when (clip, bin) pairs < 2048 x SMs and frames >= 256: 8 x 512 = 4096 pairs, 300
    # frames (chunks of 32 frames).  No fused kernel: 8 clips are below every chain threshold, and warm-up segments
    # would be 300 / (148 / 8) -> 20 frames, shorter than the 464-frame warm-up at tau 0.8.
    Case(1024, 256, 8, [2, 300, 1, 1], 0.8, lambda out, f: ("p16" if f >= 4 else "wreg", 3), bursts=(0,)),
    Case(400, 160, FEW, SMALL, 0.8, two("r400"), bursts=(2,), custom=True, outs=WITH_RGBA),
    Case(32768, 8192, FEW, SMALL, 0.8, two("smem"), bursts=(2,)),
]

# E: tau > 0, few channels, one large push: independent segments with a warm-up, segment 0 from the carried state.
# The short pushes around it take the two-kernel path; the ones after it start from the state the large push handed back.
CASES_E = [
    Case(2048, 512, FEW, [10, 6000, 1, 1, 1], 0.5,
         lambda out, f: ("warp32x32x2s", 1) if f > 1000 else ("warp32x32x2", 3), outs=("mag", "u8"), bursts=(0, 2)),
    Case(1024, 256, FEW, [10, 6000, 1, 1, 1], 0.5,
         lambda out, f: ("p16s", 1) if f > 1000 else ("p16" if f >= 4 else "wreg", 3), outs=("mag", "u8"),
         bursts=(0, 2)),
]

# reset in the middle of a tau > 0 stream on fused families: the rows after it are the oracle of the later samples alone
CASES_RESET = [
    Case(2048, 512, MANY, [1] * 6 + [3, None, 1, 1, 2, 1, 4], 0.8, one("warp32x32x2s"), outs=("mag", "u8"), bursts=(6,)),
    Case(512, 128, MANY, [1] * 6 + [3, None, 1, 1, 2, 1, 4], 0.8, one("p8s"), outs=("mag", "u8"), bursts=(6,)),
    Case(8192, 2048, MANY, [1] * 6 + [3, None, 1, 1, 2, 1, 4], 0.8, one("wregs"), outs=("mag",), bursts=(6,)),
]


@gpu
@pytest.mark.parametrize("case", params(CASES_A))
def test_one_hop_pushes_per_frame_kernels(engine, sms, case):
    run_case(engine, sms, case)


@gpu
@pytest.mark.parametrize("case", params(CASES_B))
def test_ragged_pushes_pair_kernels(engine, sms, case):
    run_case(engine, sms, case)


@gpu
@pytest.mark.parametrize("case", params(CASES_C))
def test_fused_smoothing_kernels_carry_the_state_across_pushes(engine, sms, case):
    run_case(engine, sms, case)


@gpu
@pytest.mark.parametrize("case", params(CASES_D))
def test_two_kernel_smoothing_carries_the_state_across_pushes(engine, sms, case):
    run_case(engine, sms, case)


@gpu
@pytest.mark.parametrize("case", params(CASES_E))
def test_large_push_warm_up_segments_start_from_the_carried_state(engine, sms, case):
    run_case(engine, sms, case)


@gpu
@pytest.mark.parametrize("case", params(CASES_RESET))
def test_reset_mid_stream_restarts_from_zero(engine, sms, case):
    run_case(engine, sms, case)


# ----------------------------------------------------------------------------- non-finite samples
NONFINITE_FRAMES = [1, 2, 1, 4, 1, 1, 3, 1, 1, 1, 5, 1, 1]
CASES_NONFINITE = [
    Case(1024, 256, FEW, NONFINITE_FRAMES, 0.0, by_frames("p16", "wreg"), outs=("mag", "db")),
    Case(2048, 512, MANY, NONFINITE_FRAMES, 0.8, one("warp32x32x2s"), outs=("mag", "db")),
    Case(512, 128, MANY, NONFINITE_FRAMES, 0.8, one("p8s"), outs=("mag", "db")),
    # the two-kernel path: the recurrence restarts on the frames poison_flags_kernel marks ...
    Case(1024, 256, FEW, NONFINITE_FRAMES, 0.8, lambda out, f: ("p16" if f >= 4 else "wreg", 3), outs=("mag", "db")),
    # ... also in the chunked scan (the NaN lands in the middle chunk of a 300-frame push)
    Case(1024, 256, 8, [1, 2, 1, 300, 1, 1, 3, 1, 1, 1], 0.8, lambda out, f: ("p16" if f >= 4 else "wreg", 3),
         outs=("mag", "db")),
]
@gpu
@pytest.mark.parametrize("inf", [np.inf, -np.inf], ids=["+inf", "-inf"])
@pytest.mark.parametrize("case", params(CASES_NONFINITE))
def test_non_finite_samples_zero_exactly_their_frames(engine, sms, case, inf):
    """One NaN (channel 1, push 3) and one infinity (channel 2, push 6): exactly the frames that hold the bad sample are
    zero (-inf dB), the state restarts from zero as the oracle's does, and every other channel is bit for bit what it is
    without the bad samples."""
    n, hop = case.n_fft, case.hop
    channels = 2 * sms if case.channels == MANY else case.channels
    starts = np.cumsum([0] + [f * hop for f in case.frames])
    clean = make_signal(channels, int(starts[-1]), n + hop)
    x = clean.copy()
    bad = {1: starts[3] + (case.frames[3] // 2) * hop + hop // 2 + 1, 2: starts[6] + 2 * hop + 3}     # channel -> sample
    x[1, bad[1]] = np.nan
    x[2, bad[2]] = inf
    ref = run_signal(engine, case, clean, channels, keep_all=True)
    got = run_signal(engine, case, x, channels, keep_all=True, also=(1, 2))
    total = int(starts[-1]) // hop
    ends = (np.arange(total) + 1) * hop                                  # frame t holds samples [end - n, end)
    for out in case.outs:
        a, b = np.concatenate(got[out], axis=1), np.concatenate(ref[out], axis=1)
        others = np.setdiff1d(np.arange(channels), [1, 2])
        assert np.array_equal(a[others], b[others]), f"{out}: a bad sample changed another channel"
        for ch, pos in bad.items():
            hit = (ends - n <= pos) & (pos < ends)
            assert hit.sum() == min(-(-n // hop), total)
            zero = np.isneginf(a[ch]).all(-1) if out == "db" else (a[ch] == 0).all(-1)
            assert np.array_equal(zero, hit), f"{out} channel {ch}: zero rows {np.flatnonzero(zero)}, expected {np.flatnonzero(hit)}"
