"""Sample-rate conversion in front of the path: decodeAudioData resamples a file to its context's rate, so the
AnalyserNode's bin k is k*contextRate/fftSize Hz whatever the file's rate.  The resampler is rational polyphase
resampling equal to scipy.signal.resample_poly with its default filter; tests/resample_oracle.py restates it as a
direct float64 sum, pinned here against scipy, and the GPU results are checked against that oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import analyser_oracle as ao
from oracle import pcm_oracle as po
from test_pcm_ingest import FMT_NAMES, random_pcm, wav_file
import resample_oracle as ro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATIOS = [(44100, 48000), (48000, 44100), (8000, 44100), (96000, 16000), (11025, 192000), (192000, 11025)]


def taps_per_phase(in_rate, out_rate):
    up, down = ro.resample_ratio(in_rate, out_rate)
    return -(-(20 * max(up, down) + 1) // up)


# ------------------------------------------------------------------ CPU ---------------------------
@pytest.mark.parametrize("in_rate,out_rate", RATIOS)
def test_oracle_equals_scipy_resample_poly(in_rate, out_rate):
    from scipy.signal import resample_poly

    up, down = ro.resample_ratio(in_rate, out_rate)
    rng = np.random.default_rng(in_rate + out_rate)
    for n in (0, 1, taps_per_phase(in_rate, out_rate) - 1, 4000):
        x = rng.standard_normal(n)
        y = ro.resample(x, in_rate, out_rate)
        assert y.size == -(-n * up // down)
        if n:
            np.testing.assert_allclose(y, resample_poly(x, up, down), rtol=0, atol=1e-12)


def test_oracle_filter_is_scipys_firwin_in_float32():
    from scipy.signal import firwin

    for in_rate, out_rate in RATIOS:
        up, down = ro.resample_ratio(in_rate, out_rate)
        h = ro.resample_filter(up, down)
        want = firwin(h.size, 1.0 / max(up, down), window=("kaiser", 5.0)) * up
        np.testing.assert_allclose(h, want, rtol=0, atol=1e-14)
        assert np.array_equal(h.astype(np.float32), want.astype(np.float32))


def test_num_frames_matches_resample_poly_lengths():
    import spectrogram_b200 as sg
    from scipy.signal import resample_poly

    rates = [8000, 11025, 16000, 22050, 44100, 47999, 48000, 96000, 192000, 768000]
    for a in rates:
        for b in rates:
            up, down = ro.resample_ratio(a, b)
            if max(up, down) > 16384:
                continue
            for n in (0, 1, 2, 147, 160, 1001):
                want = len(resample_poly(np.zeros(n), up, down)) if n else 0
                assert sg.resample_num_frames(n, a, b) == want, (a, b, n)
    assert sg.resample_num_frames(12_000_000, 44100, 48000) == 13_061_225
    assert sg.resample_num_frames(10, 11025, 768000) == 697                 # 10240/147


def test_num_frames_rejects_bad_rates_and_too_fine_ratios():
    import spectrogram_b200 as sg
    from spectrogram_b200 import _lib as L

    lib = L.load()
    for a, b in ((2999, 48000), (44100, 768001), (0, 48000), (-44100, 48000), (44100, 48001), (44099, 48000)):
        assert lib.sg_resample_num_frames(100, a, b) == L.SG_ERR_INDEX_SIZE
        msg = L.last_error()
        assert str(a) in msg and str(b) in msg, msg
        with pytest.raises(sg.IndexSizeError):
            sg.resample_num_frames(100, a, b)
    assert lib.sg_resample_num_frames(-1, 44100, 48000) == L.SG_ERR_INVALID_ARG


def test_entry_points_reject_bad_arguments_before_touching_a_device():
    from spectrogram_b200 import _lib as L

    lib = L.load()
    ok = L.PcmInfo(L.PCM_S16, 2, 44100, 441, 0)
    buf = (C.c_uint8 * 4096)()
    cfg = L.StftConfig()
    lib.sg_stft_config_default(C.byref(cfg))
    n_out = lib.sg_resample_num_frames(441, 44100, 48000)
    assert n_out == 480

    def calls(info, layout, rate, stride, pcm, out):
        return [lib.sg_pcm_ingest_resampled(None, pcm, 1, C.byref(info), layout, rate, out),
                lib.sg_pcm_ingest_resampled_device(None, pcm, 1, C.byref(info), layout, rate, out, stride, None),
                lib.sg_stft_pcm_resampled(None, pcm, 1, C.byref(info), layout, rate, C.byref(cfg), out)]

    assert calls(ok, 7, 48000, n_out, buf, buf) == [L.SG_ERR_INVALID_ARG] * 3                  # bad layout
    assert "layout" in L.last_error()
    assert calls(ok, L.PCM_PLANAR, 48000, n_out, None, None) == [L.SG_ERR_INVALID_ARG] * 3     # null buffers
    assert "null" in L.last_error()
    assert calls(ok, L.PCM_PLANAR, 48001, n_out, buf, buf) == [L.SG_ERR_INDEX_SIZE] * 3        # 48001/44100
    assert "48001" in L.last_error()
    no_rate = L.PcmInfo(L.PCM_S16, 2, 0, 441, 0)                                               # source rate missing
    assert calls(no_rate, L.PCM_PLANAR, 48000, n_out, buf, buf) == [L.SG_ERR_INDEX_SIZE] * 3
    rc = lib.sg_pcm_ingest_resampled_device(None, buf, 1, C.byref(ok), L.PCM_PLANAR, 48000, buf, n_out - 1, None)
    assert rc == L.SG_ERR_INVALID_ARG and "out_stride" in L.last_error()                       # short out_stride
    assert calls(ok, L.PCM_PLANAR, 48000, n_out, buf, buf) == [L.SG_ERR_INVALID_ARG] * 3       # engine is null
    assert "engine" in L.last_error()


def test_js_facade_and_shim_expose_resampling():
    text = open(os.path.join(ROOT, "spectrogram_b200", "js", "index.js")).read()
    for name in ("native.pcmDecodeResampled", "native.stftPcmResampled", "native.resampleNumFrames", "o.sampleRate"):
        assert name in text, name
    shim = open(os.path.join(ROOT, "spectrogram_b200", "js", "napi_shim.c")).read()
    for name in ('"pcmDecodeResampled"', '"stftPcmResampled"', '"resampleNumFrames"'):
        assert name in shim, name


# ------------------------------------------------------------------ GPU -----------------------------
def check_against_oracle(got, x32, in_rate, out_rate):
    """per-sample float32 dot-product bound: (J+2) u sum|h x| + u |y|, u = 2^-24"""
    J = taps_per_phase(in_rate, out_rate)
    x = x32.astype(np.float64)
    want = ro.resample(x, in_rate, out_rate)
    scale = ro.resample(x, in_rate, out_rate, absolute=True)
    bound = (J + 2) * 2.0 ** -24 * scale + 2.0 ** -24 * np.abs(want)
    assert got.shape == want.shape
    err = np.abs(got.astype(np.float64) - want)
    assert np.all(err <= bound), (in_rate, out_rate, float((err - bound).max()), int(np.argmax(err - bound)))


@pytest.mark.gpu
@pytest.mark.parametrize("in_rate,out_rate", RATIOS)
def test_impulse_response_is_the_float32_filter_at_the_predicted_indices(engine, in_rate, out_rate):
    """a unit impulse at n0 gives y[k] = float32(h[k down + half - n0 up]): pins the filter design and the phases"""
    from scipy.signal import firwin

    up, down = ro.resample_ratio(in_rate, out_rate)
    half = 10 * max(up, down)
    h32 = (firwin(2 * half + 1, 1.0 / max(up, down), window=("kaiser", 5.0)) * up).astype(np.float32)
    frames = 3 * taps_per_phase(in_rate, out_rate) + 2 * down
    for n0 in (0, frames // 2 + 1, frames - 1):
        x = np.zeros(frames, dtype="<f4")
        x[n0] = 1.0
        got = engine.decode_pcm(x.tobytes(), "f32", 1, in_rate, context_rate=out_rate).getChannelData(0)
        k = np.arange(got.size)
        idx = k * down + half - n0 * up
        want = np.where((idx >= 0) & (idx <= 2 * half), h32[np.clip(idx, 0, 2 * half)], np.float32(0))
        np.testing.assert_array_equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("in_rate,out_rate", RATIOS)
@pytest.mark.parametrize("fmt", [po.U8, po.S16, po.S24, po.S32, po.F32])
def test_resampled_planes_follow_the_oracle(engine, in_rate, out_rate, fmt):
    """every format, 1/2/6/32 channels, mono mix and planar, several clips, an unaligned source"""
    n_clips, frames = 2, 2500
    for i, channels in enumerate((1, 2, 6, 32)):
        raw = random_pcm(fmt, channels, n_clips * frames, seed=fmt * 1000 + channels + in_rate)
        src = np.frombuffer(b"\x55" * 5 + raw, dtype=np.uint8)[5:]              # odd source address
        for mix in ((True, False) if (i + fmt) % 2 == 0 or channels == 1 else (False, True)):
            if channels == 32 and mix:
                continue
            x = engine.decode_pcm(src, FMT_NAMES[fmt], channels, in_rate, n_clips=n_clips, mix=mix).planes
            buf = engine.decode_pcm(src, FMT_NAMES[fmt], channels, in_rate, n_clips=n_clips, mix=mix, context_rate=out_rate)
            assert buf.sampleRate == out_rate and buf.length == ro.resample(np.zeros(frames), in_rate, out_rate).size
            for c in range(n_clips):
                for p in range(x.shape[1]) if channels < 32 else (0, 13, 31):
                    check_against_oracle(buf.planes[c, p], x[c, p], in_rate, out_rate)


@pytest.mark.gpu
def test_equal_rates_are_the_plain_ingest_bit_for_bit(engine):
    import spectrogram_b200 as sg

    raw = random_pcm(po.S24, 2, 3 * 7000, seed=4)
    for mix in (True, False):
        a = engine.decode_pcm(raw, "s24", 2, 44100, n_clips=3, mix=mix)
        b = engine.decode_pcm(raw, "s24", 2, 44100, n_clips=3, mix=mix, context_rate=44100)
        assert b.sampleRate == 44100
        assert np.array_equal(a.planes, b.planes)
        opts = sg.Options(fftSize=1024, hop=256)
        s1 = engine.spectrogram_pcm(raw, "s24", 2, n_clips=3, mix=mix, opts=opts)
        s2 = engine.spectrogram_pcm(raw, "s24", 2, n_clips=3, mix=mix, opts=opts, sample_rate=44100, context_rate=44100)
        assert np.array_equal(s1, s2)


@pytest.mark.gpu
@pytest.mark.parametrize("in_rate,out_rate", [(44100, 48000), (96000, 16000), (192000, 11025)])
def test_host_and_device_entry_points_agree_bit_for_bit(engine, in_rate, out_rate):
    import torch
    from spectrogram_b200 import _lib as L

    lib = L.load()
    n_clips, frames, channels = 3, 9001, 2
    raw = random_pcm(po.S16, channels, n_clips * frames, seed=31)
    host = engine.decode_pcm(raw, "s16", channels, in_rate, n_clips=n_clips, context_rate=out_rate).planes
    n_out = host.shape[-1]
    src = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    stride = n_out + 5
    dst = torch.full((n_clips * channels, stride), -7.0, dtype=torch.float32, device="cuda")
    info = L.PcmInfo(L.PCM_S16, channels, in_rate, frames, 0)
    launches = engine.launch_count
    L.check(lib.sg_pcm_ingest_resampled_device(engine.handle, C.c_void_p(src.data_ptr()), n_clips, C.byref(info), L.PCM_PLANAR,
                                               out_rate, C.c_void_p(dst.data_ptr()), stride, None))
    engine.synchronize()
    assert engine.launch_count == launches + 1
    got = dst.cpu().numpy()
    assert np.array_equal(got[:, :n_out].reshape(host.shape), host)
    assert np.all(got[:, n_out:] == -7.0)                                    # nothing written past the planes


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,channels,mix,in_rate,out_rate", [
    (po.S16, 2, True, 44100, 48000), (po.S24, 6, False, 48000, 44100), (po.U8, 1, True, 96000, 16000),
    (po.F32, 2, True, 192000, 11025), (po.S32, 2, False, 8000, 44100)])
def test_fused_resampled_pipeline_equals_resampled_ingest_then_batch(engine, fmt, channels, mix, in_rate, out_rate):
    import spectrogram_b200 as sg

    n_clips, frames = 3, 30000
    raw = random_pcm(fmt, channels, n_clips * frames, seed=19)
    opts = sg.Options(fftSize=1024, hop=256)
    got = engine.spectrogram_pcm(raw, FMT_NAMES[fmt], channels, n_clips=n_clips, mix=mix, opts=opts,
                                 sample_rate=in_rate, context_rate=out_rate)
    buf = engine.decode_pcm(raw, FMT_NAMES[fmt], channels, in_rate, n_clips=n_clips, mix=mix, context_rate=out_rate)
    two = engine.spectrogram(buf.planes.reshape(-1, buf.length), opts)
    np.testing.assert_array_equal(got.reshape(two.shape), two)
    x = engine.decode_pcm(raw, FMT_NAMES[fmt], channels, in_rate, n_clips=n_clips, mix=mix).planes[0, 0]
    want = ao.spectrogram(ro.resample(x.astype(np.float64), in_rate, out_rate), ao.Config(n_fft=1024, hop=256))[0]
    assert np.abs(got[0, 0].astype(int) - want.astype(int)).max() <= 1


@pytest.mark.gpu
def test_fused_resampled_pipeline_on_one_long_stereo_clip(engine):
    """a clip larger than the pipeline's chunk: frame-range chunks, each uploading its source range plus the halo"""
    import spectrogram_b200 as sg

    frames = 12_000_000
    rng = np.random.default_rng(2)
    raw = (rng.standard_normal(2 * frames) * 3000).astype("<i2")
    opts = sg.Options(fftSize=512, hop=160, output="db")
    got = engine.spectrogram_pcm(raw, "s16", 2, mix=False, opts=opts, sample_rate=44100, context_rate=48000)
    planes = engine.decode_pcm(raw, "s16", 2, 44100, context_rate=48000).planes
    assert planes.shape == (2, 13_061_225)
    two = engine.spectrogram(planes, opts)
    assert got.shape == (1, 2) + two.shape[1:]
    np.testing.assert_array_equal(got[0], two)
    # and the long host ingest (output-range chunks) matches the oracle on a window deep inside the clip
    lo = 147 * 74830                                                       # output lo*160/147 has phase 0
    xw = engine.decode_pcm(raw[2 * lo:2 * (lo + 4410)], "s16", 2, 44100).planes[1].astype(np.float64)
    yw = ro.resample(xw, 44100, 48000)
    k0 = lo * 48000 // 44100
    inner = slice(200, yw.size - 200)                                      # away from the window's zero padding
    np.testing.assert_allclose(planes[1, k0:k0 + yw.size][inner], yw[inner], rtol=0, atol=2e-5)


@pytest.mark.gpu
def test_fused_resampled_pipeline_with_smoothing_keeps_one_state_per_plane(engine):
    import spectrogram_b200 as sg

    n_clips, frames = 2, 20000
    raw = random_pcm(po.S16, 2, n_clips * frames, seed=29)
    opts = sg.Options(fftSize=512, hop=128, smoothingTimeConstant=0.8, output="db")
    got = engine.spectrogram_pcm(raw, "s16", 2, n_clips=n_clips, mix=False, opts=opts, sample_rate=44100, context_rate=48000)
    buf = engine.decode_pcm(raw, "s16", 2, 44100, n_clips=n_clips, context_rate=48000)
    two = engine.spectrogram(buf.planes.reshape(-1, buf.length), opts)
    np.testing.assert_array_equal(got.reshape(two.shape), two)


@pytest.mark.gpu
def test_decode_audio_data_resamples_to_the_context_rate(engine):
    raw = random_pcm(po.S16, 2, 44100, seed=3)
    buf = engine.decode_audio_data(wav_file(raw, po.S16, 2, 44100, junk=True), context_rate=48000)
    assert (buf.numberOfChannels, buf.length, buf.sampleRate, buf.duration) == (2, 48000, 48000, 1.0)
    x = po.decode_interleaved(raw, po.S16, 2).astype(np.float32)
    for c in range(2):
        check_against_oracle(buf.getChannelData(c), x[c], 44100, 48000)
    mono = engine.decode_audio_data(wav_file(raw, po.S16, 2, 44100), mix=True, context_rate=16000)
    assert (mono.numberOfChannels, mono.length, mono.sampleRate) == (1, 16000, 16000)


@pytest.mark.gpu
def test_napi_resampling_natives_match_the_ctypes_path(tmp_path, engine):
    """tests/napi_host/fake_napi_host_resample.c drives the resampling natives through the fake Node runtime"""
    import spectrogram_b200 as sg
    from test_napi_shim import ADDON, build

    build()
    host = tmp_path / "fake_napi_host_resample"
    subprocess.check_call(["gcc", "-O1", "-Wall", "-Wextra", "-std=gnu11", "-rdynamic", "-o", str(host),
                           os.path.join(ROOT, "tests", "napi_host", "fake_napi_host_resample.c"), "-ldl", "-lm"])
    out = tmp_path / "napi_resample.bin"
    r = subprocess.run([str(host), ADDON, str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    blob = out.read_bytes()
    n, length = 44100, 48000
    state, vals = 12345, np.empty(2 * n, dtype=np.int64)
    for i in range(2 * n):
        state = (state * 1664525 + 1013904223) & 0xFFFFFFFF
        vals[i] = state >> 16
    s16 = vals.astype(np.uint16).view("<i2")
    dec = np.frombuffer(blob[:4 * length], dtype=np.float32)
    want = engine.decode_pcm(s16, "s16", 2, 44100, mix=True, context_rate=48000).getChannelData(0)
    assert np.array_equal(dec, want)
    spec = np.frombuffer(blob[4 * length:], dtype=np.uint8).reshape(-1, 1024)
    ref = engine.spectrogram_pcm(s16, "s16", 2, mix=True, opts=sg.Options(), sample_rate=44100, context_rate=48000)[0, 0]
    assert np.array_equal(spec, ref) and spec.shape[0] == 1 + (length - 2048) // 512
