"""BiquadFilterNode on the GPU (include/sgcore.h "biquad filter"): the coefficient table, its degenerate edges and
validation on the host; on the GPU the float64 direct-form-I recurrence run along time in parallel, within
max(1 float32 ulp, 2^-30 max|x|) of the sequential float64 oracle (tests/biquad_oracle.py), and the streaming bank's
filter, bit for bit against a bank fed pre-filtered chunks."""
import functools
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import signal

import biquad_oracle as BO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS = 48000


def lib_coef(type, **kw):
    import spectrogram_b200 as sg
    return sg.biquad_coefficients(type, **kw)


PARAM_SETS = [dict(frequency=f, Q=q, gain=g, detune=d, sample_rate=fs)
              for f, q, g, d, fs in ((350, 1, 0, 0, 48000), (1000, 10, 6, 0, 48000), (20, 30, -12, 0, 44100),
                                     (15000, 0.3, 18, -700, 96000), (440, 0.01, -3, 1200, 16000), (3000, -4, 40, 50, 3000),
                                     (8000, 45, -40, 0, 768000), (1e-3, 2, 1, 0, 22050))]


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("type", BO.TYPES)
def test_coefficients_equal_the_table(type):
    for kw in PARAM_SETS:
        got, want = lib_coef(type, **kw), BO.coefficients(type, **kw)
        np.testing.assert_allclose(got, want, rtol=1e-15, atol=1e-15 * np.abs(want).max(), err_msg=str(kw))


def test_degenerate_edges_are_the_limits_of_h():
    a2 = 10.0 ** (6 / 20)   # A^2 at gain 6 dB
    at0 = {"lowpass": 0, "bandpass": 0, "highpass": 1, "lowshelf": 1, "peaking": 1, "notch": 1, "allpass": 1, "highshelf": a2}
    atn = {"lowpass": 1, "highshelf": 1, "peaking": 1, "notch": 1, "allpass": 1, "highpass": 0, "bandpass": 0, "lowshelf": a2}
    q0 = {"bandpass": 1, "notch": 0, "allpass": -1, "peaking": a2}
    for type in BO.TYPES:
        for f, table in ((0.0, at0), (FS / 2, atn), (-5.0, at0), (1e9, atn)):
            np.testing.assert_allclose(lib_coef(type, frequency=f, Q=3, gain=6), [table[type], 0, 0, 0, 0], rtol=1e-15)
    for type, k in q0.items():
        for q in (0.0, -2.0):
            np.testing.assert_allclose(lib_coef(type, frequency=1000, Q=q, gain=6), [k, 0, 0, 0, 0], rtol=1e-15)
    # lowpass and highpass take any Q (10^(Q/20) > 0); the shelves ignore it
    assert lib_coef("lowpass", frequency=1000, Q=-10)[3] != 0
    np.testing.assert_array_equal(lib_coef("lowshelf", frequency=1000, Q=-3, gain=6), lib_coef("lowshelf", frequency=1000, Q=7, gain=6))


def test_detune_and_clamping_of_f0():
    np.testing.assert_array_equal(lib_coef("bandpass", frequency=1000, Q=5, detune=1200), lib_coef("bandpass", frequency=2000, Q=5))
    np.testing.assert_array_equal(lib_coef("peaking", frequency=0, Q=5, gain=3, detune=1e7), lib_coef("peaking", frequency=0, gain=3))
    np.testing.assert_array_equal(lib_coef("lowpass", frequency=1000, detune=1e7), lib_coef("lowpass", frequency=FS / 2))
    np.testing.assert_array_equal(lib_coef("notch", frequency=1000, gain=20), lib_coef("notch", frequency=1000, gain=-20))


def _h(c, f, fs):
    return np.abs(signal.freqz(c[:3], [1.0, c[3], c[4]], worN=np.atleast_1d(np.asarray(f, np.float64)), fs=fs)[1])


@pytest.mark.parametrize("fs", [16000, 48000, 96000])
def test_frequency_response_checks_that_do_not_read_the_table(fs):
    grid = np.linspace(0, fs / 2, 257)
    for f0 in (30.0, 1000.0, 0.3 * fs):
        for q in (0.5, 10.0):
            for gain in (-12.0, 6.0):
                A = 10 ** (gain / 40)
                kw = dict(frequency=f0, Q=q, gain=gain, sample_rate=fs)
                np.testing.assert_allclose(_h(lib_coef("bandpass", **kw), f0, fs), 1.0, rtol=1e-9)
                assert _h(lib_coef("notch", **kw), f0, fs)[0] < 1e-9
                np.testing.assert_allclose(_h(lib_coef("allpass", **kw), grid, fs), 1.0, rtol=1e-9)
                np.testing.assert_allclose(_h(lib_coef("peaking", **kw), f0, fs), 10 ** (gain / 20), rtol=1e-9)
                for t in ("lowpass", "highpass"):
                    np.testing.assert_allclose(_h(lib_coef(t, **kw), f0, fs), 10 ** (q / 20), rtol=1e-9)
                ls, hs = lib_coef("lowshelf", **kw), lib_coef("highshelf", **kw)
                np.testing.assert_allclose(_h(ls, [0, fs / 2], fs), [A * A, 1.0], rtol=1e-9)
                np.testing.assert_allclose(_h(hs, [0, fs / 2], fs), [1.0, A * A], rtol=1e-9)
                np.testing.assert_allclose(_h(ls, f0, fs), A, rtol=1e-9)
                np.testing.assert_allclose(_h(hs, f0, fs), A, rtol=1e-9)


def test_oracle_equals_the_plain_recurrence():
    rng = np.random.default_rng(1)
    for type in BO.TYPES:
        c = BO.coefficients(type, frequency=2000, Q=4, gain=5)
        x = rng.standard_normal((3, 300)).astype(np.float32)
        st = rng.standard_normal((3, 4))
        y, fin = BO.filter_df1(c, x, st)
        for ch in range(3):
            want, want_st = BO.filter_loop(c, x[ch], st[ch])
            np.testing.assert_allclose(y[ch], want, rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(fin[ch], want_st, rtol=1e-12, atol=1e-12)
        y1, s1 = BO.filter_df1(c, x[:, :100], st)     # split with the state carried
        y2, s2 = BO.filter_df1(c, x[:, 100:], s1)
        np.testing.assert_allclose(np.concatenate([y1, y2], axis=1), y, rtol=1e-12, atol=1e-12)


def test_validation_errors():
    import spectrogram_b200 as sg
    bad = [dict(sample_rate=2999), dict(sample_rate=768001), dict(sample_rate=44100.5), dict(sample_rate=math.nan),
           dict(frequency=math.nan), dict(frequency=math.inf), dict(Q=-math.inf), dict(gain=math.nan), dict(detune=math.inf)]
    for kw in bad:
        with pytest.raises(TypeError):
            sg.biquad_coefficients("bandpass", **kw)
    for kw in (dict(sample_rate=3000), dict(sample_rate=768000), dict(Q=-1e300, gain=-1e3)):
        sg.biquad_coefficients("peaking", **kw)
    import ctypes as C
    from spectrogram_b200 import _lib as L
    out = np.zeros(5)
    for t in (-1, 8):
        p = L.BiquadParams(t, 48000.0, 350.0, 1.0, 0.0, 0.0)
        assert L.load().sg_biquad_coefficients(C.byref(p), out.ctypes.data) == L.SG_ERR_INVALID_ARG
    node = sg.BiquadFilterNode()
    with pytest.raises(TypeError):
        node.type = "bogus"
    with pytest.raises(TypeError):
        node.frequency.value = math.nan
    assert node.type == "lowpass" and node.frequency.value == 350 and node.Q.value == 1
    assert node.gain.value == 0 and node.detune.value == 0


def test_header_documents_the_table_and_the_errors():
    text = open(os.path.join(ROOT, "include", "sgcore.h")).read()
    for s in ("int sg_biquad_coefficients(const sg_biquad_params* p, double coef[5]);",
              "int sg_biquad_filter(sg_engine* e, const sg_biquad_params* p, const float* in, int64_t n_channels, int64_t len,",
              "int sg_biquad_filter_device(sg_engine* e, const sg_biquad_params* p, const float* in_dev, int64_t n_channels,",
              "int sg_stream_set_filter(sg_stream* s, const sg_biquad_params* p);",
              "SG_ERR_INVALID_ARG", "integer in [3000, 768000]",
              "f0 = 0:       lowpass, bandpass -> 0;  highpass, lowshelf, peaking, notch, allpass -> 1;  highshelf -> A^2",
              "f0 = Fs/2:    lowpass, highshelf, peaking, notch, allpass -> 1;  highpass, bandpass -> 0;  lowshelf -> A^2",
              "q <= 0 with 0 < f0 < Fs/2:  bandpass -> 1;  notch -> 0;  allpass -> -1;  peaking -> A^2",
              "bandpass   aQ                       0                   -aQ                      1+aQ"):
        assert s in text, s


def test_js_facade_exposes_the_node():
    text = open(os.path.join(ROOT, "spectrogram_b200", "js", "index.js")).read()
    for s in ("class BiquadFilterNode", "process(samples, out)", "setFilter(node)", "native.biquadFilter",
              "native.biquadCoefficients", "native.streamSetFilter", "BIQUAD_TYPES.includes(value)"):
        assert s in text, s


def _napi_host(tmp_path):
    from test_napi_shim import ADDON, build
    build()
    host = tmp_path / "fake_napi_host_biquad"
    subprocess.check_call(["gcc", "-O1", "-Wall", "-Wextra", "-std=gnu11", "-rdynamic", "-o", str(host),
                           os.path.join(ROOT, "tests", "napi_host", "fake_napi_host_biquad.c"), "-ldl", "-lm"])
    return str(host), ADDON


def test_napi_biquad_natives_check_lengths(tmp_path):
    host, addon = _napi_host(tmp_path)
    r = subprocess.run([host, addon, "cpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "FAIL" not in r.stdout and "0 failure(s)" in r.stdout


# ---------------------------------------------------------------------------------------------------------------- GPU
@functools.lru_cache(maxsize=2)
def _signal(channels, n, seed, fs=FS):
    """Seeded noise plus a sine per channel (cached: callers must not modify it)."""
    rng = np.random.default_rng(seed)
    x = 0.25 * rng.standard_normal((channels, n)).astype(np.float32)
    t = np.arange(n, dtype=np.float64) / fs
    f = rng.uniform(20.0, 0.45 * fs, size=(channels, 1))
    x += (0.5 * np.sin(2 * np.pi * f * t)).astype(np.float32)
    return x


def _params(type):
    return dict(frequency=1000.0, Q=10.0 if type in ("bandpass", "notch", "peaking") else 0.7, gain=6.0)


def _node(engine, type, channels, **kw):
    import spectrogram_b200 as sg
    node = sg.BiquadFilterNode(engine, sample_rate=kw.pop("sample_rate", FS), channels=channels)
    node.type = type
    for k, v in kw.items():
        getattr(node, k).value = v
    return node


def _check(got, x, type, state=None, **kw):
    c = BO.coefficients(type, sample_rate=kw.pop("sample_rate", FS), **kw)
    want, fin = BO.filter_df1(c, x, state)
    assert BO.bound_violations(got, want, x) == 0
    return fin


@pytest.mark.gpu
@pytest.mark.parametrize("type", BO.TYPES)
def test_long_channels_follow_the_oracle(engine, type):
    for channels, n in ((1, 3600 * FS), (64, 30 * FS)):
        x = _signal(channels, n, 7)
        node = _node(engine, type, channels, **_params(type))
        y = node.process(x)
        fin = _check(y, x, type, **_params(type))
        np.testing.assert_allclose(node.state, fin, rtol=1e-12, atol=1e-12 * np.abs(x).max())


@pytest.mark.gpu
@pytest.mark.parametrize("type", BO.TYPES)
def test_many_short_channels(engine, type):
    for n in (1, 2, 3, 127):
        x = _signal(4096, n, n)
        node = _node(engine, type, 4096, **_params(type))
        st = np.random.default_rng(n).standard_normal((4096, 4)) * 0.1
        node._state[:] = st
        y = node.process(x)
        fin = _check(y, x, type, state=st, **_params(type))
        np.testing.assert_allclose(node.state, fin, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("type,kw", [("bandpass", dict(frequency=20.0, Q=30.0)), ("allpass", dict(frequency=10.0, Q=1.0))])
def test_poles_near_the_unit_circle(engine, type, kw):
    x = _signal(4, 2_000_003, 11)
    y = _node(engine, type, 4, **kw).process(x)
    _check(y, x, type, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("pieces", [1, 2, 7])
def test_split_calls_carry_the_state(engine, pieces):
    x = _signal(5, 1_234_567, 3)
    node = _node(engine, "bandpass", 5, frequency=700.0, Q=10.0)
    edges = np.linspace(0, x.shape[1], pieces + 1).astype(int)
    edges[1:-1] += 4097 % 13                       # pieces of uneven, non-tile-multiple lengths
    y = np.concatenate([node.process(x[:, a:b]) for a, b in zip(edges[:-1], edges[1:])], axis=1)
    fin = _check(y, x, "bandpass", frequency=700.0, Q=10.0)
    np.testing.assert_allclose(node.state, fin, rtol=1e-12, atol=1e-12 * np.abs(x).max())


@pytest.mark.gpu
def test_device_entry_strided_in_place_and_equal_to_host(engine):
    import torch
    x = _signal(6, 50_001, 5)
    node = _node(engine, "peaking", 6, frequency=3000.0, Q=2.0, gain=-9.0)
    host = node.process(x)
    dev = torch.zeros((6, 50_007), dtype=torch.float32, device="cuda")
    dev[:, 1:50_002] = torch.from_numpy(x).cuda()
    out = torch.zeros((6, 50_010), dtype=torch.float32, device="cuda")
    state = torch.zeros((6, 4), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    # strided, unaligned input (offset of one float), out of place
    engine.biquad_device(node, dev.data_ptr() + 4, 6, 50_001, 50_007, out.data_ptr(), 50_010, state.data_ptr())
    engine.synchronize()
    assert np.array_equal(out[:, :50_001].cpu().numpy(), host)
    assert np.array_equal(state.cpu().numpy(), node.state)
    # in place, from the carried state, against the host call
    y2 = node.process(x)
    engine.biquad_device(node, dev.data_ptr() + 4, 6, 50_001, 50_007, dev.data_ptr() + 4, 50_007, state.data_ptr())
    engine.synchronize()
    assert np.array_equal(dev[:, 1:50_002].cpu().numpy(), y2)
    assert np.array_equal(state.cpu().numpy(), node.state)
    _check(np.concatenate([host, y2], axis=1), np.concatenate([x, x], axis=1), "peaking", frequency=3000.0, Q=2.0, gain=-9.0)
    # equal inputs and shapes: equal bits
    assert np.array_equal(_node(engine, "peaking", 6, frequency=3000.0, Q=2.0, gain=-9.0).process(x), host)


def _bank(engine, channels, **kw):
    import spectrogram_b200 as sg
    opts = sg.Options(fftSize=1024, hop=128, output="u8", smoothingTimeConstant=0.8)
    return sg.StreamBank(channels, opts, max_chunk=8192, engine=engine, **kw)


def _same(a, b):
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


@pytest.mark.gpu
def test_bank_filter_equals_a_bank_fed_filtered_chunks(engine):
    ch = 32
    chunks = [_signal(ch, n, k) for k, n in enumerate((128, 1024, 128, 8192, 512, 128, 4224))]
    node = _node(engine, "bandpass", ch, frequency=1500.0, Q=10.0)
    pre = _node(engine, "bandpass", ch, frequency=1500.0, Q=10.0)
    a, b = _bank(engine, ch, history_rows=64, filter=node), _bank(engine, ch, history_rows=64)
    for k, x in enumerate(chunks):
        if k == 3:                       # dragging in draw mode: a new frequency, the state carries on
            node.frequency.value = pre.frequency.value = 4000.0
        if k == 5:
            node.Q.value = pre.Q.value = 3.0
        _same(a.push(x, want_rgba=True), b.push(pre.process(x), want_rgba=True))
    assert np.array_equal(a.history(), b.history())
    assert np.array_equal(a.view(320, 96), b.view(320, 96))
    # reset zeroes the filter state and keeps the parameters
    a.reset(); b.reset(); pre.reset()
    x = chunks[1]
    _same(a.push(x, want_rgba=True), b.push(pre.process(x), want_rgba=True))
    # detach: unfiltered samples from then on
    a.set_filter(None)
    assert np.array_equal(a.push(chunks[2]), b.push(chunks[2]))
    # re-attach: from zero state
    a.set_filter(node)
    pre.reset()
    for x in chunks[:3]:
        assert np.array_equal(a.push(x), b.push(pre.process(x)))
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("output", ["db", "mag"])
def test_bank_filter_with_float_outputs_and_no_history(engine, output):
    import spectrogram_b200 as sg
    opts = sg.Options(fftSize=1024, hop=128, output=output)
    node = _node(engine, "lowshelf", 8, frequency=300.0, gain=12.0)
    pre = _node(engine, "lowshelf", 8, frequency=300.0, gain=12.0)
    a = sg.StreamBank(8, opts, max_chunk=1024, engine=engine, filter=node)
    b = sg.StreamBank(8, opts, max_chunk=1024, engine=engine)
    for k in range(4):
        x = _signal(8, 1024, 40 + k)
        assert np.array_equal(a.push(x), b.push(pre.process(x)))
    a.close(); b.close()


@pytest.mark.gpu
def test_filter_adds_one_launch_per_push(engine):
    x = _signal(256, 128, 9)
    a = _bank(engine, 256, filter=_node(engine, "bandpass", 256, frequency=1000.0, Q=10.0))
    b = _bank(engine, 256)
    for bank in (a, b):
        bank.push(x)
    n0 = engine.launch_count
    a.push(x)
    n1 = engine.launch_count
    b.push(x)
    n2 = engine.launch_count
    assert (n1 - n0) - (n2 - n1) == 1
    a.close(); b.close()


@pytest.mark.gpu
def test_napi_biquad_natives_match_the_python_path(tmp_path, engine):
    """tests/napi_host/fake_napi_host_biquad.c: 3 channels of LCG samples through biquadFilter in two calls with the
    state carried, then a 4-channel bank with a bandpass; its bytes equal the Python path's."""
    import spectrogram_b200 as sg
    from test_stream_history import lcg_chunks
    host, addon = _napi_host(tmp_path)
    out = tmp_path / "napi_biquad.bin"
    r = subprocess.run([host, addon, "gpu", str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = open(out, "rb").read()
    chunks = list(lcg_chunks(3, [5000, 3000]))
    node = _node(engine, "bandpass", 3, frequency=1200.0, Q=10.0)
    y = np.concatenate([node.process(c) for c in chunks], axis=1)
    n_y = y.size * 4
    assert np.frombuffer(raw[:n_y], np.float32).reshape(3, 8000).tobytes() == y.tobytes()
    assert np.frombuffer(raw[n_y:n_y + 96], np.float64).reshape(3, 4).tobytes() == node.state.tobytes()
    bank = sg.StreamBank(4, sg.Options(fftSize=1024, hop=128, output="u8"), max_chunk=1024, engine=engine,
                         filter=_node(engine, "bandpass", 4, frequency=2500.0, Q=10.0))
    rows = b"".join(bank.push(c).tobytes() for c in lcg_chunks(4, [1024, 512, 1024], seed=77))
    assert raw[n_y + 96:] == rows
    bank.close()
