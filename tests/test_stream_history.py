"""Sonogram history of the streaming bank (sg_stream_set_history, sg_stream_view): per channel, the state of a
``SonogramRing(bins, rows)`` fed every push's byte rows, kept and filled on the device, with every channel's picture
rendered in one launch.  The contract is the existing objects, bit for bit: the texture, yoffset and view pixels of
per-channel rings fed the rows each push returned."""
import os
import subprocess

import numpy as np
import pytest

from oracle import analyser_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class BankHistory:
    """Numpy model of a bank's history: [channels][rows][bins] bytes and one shared yoffset.  A push of F frames writes
    them at yoffset .. yoffset+F-1 (mod rows); when F > rows only the last rows frames survive."""

    def __init__(self, channels, bins, rows):
        self.rows = rows
        self.tex = np.zeros((channels, rows, bins), np.uint8)
        self.yoffset = 0

    def append(self, frames):          # frames: [channels][F][bins]
        f = frames.shape[1]
        skip = max(0, f - self.rows)
        idx = (self.yoffset + np.arange(skip, f)) % self.rows
        self.tex[:, idx] = frames[:, skip:]
        self.yoffset = (self.yoffset + f) % self.rows


def lcg_chunks(channels, lengths, seed=2024):
    """The samples tests/napi_host/fake_napi_host_history.c generates: a 32-bit LCG, [channel][len] per chunk."""
    state = seed
    for n in lengths:
        x = np.empty(channels * n, np.float32)
        for i in range(x.size):
            state = (state * 1664525 + 1013904223) & 0xFFFFFFFF
            x[i] = (state >> 8) / 16777216.0 - 0.5
        yield x.reshape(channels, n)


def test_bank_history_model_equals_per_channel_rings():
    rng = np.random.default_rng(3)
    for rows in (2, 5, 17):
        model = BankHistory(3, 7, rows)
        rings = [O.Ring(7, rows) for _ in range(3)]
        for f in (1, 3, rows, rows + 4, 2 * rows + 1, 2):
            frames = rng.integers(0, 256, size=(3, f, 7), dtype=np.uint8)
            model.append(frames)
            for c, ring in enumerate(rings):
                ring.append(frames[c])
            assert model.yoffset == rings[0].yoffset
            assert np.array_equal(model.tex, np.stack([r.tex for r in rings]))


def test_history_header_documents_the_errors():
    text = open(os.path.join(ROOT, "include", "sgcore.h")).read()
    for name in ("int sg_stream_set_history(sg_stream* s, int rows);",
                 "int sg_stream_history_info(const sg_stream* s, int* rows, int* yoffset);",
                 "int sg_stream_history_read(sg_stream* s, int first, int count, uint8_t* dst);",
                 "int sg_stream_view(sg_stream* s, int first, int count, int width, int height, uint32_t* rgba_out);",
                 "SG_ERR_STATE when no history is attached"):
        assert name in text, name


def test_js_facade_exposes_the_history():
    text = open(os.path.join(ROOT, "spectrogram_b200", "js", "index.js")).read()
    for name in ("historyRows", "get historyYoffset()", "history(options)", "view(width, height, options)",
                 "native.streamView", "native.streamHistoryRead", "native.streamSetHistory", "native.streamHistoryInfo"):
        assert name in text, name


def _napi_host(tmp_path):
    from test_napi_shim import ADDON, build
    build()
    host = tmp_path / "fake_napi_host_history"
    subprocess.check_call(["gcc", "-O1", "-Wall", "-Wextra", "-std=gnu11", "-rdynamic", "-o", str(host),
                           os.path.join(ROOT, "tests", "napi_host", "fake_napi_host_history.c"), "-ldl", "-lm"])
    return str(host), ADDON


def test_napi_history_natives_reject_bad_handles(tmp_path):
    host, addon = _napi_host(tmp_path)
    r = subprocess.run([host, addon, "cpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "FAIL" not in r.stdout and "0 failure(s)" in r.stdout


# ---------------------------------------------------------------------------------------------------------------- GPU
def _chunks(channels, lengths, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(sum(lengths)) / 48000.0
    f = rng.uniform(200.0, 12000.0, size=(channels, 1))
    x = (0.4 * np.sin(2 * np.pi * f * t * (1.0 + 0.5 * t))
         + 0.05 * rng.standard_normal((channels, t.size))).astype(np.float32)
    x[: channels // 4] *= 0.01                      # some quiet channels: dark pictures too
    edges = np.cumsum([0] + list(lengths))
    return [x[:, a:b] for a, b in zip(edges[:-1], edges[1:])]


def _bank(engine, channels, rows, tau=0.0, max_chunk=None):
    import spectrogram_b200 as sg
    opts = sg.Options(fftSize=1024, hop=128, output="u8", smoothingTimeConstant=tau)
    return sg.StreamBank(channels, opts, max_chunk=max_chunk or 300 * 128, engine=engine, history_rows=rows)


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [256, 17])
def test_bank_history_and_views_equal_per_channel_rings(engine, rows):
    import spectrogram_b200 as sg
    channels = 64
    bank = _bank(engine, channels, rows)
    rings = [sg.SonogramRing(512, rows, engine=engine) for _ in range(channels)]
    model = BankHistory(channels, 512, rows)
    # mixed chunk sizes, one push with more frames than rows, and enough frames to wrap
    lengths = [128, 1024, 384, (rows + 9) * 128, 256, 128 * 7, 2048, 128 * 61]
    assert bank.history_rows == rows and bank.history_yoffset == 0 and not bank.history().any()
    for x in _chunks(channels, lengths, rows):
        out = bank.push(x)
        model.append(out)
        for c, ring in enumerate(rings):
            ring.append(out[c])
        assert bank.history_yoffset == rings[0].yoffset == model.yoffset
        got = bank.history()
        assert got.shape == (channels, rows, 512)
        assert np.array_equal(got, np.stack([r.texture() for r in rings]))
        assert np.array_equal(got, model.tex)
    assert np.array_equal(bank.history(5, 9), model.tex[5:14])
    for w, h in ((640, 256), (33, 7), (1, 1)):
        want = np.stack([r.view(w, h) for r in rings])
        assert np.array_equal(bank.view(w, h), want), (w, h)
        assert np.array_equal(bank.view(w, h, first=13, count=21), want[13:34]), (w, h)
        assert np.array_equal(bank.view(w, h, first=channels - 1), want[-1:]), (w, h)
    # pinned output is written by DMA directly and holds the same picture
    pin = sg.PinnedArray((4, 7, 33, 4), np.uint8)
    bank.view(33, 7, first=60, out=pin.array)
    assert np.array_equal(pin.array, np.stack([r.view(33, 7) for r in rings[60:]]))
    pin.free()
    for r in rings:
        r.close()
    bank.close()


@pytest.mark.gpu
def test_bank_views_follow_the_float64_oracle(engine):
    bank = _bank(engine, 16, 256)
    for x in _chunks(16, [128 * 100, 128 * 200], 7):
        bank.advance(x)
    tex, y = bank.history(), bank.history_yoffset
    for w, h in ((640, 256), (33, 7), (1, 1)):
        got = bank.view(w, h)
        for c in (0, 5, 15):
            d = np.abs(got[c].astype(np.int32) - O.sonogram_view(tex[c], y, w, h).astype(np.int32))
            assert d.max() <= 1, f"channel {c} {w}x{h}: max {d.max()} LSB"
            assert (d != 0).mean() < 0.02
        if w == 640:
            assert got[..., :3].max() > 100          # the tones are visible
    bank.close()


@pytest.mark.gpu
@pytest.mark.parametrize("tau", [0.0, 0.8])
def test_attaching_a_history_changes_nothing_a_push_returns(engine, tau):
    plain, hist = _bank(engine, 32, None, tau, 4096), _bank(engine, 32, 40, tau, 4096)
    for x in _chunks(32, [128, 4096, 640, 4096, 128], 11):
        a, a_rgba = plain.push(x, want_rgba=True)
        b, b_rgba = hist.push(x, want_rgba=True)
        assert np.array_equal(a, b) and np.array_equal(a_rgba, b_rgba)
        assert np.array_equal(plain.push(x), hist.push(x))
    assert plain.frames_emitted == hist.frames_emitted
    plain.close()
    hist.close()


@pytest.mark.gpu
def test_pushes_without_rows_leave_the_same_history(engine):
    a, b = _bank(engine, 24, 33, 0.8, 4096), _bank(engine, 24, 33, 0.8, 4096)
    for x in _chunks(24, [4096, 128, 1024, 4096, 384], 13):
        a.push(x)
        b.advance(x)
        assert a.history_yoffset == b.history_yoffset
        assert np.array_equal(a.history(), b.history())
    assert np.array_equal(a.view(100, 50), b.view(100, 50))
    a.close()
    b.close()


@pytest.mark.gpu
def test_reset_detach_and_bad_arguments(engine):
    import spectrogram_b200 as sg
    from spectrogram_b200 import _lib as L
    lib = L.load()
    bank = _bank(engine, 8, 16, 0.0, 1024)
    for x in _chunks(8, [1024, 512], 17):
        bank.advance(x)
    assert bank.history_yoffset == 12 and bank.history().any()
    bank.reset()
    assert bank.history_yoffset == 0 and not bank.history().any() and bank.history_rows == 16
    bank.advance(_chunks(8, [256], 19)[0])
    bank.set_history(16)                             # re-attaching starts empty too
    assert bank.history_yoffset == 0 and not bank.history().any()
    buf = np.zeros(64, np.uint32)
    for rows in (1, -1, 65537):
        assert lib.sg_stream_set_history(bank._h, rows) == L.SG_ERR_INVALID_ARG
        with pytest.raises(TypeError):
            bank.set_history(rows)
    assert bank.history_rows == 16                   # a rejected size leaves the history as it was
    for first, count in ((0, 0), (-1, 2), (7, 2), (8, 1), (0, 9)):
        assert lib.sg_stream_view(bank._h, first, count, 2, 2, buf.ctypes.data) == L.SG_ERR_INVALID_ARG
        with pytest.raises(TypeError):
            bank.view(2, 2, first, count)
        with pytest.raises(TypeError):
            bank.history(first, count)
    for w, h in ((0, 5), (5, 0), (-1, 5), (1 << 15, 1 << 15)):
        assert lib.sg_stream_view(bank._h, 0, 1, w, h, buf.ctypes.data) == L.SG_ERR_INVALID_ARG
    assert lib.sg_stream_view(bank._h, 0, 8, 1 << 14, 1 << 14, buf.ctypes.data) == L.SG_ERR_INVALID_ARG   # > 2^30 total
    assert lib.sg_stream_view(bank._h, 0, 1, 2, 2, None) == L.SG_ERR_INVALID_ARG
    x = np.zeros((8, 128), np.float32)
    assert lib.sg_stream_push(bank._h, x.ctypes.data, 128, None, buf.ctypes.data) == L.SG_ERR_INVALID_ARG
    bank.set_history(0)
    assert bank.history_rows == 0 and bank.history_yoffset == 0
    assert lib.sg_stream_view(bank._h, 0, 1, 2, 2, buf.ctypes.data) == L.SG_ERR_STATE
    with pytest.raises(sg.InvalidStateError):
        bank.view(2, 2)
    with pytest.raises(sg.InvalidStateError):
        bank.history()
    assert lib.sg_stream_push(bank._h, x.ctypes.data, 128, None, None) == L.SG_ERR_INVALID_ARG   # out needed again
    with pytest.raises(TypeError):
        bank.advance(x)
    out = bank.push(x)                               # pushes without a history work as before
    assert out.shape == (8, 1, 512)
    bank.close()
    db = sg.StreamBank(4, sg.Options(fftSize=1024, hop=128, output="db"), engine=engine)
    assert lib.sg_stream_set_history(db._h, 16) == L.SG_ERR_INVALID_ARG
    with pytest.raises(TypeError):
        db.set_history(16)
    db.close()
    with pytest.raises(TypeError):
        sg.StreamBank(4, sg.Options(fftSize=1024, hop=128, output="rgba"), engine=engine, history_rows=16)


@pytest.mark.gpu
def test_one_launch_renders_every_channel(engine):
    import spectrogram_b200 as sg
    bank = _bank(engine, 256, 256, 0.0, 1024)
    for x in _chunks(256, [1024, 1024], 23):
        bank.advance(x)
    for w, h in ((256, 128), (33, 7)):
        n = engine.launch_count
        img = bank.view(w, h)
        assert engine.launch_count == n + 1 and engine.last_kernel == "sonogram_views"
        assert img.shape == (256, h, w, 4)
    ring = sg.SonogramRing(512, 256, engine=engine)
    ring.view(8, 8)
    assert engine.last_kernel == "sonogram_view"
    ring.close()
    bank.close()


@pytest.mark.gpu
def test_napi_history_natives_match_the_ctypes_path(tmp_path, engine):
    """tests/napi_host/fake_napi_host_history.c: 8 channels, n_fft 1024, hop 128, 24 rows, pushes alternating with and
    without an out array; the texture and two views it writes equal what the Python binding makes of the same input."""
    import spectrogram_b200 as sg
    host, addon = _napi_host(tmp_path)
    out = tmp_path / "napi_history.bin"
    r = subprocess.run([host, addon, "gpu", str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(out, dtype=np.uint8)
    n_tex, n_v1 = 8 * 24 * 512, 8 * 32 * 64 * 4
    bank = sg.StreamBank(8, sg.Options(fftSize=1024, hop=128, output="u8"), max_chunk=1024, engine=engine,
                         history_rows=24)
    for k, x in enumerate(lcg_chunks(8, [256, 1024, 128, 1024, 1024, 512, 1024, 1024])):
        if k % 2:
            bank.advance(x)
        else:
            bank.push(x)
    assert bank.history_yoffset == 47 % 24
    assert np.array_equal(raw[:n_tex].reshape(8, 24, 512), bank.history())
    assert np.array_equal(raw[n_tex:n_tex + n_v1].reshape(8, 32, 64, 4), bank.view(64, 32))
    assert np.array_equal(raw[n_tex + n_v1:].reshape(3, 7, 33, 4), bank.view(33, 7, first=2, count=3))
    bank.close()
