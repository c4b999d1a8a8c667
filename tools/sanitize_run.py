#!/usr/bin/env python
"""One small call into every kernel family and every object of the C ABI.  Run against the SG_DEBUG build of the
library (make -C spectrogram_b200/csrc debug; SG_LIBSGCORE=spectrogram_b200/libsgcore_debug.so) it arms the epoch
tags beside the shared-memory hand-offs (spectrogram_b200/csrc/common.cuh) and prints the mismatch counts as a JSON
line; tests/test_debug_build.py drives it that way.  (compute-sanitizer is closed on this pool.)"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import spectrogram_b200 as sg  # noqa: E402

eng = sg.Engine(0)
rng = np.random.default_rng(0)
x = (0.1 * rng.standard_normal((3, 9000))).astype(np.float32)
seen = set()
for n_fft, hop, align in ((2048, 512, "valid"), (2048, 512, "analyser"), (2048, 300, "valid"), (400, 160, "valid"),
                          (400, 77, "analyser"), (512, 160, "valid"), (256, 64, "analyser"), (1024, 128, "valid"),
                          (4096, 1024, "valid"), (8192, 2048, "analyser"), (600, 150, "valid")):
    for out in ("u8", "db", "rgba", "mag"):
        for tau in (0.0, 0.8):
            o = sg.Options(fftSize=n_fft, hop=hop, align=align, output=out, smoothingTimeConstant=tau)
            y = eng.spectrogram(x, o)
            seen.add(eng.last_kernel)
for v in (1, 2, 4, 6):
    eng.set_kernel_variant(v)
    eng.spectrogram(x, sg.Options())
    seen.add(eng.last_kernel)
eng.set_kernel_variant(0)
bank = sg.StreamBank(4, sg.Options(fftSize=1024, hop=128, output="u8"), max_chunk=256, engine=eng)
for _ in range(3):
    bank.push(x[:, :256].repeat(2, axis=0)[:4].copy(), want_rgba=True)
bank.close()
ring = sg.SonogramRing(1024, 256, engine=eng)
ring.append(eng.spectrogram(x[0], sg.Options()).reshape(-1, 1024))
ring.view(64, 32)
ring.close()
an = sg.AnalyserNode(eng)
an.push(x[0, :4096])
buf = np.zeros(an.frequencyBinCount, np.uint8)
an.getByteFrequencyData(buf)
an.close()
# larger batches: every warp of every CTA runs several pairs, clips end inside CTAs, and the fused smoothing kernel runs in
# both of its modes (chained segments, look-back)
big = (0.1 * rng.standard_normal((160, 2048 + 90 * 512))).astype(np.float32)
for out in ("u8", "db"):
    eng.spectrogram(big, sg.Options(output=out))
    seen.add(eng.last_kernel)
eng.set_kernel_variant(7)
for clips in (160, 3):
    eng.spectrogram(big[:clips], sg.Options(smoothingTimeConstant=0.8))
    seen.add(eng.last_kernel)
# ... and the fused smoothing kernels of n_fft 4096 / 1024 / 512 / 256: several steps per warp, chained segments
for n_fft, clips in ((4096, 160), (1024, 160), (512, 40), (256, 3)):
    eng.spectrogram(big[:clips], sg.Options(fftSize=n_fft, hop=n_fft // 4, smoothingTimeConstant=0.8))
    seen.add(eng.last_kernel)
eng.set_kernel_variant(0)
# the biquad filter: one tile per channel (one launch), and channels of several tiles (tile aggregates, carry scan, emit)
bq = sg.BiquadFilterNode(eng, channels=3)
bq.type = "bandpass"
for n in (300, 3 * 4096 + 77):
    bq.process(x[:, :n] if n <= x.shape[1] else np.tile(x, (1, 2))[:, :n])
    seen.add(eng.last_kernel)
lib = sg._lib.load()
if hasattr(lib, "sg_debug_counts"):
    counts = (C.c_ulonglong * 16)()
    lib.sg_debug_counts.argtypes = [C.c_void_p, C.c_void_p]
    assert lib.sg_debug_counts(eng.handle, counts) == 0
    print(json.dumps({"debug_counts": list(counts), "kernels": sorted(seen)}))
eng.close()
print("sanitize_run ok; kernels:", sorted(seen))
