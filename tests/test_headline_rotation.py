"""The headline kernel (``stft_w32x2p_kernel``) runs the warps of each scheduler in a rotation: three sections per
frame pair, one group barrier per step, and every warp of a group executing the same number of barriers
(kernel_w32x2p.cuh).  Two things are checked here.

CPU: the closed-form pair and step counts the kernel takes its barrier count from equal a brute-force play of the
rotation over a sweep of (total frames, grid, warps per CTA).  A wrong count would leave a warp waiting at a barrier
the others never reach.

GPU: at smoothingTimeConstant 0 every frame is independent of the warp, the pair and the grid it lands on, so batches
that change the grid, the per-warp pair counts, the pairing of frames (odd frames per clip: pairs straddle clips)
and the number of idle warps give byte-identical rows to the same clips cut out of one large batch, and stay within
the oracle tolerance of tests/_tol.py."""
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "spectrogram_b200", "csrc")

BRUTE = r"""
#include <cstdio>
#include "kernel_w32x2p.cuh"
using namespace sg;

int main() {
  long long groups = 0, bad = 0;
  const int grids[] = {1, 2, 3, 7, 148};
  for (int nw = 8; nw <= 12; nw += 4)
    for (int grid : grids)
      for (long long total = 0; total <= 4000; total += total < 300 ? 1 : 97)
        for (int block = 0; block < grid; ++block)
          for (int group = 0; group < 4; ++group, ++groups) {
            // each member's pairs, enumerated the way the kernel's loop advances
            long long left[3] = {0, 0, 0}, own[3] = {0, 0, 0};
            for (int k = 0; k < nw / 4; ++k) {
              const int warp = group + 4 * k;
              for (long long fa = 2 * ((long long)block * nw + warp); fa < total; fa += 2LL * grid * nw) ++left[k];
              if (left[k] != xp_warp_pairs(total, grid, nw, block, warp)) ++bad;
            }
            // the rotation: at step s rank k runs section (s + k) % 3 and starts a pair only at a section-A step;
            // the group's count is one past the last step in which any member still runs a section
            long long last = -1, in_pair[3] = {0, 0, 0};
            for (long long s = 0; left[0] + left[1] + left[2] + in_pair[0] + in_pair[1] + in_pair[2] > 0; ++s) {
              for (int k = 0; k < nw / 4; ++k) {
                const int sec = (int)((s + k) % 3);
                if (sec == 0 && left[k] > 0) { --left[k]; in_pair[k] = 1; }
                if (in_pair[k]) {
                  last = s;
                  if (sec == 2) { in_pair[k] = 0; ++own[k]; }
                }
              }
            }
            const long long steps = xp_group_steps(total, grid, nw, block, group);
            if (steps != last + 1) ++bad;
            for (int k = 0; k < nw / 4; ++k)   // barriers: lead + 3 per pair + tail, never a negative tail
              if (xp_warp_steps(total, grid, nw, block, group + 4 * k) > steps ||
                  own[k] != xp_warp_pairs(total, grid, nw, block, group + 4 * k))
                ++bad;
          }
  printf("groups %lld mismatches %lld\n", groups, bad);
  return bad != 0;
}
"""


def _nvcc():
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    pytest.skip("nvcc not found")


def test_rotation_step_count_matches_brute_force(tmp_path):
    src = tmp_path / "rotation_brute.cu"
    src.write_text(BRUTE)
    exe = tmp_path / "rotation_brute"
    subprocess.run([_nvcc(), "-std=c++17", "--expt-relaxed-constexpr", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-I", CSRC, "-o", str(exe), str(src)], check=True, capture_output=True, timeout=600)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches 0" in r.stdout


# ----------------------------------------------------------------------------------------------------------- GPU
import spectrogram_b200 as sg  # noqa: E402
from oracle import analyser_oracle as O  # noqa: E402
from _tol import assert_bytes_close, assert_db_close  # noqa: E402

BIG = 512


def _clips(n, clip_len, seed):
    rng = np.random.default_rng(seed)
    x = (rng.random((n, clip_len), dtype=np.float32) - 0.5)
    x[:, ::997] *= 40.0                                      # loud clicks: bytes at both ends of the range
    t = np.arange(clip_len, dtype=np.float32) / 44100.0
    x[::5] += 0.3 * np.sin(2 * np.pi * (200.0 + 3000.0 * t) * t).astype(np.float32)
    return x


# (clip_len, hop, output, align): 44100 samples give 83 frames per clip at hop 512 -- odd, so frame pairs straddle clips
# and a clip's first frame is frame A in one batch and frame B in another; 2560 samples give 2 frames, so a few clips
# leave most warps of the CTA without a pair
SHAPES = [(44100, 512, "u8", "valid"), (44100, 256, "u8", "valid"), (44100, 512, "u8", "analyser"),
          (2560, 512, "u8", "valid"), (44100, 256, "db", "valid"), (22050, 256, "rgba", "analyser")]
# (first clip, clip count) cut out of the big batch
CUTS = [(0, 1), (3, 2), (11, 7), (100, 149), (201, 150), (0, BIG)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}-hop{s[1]}-{s[2]}-{s[3]}")
def test_rows_independent_of_batch(engine, shape):
    clip_len, hop, out, align = shape
    engine.set_kernel_variant(0)
    opts = sg.Options(fftSize=2048, hop=hop, output=out, align=align)
    x = _clips(BIG, clip_len, seed=clip_len + hop)
    big = engine.spectrogram(x, opts)
    assert engine.last_kernel == "warp32x32x2p"
    for first, n in CUTS:
        got = engine.spectrogram(x[first:first + n], opts)
        assert engine.last_kernel == "warp32x32x2p"
        assert np.array_equal(got, big[first:first + n]), f"clips [{first}, {first + n}) differ from the big batch"
    # the big batch itself against the float64 oracle, on a spread of clips
    pick = [0, 1, 2, 5, 149, 150, 299, BIG - 1]
    cfg = O.Config(n_fft=2048, hop=hop, align=O.ALIGN_ANALYSER if align == "analyser" else O.ALIGN_VALID,
                   output=O.OUT_F32_MAG)
    ref_mag = O.spectrogram(x[pick], cfg)
    if out == "db":
        assert_db_close(big[pick], ref_mag)
    else:
        ref_u8 = O.finish(ref_mag, O.Config(**{**cfg.__dict__, "output": O.OUT_U8}))
        got_u8 = big[pick]
        if out == "rgba":   # the colour map applied to the kernel's own bytes is exact
            got_u8 = engine.spectrogram(x[pick], sg.Options(fftSize=2048, hop=hop, output="u8", align=align))
            assert np.array_equal(big[pick], O.colormap_lut()[got_u8])
        assert_bytes_close(got_u8, ref_u8)


@pytest.mark.gpu
def test_eight_warp_form_rows_independent_of_batch(engine):
    """Variant 6 runs the same kernel with 8 warps, two per rotation group (hop 512: u8, dB)."""
    x = _clips(150, 44100, seed=6)
    try:
        engine.set_kernel_variant(6)
        for out in ("u8", "db"):
            opts = sg.Options(fftSize=2048, hop=512, output=out)
            ref = engine.spectrogram(x, opts)
            assert engine.last_kernel == "warp32x32x2p"
            for first, n in [(1, 7), (149, 1), (0, 149)]:
                assert np.array_equal(engine.spectrogram(x[first:first + n], opts), ref[first:first + n])
            ref_mag = O.spectrogram(x[[0, 77, 149]], O.Config(n_fft=2048, hop=512, output=O.OUT_F32_MAG))
            if out == "db":
                assert_db_close(ref[[0, 77, 149]], ref_mag)
            else:
                assert_bytes_close(ref[[0, 77, 149]], O.finish(ref_mag, O.Config(n_fft=2048, hop=512)))
    finally:
        engine.set_kernel_variant(0)
