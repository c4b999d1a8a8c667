"""Host-side logic that needs no GPU: options mapping, sharding, the multi-process bench plumbing, bench.py's output dump
(the GPU arm's under ``-m gpu``)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import spectrogram_b200 as sg
from spectrogram_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_bounds_cover_and_partition():
    for n, g in [(4096, 8), (4096, 3), (5, 8), (0, 4), (256, 2)]:
        b = sg.shard_bounds(n, g)
        assert b[0][0] == 0 and b[-1][1] == n
        assert all(b[i][1] == b[i + 1][0] for i in range(g - 1))
        sizes = [hi - lo for lo, hi in b]
        assert max(sizes) - min(sizes) <= 1


def test_options_map_to_the_c_struct():
    cfg, _keep = sg.Options(fftSize=512, hop=160, window="hann", output="db", align="analyser",
                            minDecibels=-90, maxDecibels=-10, smoothingTimeConstant=0.8).to_c()
    assert (cfg.n_fft, cfg.hop, cfg.window, cfg.output, cfg.align) == (512, 160, _lib.WINDOW_HANN, _lib.OUT_F32_DB, _lib.ALIGN_ANALYSER)
    assert (cfg.min_db, cfg.max_db) == (-90.0, -10.0) and abs(cfg.smoothing - 0.8) < 1e-7
    w = np.hanning(512).astype(np.float32)
    cfg, keep = sg.Options(fftSize=512, window=w).to_c()
    assert cfg.window == _lib.WINDOW_CUSTOM and keep
    with pytest.raises(TypeError):
        sg.Options(window="kaiser").to_c()
    with pytest.raises(TypeError):
        sg.Options(output="png").to_c()
    with pytest.raises(TypeError):
        sg.Options(fftSize=512, window=np.ones(100, np.float32)).to_c()


def test_status_codes_map_to_web_audio_exceptions():
    with pytest.raises(sg.IndexSizeError):
        _lib.check(_lib.SG_ERR_INDEX_SIZE)
    with pytest.raises(TypeError):
        _lib.check(_lib.SG_ERR_INVALID_ARG)
    with pytest.raises(MemoryError):
        _lib.check(_lib.SG_ERR_OOM)
    with pytest.raises(sg.EngineError):
        _lib.check(_lib.SG_ERR_CUDA)
    assert sg.IndexSizeError.name == "IndexSizeError"


def test_bench_shard_plan_world_size_2_gloo(tmp_path):
    """The N>1 path of bench.py (clip sharding, barrier, max-over-ranks reduction) on CPU/gloo."""
    script = tmp_path / "gloo_ranks.py"
    script.write_text(r"""
import sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
import bench
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
plan = bench.shard_plan(total_clips=10, world=world, rank=rank)
t = torch.tensor([float(plan["n_clips"])])
dist.all_reduce(t)
assert int(t.item()) == 10, t
ms = bench.max_over_ranks(5.0 + rank, device="cpu")
assert ms == 6.0, ms
frames = bench.sum_over_ranks(100 * (rank + 1), device="cpu")
assert frames == 300, frames
bench.barrier()
dist.destroy_process_group()
print("ok", rank)
""" % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29517", str(script)],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.count("ok") == 2


def test_reference_arm_prints_the_contract_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--clips-per-gpu", "8", "--dump-outputs", str(tmp_path / "dump")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "stft_frames_per_s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["n_fft"] == 2048
    assert line["config"]["clips_per_gpu"] == 8      # the CPU arm runs the GPU arm's batch, clip for clip
    # 8 clips x 858 frames is below the dump's row budget: every row of the timed step's output, in order
    import bench
    from oracle import analyser_oracle as O
    from oracle import cref
    dump = np.load(tmp_path / "dump" / "spectrogram.npy")
    want = cref.stft_batch(bench.synth_clips_cpu(8), O.Config(window=O.WINDOW_BLACKMAN, output=O.OUT_U8))
    assert dump.dtype == np.float32 and np.array_equal(dump, want.reshape(-1, 1024))


@pytest.mark.gpu
def test_gpu_arm_times_the_given_steps_and_dumps_the_same_outputs_every_run(tmp_path):
    import json
    from oracle import analyser_oracle as O
    from _tol import assert_bytes_close
    lines, dumps = [], []
    for run in range(2):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--clips-per-gpu", "8",
                            "--e2e-clips", "0", "--no-cpu-baseline", "--no-configs", "--dump-outputs", str(tmp_path / str(run))],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
        dumps.append(np.load(tmp_path / str(run) / "spectrogram.npy"))
    assert lines[0]["steps"] == 3 and lines[0]["gpu_launches"] == 3      # one launch per step
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (8 * 858, 1024)   # every row: 8 clips are below the budget
    assert np.array_equal(dumps[0], dumps[1])
    import bench
    ref = O.spectrogram(bench.synth_clips_cpu(1, first_clip=7)[0], O.Config())[0]
    assert_bytes_close(dumps[0][7 * 858:], ref)


def test_dump_is_a_fixed_sample_of_whole_rows_within_64_mb(tmp_path):
    import torch
    import bench
    n = 40000                                    # rows: more than the dump keeps; each row holds its own index
    out = torch.arange(n, dtype=torch.int32)[:, None].expand(n, 1024).reshape(40, 1000, 1024)
    bench.dump_outputs(str(tmp_path / "a"), out)
    bench.dump_outputs(str(tmp_path / "b"), out)
    a, b = np.load(tmp_path / "a" / "spectrogram.npy"), np.load(tmp_path / "b" / "spectrogram.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_ROWS, 1024) and a.nbytes <= 64 << 20
    assert np.array_equal(a, b)
    rows = a[:, 0]
    assert np.all(a == rows[:, None]) and np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < n
