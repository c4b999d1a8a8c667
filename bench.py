#!/usr/bin/env python
"""bench.py -- headline benchmark of the frame-producing hot path (BASELINE.json metric:
STFT frames/s & audio-sec/s at n_fft 2048 / hop 512, HBM GB/s fraction).

A "step" is one pass of the fused window -> real FFT -> |X|^2 -> dB -> byte kernel over one batch of
synthetic clips (config 1's shape tiled to a batch, SURVEY.md 8(d)): CLIPS_PER_GPU clips x 10 s x
44.1 kHz, n_fft 2048, hop 512, Blackman (the AnalyserNode window), u8 output.

  python bench.py [--gpus N] [--steps K] [--warmup W]          this repo's CUDA path
  python bench.py ... --dump-outputs DIR                        also writes a seeded sample of the last timed step's
                                                               output to DIR/spectrogram.npy (float32, rank 0)
  python bench.py --impl reference ...                          the CPU arm (oracle port, all host threads)
  torchrun ... bench.py --gpus N ...                            one rank per GPU, clips sharded, no collective
                                                               on the data path (shards are independent)
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_FFT, HOP, SR = 2048, 512, 44100
CLIP_LEN = 441000            # 10 s at 44.1 kHz (BASELINE config 1)
CLIPS_PER_GPU = 512          # 903 MB of float32 input per step: far larger than the 126 MB L2
BYTES_PER_FRAME = 4 * HOP + 1 * (N_FFT // 2)   # algorithmic: each input sample once + one byte per bin = 3072
FALLBACK_HBM_GBS = 6650.0    # B200_PROFILING.md fallback, used only if MEASURED_PEAKS.json is absent


# ------------------------------------------------------------------------------------------------
# multi-rank plumbing (also exercised on CPU/gloo by tests/test_host_logic.py)
# ------------------------------------------------------------------------------------------------
def shard_plan(total_clips: int, world: int, rank: int) -> dict:
    """Contiguous block of clips for this rank (SURVEY 8(e)): clip i -> rank floor(i*world/total)."""
    lo, hi = total_clips * rank // world, total_clips * (rank + 1) // world
    return {"lo": lo, "hi": hi, "n_clips": hi - lo}


def _dist():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


def max_over_ranks(value: float, device="cuda") -> float:
    import torch
    d = _dist()
    if d is None:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    d.all_reduce(t, op=d.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value: float, device="cuda") -> float:
    import torch
    d = _dist()
    if d is None:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    d.all_reduce(t, op=d.ReduceOp.SUM)
    return float(t.item())


def barrier():
    d = _dist()
    if d is not None:
        d.barrier()


# ------------------------------------------------------------------------------------------------
# clocks: sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.005)

    def start(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self) -> dict | None:
        if self._thread is None:
            return None
        self._stop.set()
        self._thread.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/analyser_ref.c) on the host cores
# ------------------------------------------------------------------------------------------------
def synth_clips_cpu(n_clips: int, first_clip: int = 0):
    """Same family as the GPU batch: linear chirp 20 Hz -> 20 kHz, amplitude 0.5, plus per-clip phase
    (sin(base + ph) expanded so the transcendental work is done once, not once per clip)."""
    import numpy as np
    t = np.arange(CLIP_LEN, dtype=np.float64) / SR
    dur = CLIP_LEN / SR
    base = 2 * np.pi * (20.0 * t + 0.5 * (20000.0 - 20.0) / dur * t * t)
    sb, cb = 0.5 * np.sin(base), 0.5 * np.cos(base)
    out = np.empty((n_clips, CLIP_LEN), dtype=np.float32)
    for c in range(n_clips):
        ph = 0.37 * (first_clip + c)
        out[c] = (sb * np.cos(ph) + cb * np.sin(ph)).astype(np.float32)
    return out


def cpu_arm(x, steps: int, warmup: int, threads: int = 0) -> dict:
    """Times the oracle's C port (oracle/analyser_ref.c, float32, Chromium's arithmetic widths) on `x` [clips, CLIP_LEN]
    with `threads` host threads (0 = all)."""
    from oracle import analyser_oracle as O
    from oracle import cref
    cores = cref.max_threads() if threads == 0 else threads
    n_clips = x.shape[0]
    cfg = O.Config(n_fft=N_FFT, hop=HOP, window=O.WINDOW_BLACKMAN, output=O.OUT_U8)
    frames = O.num_frames(CLIP_LEN, N_FFT, HOP, O.ALIGN_VALID) * n_clips
    for _ in range(warmup):
        cref.stft_batch(x, cfg, threads)
    times = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        y = cref.stft_batch(x, cfg, threads)
        times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return {"value": frames / dt, "unit": "frames/s", "cores": cores, "kind": "port", "out": y,
            "sample": f"{n_clips} clips x 10 s x 44.1 kHz ({frames} frames) per step, {len(times)} steps, "
                      f"oracle/analyser_ref.c float32, {cores} thread{'s' if cores != 1 else ''}",
            "ms_per_step": dt * 1e3, "ms_min": min(times) * 1e3, "ms_max": max(times) * 1e3, "frames": frames}


def cpu_pocketfft_point(x, steps: int = 3) -> dict:
    """Second CPU point (SURVEY 8(d)): the same path vectorised over frames with numpy's pocketfft
    (float32 window multiply, rfft, |X|/N, 20 log10, truncating byte), one thread."""
    import numpy as np
    from oracle import analyser_oracle as O
    w = O.make_window(O.WINDOW_BLACKMAN, N_FFT).astype(np.float32)
    n_clips = x.shape[0]
    fpc = 1 + (CLIP_LEN - N_FFT) // HOP
    times = []
    for _ in range(steps + 1):
        t0 = time.perf_counter()
        for c in range(n_clips):
            fr = np.lib.stride_tricks.sliding_window_view(x[c], N_FFT)[::HOP][:fpc]
            spec = np.fft.rfft(fr * w, axis=-1)[:, :N_FFT // 2]
            mag = np.abs(spec) * np.float32(1.0 / N_FFT)
            with np.errstate(divide="ignore"):
                db = 20.0 * np.log10(mag)
            np.clip((255.0 / 70.0) * (db + 100.0), 0, 255).astype(np.uint8)
        times.append(time.perf_counter() - t0)
    dt = sum(times[1:]) / steps
    return {"value": n_clips * fpc / dt, "unit": "frames/s", "cores": 1, "kind": "numpy pocketfft (rfft over sliding frames)",
            "sample": f"{n_clips} clips, {steps} steps", "ms_per_step": dt * 1e3}


def cpu_baseline_block(x_all, steps: int) -> dict:
    """cpu_baseline of the bench line: all host threads on the SAME clips the GPU arm times, plus the single-thread
    figure (what a browser main thread does) and the pocketfft point on a 16-clip sample."""
    r = cpu_arm(x_all, steps=steps, warmup=1)
    out = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "ms_per_step", "ms_min", "ms_max")}
    small = x_all[:16]
    r1 = cpu_arm(small, steps=3, warmup=1, threads=1)
    out["single_thread"] = {k: r1[k] for k in ("value", "unit", "cores", "sample", "ms_per_step")}
    out["pocketfft"] = cpu_pocketfft_point(small)
    return out


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the CPU arm runs once per box
    n_clips = args.clips_per_gpu                  # the GPU arm's batch, clip for clip (same `config`)
    x = synth_clips_cpu(n_clips)
    r = cpu_arm(x, args.steps, args.warmup)
    if args.dump_outputs:
        import torch
        dump_outputs(args.dump_outputs, torch.from_numpy(r["out"]))
    line = {
        "impl": "reference", "metric": "stft_frames_per_s", "value": r["value"], "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "audio_s_per_s": r["value"] * HOP / SR,
        "config": workload_config(n_clips),
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "ms_min", "ms_max")},
        "e2e": {"value": r["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU arm: the oracle's C port of the AnalyserNode algorithm on all host threads (the reference's own "
                "implementation is the browser's, which cannot run here -- DESIGN.md)",
    }
    print(json.dumps(line), flush=True)


def workload_config(clips_per_gpu: int) -> dict:
    cfg = {
        "workload": "config 1 tiled: batch of 10 s mono 44.1 kHz chirps, n_fft 2048, hop 512, u8 dB bytes",
        "n_fft": N_FFT, "hop": HOP, "window": "blackman (AnalyserNode parity window)", "output": "u8",
        "min_db": -100, "max_db": -30, "smoothing": 0.0, "clips_per_gpu": clips_per_gpu, "clip_len": CLIP_LEN,
        "frames_per_clip": 1 + (CLIP_LEN - N_FFT) // HOP, "sharding": "contiguous clip blocks per rank, no collective",
        "l2": f"inputs larger than L2 ({clips_per_gpu * CLIP_LEN * 4 / 1e6:.0f} MB read per step, no flush needed)",
    }
    return cfg


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def synth_clips_gpu(torch, n_clips: int, first_clip: int, device):
    t = torch.arange(CLIP_LEN, dtype=torch.float64, device=device) / SR
    dur = CLIP_LEN / SR
    base = 2 * torch.pi * (20.0 * t + 0.5 * (20000.0 - 20.0) / dur * t * t)
    x = torch.empty((n_clips, CLIP_LEN), dtype=torch.float32, device=device)
    for c0 in range(0, n_clips, 32):
        c1 = min(n_clips, c0 + 32)
        ph = 0.37 * torch.arange(first_clip + c0, first_clip + c1, dtype=torch.float64, device=device)
        x[c0:c1] = (0.5 * torch.sin(base[None, :] + ph[:, None])).to(torch.float32)
    return x


DUMP_ROWS = 12288            # 48 MB as float32: under the 64 MB a dump may take


def dump_outputs(dirname: str, out, rows: int = DUMP_ROWS, seed: int = 0) -> None:
    """Writes `rows` output rows of `out` (all of them if it has fewer; [clip, frame] pairs drawn without replacement by a
    fixed seed, in flattened order) as float32 to dirname/spectrogram.npy, so that two builds run with the same arguments
    compare row for row."""
    import numpy as np
    import torch
    flat = out.reshape(-1, out.shape[-1])
    idx = np.sort(np.random.default_rng(seed).choice(flat.shape[0], min(rows, flat.shape[0]), replace=False))
    sample = flat[torch.from_numpy(idx).to(flat.device)].float().cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "spectrogram.npy"), sample)


def bind_near_gpu(index: int) -> str:
    """Pin this rank's host threads to the cores closest to its GPU (NVML's ideal CPU affinity), so the pinned
    staging buffers it allocates next are first-touched on that NUMA node.  Matters for the end-to-end number at
    4-8 GPUs, where every rank streams ~1.3 GB per step over PCIe."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return f"{len(os.sched_getaffinity(0))} cores"
    except Exception as e:  # no NVML / not permitted: run unbound
        return f"unbound ({type(e).__name__})"


def fp32_bound(clocks: dict, frames_per_s_per_gpu: float) -> dict:
    """The kernel's real ceiling (DESIGN.md): one frame pair costs 2430 FP32-pipe cycles on one of the 4 x 148
    schedulers (1064 packed FFMA2/FADD2 ops at 2 cycles + 300 scalar), counted from the SASS of
    stft_w32x2p_kernel and confirmed by tools/microbench/pipe_bench.cu (2.05 cycles per packed op)."""
    mhz = float(clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0)
    cap = 148 * 4 * mhz * 1e6 / 2430.0 * 2.0
    return {"cycles_per_frame_pair": 2430, "cap_frames_per_s": cap, "frac_of_cap": frames_per_s_per_gpu / cap,
            "cap_as_hbm_frac": cap * BYTES_PER_FRAME / 1e9 / 6551.4}


# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configs (2-5), driver-measured inside the same run: one entry each in `configs`
# ------------------------------------------------------------------------------------------------
L2_FLUSH_BYTES = 256 << 20


def timed_region(torch, fn, stream, dev_index: int, min_seconds: float = 0.12, flush_buf=None, max_steps: int = 400) -> dict:
    """W = 3 warm-up calls, then K calls timed with CUDA events on `stream` (K sized so the region lasts >= min_seconds,
    long enough for the NVML clock sampler).  flush_buf: inputs fit in L2 -> write a 256 MB buffer before every timed
    call and time each call with its own event pair."""
    for _ in range(3):
        fn()
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    stream.synchronize()
    est = max(e0.elapsed_time(e1) * 1e-3, 1e-6)
    steps = int(min(max_steps, max(5, -(-min_seconds // est))))
    sampler = ClockSampler(dev_index)
    sampler.start()
    if flush_buf is None:
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        stream.synchronize()
        ms = e0.elapsed_time(e1) / steps
    else:
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        with torch.cuda.stream(stream):
            for a, b in pairs:
                flush_buf.fill_(1)
                a.record(stream)
                fn()
                b.record(stream)
        stream.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in pairs) / steps
    clocks = sampler.stop()
    return {"ms": ms, "steps": steps, "clocks": clocks}


def measure_configs(torch, sg, eng, dev, stream, peak: float, quick: bool = False) -> dict:
    import numpy as np
    out = {}
    di = dev.index or 0
    gen = torch.Generator(device=dev).manual_seed(1234)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def entry(n_clips, clip_len, opts, sr, elem_bytes, dtype, flush_l2, sigma=0.1):
        # every entry starts from fresh device allocations: a tensor carved out of a block the caching allocator kept from
        # an earlier, larger entry can land where the same call runs 1.7x slower (measured: 64 x 60 s clips at n_fft 2048,
        # tau 0.8: 0.98 ms in fresh buffers, 1.7-1.8 ms in recycled ones; tools/bimodal_probe6.py)
        torch.cuda.empty_cache()
        frames = eng.num_frames(opts, clip_len)
        bins = opts.fftSize // 2
        x = (torch.randn((n_clips, clip_len), device=dev, generator=gen) * sigma).float()
        o = torch.empty((n_clips, frames, bins), dtype=dtype, device=dev)
        l0 = eng.launch_count

        def fn():
            eng.spectrogram_device(x.data_ptr(), n_clips, clip_len, clip_len, opts, o.data_ptr(), stream.cuda_stream)
        fn()
        launches = eng.launch_count - l0
        r = timed_region(torch, fn, stream, di, flush_buf=flush if flush_l2 else None)
        total = n_clips * frames
        bpf = 4 * opts.hop + elem_bytes * bins
        e = {"n_fft": opts.fftSize, "hop": opts.hop, "output": opts.output, "tau": opts.smoothingTimeConstant,
             "clips": n_clips, "clip_len": clip_len, "frames": total, "ms": r["ms"], "steps": r["steps"],
             "frames_per_s": total / r["ms"] * 1e3, "audio_s_per_s": total * opts.hop / sr / r["ms"] * 1e3,
             "bytes_per_frame": bpf, "frac": total * bpf / r["ms"] / 1e6 / peak, "kernel": eng.last_kernel,
             "launches_per_step": launches, "clocks": r["clocks"],
             "l2": "L2 flushed (256 MB write) before every timed call" if flush_l2 else "inputs larger than L2"}
        del x, o
        return e

    # the headline batch with smoothingTimeConstant 0.8 (AnalyserNode's default): the fused one-pass kernel
    out["config1_tau"] = entry(512, CLIP_LEN, sg.Options(fftSize=N_FFT, hop=HOP, output="u8", smoothingTimeConstant=0.8),
                               SR, 1, torch.uint8, False)
    # the same batch shape at the other sizes (hop n/4): their fused one-pass kernels (kernel_pair_s.cuh, kernel_w32eo_s.cuh, kernel_wreg_s.cuh)
    out["config1_tau_sizes"] = {str(n): entry(512, CLIP_LEN, sg.Options(fftSize=n, hop=n // 4, output="u8", smoothingTimeConstant=0.8),
                                              SR, 1, torch.uint8, False) for n in (256, 512, 1024, 4096, 8192)}
    # config 2: 1 h mono 16 kHz, n_fft 512, hop 160, float dB (Hann, as BASELINE.json names it)
    out["config2"] = entry(1, 16000 * (600 if quick else 3600), sg.Options(fftSize=512, hop=160, window="hann", output="db"),
                           16000, 4, torch.float32, False)
    # config 3 as named: 60 s stereo 48 kHz (two channels = two clips), smoothingTimeConstant 0.8, hop n/4, bytes
    out["config3"] = {str(n): entry(2, 48000 * 60, sg.Options(fftSize=n, hop=n // 4, output="u8", smoothingTimeConstant=0.8,
                                                                 align="analyser"), 48000, 1, torch.uint8, True)
                      for n in (256, 512, 1024, 2048, 4096, 8192)}
    # config 3b: the same sweep as a batch (64 channels, tau 0 and tau 0.8) -- where each size's kernel stands
    out["config3b"] = {str(n): entry(64, 48000 * 60, sg.Options(fftSize=n, hop=n // 4, output="u8"), 48000, 1, torch.uint8, False)
                       for n in (256, 512, 1024, 2048, 4096, 8192)}
    out["config3b_tau"] = {str(n): entry(64, 48000 * 60, sg.Options(fftSize=n, hop=n // 4, output="u8", smoothingTimeConstant=0.8),
                                         48000, 1, torch.uint8, False) for n in (1024, 2048)}
    # odd hop (441 samples = 10 ms at 44.1 kHz) against the aligned hop on the same clips
    out["hop441"] = {"hop441": entry(64, 441000, sg.Options(fftSize=2048, hop=441, output="u8"), 44100, 1, torch.uint8, False),
                     "hop512": entry(64, 441000, sg.Options(fftSize=2048, hop=512, output="u8"), 44100, 1, torch.uint8, False)}
    # config 4: 4096 x 30 s x 16 kHz, n_fft 400, hop 160, float dB
    out["config4"] = entry(512 if quick else 4096, 480000, sg.Options(fftSize=400, hop=160, window="hann", output="db"),
                           16000, 4, torch.float32, False)
    del flush
    torch.cuda.empty_cache()
    # config 5: 256 concurrent 48 kHz channels, n_fft 1024, hop 128, one render quantum per push, u8 + RGBA, host to host
    opts = sg.Options(fftSize=1024, hop=128, output="u8")
    bank = sg.StreamBank(256, opts, max_chunk=128, engine=eng)
    chunk = sg.PinnedArray((256, 128), np.float32)
    chunk.array[...] = (0.1 * np.random.default_rng(0).standard_normal((256, 128))).astype(np.float32)
    o8 = sg.PinnedArray((256, 1, 512), np.uint8)
    o32 = sg.PinnedArray((256, 1, 512, 4), np.uint8)
    for _ in range(50):
        bank.push(chunk.array, out=o8.array, out_rgba=o32.array)
    sampler = ClockSampler(di)
    sampler.start()
    lat = []
    l0 = eng.launch_count
    n_push = 300 if quick else 2000
    for _ in range(n_push):
        t0 = time.perf_counter()
        bank.push(chunk.array, out=o8.array, out_rgba=o32.array)
        lat.append((time.perf_counter() - t0) * 1e6)
    clocks = sampler.stop()
    lat = np.sort(np.array(lat))
    out["config5"] = {"channels": 256, "n_fft": 1024, "hop": 128, "outputs": "u8 + rgba8", "pushes": n_push,
                      "p50_us": float(lat[len(lat) // 2]), "p99_us": float(lat[int(len(lat) * 0.99)]),
                      "chunks_per_s": 1e6 / float(lat.mean()), "frames_per_s": 256 * 1e6 / float(lat.mean()),
                      "realtime_factor": (128 / 48000) / (float(lat.mean()) * 1e-6), "kernel": eng.last_kernel,
                      "launches_per_push": (eng.launch_count - l0) / n_push, "clocks": clocks,
                      "bytes_per_frame": 4 * 128 + 512 + 4 * 512, "timing": "host perf_counter around the synchronous push (H2D + kernels + 2 x D2H)"}
    bank.close()
    chunk.free(); o8.free(); o32.free()
    return out


def run_gpu(args) -> None:
    import numpy as np
    import torch

    import spectrogram_b200 as sg
    from spectrogram_b200 import _lib

    _lib.load()  # fails loudly if the CUDA library has not been built
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (this engine has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = bind_near_gpu(local) if world > 1 else "all cores"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    clips = args.clips_per_gpu
    plan = shard_plan(clips * world, world, rank)
    eng = sg.Engine(local)
    opts = sg.Options(fftSize=N_FFT, hop=HOP, window="blackman", output="u8")
    frames_per_clip = eng.num_frames(opts, CLIP_LEN)
    frames = frames_per_clip * plan["n_clips"]

    x = synth_clips_gpu(torch, plan["n_clips"], plan["lo"], dev)
    out = torch.empty((plan["n_clips"], frames_per_clip, N_FFT // 2), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)   # the kernels and the timing events share this stream

    def step():
        eng.spectrogram_device(x.data_ptr(), plan["n_clips"], CLIP_LEN, CLIP_LEN, opts, out.data_ptr(), stream.cuda_stream)

    # ---- device-resident timing: W warm-up steps, K timed steps between barriers + synchronize
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    torch.cuda.synchronize()
    barrier()
    ms_local = ev0.elapsed_time(ev1) / args.steps
    launches = eng.launch_count - launches0
    headline_kernel = eng.last_kernel
    clocks = sampler.stop()
    ms = max_over_ranks(ms_local, dev)
    total_frames = sum_over_ranks(frames, dev)
    value = total_frames / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)     # `out` still holds the last timed step's result

    # ---- parity spot check of what was just timed (rank 0, first clip) against the oracle
    parity = None
    if rank == 0:
        from oracle import analyser_oracle as O
        ref = O.spectrogram(x[0].cpu().numpy(), O.Config())[0]
        got = out[0].cpu().numpy()
        d = np.abs(ref.astype(np.int32) - got.astype(np.int32))
        parity = {"max_lsb": int(d.max()), "mismatch_frac": float((d != 0).mean()), "frames_checked": int(ref.shape[0])}
        if d.max() > 1:
            raise SystemExit(f"parity failure in the timed kernel: {parity}")

    # ---- the same kernel with float dB output (getFloatFrequencyData rows, 6144 algorithmic bytes per frame):
    #      secondary figure, rank 0 at N = 1 only; the headline above stays the byte output BASELINE.json names
    float_db = None
    if world == 1:
        opts_db = sg.Options(fftSize=N_FFT, hop=HOP, window="blackman", output="db")
        n_db = min(plan["n_clips"], 512)
        out_db = torch.empty((n_db, frames_per_clip, N_FFT // 2), dtype=torch.float32, device=dev)

        def step_db():
            eng.spectrogram_device(x.data_ptr(), n_db, CLIP_LEN, CLIP_LEN, opts_db, out_db.data_ptr(), stream.cuda_stream)

        for _ in range(3):
            step_db()
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record(stream)
        for _ in range(args.steps):
            step_db()
        d1.record(stream)
        torch.cuda.synchronize()
        ms_db = d0.elapsed_time(d1) / args.steps
        fps_db = n_db * frames_per_clip / (ms_db * 1e-3)
        float_db = {"value": fps_db, "unit": "frames/s", "ms_per_step": ms_db, "bytes_per_frame": 4 * HOP + 4 * (N_FFT // 2),
                    "achieved_gbs": fps_db * (4 * HOP + 4 * (N_FFT // 2)) / 1e9, "kernel": eng.last_kernel, "clips": n_db}
        del out_db
        step()                      # leave the engine on the byte kernel (last_kernel, parity check below)
        torch.cuda.synchronize()

    # ---- end to end through the public host API: pinned host buffers, H2D + kernel + D2H every step
    e2e = None
    e2e_clips = min(plan["n_clips"], args.e2e_clips)
    if e2e_clips > 0:
        pin_in = sg.PinnedArray((e2e_clips, CLIP_LEN), np.float32)
        pin_out = sg.PinnedArray((e2e_clips, frames_per_clip, N_FFT // 2), np.uint8)
        pin_in.array[...] = x[:e2e_clips].cpu().numpy()
        for _ in range(2):
            eng.spectrogram(pin_in.array, opts, out=pin_out.array)
        barrier()
        e2e_steps = max(2, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.spectrogram(pin_in.array, opts, out=pin_out.array)   # synchronous: returns when out is filled
        dt_local = (time.perf_counter() - t0) / e2e_steps
        barrier()
        dt = max_over_ranks(dt_local, dev)
        e2e_frames = sum_over_ranks(e2e_clips * frames_per_clip, dev)
        if rank == 0:
            assert np.array_equal(pin_out.array[0], out[0].cpu().numpy()), "host-API result differs from device-API result"
        # the copy-only ceiling of the same host path: the step's bytes moved with plain cudaMemcpyAsync, both directions
        # at once, every rank concurrently, no kernel (tools/host_path_ceiling.py)
        ceiling = None
        try:
            from tools import host_path_ceiling as hpc
            c = hpc.measure(dev, e2e_clips, 3, 4, barrier)
            t_both = max_over_ranks(c["t_both"], dev)
            ceiling = {"frames_per_s": e2e_frames / t_both, "ms_per_step": t_both * 1e3,
                       "h2d_gbs_per_gpu": c["h2d_bytes"] / max_over_ranks(c["t_h2d"], dev) / 1e9,
                       "d2h_gbs_per_gpu": c["d2h_bytes"] / max_over_ranks(c["t_d2h"], dev) / 1e9,
                       "aggregate_gbs": world * (c["h2d_bytes"] + c["d2h_bytes"]) / t_both / 1e9,
                       "how": "plain concurrent cudaMemcpyAsync H2D + D2H of the step's bytes between pinned host and device buffers, no kernel, all ranks at once"}
        except Exception as ex:  # the ceiling is a diagnostic, never a reason to lose the bench line
            ceiling = {"error": f"{type(ex).__name__}: {ex}"}
        e2e = {"value": e2e_frames / dt, "unit": "frames/s", "h2d_bytes_per_step": int(world * e2e_clips * CLIP_LEN * 4),
               "d2h_bytes_per_step": int(world * e2e_clips * frames_per_clip * (N_FFT // 2)), "ms_per_step": dt * 1e3,
               "api": "spectrogram_b200.Engine.spectrogram -> sg_stft_batch (pinned host in/out)",
               "host_affinity": affinity, "host_ceiling": ceiling,
               "frac_of_host_ceiling": (e2e_frames / dt) / ceiling["frames_per_s"] if ceiling and "frames_per_s" in ceiling else None}
        # secondary: the same clips as 16-bit PCM through sg_stft_pcm (ingest on the GPU, 2 bytes per sample over PCIe)
        if world == 1:
            from spectrogram_b200 import _lib as L
            import ctypes as C
            pin_s16 = sg.PinnedArray((e2e_clips, CLIP_LEN), np.int16)
            pin_s16.array[...] = np.clip(np.rint(pin_in.array * 32767.0), -32768, 32767).astype(np.int16)
            cfg_c, _keep = opts.to_c()
            info = L.PcmInfo(L.PCM_S16, 1, int(SR), CLIP_LEN, 0)
            lib = L.load()

            def pcm_step():
                L.check(lib.sg_stft_pcm(eng.handle, pin_s16.array.ctypes.data, e2e_clips, C.byref(info), L.PCM_MONO_MIX,
                                        C.byref(cfg_c), pin_out.array.ctypes.data))
            for _ in range(2):
                pcm_step()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                pcm_step()
            dt16 = (time.perf_counter() - t0) / e2e_steps
            e2e["pcm16_input"] = {"value": e2e_clips * frames_per_clip / dt16, "unit": "frames/s", "ms_per_step": dt16 * 1e3,
                                  "h2d_bytes_per_step": int(e2e_clips * CLIP_LEN * 2),
                                  "api": "sg_stft_pcm (16-bit mono PCM, pinned host in/out)"}
            pin_s16.free()
        pin_in.free()
        pin_out.free()

    if rank == 0:
        peak, peak_src = FALLBACK_HBM_GBS, "fallback"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peak, peak_src = float(json.load(f)["hbm_gbs"]), "measured"
        except Exception:
            pass
        achieved = frames * BYTES_PER_FRAME / (ms_local * 1e-3) / 1e9   # this rank's kernel: bytes per launch / launch time
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                tr = json.load(f)
                traffic = tr["dram_bytes_per_frame"] * frames
        except Exception:
            pass
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_block(x.cpu().numpy(), steps=5)     # the very clips the GPU arm timed
        configs = None
        if world == 1 and not args.no_configs:
            del out
            torch.cuda.empty_cache()
            configs = measure_configs(torch, sg, eng, dev, stream, peak, quick=args.quick_configs)
        line = {
            "metric": "stft_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "audio_s_per_s": value * HOP / SR,
            "config": workload_config(clips),
            "kernel": headline_kernel,
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "bytes_per_frame": BYTES_PER_FRAME,
                         "frames_per_launch": frames,
                         "fp32_pipe": fp32_bound(clocks, value / max(world, 1)),
                         "note": "co-bound by the FP32 pipe: 2430 FP32-pipe cycles per frame pair per scheduler cap the kernel at 43% of HBM peak (DESIGN.md)"},
            "cpu_baseline": cpu,
            "parity": parity,
            "configs": configs,
        }
        if float_db is not None:
            float_db["frac_of_hbm_peak"] = float_db["achieved_gbs"] / peak
            line["float_db_output"] = float_db
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips-per-gpu", type=int, default=CLIPS_PER_GPU)
    ap.add_argument("--e2e-clips", type=int, default=CLIPS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 2-5 block (N = 1 only anyway)")
    ap.add_argument("--quick-configs", action="store_true", help="smaller config 2 / 4 / 5 workloads (development)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's output to "
                                                          "DIR/spectrogram.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
