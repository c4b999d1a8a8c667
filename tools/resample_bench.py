"""Fused ingest + resampling kernel against the plain ingest kernel on the same device-resident bytes, and the whole
host path (sg_stft_pcm_resampled against sg_stft_pcm).  One JSON line per case, on stdout and appended to --out.

Inputs are larger than L2 (126 MB): by default 256 clips x 30 s of s16 stereo, so every timed pass reads its bytes
from HBM.  Kernel cases alternate resample / ingest launches in one process and time each with CUDA events.
Algorithmic bytes: the PCM bytes read + 4 bytes per output sample per plane written.

  python tools/resample_bench.py [--clips 256] [--seconds 30] [--reps 20] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spectrogram_b200 as sg  # noqa: E402
from spectrogram_b200 import _lib as L  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def kernel_case(eng, lib, in_rate, out_rate, mix, clips, seconds, reps, base):
    channels, frames = 2, int(in_rate * seconds)
    planes = 1 if mix else channels
    layout = L.PCM_MONO_MIX if mix else L.PCM_PLANAR
    n_out = sg.resample_num_frames(frames, in_rate, out_rate)
    src = torch.randint(-32768, 32768, (clips * frames * channels,), dtype=torch.int16, device="cuda")
    dst_rs = torch.empty((clips * planes, n_out), dtype=torch.float32, device="cuda")
    dst_in = torch.empty((clips * planes, frames), dtype=torch.float32, device="cuda")
    info = L.PcmInfo(L.PCM_S16, channels, in_rate, frames, 0)
    stream = torch.cuda.Stream()            # a stream of our own: a null handle would mean the engine's stream
    st = stream.cuda_stream
    torch.cuda.synchronize()

    def resample():
        L.check(lib.sg_pcm_ingest_resampled_device(eng.handle, C.c_void_p(src.data_ptr()), clips, C.byref(info), layout,
                                                   out_rate, C.c_void_p(dst_rs.data_ptr()), n_out, C.c_void_p(st)))

    def ingest():
        L.check(lib.sg_pcm_ingest_device(eng.handle, C.c_void_p(src.data_ptr()), clips, C.byref(info), layout,
                                         C.c_void_p(dst_in.data_ptr()), frames, C.c_void_p(st)))

    for f in (resample, ingest, resample, ingest):
        f()
    torch.cuda.synchronize()
    times = {"resample": [], "ingest": []}
    for _ in range(reps):
        for name, f in (("resample", resample), ("ingest", ingest)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            f()
            e1.record(stream)
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e-3)
    in_bytes = clips * frames * channels * 2
    rs_t, in_t = float(np.median(times["resample"])), float(np.median(times["ingest"]))
    rs_out, in_out = clips * planes * n_out, clips * planes * frames
    rec = dict(base, case="kernel", in_rate=in_rate, out_rate=out_rate, layout="mono_mix" if mix else "planar", clips=clips,
               seconds=seconds, in_bytes=in_bytes, reps=reps,
               resample_ms=rs_t * 1e3, resample_ms_min=min(times["resample"]) * 1e3,
               resample_out_frames_per_s=rs_out / rs_t, resample_bytes_per_s=(in_bytes + 4 * rs_out) / rs_t,
               ingest_ms=in_t * 1e3, ingest_ms_min=min(times["ingest"]) * 1e3,
               ingest_out_frames_per_s=in_out / in_t, ingest_bytes_per_s=(in_bytes + 4 * in_out) / in_t)
    rec["out_frames_ratio"] = rec["resample_out_frames_per_s"] / rec["ingest_out_frames_per_s"]
    del src, dst_rs, dst_in
    torch.cuda.empty_cache()
    return rec


def e2e_case(eng, clips, seconds, reps, base):
    in_rate, out_rate, channels = 44100, 48000, 2
    frames = int(in_rate * seconds)
    rng = np.random.default_rng(0)
    raw = rng.integers(-32768, 32768, clips * frames * channels, dtype=np.int64).astype("<i2")
    opts = sg.Options(fftSize=2048, hop=512, output="u8")

    def run(resampled):
        t0 = time.perf_counter()
        if resampled:
            eng.spectrogram_pcm(raw, "s16", channels, n_clips=clips, mix=True, opts=opts, sample_rate=in_rate, context_rate=out_rate)
        else:
            eng.spectrogram_pcm(raw, "s16", channels, n_clips=clips, mix=True, opts=opts)
        return time.perf_counter() - t0

    run(True), run(False)
    t = {"resampled": [], "plain": []}
    for _ in range(reps):
        t["resampled"].append(run(True))
        t["plain"].append(run(False))
    rs, pl = float(np.median(t["resampled"])), float(np.median(t["plain"]))
    return dict(base, case="e2e_stft_pcm", in_rate=in_rate, out_rate=out_rate, layout="mono_mix", clips=clips, seconds=seconds,
                n_fft=2048, hop=512, output="u8", in_bytes=raw.nbytes, reps=reps,
                stft_pcm_resampled_s=rs, stft_pcm_s=pl, resampled_in_bytes_per_s=raw.nbytes / rs, plain_in_bytes_per_s=raw.nbytes / pl,
                resampled_out_frames_per_s=clips * sg.resample_num_frames(frames, in_rate, out_rate) / rs,
                plain_out_frames_per_s=clips * frames / pl)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--e2e-clips", type=int, default=64)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resample_bench needs a CUDA device")
    name, power = card()
    base = {"card": name, "power_limit": power}
    eng = sg.Engine(0)
    lib = L.load()
    for in_rate, out_rate, mix in ((44100, 48000, True), (44100, 48000, False), (48000, 16000, True), (192000, 11025, True)):
        clips = max(1, int(a.clips * 44100 / in_rate))          # about the same input bytes in every case
        emit(kernel_case(eng, lib, in_rate, out_rate, mix, clips, a.seconds, a.reps, base), a.out)
    emit(e2e_case(eng, a.e2e_clips, a.seconds, a.e2e_reps, base), a.out)
    eng.close()


if __name__ == "__main__":
    main()
