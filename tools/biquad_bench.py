#!/usr/bin/env python
"""Biquad filter on the GPU (sg_biquad_filter_device) against a device-to-device cudaMemcpyAsync of the same in + out
bytes, timed alternately in one process with CUDA events, and the streaming bank's push latency (BASELINE config 5:
256 channels, n_fft 1024, hop 128, 128-sample pushes) with and without a bandpass attached.  Writes one JSON line per
measurement to --out (default profiles/r05_biquad_bench.jsonl), each with the card's name and power limit read in the
same run.  Needs a GPU: without one it fails."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = (s.strip() for s in q[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_biquad_bench.jsonl"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--pushes", type=int, default=2000)
    args = ap.parse_args()
    import torch
    import spectrogram_b200 as sg
    info = card()
    eng = sg.Engine(0)
    node = sg.BiquadFilterNode(eng, sample_rate=48000)
    node.type, node.Q.value, node.frequency.value = "bandpass", 10.0, 1000.0
    # a stream of its own: handle 0 (torch's legacy default stream) would mean "the engine's stream" to the library,
    # and the events would then time only the enqueue
    stream = torch.cuda.Stream()
    rows = []
    for name, ch, n in (("256ch_60s_48k", 256, 60 * 48000), ("1ch_1h_48k", 1, 3600 * 48000), ("4096ch_30s_16k", 4096, 30 * 16000)):
        x = torch.randn(ch, n, device="cuda", dtype=torch.float32)
        y = torch.empty_like(x)
        state = torch.zeros(ch, 4, device="cuda", dtype=torch.float64)
        torch.cuda.synchronize()
        nbytes = x.numel() * 4

        def filt():
            eng.biquad_device(node, x.data_ptr(), ch, n, n, y.data_ptr(), n, state.data_ptr(), stream.cuda_stream)

        def copy():
            with torch.cuda.stream(stream):
                y.copy_(x)
        for f in (filt, copy):   # warm-up
            f()
        torch.cuda.synchronize()
        t = {"filter": [], "copy": []}
        for _ in range(args.reps):
            for key, f in (("filter", filt), ("copy", copy)):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                f()
                b.record(stream)
                b.synchronize()
                t[key].append(a.elapsed_time(b))
        kf, kc = float(np.median(t["filter"])), float(np.median(t["copy"]))
        rows.append(dict(info, kind="kernel_vs_copy", shape=name, channels=ch, samples=n, filter_ms=kf, copy_ms=kc,
                         filter_gbps=2 * nbytes / kf / 1e6, copy_gbps=2 * nbytes / kc / 1e6, ratio_of_copy_rate=kc / kf,
                         launches=3 if n > 4096 else 1, reps=args.reps))
        print(json.dumps(rows[-1]), flush=True)
        del x, y, state
        torch.cuda.empty_cache()
    opts = sg.Options(fftSize=1024, hop=128, output="u8")
    chunk = (0.1 * np.random.default_rng(0).standard_normal((256, 128))).astype(np.float32)
    pin = sg.PinnedArray((256, 128), np.float32)
    pin.array[:] = chunk
    out = sg.PinnedArray((256, 1, 512), np.uint8)
    for label, filt in (("no_filter", None), ("bandpass", node)):
        bank = sg.StreamBank(256, opts, max_chunk=128, engine=eng, filter=filt)
        for _ in range(100):
            bank.push(pin.array, out=out.array)
        lat = []
        for _ in range(args.pushes):
            t0 = time.perf_counter()
            bank.push(pin.array, out=out.array)
            lat.append((time.perf_counter() - t0) * 1e6)
        bank.close()
        rows.append(dict(info, kind="push_latency", config="cfg5_256ch_n1024_hop128_chunk128", filter=label,
                         p50_us=float(np.percentile(lat, 50)), p99_us=float(np.percentile(lat, 99)), pushes=args.pushes))
        print(json.dumps(rows[-1]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
