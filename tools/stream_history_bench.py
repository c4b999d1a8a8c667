"""Cost of the streaming bank's sonogram history (sg_stream_set_history / sg_stream_view) at BASELINE config 5
(256 channels, n_fft 1024, hop 128, one 128-sample chunk per push).  One JSON line per case, on stdout and appended to
--out; the card's name and power limit are read in the same run and written into every line.

  push     push latency p50/p99 of a bank without a history, one with a 256-row history (rows still returned), and
           the same history bank pushing without rows (advance); the three alternate push by push in one process
  refresh  one picture refresh of all 256 channels: bank.view (one launch, one copy) against the host loop a client
           needs without it (per channel SonogramRing.append of the pushed row, then SonogramRing.view), on the same
           rows; both outputs are compared
  kernel   (--profile, a run of its own) device time of sonogram_views_kernel from torch.profiler's CUDA activity

  python tools/stream_history_bench.py [--pushes 3000] [--refreshes 20] [--out FILE] [--profile]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spectrogram_b200 as sg  # noqa: E402

CH, NFFT, HOP, ROWS = 256, 1024, 128, 256
SIZES = ((256, 128), (512, 256))


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


def pct(v):
    v = np.sort(np.asarray(v))
    return {"p50_us": round(float(v[len(v) // 2]), 2), "p99_us": round(float(v[int(len(v) * 0.99)]), 2),
            "mean_us": round(float(v.mean()), 2), "n": int(v.size)}


def banks(eng):
    opts = sg.Options(fftSize=NFFT, hop=HOP, output="u8")
    return sg.StreamBank(CH, opts, max_chunk=HOP, engine=eng), sg.StreamBank(CH, opts, max_chunk=HOP, engine=eng,
                                                                             history_rows=ROWS)


def chunks(n, seed=0):
    rng = np.random.default_rng(seed)
    chunk = sg.PinnedArray((CH, HOP), np.float32)
    base = (0.1 * rng.standard_normal((CH, HOP * 64))).astype(np.float32)
    for i in range(n):
        chunk.array[...] = base[:, (i % 64) * HOP:(i % 64 + 1) * HOP]
        yield chunk.array


def push_case(eng, n, base, out):
    plain, hist = banks(eng)
    rows = sg.PinnedArray((CH, 1, NFFT // 2), np.uint8)
    lat = {"no_history": [], "history": [], "history_no_rows": []}

    def timed(key, fn):
        t0 = time.perf_counter()
        fn()
        lat[key].append((time.perf_counter() - t0) * 1e6)

    for i, x in enumerate(chunks(n + 100)):
        keep = i >= 100                                     # the first 100 rounds warm up
        for key, fn in (("no_history", lambda: plain.push(x, out=rows.array)),
                        ("history", lambda: hist.push(x, out=rows.array)),
                        ("history_no_rows", lambda: hist.advance(x))):
            if keep:
                timed(key, fn)
            else:
                fn()
    for key, v in lat.items():
        emit(dict(base, case="push", variant=key, channels=CH, n_fft=NFFT, hop=HOP, chunk=HOP,
                  history_rows=0 if key == "no_history" else ROWS, **pct(v)), out)
    plain.close()
    hist.close()


def refresh_case(eng, reps, base, out):
    _, hist = banks(eng)
    rings = [sg.SonogramRing(NFFT // 2, ROWS, engine=eng) for _ in range(CH)]
    rows = sg.PinnedArray((CH, 1, NFFT // 2), np.uint8)
    feed = chunks(ROWS + 20 + reps * 2 * len(SIZES))
    for _ in range(ROWS + 20):                              # fill and wrap every texture
        hist.push(next(feed), out=rows.array)
        for c in range(CH):
            rings[c].append(rows.array[c])
    for w, h in SIZES:
        pinned = sg.PinnedArray((CH, h, w, 4), np.uint8)
        host = [np.empty((h, w, 4), np.uint8) for _ in range(CH)]
        t_bank, t_bank_pageable, t_loop = [], [], []
        hist.view(w, h, out=pinned.array)                  # warm the shape
        for _ in range(reps):
            hist.push(next(feed), out=rows.array)
            t0 = time.perf_counter()
            for c in range(CH):                            # the client loop without a device-side history
                rings[c].append(rows.array[c])
                rings[c].view(w, h, out=host[c])
            t_loop.append((time.perf_counter() - t0) * 1e6)
            t0 = time.perf_counter()
            hist.view(w, h, out=pinned.array)
            t_bank.append((time.perf_counter() - t0) * 1e6)
            t0 = time.perf_counter()
            pageable = hist.view(w, h)
            t_bank_pageable.append((time.perf_counter() - t0) * 1e6)
        same = bool(np.array_equal(np.stack(host), pinned.array) and np.array_equal(pageable, pinned.array))
        # 4 bytes per pixel leave the device once for bank.view; the loop also sends each row up and its picture down
        mb = CH * w * h * 4 / 1e6
        for variant, v in (("bank.view pinned out", t_bank), ("bank.view pageable out", t_bank_pageable),
                           ("host loop ring.append + ring.view", t_loop)):
            emit(dict(base, case="refresh", variant=variant, channels=CH, width=w, height=h, image_mb=round(mb, 2),
                      identical_to_rings=same, **pct(v)), out)
        pinned.free()
    for r in rings:
        r.close()
    hist.close()


def kernel_case(eng, reps, base, out, trace_dir):
    from torch.profiler import ProfilerActivity, profile
    _, hist = banks(eng)
    for x in chunks(ROWS + 20):
        hist.advance(x)
    for w, h in SIZES:
        pinned = sg.PinnedArray((CH, h, w, 4), np.uint8)
        for _ in range(5):
            hist.view(w, h, out=pinned.array)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                hist.view(w, h, out=pinned.array)
        ev = [e for e in prof.events() if "sonogram_views_kernel" in e.name]
        dur = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in ev]
        if trace_dir:
            prof.export_chrome_trace(os.path.join(trace_dir, f"stream_views_{w}x{h}.json"))
        px = CH * w * h
        rec = dict(base, case="kernel", kernel="sonogram_views_kernel", channels=CH, width=w, height=h,
                   launches_seen=len(dur), source="torch.profiler CUDA activity")
        if dur:
            us = float(np.median(dur))
            rec.update(median_us=round(us, 2), min_us=round(float(np.min(dur)), 2),
                       store_gb_per_s=round(px * 4 / (us * 1e-6) / 1e9, 1), gpixel_per_s=round(px / (us * 1e-6) / 1e9, 2))
        emit(rec, out)
        pinned.free()
    hist.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pushes", type=int, default=3000)
    ap.add_argument("--refreshes", type=int, default=20)
    ap.add_argument("--out", default=os.path.join("profiles", "r04_stream_history.jsonl"))
    ap.add_argument("--profile", action="store_true", help="only the kernel case, under torch.profiler")
    ap.add_argument("--trace-dir", default=None)
    a = ap.parse_args()
    name, power = card()
    base = {"gpu": name, "power_limit": power}
    eng = sg.Engine(0)
    if a.profile:
        kernel_case(eng, a.refreshes, base, a.out, a.trace_dir)
    else:
        push_case(eng, a.pushes, base, a.out)
        refresh_case(eng, a.refreshes, base, a.out)
    eng.close()


if __name__ == "__main__":
    main()
