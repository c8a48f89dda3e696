#!/usr/bin/env python
"""bench_scan.py -- band scan (rfm_scan_*, BandScan) on the C5 capture: 100 FM stations on the 200 kHz raster of one
shared 50 MS/s u8 capture, `--calls` demodulator calls long (24 = 0.98 s), made on the device; raster 100 kHz from
-24.9 to +24.9 MHz.  One warm-up scan, then `--repeat` timed scans, then WidebandReceiver(mixer="osc") on the same 100
frequencies for the same calls, in the same job.  Prints one JSON line:

    spectrum_ms      k_scan_psd + k_scan_reduce (CUDA events), with the FFT rate 5 N log2 N flop per segment
    confirm_ms       front end + demodulator over every call (CUDA events), per call
    total_ms, rtf    wall time of the whole blocking scan (receiver creation included) and capture seconds / that
    wideband_osc     WidebandReceiver(osc) per call (host clock around synchronised calls)
    device           name and power limit (read-only nvidia-smi query)
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS, N_CALL, N = 50.0e6, 2048000, 4096


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=24)
    ap.add_argument("--stations", type=int, default=100)
    ap.add_argument("--repeat", type=int, default=3)
    args = ap.parse_args()

    import torch
    from __graft_entry__ import load_package
    rfm = load_package()
    sd = importlib.import_module("radiofm_b200.synth_device")
    wideband = importlib.import_module("radiofm_b200.wideband")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    freqs = [(k - args.stations // 2) * 200000.0 for k in range(args.stations)]
    n = args.calls * N_CALL
    cap = sd.make_wideband_u8(torch, FS, n, freqs, dev)
    torch.cuda.synchronize()

    s = rfm.BandScan(FS, -24.9e6, 100e3, 499, device=0)
    s.run_device(cap.data_ptr(), n)                       # warm-up
    found = len(s.stations())
    runs = []
    for _ in range(args.repeat):
        t0 = time.perf_counter()
        s.run_device(cap.data_ptr(), n)
        wall = (time.perf_counter() - t0) * 1e3
        runs.append((wall,) + s.timing())
    s.close()
    wall, spec_ms, conf_ms = (min(r[i] for r in runs) for i in range(3))
    n_seg = (n - N) // (N // 2) + 1
    flop = 5.0 * N * math.log2(N) * n_seg

    wb = wideband.WidebandReceiver(torch, freqs, FS, 32000, 64, mixer="osc", device=0)
    wb.process_device(cap.data_ptr())                     # warm-up call
    wb.wait()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for c in range(args.calls):
        wb.process_device(cap.data_ptr() + 2 * c * N_CALL)
    wb.wait()
    torch.cuda.synchronize()
    wb_ms = (time.perf_counter() - t0) * 1e3
    wb.close()

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(json.dumps({
        "workload": f"{args.stations} stations, {args.calls} calls x {N_CALL} samples at 50 MS/s ({n / FS:.3f} s)",
        "stations_found": found,
        "spectrum_ms": round(spec_ms, 4),
        "spectrum_gflops": round(flop / (spec_ms * 1e-3) / 1e9, 1),
        "spectrum_segments": n_seg,
        "confirm_ms": round(conf_ms, 2),
        "confirm_ms_per_call": round(conf_ms / args.calls, 3),
        "total_ms": round(wall, 2),
        "rtf": round(n / FS / (wall * 1e-3), 3),
        "spectrum_share_of_confirm": round(spec_ms / conf_ms, 5) if conf_ms else None,
        "wideband_osc_ms_per_call": round(wb_ms / args.calls, 3),
        "scan_over_wideband_per_call": round(conf_ms / wb_ms, 4),
        "runs_ms": [[round(v, 3) for v in r] for r in runs],
        "device": q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0),
    }))


if __name__ == "__main__":
    main()
