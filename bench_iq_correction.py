"""IQ correction on one B200 (DESIGN.md section 14): what the estimate and the corrected conversion cost.

    estimate  rfm_iq_estimate over 1 s at 50 MS/s (50 M samples, device input) in u8 / s8 / s16 / cf32: wall time of
              the blocking call (statistics pass, scratch allocation, read-back of the five sums), best and median of
              10 after 2 of warm-up, and the input bytes over the best time
    c5        WidebandReceiver, 100 stations of one 50 MS/s cs8 capture, mixers freqshift and osc, ms per demodulator
              call (2 048 000 capture samples), without / with / without correction in one job
    scan      the band scan's spectrum stage (rfm_scan_timing), 100 stations, 24 calls (0.98 s at 50 MS/s) of cs8:
              correction off, fixed (mode 2) and estimated per run (mode 1: the statistics pass is inside the stage)
    device    name and power limit (read-only nvidia-smi query)

Prints one JSON line.  usage: python bench_iq_correction.py [--calls K]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import time

import numpy as np

from __graft_entry__ import load_package
from bench_iq_formats import BLK5, BPC5, FREQS5, FS5, N_CALL5, convert


def bench_estimate(torch, rfm, synth_device):
    dev = torch.device("cuda", 0)
    n = int(FS5)
    u8 = synth_device.make_wideband_u8(torch, FS5, n, FREQS5, dev)
    out = {}
    for fmt in ("u8", "s8", "s16", "cf32"):
        cap = convert(torch, u8, fmt).contiguous()
        torch.cuda.synchronize()
        ts = []
        for i in range(12):
            t0 = time.perf_counter()
            c = rfm.estimate_iq_correction(cap)
            t1 = time.perf_counter()
            if i >= 2:
                ts.append((t1 - t0) * 1e3)
        best = min(ts)
        nbytes = n * rfm.iq_format_bytes(fmt)
        out[fmt] = {"best_ms": round(best, 4), "median_ms": round(float(np.median(ts)), 4),
                    "input_mb": round(nbytes / 1e6, 1), "gb_per_s_at_best": round(nbytes / (best * 1e-3) / 1e9, 1),
                    "coefficients": [float(c.dc_i), float(c.dc_q), float(c.a), float(c.b)]}
        del cap
        torch.cuda.empty_cache()
    return out


def bench_c5(torch, rfm, synth_device, K, W):
    wb_mod = __import__("radiofm_b200.wideband", fromlist=["WidebandReceiver"])
    dev = torch.device("cuda", 0)
    ncalls = 4
    cap = convert(torch, synth_device.make_wideband_u8(torch, FS5, ncalls * N_CALL5, FREQS5, dev), "s8").contiguous()
    corr = rfm.estimate_iq_correction(cap)
    out = {}
    for mixer in ("freqshift", "osc"):
        for label, c in (("off", None), ("corrected", corr), ("off_again", None)):
            wb = wb_mod.WidebandReceiver(torch, FREQS5, FS5, BLK5, BPC5, mixer=mixer, device=0, input_format="s8",
                                         iq_correction=c)
            for i in range(W):
                wb.process_device(cap.data_ptr() + 2 * (i % ncalls) * N_CALL5)
            wb.wait()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(K):
                wb.process_device(cap.data_ptr() + 2 * ((W + i) % ncalls) * N_CALL5)
            wb.wait()
            e1.record()
            torch.cuda.synchronize()
            out[f"{mixer}_{label}_ms_per_call"] = round(e0.elapsed_time(e1) / K, 3)
            wb.close()
    return out


def bench_scan(torch, rfm, synth_device):
    dev = torch.device("cuda", 0)
    cap = convert(torch, synth_device.make_wideband_u8(torch, FS5, 24 * N_CALL5, FREQS5, dev), "s8").contiguous()
    torch.cuda.synchronize()
    corr = rfm.estimate_iq_correction(cap)
    out = {}
    for label, c in (("off", None), ("fixed", corr), ("estimate", "estimate"), ("off_again", None)):
        s = rfm.BandScan(FS5, -24.9e6, 100e3, 499, device=0, iq_correction=c)
        s.run(cap)        # first run: module load and allocations
        s.run(cap)
        spec_ms, conf_ms = s.timing()
        out[label] = {"spectrum_ms": round(spec_ms, 4), "stations": len(s.stations())}
        s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    import importlib
    import torch
    rfm = load_package()
    synth_device = importlib.import_module("radiofm_b200.synth_device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res = {"device": q.stdout.strip() or "unknown"}
    res["estimate"] = bench_estimate(torch, rfm, synth_device)
    res["c5"] = bench_c5(torch, rfm, synth_device, args.calls, 3)
    res["scan"] = bench_scan(torch, rfm, synth_device)
    print(json.dumps(res))


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
