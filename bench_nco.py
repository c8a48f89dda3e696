"""The phase-accumulator NCO on one B200 (DESIGN.md section 15): what C5 and the band scan cost with each mixer.

    c5        WidebandReceiver, 100 stations on the 200 kHz raster of one 50 MS/s capture, u8 and cs16, mixers osc,
              freqshift and nco (then freqshift and nco again, for the spread), ms per demodulator call (2 048 000
              capture samples), K calls after W of warm-up, CUDA events around the calls
    offgrid   the nco receiver with the same 100 stations moved 12 345.6 Hz off the raster (not phase-coherent with
              32000-sample blocks, so freqshift cannot take them), u8
    scan      the band scan of 24 calls (0.98 s) of the same u8 capture, mixers osc and nco: wall time of the blocking
              run and its confirmation stage (rfm_scan_timing), the second of two runs
    device    name and power limit (read-only nvidia-smi query)

Prints one JSON line.  usage: python bench_nco.py [--calls K]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import time

import numpy as np

from __graft_entry__ import load_package
from bench_iq_formats import BLK5, BPC5, FREQS5, FS5, N_CALL5, convert

OFFGRID = 12345.6


def bench_c5(torch, wb_mod, cap, fmt, freqs, mixer, K, W, ncalls):
    esz = {"u8": 2, "s16": 4}[fmt]
    wb = wb_mod.WidebandReceiver(torch, freqs, FS5, BLK5, BPC5, mixer=mixer, device=0, input_format=fmt)
    for i in range(W):
        wb.process_device(cap.data_ptr() + esz * (i % ncalls) * N_CALL5)
    wb.wait()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        wb.process_device(cap.data_ptr() + esz * ((W + i) % ncalls) * N_CALL5)
    wb.wait()
    e1.record()
    torch.cuda.synchronize()
    wb.close()
    return round(e0.elapsed_time(e1) / K, 3)


def bench_scan(torch, rfm, cap, mixer):
    s = rfm.BandScan(FS5, -24.9e6, 100e3, 499, device=0, mixer=mixer)
    s.run(cap)          # first run: module load and allocations
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s.run(cap)
    wall = (time.perf_counter() - t0) * 1e3
    spec_ms, conf_ms = s.timing()
    st = s.stations()
    s.close()
    return {"run_ms": round(wall, 1), "confirm_ms": round(conf_ms, 1), "confirm_ms_per_call": round(conf_ms / 24, 3),
            "spectrum_ms": round(spec_ms, 3), "stations": len(st), "stereo": sum(d["stereo"] for d in st),
            "with_ps": sum(d["ps"] != "" for d in st)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    import importlib
    import torch
    rfm = load_package()
    synth_device = importlib.import_module("radiofm_b200.synth_device")
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res = {"device": q.stdout.strip() or "unknown"}
    dev = torch.device("cuda", 0)
    K, W, ncalls = args.calls, 3, 4
    u8 = synth_device.make_wideband_u8(torch, FS5, 24 * N_CALL5, FREQS5, dev)
    c5 = {}
    for fmt in ("u8", "s16"):
        cap = convert(torch, u8[:ncalls * N_CALL5], fmt).contiguous()
        for label, mixer in (("osc", "osc"), ("freqshift", "freqshift"), ("nco", "nco"), ("freqshift_again", "freqshift"),
                             ("nco_again", "nco")):
            c5[f"{fmt}_{label}_ms_per_call"] = bench_c5(torch, wb_mod, cap, fmt, FREQS5, mixer, K, W, ncalls)
        del cap
    res["c5"] = c5
    off = [f + OFFGRID for f in FREQS5]
    res["offgrid"] = {"u8_nco_ms_per_call": bench_c5(torch, wb_mod, u8, "u8", off, "nco", K, W, ncalls)}
    torch.cuda.synchronize()
    res["scan"] = {m: bench_scan(torch, rfm, u8, m) for m in ("osc", "nco")}
    print(json.dumps(res))


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
