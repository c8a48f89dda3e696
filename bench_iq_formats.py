"""IQ input formats on one B200 (DESIGN.md section 13): the cost of each rfm_iq_format where the format is read.

    c4       the device-resident 4096-stream decoder step at 2.4 MS/s (downsample 11, 65472 samples per block), timed as
             bench.py times its value leg: K steps enqueued on one stream between two CUDA events, the decoder's wait()
             inside the window; u8 / s8 / s16 / cf32 rows of the same stations, 12 blocks resident in HBM
    c5       WidebandReceiver, 100 stations of one 50 MS/s capture, mixers freqshift and osc, ms per demodulator call
             (2 048 000 capture samples), u8 / s8 / s16
    scan     the band scan's spectrum stage (rfm_scan_timing), 100 stations, 24 calls (0.98 s at 50 MS/s), all four
    device   name and power limit (read-only nvidia-smi query)

Prints one JSON line.  usage: python bench_iq_formats.py [--steps K] [--calls K]
"""
from __future__ import annotations

import argparse
import json
import subprocess

import numpy as np

from __graft_entry__ import load_package

FS4, DS4, BLK4, S4 = 2.4e6, 11, 65472, 4096
FS5, BLK5, BPC5 = 50.0e6, 32000, 64
N_CALL5 = BLK5 * BPC5
FREQS5 = [(k - 50) * 200000.0 for k in range(100)]


def convert(torch, u8, fmt):
    """The same samples in each container (s8 = u - 128, s16 = 256 (u - 128), cf32 = u / 127.5 - 1)."""
    v = u8.to(torch.int16) - 128
    if fmt == "u8":
        return u8
    if fmt == "s8":
        return v.to(torch.int8)
    if fmt == "s16":
        return v * 256
    return u8.to(torch.float32) / 127.5 - 1.0


def bench_c4(torch, rfm, synth_device, K, W):
    dev = torch.device("cuda", 0)
    nres = 12
    u8 = synth_device.make_batch_u8(torch, S4, FS4, nres * BLK4, dev)
    out = {}
    for fmt in ("u8", "s8", "s16", "cf32", "u8"):
        iq = convert(torch, u8, fmt).contiguous()
        esz = rfm.iq_format_bytes(fmt)
        dec = rfm.FmDecoderBatch(FS4, -0.15 * FS4, downsample=DS4, n_streams=S4, max_block_len=BLK4, device=0)
        stride = dec.max_audio_floats(BLK4)
        audio = torch.zeros((S4, stride), dtype=torch.float32, device=dev)
        stream = torch.cuda.Stream()

        def step(i):
            b = i % nres
            return dec.process_iq_device(fmt, iq.data_ptr() + b * BLK4 * esz, nres * BLK4, BLK4, audio.data_ptr(),
                                         stride, stream.cuda_stream)

        with torch.cuda.stream(stream):
            for i in range(W):
                step(i)
            dec.wait(stream.cuda_stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for i in range(K):
                step(W + i)
            dec.wait(stream.cuda_stream)
            e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / K
        key = fmt if fmt not in out else fmt + "_again"
        out[key] = {"ms_per_step": round(ms, 4), "input_gb_per_step": round(S4 * BLK4 * esz / 1e9, 3),
                    "msps": round(S4 * BLK4 / (ms * 1e-3) / 1e6, 1)}
        dec.close()
        del iq, audio
        torch.cuda.empty_cache()
    return out


def bench_c5(torch, rfm, synth_device, K, W):
    wb_mod = __import__("radiofm_b200.wideband", fromlist=["WidebandReceiver"])
    dev = torch.device("cuda", 0)
    ncalls = 4
    u8 = synth_device.make_wideband_u8(torch, FS5, ncalls * N_CALL5, FREQS5, dev)
    out = {}
    for mixer in ("freqshift", "osc"):
        for fmt in ("u8", "s8", "s16"):
            cap = convert(torch, u8, fmt).contiguous()
            esz = rfm.iq_format_bytes(fmt)
            wb = wb_mod.WidebandReceiver(torch, FREQS5, FS5, BLK5, BPC5, mixer=mixer, device=0, input_format=fmt)
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
            out[f"{mixer}_{fmt}_ms_per_call"] = round(e0.elapsed_time(e1) / K, 3)
            wb.close()
            del cap
    return out


def bench_scan(torch, rfm, synth_device):
    dev = torch.device("cuda", 0)
    u8 = synth_device.make_wideband_u8(torch, FS5, 24 * N_CALL5, FREQS5, dev)
    out = {}
    for fmt in ("u8", "s8", "s16", "cf32"):
        cap = convert(torch, u8, fmt).contiguous()
        torch.cuda.synchronize()
        s = rfm.BandScan(FS5, -24.9e6, 100e3, 499, device=0)
        s.run(cap)        # first run: module load and allocations
        s.run(cap)
        spec_ms, conf_ms = s.timing()
        out[fmt] = {"spectrum_ms": round(spec_ms, 4), "stations": len(s.stations())}
        s.close()
        del cap
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    import importlib
    import torch
    rfm = load_package()
    synth_device = importlib.import_module("radiofm_b200.synth_device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res = {"device": q.stdout.strip() or "unknown"}
    res["c4"] = bench_c4(torch, rfm, synth_device, args.steps, args.warmup)
    res["c5"] = bench_c5(torch, rfm, synth_device, args.calls, 3)
    res["scan"] = bench_scan(torch, rfm, synth_device)
    print(json.dumps(res))


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
