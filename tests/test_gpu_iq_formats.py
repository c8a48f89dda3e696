"""Signed 8- and 16-bit IQ on the device.  The input format is not a reference concept: the reference's classes take
ComplexType.  So every s8 / s16 path must give, bit for bit, what the cf32 path gives for the converted samples
(test_iq_formats.s8_to_cf32 / s16_to_cf32), and the cf32 paths are the ones pinned to the reference elsewhere."""
import ctypes as C
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import RATES, ROOT, bits_equal, station
from oracle import scan
from test_iq_formats import build_iq_driver, to_cf32, welch_psd_iq

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

pytestmark = pytest.mark.gpu

FMTS = ["s8", "s16"]
RFM_ERR_INVALID = -1


def requantise(u8: np.ndarray, fmt: str, seed: int = 0) -> np.ndarray:
    """The same station in a signed container: s8 = u - 128; s16 = 256 (u - 128) + random low byte (every s16 code can
    occur, so the low bits are exercised too)."""
    v = u8.astype(np.int32) - 128
    if fmt == "s8":
        return v.astype(np.int8)
    low = np.random.default_rng(seed).integers(0, 256, size=v.shape)
    return (v * 256 + low).astype(np.int16)


def _torch():
    import torch
    return torch


# ---------------------------------------------------------------------------------------------------------------------
# 1. the conversion itself, exhaustively, through rfm_freqshift at 0 Hz (x * 1 - y * 0, x * 0 + y * 1: the identity)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", FMTS)
def test_every_code_converts_exactly_through_the_product(rfm, fmt):
    torch = _torch()
    v = np.arange(-128, 128) if fmt == "s8" else np.arange(-32768, 32768)
    dt = np.int8 if fmt == "s8" else np.int16
    cap = np.stack([v, v[::-1]], axis=1).astype(dt)
    want = to_cf32(cap)
    assert np.array_equal(want[:, 0].astype(np.float64), v / (128.0 if fmt == "s8" else 32768.0))
    n = cap.shape[0]
    fs = rfm.FreqShiftBatch([0.0, 0.0], 2.4e6, max_len=n, device=0)
    out = fs.process_iq(cap, shared_capture=True)                       # host, shared capture
    assert bits_equal(out[0], want) and bits_equal(out[1], want)
    fs.reset()
    rows = np.stack([cap, cap[::-1]])
    out = fs.process_iq(rows, shared_capture=False)                     # host, one row each
    assert bits_equal(out[0], want) and bits_equal(out[1], to_cf32(cap[::-1]))
    fs.reset()
    d_in = torch.from_numpy(rows).cuda()
    d_out = torch.empty((2, n, 2), dtype=torch.float32, device="cuda")
    fs.process_iq_device(fmt, False, d_in.data_ptr(), n, d_out.data_ptr(), n, n)
    torch.cuda.synchronize()
    assert bits_equal(d_out[0].cpu().numpy(), want)
    # a device pointer that is not aligned to the sample size is refused with the reason
    if fmt == "s16":
        with pytest.raises(rfm.RadioFmError):
            fs.process_iq_device(fmt, True, d_in.data_ptr() + 2, n, d_out.data_ptr(), n, 16)
    fs.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. decoder: host, submit and device entry points against rfm_decoder_process_cf32 of the converted samples
# ---------------------------------------------------------------------------------------------------------------------
DECODERS = {   # label -> (rate of the synthetic station, fs, downsample, block)
    "1.0M": ("1.0M",) + RATES["1.0M"],
    "1.2M": ("1.2M",) + RATES["1.2M"],
    "2.4M": ("2.4M",) + RATES["2.4M"],
    "390k": ("390k",) + RATES["390k"],
    "1.2M/3": ("1.2M", 1.2e6, 3, 65520),        # a downsample the tiled front ends are not built for: k_front
}


def _all_outputs(d, S):
    out = []
    for s in range(S):
        out.append((d.take_bits(s), d.take_groups(s), d.take_uecp(s), d.status(s)))
    return out


def _same_outputs(a, b, label):
    for s, ((ba, ga, ua, sa), (bb, gb, ub, sb)) in enumerate(zip(a, b)):
        assert np.array_equal(ba, bb), (label, s, "bits")
        assert np.array_equal(ga, gb), (label, s, "groups")
        assert ua == ub, (label, s, "uecp")
        assert all(np.float32(sa[k]) == np.float32(sb[k]) for k in sa), (label, s, sa, sb)


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("cfg", list(DECODERS))
def test_decoder_formats_equal_cf32_of_the_converted_samples(rfm, fmt, cfg):
    torch = _torch()
    rate, fs, ds, blk = DECODERS[cfg]
    S, nblk = 3, 3
    raw = np.stack([requantise(station(rate, nblk, stream_id=20 + s)[0][:nblk * blk], fmt, seed=s) for s in range(S)])
    conv = to_cf32(raw)
    kw = dict(downsample=ds, n_streams=S, max_block_len=blk, device=0)
    ref, host, sub, dev = (rfm.FmDecoderBatch(fs, -0.15 * fs, **kw) for _ in range(4))
    # device rows with an odd pitch (n + 3 samples): u8 / s8 rows a tensor map cannot describe take the tiled kernel
    pitch = blk + 3
    d_iq = torch.zeros((S, pitch, 2), dtype=torch.int8 if fmt == "s8" else torch.int16, device="cuda")
    stride = max(dev.max_audio_floats(blk), 2)
    stride += stride & 1
    d_audio = torch.zeros((S, stride), dtype=torch.float32, device="cuda")
    for b in range(nblk):
        sl = slice(b * blk, (b + 1) * blk)
        a_ref = ref.process_cf32(conv[:, sl])
        a_host = host.process_iq(raw[:, sl])
        a_sub = sub.process_iq(raw[:, sl], submit=True)
        sub.synchronize()
        d_iq[:, :blk] = torch.from_numpy(np.ascontiguousarray(raw[:, sl])).cuda()
        torch.cuda.synchronize()
        k = dev.process_iq_device(fmt, d_iq.data_ptr(), pitch, blk, d_audio.data_ptr(), stride)
        dev.synchronize()
        a_dev = d_audio[:, :k].cpu().numpy()
        for label, a in (("host", a_host), ("submit", a_sub), ("device", a_dev)):
            assert bits_equal(a, a_ref), (cfg, fmt, label, b)
    assert float(np.max(np.abs(a_ref))) > 0.02
    want = _all_outputs(ref, S)
    assert sum(len(b) for b, _, _, _ in want) > 0, "RDS bits decoded"
    for label, d in (("host", host), ("submit", sub), ("device", dev)):
        _same_outputs(_all_outputs(d, S), want, (cfg, fmt, label))
    for d in (ref, host, sub, dev):
        d.close()


@pytest.mark.parametrize("fmt", FMTS)
def test_decoder_odd_and_short_blocks(rfm, fmt):
    """test_default_rtlsdr_block_at_1200k_and_odd_short_blocks's block sizes at 1.2 MS/s, two streams."""
    from make_golden_ref_cases import ODD_SIZES
    fs, ds = 1.2e6, 5
    iq = np.stack([station("1.2M", 12, stream_id=s)[0] for s in range(2)])
    raw = requantise(iq, fmt, seed=7)
    conv = to_cf32(raw)
    kw = dict(downsample=ds, n_streams=2, max_block_len=65536, device=0)
    ref, host = rfm.FmDecoderBatch(fs, -0.15 * fs, **kw), rfm.FmDecoderBatch(fs, -0.15 * fs, **kw)
    pos = 0
    for n in ODD_SIZES:
        if n < 8 * ds:
            for d, x in ((ref, conv), (host, raw)):
                with pytest.raises(rfm.RadioFmError):
                    d.process_iq(x[:, pos:pos + n]) if d is host else d.process_cf32(x[:, pos:pos + n])
            continue
        assert bits_equal(host.process_iq(raw[:, pos:pos + n]), ref.process_cf32(conv[:, pos:pos + n])), (fmt, n)
        pos += n
    _same_outputs(_all_outputs(host, 2), _all_outputs(ref, 2), (fmt, "odd sizes"))
    ref.close()
    host.close()


def test_unknown_format_and_misaligned_device_input_are_refused(rfm):
    torch = _torch()
    L = rfm.lib()
    d = rfm.FmDecoderBatch(1.0e6, -0.15e6, downsample=4, n_streams=1, max_block_len=4096, device=0)
    x = torch.zeros((4096, 2), dtype=torch.int16, device="cuda")
    a = torch.zeros(8192, dtype=torch.float32, device="cuda")
    k = C.c_uint32(0)
    for f in (-1, 4):
        assert L.rfm_decoder_process_iq_device(d._h, f, C.c_void_p(x.data_ptr()), 4096, 4096, C.c_void_p(a.data_ptr()),
                                               8192, C.byref(k), None) == RFM_ERR_INVALID
        assert b"format" in L.rfm_last_error()
    assert L.rfm_decoder_process_iq_device(d._h, rfm.IQ_S16, C.c_void_p(x.data_ptr() + 2), 4096, 4000,
                                           C.c_void_p(a.data_ptr()), 8192, C.byref(k), None) == RFM_ERR_INVALID
    assert b"aligned" in L.rfm_last_error()
    h = np.zeros((4096, 2), dtype=np.int16)
    assert L.rfm_decoder_process_iq(d._h, 7, h.ctypes.data_as(C.c_void_p), 4096, None, 0, None) == RFM_ERR_INVALID
    d.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. wideband front end and WidebandReceiver
# ---------------------------------------------------------------------------------------------------------------------
FS, BLK, BPC = 50.0e6, 32000, 64
FREQS = [-1.0e6, 200000.0, 7.0e6]
N_CALL = BLK * BPC


@pytest.fixture(scope="module")
def wide_u8(synth):
    return synth.make_wideband_u8(FS, 2 * N_CALL, FREQS)


def _oracle_baseband(o, x):
    """OracleStation.baseband on a float capture [n, 2] (the oracle's own loop without its u8 conversion)."""
    from oracle.wideband import _P
    out = []
    for b in range(x.shape[0] // o.front_block):
        z = np.array(x[b * o.front_block:(b + 1) * o.front_block], dtype=np.float32, order="C")
        if o.shift:
            o.L.rfo_freqshift_reset(o.shift)
            o.L.rfo_freqshift_process(o.shift, _P(z), z.shape[0])
        y = np.zeros_like(z)
        k = o.L.rfo_rdsdc_process(o.dc, z.shape[0], _P(z), _P(y))
        out.append(y[:k].copy())
    return np.concatenate(out)


@pytest.mark.parametrize("fmt", FMTS)
def test_downconvert_shared_capture_equals_cf32_rows(rfm, wide_u8, fmt):
    torch = _torch()
    raw = requantise(wide_u8[:N_CALL], fmt)
    conv = to_cf32(raw)
    nco = -np.asarray(FREQS)
    outs = {}
    for label in ("iq shared", "cf32 stride 0", "cf32 rows"):
        dc = rfm.DownConvertBatch(nco, FS, 100000.0, wfm=True, max_len=N_CALL, device=0)
        m = N_CALL >> dc.n_stages
        out = torch.empty((3, m, 2), dtype=torch.float32, device="cuda")
        if label == "iq shared":
            x = torch.from_numpy(raw).cuda()
            k = dc.process_iq_device(fmt, True, x.data_ptr(), 0, out.data_ptr(), m, N_CALL)
        elif label == "cf32 stride 0":
            x = torch.from_numpy(conv).cuda()
            k = dc.process_iq_device("cf32", False, x.data_ptr(), 0, out.data_ptr(), m, N_CALL)
        else:
            x = torch.from_numpy(np.stack([conv] * 3)).cuda()
            k = dc.process_iq_device("cf32", False, x.data_ptr(), N_CALL, out.data_ptr(), m, N_CALL)
        torch.cuda.synchronize()
        assert k == m
        outs[label] = out.cpu().numpy()
        # the host form of the same call
        dc.reset()
        outs[label + " host"] = dc.process_iq(raw if label == "iq shared" else conv, shared_capture=True)
        dc.close()
    for label, o in outs.items():
        assert bits_equal(o, outs["cf32 rows"]), (fmt, label)
    assert float(np.max(np.abs(outs["cf32 rows"]))) > 1e-3


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("mixer", ["osc", "freqshift", "freqshift_unfused"])
def test_wideband_receiver_input_format(rfm, port, wide_u8, fmt, mixer):
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    from oracle.wideband import OracleStation
    raw = requantise(wide_u8, fmt, seed=3)
    conv = to_cf32(raw)
    wb = wb_mod.WidebandReceiver(torch, FREQS, FS, BLK, BPC, mixer=mixer, device=0, input_format=fmt)
    oracles = [OracleStation(f, FS, BLK, BPC, mixer=mixer.split("_")[0]) for f in FREQS]
    for c in range(2):
        sl = slice(c * N_CALL, (c + 1) * N_CALL)
        audio = wb.process_iq(raw[sl])
        bb = wb.bb.cpu().numpy()
        for s, o in enumerate(oracles):
            ref_bb = _oracle_baseband(o, conv[sl])
            assert bits_equal(bb[s], ref_bb), (fmt, mixer, c, s, "baseband")
            assert bits_equal(audio[s], o.dec.process_cf32(ref_bb)), (fmt, mixer, c, s, "audio")
    for s, o in enumerate(oracles):
        assert np.array_equal(wb.dec.take_bits(s), o.dec.take_bits())
        so, sd = o.dec.status(), wb.dec.status(s)
        assert all(np.float32(so[k]) == np.float32(sd[k]) for k in so), (so, sd)
        o.close()
    wb.close()


@pytest.mark.parametrize("fmt", FMTS)
def test_wideband_100_stations_freqshift(rfm, port, fmt):
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    synth_device = importlib.import_module("radiofm_b200.synth_device")
    from oracle.wideband import OracleStation
    freqs = [(k - 50) * 200000.0 for k in range(100)]
    checked = [0, 49, 50, 99]
    cap = requantise(synth_device.make_wideband_u8(torch, FS, 2 * N_CALL, freqs, torch.device("cuda", 0)).cpu().numpy(),
                     fmt, seed=5)
    conv = to_cf32(cap)
    wb = wb_mod.WidebandReceiver(torch, freqs, FS, BLK, BPC, mixer="freqshift", device=0, input_format=fmt)
    oracles = {s: OracleStation(freqs[s], FS, BLK, BPC, mixer="freqshift") for s in checked}
    for c in range(2):
        sl = slice(c * N_CALL, (c + 1) * N_CALL)
        audio = wb.process_iq(cap[sl])
        bb = wb.bb.cpu().numpy()
        for s, o in oracles.items():
            ref_bb = _oracle_baseband(o, conv[sl])
            assert bits_equal(bb[s], ref_bb), (fmt, c, s)
            assert bits_equal(audio[s], o.dec.process_cf32(ref_bb)), (fmt, c, s)
        assert np.all(np.max(np.abs(audio), axis=1) > 1e-3)
    for s, o in oracles.items():
        assert np.array_equal(wb.dec.take_bits(s), o.dec.take_bits())
        o.close()
    wb.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. band scan
# ---------------------------------------------------------------------------------------------------------------------
RASTER_50M = (-24.9e6, 100e3, 499)


@pytest.fixture(scope="module")
def scan_u8():
    torch = _torch()
    sd = importlib.import_module("radiofm_b200.synth_device")
    return sd.make_wideband_u8(torch, FS, 2 * N_CALL, FREQS, torch.device("cuda", 0)).cpu().numpy()


def _capture(u8, fmt):
    if fmt == "cf32":
        return to_cf32(u8)
    return requantise(u8, fmt, seed=11)


@pytest.mark.parametrize("fmt", ["s8", "s16", "cf32"])
def test_scan_formats(rfm, scan_u8, fmt):
    torch = _torch()
    cap = _capture(scan_u8, fmt)
    s = rfm.BandScan(FS, *RASTER_50M, device=0)
    s.run(cap)
    psd, chan, st = s.spectrum(), s.channel_power(), s.stations()
    # spectrum: within test_gpu_scan.py's bounds of the float64 restatement
    ref = welch_psd_iq(cap)
    tot = float(ref.sum())
    assert float(np.max(np.abs(psd.astype(np.float64) - ref))) <= 1e-6 * tot
    bins = scan.channel_bins(FS, *RASTER_50M)
    c_ref = scan.channel_powers(ref, bins)
    sel = c_ref >= scan.noise_floor(c_ref)
    assert float(np.max(np.abs(scan.channel_powers(psd, bins)[sel] - c_ref[sel]) / c_ref[sel])) <= 1e-4
    # channel powers and decisions: the restatement applied to the product's own spectrum, bit for bit
    assert np.array_equal(chan.view(np.uint64), scan.channel_powers(psd, bins).view(np.uint64))
    cand = scan.candidates(chan)
    assert [d["freq"] for d in st] == [RASTER_50M[0] + j * RASTER_50M[1] for j in cand]
    assert [d["freq"] for d in st] == FREQS
    # device input gives the same bits as host input
    d_cap = torch.from_numpy(np.ascontiguousarray(cap)).cuda()
    torch.cuda.synchronize()
    s2 = rfm.BandScan(FS, *RASTER_50M, device=0)
    s2.run(d_cap)
    assert bits_equal(s2.spectrum(), psd) and np.array_equal(s2.channel_power().view(np.uint64), chan.view(np.uint64))
    assert s2.stations() == st
    # each station: what WidebandReceiver(osc, input_format=fmt) reports after the same calls
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    wb = wb_mod.WidebandReceiver(torch, [d["freq"] for d in st], FS, BLK, BPC, mixer="osc", device=0, input_format=fmt)
    for c in range(cap.shape[0] // N_CALL):
        wb.process_iq(cap[c * N_CALL:(c + 1) * N_CALL])
    for m, d in enumerate(st):
        so, groups = wb.dec.status(m), wb.dec.take_groups(m)
        assert d["stereo"] == so["stereo"] and d["rds_groups"] == len(groups), (fmt, d, so)
        for k in ("pilot_level", "if_level", "bb_level"):
            assert bits_equal(np.atleast_1d(d[k]), np.atleast_1d(so[k])), (fmt, k)
        assert d["pi"] == (int(np.bincount(groups[:, 0]).argmax()) if len(groups) else -1)
    wb.close()
    s.close()
    s2.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. why: a station 75 dB below the strongest, found in cs16 and lost in u8
# ---------------------------------------------------------------------------------------------------------------------
FS_RTL, N_CALL_RTL = 2.4e6, 128000
RASTER_RTL = (-1.1e6, 100e3, 23)
STRONG = [(-900e3, 31), (-500e3, 32), (300e3, 33)]    # (offset, synth stream id), equal amplitude
WEAK = (800e3, 34, 10 ** (-75 / 20))


def _fm(mpx, fs, f):
    return np.exp(1j * (2.0 * np.pi * 75000.0 / fs * np.cumsum(mpx) + 2.0 * np.pi * f * np.arange(mpx.size) / fs))


@pytest.fixture(scope="module")
def weak_window(synth):
    n = int(FS_RTL)
    acc = np.zeros(n, dtype=np.complex128)
    for f, sid, amp in [(f, sid, 1.0) for f, sid in STRONG] + [WEAK]:
        p = synth.stream_params(sid)
        bits = synth.rds_bits_from_groups(synth.rds_group_stream(p["pi"], p["ps"], 16))
        mpx = synth.mpx_signal(FS_RTL, n, left=p["left"], right=p["right"], pilot=0.1, rds_level=0.05, rds_bits=bits)
        acc += amp * _fm(mpx, FS_RTL, f)
    acc *= 0.9 / float(np.max(np.abs(acc)))
    u8 = np.empty((n, 2), dtype=np.uint8)
    u8[:, 0] = np.clip(np.rint(127.5 + 127.5 * acc.real), 0, 255)
    u8[:, 1] = np.clip(np.rint(127.5 + 127.5 * acc.imag), 0, 255)
    s16 = np.empty((n, 2), dtype=np.int16)
    s16[:, 0] = np.clip(np.rint(32768.0 * acc.real), -32768, 32767)
    s16[:, 1] = np.clip(np.rint(32768.0 * acc.imag), -32768, 32767)
    return u8, s16


def test_weak_station_is_found_in_cs16_and_lost_in_u8(rfm, synth, weak_window):
    """Three stations near full scale (together 0.9 of it at the peak, each about -10.5 dBFS) and one 75 dB below them
    at +800 kHz (about -85.5 dBFS), modulated in float64 and quantised once per format.  The weak station sits 500 kHz
    from the nearest strong one and off the strong stations' third-order products (2 f_a - f_b and f_a + f_b - f_c land
    at -2.1, -1.7, -1.3, -0.1, +0.7, +1.1, +1.5 MHz: the nearest is 100 kHz away, a whole raster step).  Per 100 kHz
    channel the u8 quantisation floor is about -64 dBFS and the cs16 floor about -112 dBFS, so the weak station is some
    21 dB under the u8 floor and some 26 dB over the cs16 floor: the scan's 10 dB rule finds it in cs16 only, and the
    confirmation decodes it -- stereo, PI and PS -- from the cs16 samples."""
    u8, s16 = weak_window
    p = synth.stream_params(WEAK[1])
    s = rfm.BandScan(FS_RTL, *RASTER_RTL, device=0)
    s.run(s16)
    st = {d["freq"]: d for d in s.stations()}
    chan = s.channel_power()
    j = int(round((WEAK[0] - RASTER_RTL[0]) / RASTER_RTL[1]))
    fl = scan.noise_floor(chan)
    print(f"[weak station] cs16: weak {10 * np.log10(chan[j]):.1f} dBFS, floor {10 * np.log10(fl):.1f} dBFS")
    assert WEAK[0] in st, sorted(st)
    w = st[WEAK[0]]
    assert w["stereo"] and w["pi"] == p["pi"] and w["ps"] == p["ps"], w
    for f, sid in STRONG:
        assert f in st and st[f]["pi"] == synth.stream_params(sid)["pi"], (f, st.get(f))
    s.run(u8)
    st8 = {d["freq"]: d for d in s.stations()}
    chan8 = s.channel_power()
    print(f"[weak station] u8: weak channel {10 * np.log10(chan8[j]):.1f} dBFS, floor "
          f"{10 * np.log10(scan.noise_floor(chan8)):.1f} dBFS")
    assert WEAK[0] not in st8, st8.get(WEAK[0])
    for f, _ in STRONG:
        assert f in st8
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. the C++ driver: cs16 capture -> scan -> decode one station, C ABI only
# ---------------------------------------------------------------------------------------------------------------------
def test_iq_driver_scans_and_decodes_a_cs16_capture(rfm, synth, weak_window, tmp_path):
    exe = build_iq_driver(tmp_path)
    _, s16 = weak_window
    s16.tofile(tmp_path / "cap.cs16")
    out = subprocess.run([exe, str(tmp_path / "cap.cs16"), str(FS_RTL), *[str(v) for v in RASTER_RTL]],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    print(out.stdout)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("decoded:")][0]
    head, ps = line.split(" ps=", 1)
    fields = dict(kv.split("=", 1) for kv in head.split()[1:])
    f = float(fields["offset_hz"])
    sid = {fr: sid for fr, sid in STRONG}[f]
    p = synth.stream_params(sid)
    assert fields["stereo"] == "1" and int(fields["groups"]) > 0 and fields["pi"] == f"{p['pi']:X}"
    assert ps == p["ps"]
