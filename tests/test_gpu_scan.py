"""Band scan on the device (rfm_scan_*, BandScan): the spectrum against the float64 restatement (oracle/scan.py), the
channel decisions bit for bit, determinism, C5 at its stated length (100 stations, 1 s at 50 MS/s), the confirmation
against the oracle composition of the reference's classes, an RTL-SDR window, empty captures and the C++ driver."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits_equal
from oracle import scan

pytestmark = pytest.mark.gpu

FS = 50.0e6
N_CALL = 2048000                       # 16000 baseband samples << 7 stages
RASTER_50M = (-24.9e6, 100e3, 499)
FS_RTL, N_CALL_RTL = 2.4e6, 128000     # 16000 << 3
RASTER_RTL = (-1.1e6, 100e3, 23)


def _torch():
    import torch
    return torch


def _scan(rfm, fs, raster, capture=None, d_capture=None, n=None):
    s = rfm.BandScan(fs, *raster, device=0)
    if capture is not None:
        s.run_u8(capture)
    else:
        _torch().cuda.synchronize()
        s.run_device(d_capture.data_ptr(), n)
    return s


def _result(s):
    return s.spectrum(), s.channel_power(), s.stations()


def _same_bits(a, b):
    (pa, ca, sa), (pb, cb, sb) = a, b
    assert bits_equal(pa, pb)
    assert np.array_equal(ca.view(np.uint64), cb.view(np.uint64))
    assert len(sa) == len(sb)
    for x, y in zip(sa, sb):
        for k in x:
            if isinstance(x[k], np.floating):
                assert bits_equal(np.atleast_1d(x[k]), np.atleast_1d(y[k])), k
            else:
                assert x[k] == y[k], k


def _check_spectrum(psd, ref, fs, raster, label):
    tot = float(ref.sum())
    err = float(np.max(np.abs(psd.astype(np.float64) - ref)))
    assert err <= 1e-6 * tot, (label, err, tot)
    bins = scan.channel_bins(fs, *raster)
    c_ref = scan.channel_powers(ref, bins)
    c = scan.channel_powers(psd, bins)
    fl = scan.noise_floor(c_ref)
    sel = c_ref >= fl
    rel = float(np.max(np.abs(c[sel] - c_ref[sel]) / c_ref[sel]))
    assert rel <= 1e-4, (label, rel)
    print(f"[scan spectrum {label}] max |P - P_ref| / sum P_ref = {err / tot:.3e}, "
          f"max channel rel err (C >= floor) = {rel:.3e}")


@pytest.fixture(scope="module")
def three_stations():
    torch = _torch()
    sd = importlib.import_module("radiofm_b200.synth_device")
    return sd.make_wideband_u8(torch, FS, 2 * N_CALL, [-1.0e6, 200000.0, 7.0e6], torch.device("cuda", 0)).cpu().numpy()


@pytest.fixture(scope="module")
def c5_capture():
    """test_wideband_100_stations_on_the_raster's 100 stations, 24 calls (0.98 s), made on the device."""
    torch = _torch()
    sd = importlib.import_module("radiofm_b200.synth_device")
    freqs = [(k - 50) * 200000.0 for k in range(100)]
    cap = sd.make_wideband_u8(torch, FS, 24 * N_CALL, freqs, torch.device("cuda", 0))
    torch.cuda.synchronize()
    return freqs, cap


def _fm(mpx, fs, f):
    return np.exp(1j * (2.0 * np.pi * 75000.0 / fs * np.cumsum(mpx) + 2.0 * np.pi * f * np.arange(mpx.size) / fs))


RTL_STATIONS = [   # (offset Hz, stereo, rds, relative amplitude, synth stream id)
    (-800e3, True, True, 1.0, 11),
    (-300e3, True, False, 1.0, 12),
    (200e3, False, True, 1.0, 13),
    (700e3, True, False, 0.1, 14),
]


@pytest.fixture(scope="module")
def rtl_capture(synth):
    n = int(FS_RTL)
    acc = np.zeros(n, dtype=np.complex128)
    for f, stereo, rds, amp, sid in RTL_STATIONS:
        p = synth.stream_params(sid)
        bits = synth.rds_bits_from_groups(synth.rds_group_stream(p["pi"], p["ps"], 16)) if rds else None
        mpx = synth.mpx_signal(FS_RTL, n, left=p["left"], right=p["right"], pilot=0.1 if stereo else 0.0,
                               rds_level=0.05 if rds else 0.0, rds_bits=bits)
        acc += amp * _fm(mpx, FS_RTL, f)
    acc *= 0.8 / float(np.max(np.abs(acc)))
    out = np.empty((n, 2), dtype=np.uint8)
    out[:, 0] = np.clip(np.rint(127.5 + 127.5 * acc.real), 0, 255)
    out[:, 1] = np.clip(np.rint(127.5 + 127.5 * acc.imag), 0, 255)
    return out


def test_spectrum_matches_the_float64_restatement(rfm, three_stations):
    s = _scan(rfm, FS, RASTER_50M, three_stations)
    _check_spectrum(s.spectrum(), scan.welch_psd(three_stations), FS, RASTER_50M, "3 stations")
    assert [st["freq"] for st in s.stations()] == [-1.0e6, 200000.0, 7.0e6]
    s.close()
    # a lone tone between bins, dithered: undithered u8 quantisation of a pure tone makes discrete spurs, which are
    # spectral lines like any other and would be candidates
    n = 2 * N_CALL
    rng = np.random.default_rng(9)
    x = 0.8 * np.exp(2j * np.pi * 3.3337e6 * np.arange(n) / FS)
    x = x + (rng.standard_normal(n) + 1j * rng.standard_normal(n)) * (2.0 / 127.5)
    tone = np.stack([np.clip(np.rint(127.5 + 127.5 * x.real), 0, 255), np.clip(np.rint(127.5 + 127.5 * x.imag), 0, 255)],
                    axis=1).astype(np.uint8)
    s = _scan(rfm, FS, RASTER_50M, tone)
    _check_spectrum(s.spectrum(), scan.welch_psd(tone), FS, RASTER_50M, "tone")
    st = s.stations()
    assert [d["freq"] for d in st] == [3.3e6] and not st[0]["stereo"] and st[0]["pi"] == -1
    assert abs(st[0]["power_dbfs"] - 20 * np.log10(0.8)) < 0.05
    s.close()


def test_decisions_are_the_restatements_bit_for_bit(rfm, three_stations, rtl_capture):
    for fs, raster, cap in ((FS, RASTER_50M, three_stations), (FS_RTL, RASTER_RTL, rtl_capture)):
        s = _scan(rfm, fs, raster, cap)
        psd, chan, st = _result(s)
        ref = scan.channel_powers(psd, scan.channel_bins(fs, *raster))
        assert np.array_equal(ref.view(np.uint64), chan.view(np.uint64))
        cand = scan.candidates(ref, 10.0)
        assert [d["freq"] for d in st] == [raster[0] + float(j) * raster[1] for j in cand]
        fl = scan.noise_floor(ref)
        for d, j in zip(st, cand):
            assert d["power_dbfs"] == np.float32(10.0 * np.log10(ref[j]))
            assert d["snr_db"] == np.float32(10.0 * np.log10(ref[j] / fl))
        s.close()


def test_runs_are_deterministic_and_host_equals_device_input(rfm, three_stations):
    torch = _torch()
    s = _scan(rfm, FS, RASTER_50M, three_stations)
    a = _result(s)
    s.run_u8(three_stations)                  # the same handle again
    _same_bits(a, _result(s))
    s.close()
    d = torch.from_numpy(three_stations).to("cuda:0")
    s = _scan(rfm, FS, RASTER_50M, d_capture=d, n=three_stations.shape[0])
    _same_bits(a, _result(s))
    s.close()


def test_c5_100_stations_one_second(rfm, synth, c5_capture):
    freqs, cap = c5_capture
    s = _scan(rfm, FS, RASTER_50M, d_capture=cap, n=cap.shape[0])
    st = s.stations()
    assert [d["freq"] for d in st] == freqs
    for k, d in enumerate(st):
        p = synth.stream_params(k % 4)
        assert d["stereo"], (k, d)
        assert d["pi"] == p["pi"] and d["ps"] == p["ps"], (k, d, p["pi"], p["ps"])
    spec_ms, conf_ms = s.timing()
    print(f"[scan C5] 100 stations x 24 calls: spectrum {spec_ms:.3f} ms, confirmation {conf_ms:.1f} ms")
    s.close()


def test_c5_confirmation_is_the_oracle_receiver(rfm, port, c5_capture):
    from oracle.wideband import OracleStation
    freqs, cap = c5_capture
    s = _scan(rfm, FS, RASTER_50M, d_capture=cap, n=cap.shape[0])
    st = s.stations()
    host = cap.cpu().numpy()
    for k in (0, 50, 99):
        o = OracleStation(freqs[k], FS, 32000, 64, mixer="osc")
        for c in range(24):
            o.process_u8(host[c * N_CALL:(c + 1) * N_CALL])
        so, groups = o.dec.status(), o.dec.take_groups()
        d = st[k]
        assert d["stereo"] == bool(so["stereo"])
        for a, b in (("pilot_level", "pilot_level"), ("if_level", "if_level"), ("bb_level", "bb_level")):
            assert bits_equal(np.atleast_1d(d[a]), np.atleast_1d(np.float32(so[b]))), (k, a)
        assert d["rds_groups"] == len(groups) > 0
        vals, first, cnt = np.unique(groups[:, 0], return_index=True, return_counts=True)
        best = max(range(len(vals)), key=lambda i: (cnt[i], -first[i]))
        assert d["pi"] == int(vals[best])
        g = rfm.RdsGroupDecoder()
        g.decode(groups)
        assert d["ps"].encode("latin-1") == g.channel_name().rstrip(b"\0") and d["ps"] != ""
        g.close()
        o.close()
    s.close()


def _oracle_rtl(port, cap, f):
    from oracle.wideband import OracleStation
    o = OracleStation(f, FS_RTL, 32000, 4, mixer="osc")
    for c in range(cap.shape[0] // N_CALL_RTL):
        o.process_u8(cap[c * N_CALL_RTL:(c + 1) * N_CALL_RTL])
    return o


def test_rtlsdr_window_four_stations(rfm, port, synth, rtl_capture):
    s = _scan(rfm, FS_RTL, RASTER_RTL, rtl_capture)
    st = s.stations()
    assert [d["freq"] for d in st] == [f for f, *_ in RTL_STATIONS]
    for d, (f, stereo, rds, amp, sid) in zip(st, RTL_STATIONS):
        p = synth.stream_params(sid)
        if amp < 1.0:
            o = _oracle_rtl(port, rtl_capture, f)
            so, groups = o.dec.status(), o.dec.take_groups()
            assert d["stereo"] == bool(so["stereo"]) and d["rds_groups"] == len(groups)
            assert bits_equal(np.atleast_1d(d["pilot_level"]), np.atleast_1d(np.float32(so["pilot_level"])))
            o.close()
            continue
        assert d["stereo"] == stereo, (f, d)
        if rds:
            assert d["pi"] == p["pi"] and d["ps"] == p["ps"], (f, d)
        else:
            assert d["rds_groups"] == 0 and d["pi"] == -1 and d["ps"] == "", (f, d)
    s.close()


def test_no_stations_in_noise_or_off_a_dc_offset(rfm):
    rng = np.random.default_rng(5)
    n = 2 * N_CALL_RTL
    noise = np.clip(np.rint(127.5 + 20.0 * rng.standard_normal((n, 2))), 0, 255).astype(np.uint8)
    s = _scan(rfm, FS_RTL, RASTER_RTL, noise)
    assert s.stations() == [] and s.channel_power().min() > 0
    s.close()
    const = np.empty((n, 2), dtype=np.uint8)
    const[:, 0], const[:, 1] = 127, 128
    # a constant capture is a pure DC offset: nothing away from 0 Hz ...
    s = _scan(rfm, FS_RTL, (200e3, 100e3, 10), const)
    assert s.stations() == [] and s.timing()[1] == 0.0
    s.close()
    # ... and the 0 Hz channel, a spectral line like any carrier, is a candidate that the receiver does not confirm
    s = _scan(rfm, FS_RTL, RASTER_RTL, const)
    st = s.stations()
    assert [d["freq"] for d in st] == [0.0]
    assert not st[0]["stereo"] and st[0]["rds_groups"] == 0 and st[0]["pi"] == -1 and st[0]["ps"] == ""
    s.close()
    with pytest.raises(rfm.RadioFmError):
        _scan(rfm, FS_RTL, RASTER_RTL, const[:N_CALL_RTL - 1])


def test_cpp_driver_gives_bandscans_table(rfm, rtl_capture, tmp_path):
    lib_dir = os.path.join(ROOT, "pvr.rtl.radiofm_b200")
    exe = str(tmp_path / "host_scan_driver")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "host_scan_driver.cpp"), "-o", exe,
                           "-L", lib_dir, "-lradiofm_b200", f"-Wl,-rpath,{lib_dir}"])
    rtl_capture.tofile(tmp_path / "cap.bin")
    out = subprocess.run([exe, str(tmp_path / "cap.bin"), str(FS_RTL), *[str(v) for v in RASTER_RTL],
                          str(tmp_path / "st.bin")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    raw = (tmp_path / "st.bin").read_bytes()
    sz = C.sizeof(rfm.ScanStation)
    drv = [rfm.scan_station_dict(rfm.ScanStation.from_buffer_copy(raw[i:i + sz])) for i in range(0, len(raw), sz)]
    s = _scan(rfm, FS_RTL, RASTER_RTL, rtl_capture)
    _same_bits((np.zeros(1, np.float32), np.zeros(1), drv), (np.zeros(1, np.float32), np.zeros(1), s.stations()))
    assert len(drv) == 4
    s.close()
