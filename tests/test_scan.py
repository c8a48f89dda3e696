"""Band scan, CPU side: the restatement's channel decisions and normalisation (oracle/scan.py), argument validation of
rfm_scan_create through the C ABI, and the C++ driver built against include/ and the library.  No kernel runs here."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import scan

RFM_ERR_INVALID, RFM_ERR_NO_DEVICE = -1, -4


def test_candidate_rule_plateaus_ends_threshold_and_short_rasters():
    f = 1.0
    # plateau of two equal maxima: the first (strictly above its left, >= its right) wins, the second does not
    c = np.array([f, f, f, f, 50.0, 50.0, f, f])
    assert scan.candidates(c) == [4]
    # a three-wide plateau: only its first channel
    assert scan.candidates(np.array([f, f, f, 30.0, 30.0, 30.0, f, f])) == [3]
    # both raster ends: j = 0 needs only C_0 >= C_1, j = count - 1 only C_{j} > C_{j-1}
    c = np.array([40.0, f, f, f, f, f, f, 40.0])
    assert scan.candidates(c) == [0, 7]
    c = np.array([40.0, 40.0, f, f, f, f, f, f])
    assert scan.candidates(c) == [0]
    # exactly on the threshold (floor 1, 10 dB -> 10.0): >= accepts it; a hair below does not
    thr = 1.0 * 10.0 ** (10.0 / 10.0)
    assert scan.candidates(np.array([f, f, thr, f, f, f, f, f])) == [2]
    assert scan.candidates(np.array([f, f, np.nextafter(thr, 0.0), f, f, f, f, f])) == []
    # fewer than four channels: the floor is the smallest (index (count - 1) // 4 == 0)
    assert scan.noise_floor(np.array([5.0, 1.0, 3.0])) == 1.0
    assert scan.candidates(np.array([1.0, 20.0, 3.0])) == [1]
    assert scan.candidates(np.array([7.0])) == []            # floor = itself: 0 dB < 10 dB
    assert scan.candidates(np.array([7.0]), min_snr_db=0.0) == [0]
    assert scan.candidates(np.array([1.0, 10.0])) == [1]
    # the floor is the 25th percentile: three quarters of the raster may be occupied
    c = np.array([1.0, 100.0, 1.0, 100.0, 1.0, 100.0, 1.0, 100.0, 1.0, 100.0, 1.0, 100.0, 1.0, 1.0])
    assert scan.noise_floor(c) == 1.0 and scan.candidates(c) == [1, 3, 5, 7, 9, 11]


def test_channel_bins_follow_the_half_open_rule():
    fs = 2.4e6
    df = fs / scan.N
    bins = scan.channel_bins(fs, -1.1e6, 100e3, 23)
    f = scan.bin_freqs(fs)
    seen = np.concatenate(bins)
    assert np.unique(seen).size == seen.size                 # no bin in two channels
    for j, b in enumerate(bins):
        fj = -1.1e6 + j * 100e3
        assert np.all(np.diff(b) == 1) and np.all(f[b] >= fj - 50e3) and np.all(f[b] < fj + 50e3)
        assert b.size in (170, 171) and abs(b.size - 100e3 / df) < 1


@pytest.mark.parametrize("offset_bins", [0.0, 0.5])
def test_parseval_and_full_scale_tone(offset_bins):
    """|x| = 1 is 0 dBFS: the spectrum sums to the mean power 1; a tone on a bin centre puts 2/3 in its bin and 1/6
    in each neighbour (periodic Hann), all inside its channel; half a bin off, the channel still holds all but the
    far sidelobes."""
    fs, n = 2.4e6, 20 * scan.N
    k0 = 300
    f0 = (k0 + offset_bins) * fs / scan.N
    x = np.exp(2j * np.pi * f0 * np.arange(n) / fs)
    p = scan.welch_psd_cf(x)
    assert abs(p.sum() - 1.0) < 1e-12
    c0 = scan.N // 2 + k0
    if offset_bins == 0.0:
        assert np.allclose(p[c0 - 1:c0 + 2], [1 / 6, 2 / 3, 1 / 6], atol=1e-12)
        assert p[:c0 - 1].sum() + p[c0 + 2:].sum() < 1e-20
    bins = scan.channel_bins(fs, 100e3 * round(f0 / 100e3), 100e3, 1)
    c = scan.channel_powers(p, bins)[0]
    assert (abs(c - 1.0) < 1e-12) if offset_bins == 0.0 else (0.9999 < c <= 1.0 + 1e-12)
    assert abs(10 * np.log10(c)) < 1e-3


def test_u8_conversion_is_the_references():
    u = np.stack([np.arange(256), np.arange(256)[::-1]], axis=1).astype(np.uint8)
    x = scan.u8_to_float(u)
    want = (np.arange(256) / 127.5 - 1.0).astype(np.float32)
    assert np.array_equal(x.real.astype(np.float32), want) and np.array_equal(x.imag.astype(np.float32), want[::-1])


@pytest.mark.parametrize("fs,first,step,count", [
    (2.4e6, -1.1e6, 2000.0, 23),        # step < 4 Fs / N (2343.75 Hz)
    (2.4e6, -1.1e6, 100e3, 0),          # count < 1
    (50e6, -24.9e6, 1000e3, 4097),      # count > N
    (2.4e6, -1.2e6, 100e3, 25),         # |f| + 100 kHz > Fs / 2 at both ends
    (2.4e6, -1.0e6, 100e3, 23),         # ... at the top end only
    (300e3, 0.0, 100e3, 1),             # the WFM decimation chain has no stage (<= 400 kHz)
    (float("nan"), 0.0, 100e3, 1),
    (2.4e6, float("inf"), 100e3, 1),
])
def test_create_rejects_bad_rasters_without_a_device(rfm, fs, first, step, count):
    cfg = rfm.scan_config(fs, first, step, count)
    h = C.c_void_p()
    assert rfm.lib().rfm_scan_create(C.byref(cfg), C.byref(h)) == RFM_ERR_INVALID
    assert not h.value


def test_valid_config_needs_a_device(rfm):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    for args in ((2.4e6, -1.1e6, 100e3, 23), (50e6, -24.9e6, 100e3, 499), (2.4e6, 0.0, 4 * 2.4e6 / 4096, 1)):
        cfg = rfm.scan_config(*args)
        h = C.c_void_p()
        assert rfm.lib().rfm_scan_create(C.byref(cfg), C.byref(h)) == RFM_ERR_NO_DEVICE, args
        assert b"no CUDA device" in rfm.lib().rfm_last_error()
    with pytest.raises(rfm.RadioFmError, match="no CUDA device"):
        rfm.BandScan(2.4e6, -1.1e6, 100e3, 23)


def test_scan_driver_compiles_against_the_c_abi(rfm, tmp_path):
    lib_dir = os.path.join(ROOT, "pvr.rtl.radiofm_b200")
    exe = str(tmp_path / "host_scan_driver")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "host_scan_driver.cpp"), "-o", exe,
                           "-L", lib_dir, "-lradiofm_b200", f"-Wl,-rpath,{lib_dir}"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "usage" in out.stderr
    # the record layout the driver writes is the binding's
    assert C.sizeof(rfm.ScanStation) == 56
