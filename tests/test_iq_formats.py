"""Signed 8- and 16-bit IQ (rfm_iq_format): the exact conversions restated in numpy, the format table of the C ABI, the
binding's dtype mapping and the C++ driver's build.  No GPU needed.

The restatement (s8_to_cf32 / s16_to_cf32 / welch_psd_iq) is what the GPU tests in test_gpu_iq_formats.py feed the cf32
paths and the float64 spectrum with."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import scan

RFM_ERR_INVALID = -1


def s8_to_cf32(iq) -> np.ndarray:
    """[n, 2] int8 -> [n, 2] float32, v * 2^-7 (exact)."""
    return np.asarray(iq, dtype=np.int8).astype(np.float32) * np.float32(2.0 ** -7)


def s16_to_cf32(iq) -> np.ndarray:
    """[n, 2] int16 -> [n, 2] float32, v * 2^-15 (exact)."""
    return np.asarray(iq, dtype=np.int16).astype(np.float32) * np.float32(2.0 ** -15)


def to_cf32(iq) -> np.ndarray:
    """Any supported capture -> the float32 samples the product converts it to (u8: the reference's conversion)."""
    a = np.asarray(iq)
    if a.dtype == np.uint8:
        return scan.u8_to_float(a).astype(np.complex64).view(np.float32).reshape(a.shape)
    if a.dtype == np.int8:
        return s8_to_cf32(a)
    if a.dtype == np.int16:
        return s16_to_cf32(a)
    if a.dtype == np.complex64:
        return np.ascontiguousarray(a).view(np.float32).reshape(a.shape + (2,))
    assert a.dtype == np.float32, a.dtype
    return a


def welch_psd_iq(capture) -> np.ndarray:
    """oracle/scan.py's float64 spectrum of any supported capture."""
    x = to_cf32(capture).reshape(-1, 2).astype(np.float64)
    return scan.welch_psd_cf(x[:, 0] + 1j * x[:, 1])


def test_s8_conversion_is_exact_for_every_code():
    v = np.arange(-128, 128)
    x = s8_to_cf32(np.stack([v, v[::-1]], axis=1))
    want = v.astype(np.float64) / 128.0
    assert np.array_equal(x[:, 0].astype(np.float64), want) and np.array_equal(x[:, 1].astype(np.float64), want[::-1])
    assert x.min() == -1.0 and x.max() == np.float32(127 / 128)


def test_s16_conversion_is_exact_for_every_code():
    v = np.arange(-32768, 32768)
    x = s16_to_cf32(np.stack([v, v[::-1]], axis=1))
    want = v.astype(np.float64) / 32768.0
    assert np.array_equal(x[:, 0].astype(np.float64), want) and np.array_equal(x[:, 1].astype(np.float64), want[::-1])
    # every code lands on a distinct float32 and converts back
    assert np.array_equal((x[:, 0].astype(np.float64) * 32768.0).astype(np.int64), v)


@pytest.mark.parametrize("offset_bins", [0.0, 0.5])
def test_full_scale_cs16_tone_is_0_dbfs(offset_bins):
    """A complex tone at the cs16 container's full scale (|x| = 32767 / 32768 after rounding to codes) is 0 dBFS within
    the quantisation: Parseval on the restated spectrum, as test_scan.py checks it for the float tone."""
    fs, n = 2.4e6, 20 * scan.N
    k0 = 300
    f0 = (k0 + offset_bins) * fs / scan.N
    t = np.arange(n)
    z = 32767.0 * np.exp(2j * np.pi * f0 * t / fs)
    cap = np.stack([np.round(z.real), np.round(z.imag)], axis=1).astype(np.int16)
    p = welch_psd_iq(cap)
    # sum P = the mean windowed power: (32767 / 32768)^2 up to the rounding to codes
    assert abs(10 * np.log10(p.sum())) < 1e-3
    bins = scan.channel_bins(fs, 100e3 * round(f0 / 100e3), 100e3, 1)
    c = scan.channel_powers(p, bins)[0]
    assert abs(10 * np.log10(c)) < 1e-3


def test_to_cf32_agrees_across_formats():
    """The same codes, scaled to each container, are the same floats where they are representable in both."""
    v = np.arange(-128, 128, dtype=np.int64)
    a8 = np.stack([v, -v - 1], axis=1).astype(np.int8)
    a16 = (a8.astype(np.int16) * 256)
    assert np.array_equal(to_cf32(a8), to_cf32(a16))
    c = (to_cf32(a8)[:, 0] + 1j * to_cf32(a8)[:, 1]).astype(np.complex64)
    assert np.array_equal(to_cf32(c), to_cf32(a8))


def test_iq_format_bytes_and_unknown_formats(rfm):
    L = rfm.lib()
    assert [int(L.rfm_iq_format_bytes(f)) for f in range(4)] == [2, 2, 4, 8]
    for f in (-1, 4, 99, 1 << 30):
        assert int(L.rfm_iq_format_bytes(f)) == 0
    assert (rfm.IQ_U8, rfm.IQ_S8, rfm.IQ_S16, rfm.IQ_CF32) == (0, 1, 2, 3)


def test_binding_maps_dtypes_to_formats(rfm):
    for dt, f in ((np.uint8, 0), (np.int8, 1), (np.int16, 2), (np.float32, 3), (np.complex64, 3)):
        assert rfm.iq_format(np.dtype(dt)) == f
        assert rfm.iq_format(np.zeros(2, dtype=dt).dtype) == f
    for name, f in (("u8", 0), ("s8", 1), ("s16", 2), ("cf32", 3), ("torch.int16", 2), ("torch.complex64", 3)):
        assert rfm.iq_format(name) == f
    assert rfm.iq_format(2) == 2
    for bad in (np.int32, np.float64, np.uint16, "s12", 4, -1):
        with pytest.raises(ValueError):
            rfm.iq_format(bad)
    assert [rfm.iq_format_bytes(f) for f in ("u8", "s8", "s16", "cf32")] == [2, 2, 4, 8]


def test_scan_create_validation_is_unchanged(rfm):
    """The scan's configuration is the same struct with the same checks; the format is an argument of the run."""
    assert C.sizeof(rfm.ScanConfig) == 48
    cfg = rfm.scan_config(2.4e6, -1.1e6, 2000.0, 23)
    h = C.c_void_p()
    assert rfm.lib().rfm_scan_create(C.byref(cfg), C.byref(h)) == RFM_ERR_INVALID and not h.value


def build_iq_driver(tmp_path) -> str:
    lib_dir = os.path.join(ROOT, "pvr.rtl.radiofm_b200")
    exe = str(tmp_path / "host_iq_driver")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
                           os.path.join(ROOT, "tests", "cpp", "host_iq_driver.cpp"), "-o", exe,
                           "-L", lib_dir, "-lradiofm_b200", f"-Wl,-rpath,{lib_dir}",
                           "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath,/usr/local/cuda/lib64"])
    return exe


def test_iq_driver_compiles_against_the_c_abi(rfm, tmp_path):
    exe = build_iq_driver(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "usage" in out.stderr
