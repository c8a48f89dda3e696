"""Phase-accumulator NCO (rfm_downconvert_set_nco): the restatement in oracle/nco.py against closed forms, its phase
bookkeeping, the table-midpoint condition that makes the host tables independent of the libm, the purity of the
phasor, the binding's argument checks that need no device and the C++ driver's build.  No GPU needed.

test_freqshift_phase_error_against_the_nco restates the numpy check that motivated the feature: the float32 phase of a
cFreqShift that is Reset() every 32000 samples swings by kHz within a block at 9.8 MHz; the NCO's does not."""
from __future__ import annotations

import math
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from conftest import ROOT
from oracle import nco

FS = np.float32(50.0e6)
FREQS = [0.2e6, 2.0e6, 5.0e6, 9.8e6, 3_333_317.3]   # the last one is off the 1562.5 Hz raster of 32000-sample blocks


# ---------------------------------------------------------------------------------------------------------------------
# the word
# ---------------------------------------------------------------------------------------------------------------------
def test_word_closed_forms():
    fs = float(FS)
    assert nco.word(0.0, FS) == 0 and nco.word(-0.0, FS) == 0
    assert nco.word(fs / 4, FS) == 1 << 30
    assert nco.word(-fs / 4, FS) == (1 << 32) - (1 << 30)
    assert nco.word(fs / 2, FS) == 1 << 31 and nco.word(-fs / 2, FS) == 1 << 31
    assert nco.word(fs / 8, FS) == 1 << 29
    # in_rate is the down-converter's float rate: a rate that float32 cannot hold is rounded first
    assert nco.word(1.0e6, 2.4e6) == nco.word(1.0e6, np.float32(2.4e6))
    assert nco.word(1.0e6, 2.4e6) == nco.llround(1.0e6 / float(np.float32(2.4e6)) * 2.0 ** 32)


def test_word_rounds_halves_away_from_zero():
    rate = float(1 << 25)     # f / rate * 2^32 = 128 f: f = (k + 0.5) / 128 Hz lies exactly half-way
    for k in (0, 1, 6, 7, 1000, 1001):
        f = (k + 0.5) / 128.0
        assert f / rate * 2.0 ** 32 == k + 0.5
        assert nco.word(f, rate) == k + 1
        assert nco.word(-f, rate) == (1 << 32) - (k + 1)
    # numpy and Python round half to even: they would give k for even k
    assert round(6.5) == 6 and np.round(6.5) == 6.0 and nco.llround(6.5) == 7 and nco.llround(-6.5) == -7
    # the classic trap of floor(x + 0.5): the largest double below 0.5
    assert nco.llround(0.49999999999999994) == 0
    assert nco.llround(2.5) == 3 and nco.llround(-2.5) == -3 and nco.llround(-2.4999) == -2


def test_word_range_errors():
    fs = float(FS)
    for bad in (math.nextafter(fs / 2, math.inf), -math.nextafter(fs / 2, math.inf), 1e9, math.inf, -math.inf,
                math.nan):
        with pytest.raises(ValueError):
            nco.word(bad, FS)


def test_frequency_is_within_fs_over_2_33():
    for f in FREQS + [-f for f in FREQS] + [12_345_678.9, -24_999_999.9]:
        d = nco.word(f, FS)
        got = (d if d < 1 << 31 else d - (1 << 32)) * float(FS) / 2.0 ** 32
        assert abs(got - f) <= float(FS) / 2.0 ** 33, (f, got)


# ---------------------------------------------------------------------------------------------------------------------
# the phase
# ---------------------------------------------------------------------------------------------------------------------
def test_unequal_calls_continue_one_phase_sequence():
    d = nco.word(-9.8e6, FS)
    whole = nco.phases(d, 100_000)
    pos, parts = 0, []
    phi = 0
    for n in (1, 7, 32000, 12345, 2, 55645):
        parts.append(nco.phases(d, n, phi))
        phi = nco.advance(phi, d, n)
        pos += n
    assert pos == 100_000
    assert np.array_equal(np.concatenate(parts), whole)
    assert phi == (100_000 * d) % (1 << 32)
    # and the mixed samples likewise
    rng = np.random.default_rng(3)
    x = rng.standard_normal((100_000, 2)).astype(np.float32)
    one = nco.mix(x, -9.8e6, FS)
    o = nco.Nco(-9.8e6, FS)
    cut = [0, 1, 8, 32008, 44353, 44355, 100_000]
    assert np.array_equal(np.concatenate([o.mix(x[a:b]) for a, b in zip(cut, cut[1:])]).view(np.uint32),
                          one.view(np.uint32))
    o.reset()
    assert np.array_equal(o.mix(x[:5000]).view(np.uint32), one[:5000].view(np.uint32))


def test_phase_wraps_at_2_32():
    d = 0xFFFFFFFF                                  # one step back per sample
    assert list(nco.phases(d, 4)) == [0, 0xFFFFFFFF, 0xFFFFFFFE, 0xFFFFFFFD]
    assert nco.advance(5, d, 6) == 0xFFFFFFFF
    d = 0x80000001
    assert list(nco.phases(d, 3, 0x7FFFFFFF)) == [0x7FFFFFFF, 0, 0x80000001]
    # a whole revolution after 2^32 samples for any word, 2^32 n d mod 2^32 = 0
    assert nco.advance(0, nco.word(9.8e6, FS), 1 << 32) == 0
    big = (1 << 32) - 3
    assert nco.advance(123, d, big) == (123 + big * d) % (1 << 32)


# ---------------------------------------------------------------------------------------------------------------------
# the tables
# ---------------------------------------------------------------------------------------------------------------------
def test_no_table_entry_is_near_a_float_rounding_midpoint():
    """Each entry's double cos / sin is more than 2^-40 (relative) from every float32 rounding midpoint, so a faithfully
    rounded libm (error under 2^-52 relative) gives the same float as the exact value: the host's tables do not depend
    on its libm, and none has to be pinned."""
    closest = 1.0
    t = nco.tables()
    for m in range(3):
        for k in range(256):
            a = nco.table_angle(m, k)
            for j, v in enumerate((math.cos(a), math.sin(a))):
                assert t[m, k, j] == np.float32(v)
                if v == 0.0:
                    continue
                f = np.float32(v)
                for nb in (np.nextafter(f, np.float32(-np.inf)), np.nextafter(f, np.float32(np.inf))):
                    mid = (Fraction(float(f)) + Fraction(float(nb))) / 2
                    closest = min(closest, float(abs(Fraction(v) - mid) / abs(Fraction(v))))
    print(f"[nco tables] closest relative distance of an entry to a float midpoint: 2^{math.log2(closest):.1f}")
    assert closest > 2.0 ** -40
    assert t[0, 0].tolist() == [1.0, 0.0] and t[0, 64, 1] == 1.0 and t[0, 128, 0] == -1.0


def test_phasor_is_the_contracts_product():
    p = np.array([0, 0x01000000, 0x00010000, 0x00000100, 0x000000FF, 0x40000000, 0xFFFFFFFF, 0x12345678],
                 dtype=np.uint32)
    t = nco.tables()
    e = nco.phasor(p)
    for i, phi in enumerate(int(v) for v in p):
        a, b, c = t[0, phi >> 24], t[1, (phi >> 16) & 255], t[2, (phi >> 8) & 255]
        ab = (np.float32(a[0] * b[0]) - np.float32(a[1] * b[1]), np.float32(a[0] * b[1]) + np.float32(a[1] * b[0]))
        ab = np.float32(ab[0]), np.float32(ab[1])
        want = (np.float32(ab[0] * c[0]) - np.float32(ab[1] * c[1]), np.float32(ab[0] * c[1]) + np.float32(ab[1] * c[0]))
        assert e[i, 0] == np.float32(want[0]) and e[i, 1] == np.float32(want[1]), hex(phi)
    assert e[0].tolist() == [1.0, 0.0]
    assert np.array_equal(e[3], t[2, 1]) and np.array_equal(e[4], e[0])    # the lowest 8 bits are dropped


@pytest.mark.parametrize("f", FREQS)
def test_purity(f):
    n = 1 << 18
    d = nco.word(-f, FS)
    ph = nco.phases(d, n)
    e = nco.phasor(ph).astype(np.float64)
    e = e[:, 0] + 1j * e[:, 1]
    exact = np.exp(2j * np.pi * ph.astype(np.float64) / 2.0 ** 32)
    err = e - exact
    dbc = 10 * np.log10(np.mean(np.abs(err) ** 2))
    line = 10 * np.log10(np.max(np.abs(np.fft.fft(err)) ** 2) / float(n) ** 2)
    amp = float(np.max(np.abs(np.abs(e) - 1.0)))
    print(f"[nco purity] {f / 1e6:.6f} MHz: error {dbc:.1f} dBc, largest error line {line:.1f} dBc, "
          f"max ||e| - 1| {amp:.2e}")
    assert dbc <= -130.0, (f, dbc)
    assert amp <= 2e-7, (f, amp)


# ---------------------------------------------------------------------------------------------------------------------
# the motivating check
# ---------------------------------------------------------------------------------------------------------------------
def _freq_error_20us(phase_err: np.ndarray, fs: float) -> np.ndarray:
    w = int(round(20e-6 * fs))
    return (phase_err[w:] - phase_err[:-w]) / (2.0 * np.pi * w / fs)


def test_freqshift_phase_error_against_the_nco():
    """cFreqShift(-9.8 MHz, 50 MS/s) reset every 32000 samples: float32 phase acc += inc, never wrapped
    (FreqShift.cpp:55-69), so its increment is quantised to the ulp of a phase that grows to 2 pi f L / Fs.  Its
    frequency error averaged over 20 us swings by kHz within every block; the NCO's stays at the word's rounding."""
    f, fs, L = -9.8e6, float(FS), 32000
    inc = np.float32(2.0 * np.pi * float(np.float32(f)) / fs)
    acc = np.empty(L, dtype=np.float32)
    acc[0] = 0.0
    acc[1:] = np.add.accumulate(np.full(L - 1, inc, dtype=np.float32), dtype=np.float32)
    i = np.arange(L, dtype=np.float64)
    fe_fs = _freq_error_20us(acc.astype(np.float64) - 2.0 * np.pi * f * i / fs, fs)
    # the NCO over the same block, measured the same way from the phase of its float32 phasor
    e = nco.phasor(nco.phases(nco.word(f, FS), L)).astype(np.float64)
    ang = np.unwrap(np.arctan2(e[:, 1], e[:, 0]))
    fe_nco = _freq_error_20us(ang - 2.0 * np.pi * f * i / fs, fs)
    print(f"[nco motivation] 9.8 MHz, 20 us average within a 32000-sample block: freqshift {fe_fs.min():+.0f} .. "
          f"{fe_fs.max():+.0f} Hz, nco {fe_nco.min():+.4f} .. {fe_nco.max():+.4f} Hz")
    assert fe_fs.max() - fe_fs.min() > 10e3
    assert float(np.max(np.abs(fe_nco))) < 0.05
    # and the freqshift's phase jumps at every reset: the phase error at the end of a block is not the start's
    assert abs(float(acc[-1]) + float(inc) - 2.0 * np.pi * f * L / fs) > 1e-3


# ---------------------------------------------------------------------------------------------------------------------
# the binding's argument checks, no device
# ---------------------------------------------------------------------------------------------------------------------
def test_mixer_strings_are_checked_before_any_device_work(rfm):
    import importlib
    import torch
    wb = importlib.import_module("radiofm_b200.wideband")
    for bad in ("NCO", "nco ", "phasor", ""):
        with pytest.raises(ValueError):
            wb.WidebandReceiver(torch, [1.0e6], mixer=bad)
        with pytest.raises(ValueError):
            rfm.BandScan(50.0e6, -24.9e6, 100e3, 499, mixer=bad)
    with pytest.raises(ValueError):
        rfm.BandScan(50.0e6, -24.9e6, 100e3, 499, mixer=1)
    assert rfm.scan_mixer("osc") == 0 and rfm.scan_mixer("nco") == 1
    for sym in ("rfm_downconvert_set_nco", "rfm_scan_set_mixer"):
        assert sym in rfm.EXPORTED_SYMBOLS
        getattr(rfm.lib(), sym)


def build_nco_driver(tmp_path) -> str:
    lib_dir = os.path.join(ROOT, "pvr.rtl.radiofm_b200")
    exe = str(tmp_path / "host_nco_driver")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
                           os.path.join(ROOT, "tests", "cpp", "host_nco_driver.cpp"), "-o", exe,
                           "-L", lib_dir, "-lradiofm_b200", f"-Wl,-rpath,{lib_dir}",
                           "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath,/usr/local/cuda/lib64"])
    return exe


def test_nco_driver_compiles_against_the_c_abi(rfm, tmp_path):
    exe = build_nco_driver(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "usage" in out.stderr
