"""IQ correction (rfm_iq_correction): the restatement in oracle/iqcorr.py against closed forms, the argument checks of
rfm_iq_estimate that need no device, the binding's types and the C++ driver's build.  No GPU needed.

test_correction_removes_mirror_and_dc_in_a_cs8_window restates the numpy check that motivated the feature: a zero-IF
window with 1 dB / 3 degrees of imbalance and a DC offset, quantised to cs8, estimated blindly and corrected."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import iqcorr, scan
from test_iq_formats import to_cf32

RFM_ERR_INVALID = -1


def imbalanced(z: np.ndarray, gain_db: float, phase_deg: float, dc=(0.0, 0.0)) -> np.ndarray:
    """A receiver's I, Q of the proper signal z: I = Re z, Q = g (sin(phi) Re z + cos(phi) Im z), plus DC.  The exact
    correction is a = 1 / (g cos(phi)), b = -tan(phi)."""
    g, ph = 10 ** (gain_db / 20), np.deg2rad(phase_deg)
    i = z.real + dc[0]
    q = g * (np.sin(ph) * z.real + np.cos(ph) * z.imag) + dc[1]
    return np.stack([i, q], axis=1)


def quantise(x: np.ndarray, fmt: str) -> np.ndarray:
    if fmt == "s8":
        return np.clip(np.rint(128.0 * x), -128, 127).astype(np.int8)
    if fmt == "s16":
        return np.clip(np.rint(32768.0 * x), -32768, 32767).astype(np.int16)
    if fmt == "u8":
        return np.clip(np.rint(127.5 + 127.5 * x), 0, 255).astype(np.uint8)
    return x.astype(np.float32)


def test_pure_dc_is_found_exactly_and_leaves_no_imbalance_estimate():
    for fmt, cap, want in (("s16", np.full((1001, 2), [-1200, 3000], dtype=np.int16), (-1200 / 32768, 3000 / 32768)),
                           ("s8", np.full((7, 2), [5, -128], dtype=np.int8), (5 / 128, -1.0)),
                           ("u8", np.full((3, 2), [128, 0], dtype=np.uint8), (np.float32(128 / 127.5 - 1), -1.0))):
        dc_i, dc_q, a, b, ok = iqcorr.estimate(cap)
        assert (dc_i, dc_q) == (np.float32(want[0]), np.float32(want[1])), fmt
        assert (a, b, ok) == (1.0, 0.0, False), fmt      # v_I = 0: degenerate
    # a constant cf32 capture: the float64 moments cancel to (about) zero, never to a usable imbalance
    x = np.full((4096, 2), [0.3, -0.1], dtype=np.float32)
    dc_i, dc_q, a, b, ok = iqcorr.estimate(x)
    assert (dc_i, dc_q) == (np.float32(0.3), np.float32(-0.1)) and (a, b, ok) == (1.0, 0.0, False)


@pytest.mark.parametrize("fmt", ["u8", "s8", "s16", "cf32"])
def test_known_gain_and_phase_of_a_proper_signal(fmt):
    rng = np.random.default_rng(1)
    n = 1 << 18
    z = 0.2 * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2)
    x = imbalanced(z, 1.0, 3.0, dc=(0.02, -0.015))
    cap = quantise(x, fmt)
    dc_i, dc_q, a, b, ok = iqcorr.estimate(cap)
    g, ph = 10 ** (1 / 20), np.deg2rad(3.0)
    tol = 4.0 / np.sqrt(n)            # sampling error of the moments
    assert ok
    assert abs(a - 1 / (g * np.cos(ph))) < tol and abs(b + np.tan(ph)) < tol, (fmt, a, b)
    dtol = 1e-3 if fmt in ("u8", "s8") else 1e-5      # the rounding to codes, averaged
    assert abs(dc_i - x[:, 0].mean()) < dtol and abs(dc_q - x[:, 1].mean()) < dtol, (fmt, dc_i, dc_q)
    # the corrected samples are proper: equal powers, uncorrelated parts (to the sample, not only in expectation)
    y = iqcorr.apply(to_cf32(cap).reshape(-1, 2), dc_i, dc_q, a, b).astype(np.float64)
    yi, yq = y[:, 0] - y[:, 0].mean(), y[:, 1] - y[:, 1].mean()
    assert abs(np.mean(yi * yq)) < 1e-5 * np.mean(yi * yi) and abs(np.mean(yq * yq) / np.mean(yi * yi) - 1) < 1e-5
    # the integer path and the float64 path describe the same statistics
    if fmt != "cf32":
        f64 = iqcorr.coefficients_float64(to_cf32(cap))
        for u, v in zip((dc_i, dc_q, a, b), f64[:4]):
            assert abs(float(u) - float(v)) <= 1e-6 * max(1.0, abs(float(v))), (fmt, u, v)


def test_degenerate_inputs():
    # Q = 2 I: v_I v_Q - c^2 = 0 exactly in integers
    i = np.arange(-50, 50, dtype=np.int64)
    cap = np.stack([i, 2 * i], axis=1).astype(np.int8)
    assert iqcorr.estimate(cap)[2:] == (1.0, 0.0, False)
    # Q constant: v_Q = 0
    cap = np.stack([i, np.full_like(i, 7)], axis=1).astype(np.int16)
    assert iqcorr.estimate(cap)[2:] == (1.0, 0.0, False)
    # one sample
    assert iqcorr.estimate(np.array([[3, 4]], dtype=np.int16))[2:] == (1.0, 0.0, False)
    with pytest.raises(ValueError):
        iqcorr.estimate(np.zeros((0, 2), dtype=np.int16))


def test_integer_sums_are_exact_at_the_2_32_boundary():
    """n = 2^32 full-scale cs16 samples: every 64-bit sum and every 128-bit centred moment is in range, and the
    estimate of the quadrature pattern (A, 0), (0, A), (-A, 0), (0, -A) is exactly a = 1, b = 0."""
    n, A = 1 << 32, 32767
    assert n * 32768 ** 2 < 2 ** 63 and n * (n * 32768 ** 2) < 2 ** 127
    sums = (n, 0, 0, n // 2 * A * A, n // 2 * A * A, 0)
    dc_i, dc_q, a, b, ok = iqcorr.coefficients_from_integer_sums(iqcorr.S16, sums)
    assert (dc_i, dc_q, a, b, ok) == (0.0, 0.0, 1.0, 0.0, True)
    # the largest s8 cross product sum, all samples (-128, -128): degenerate, DC exactly -1
    sums = (n, -128 * n, -128 * n, 16384 * n, 16384 * n, 16384 * n)
    assert iqcorr.coefficients_from_integer_sums(iqcorr.S8, sums) == (-1.0, -1.0, 1.0, 0.0, False)


def test_estimate_refuses_bad_arguments_before_touching_a_device(rfm):
    """Unknown format, n = 0, n > 2^32 and a misaligned device pointer are refused by argument checks alone."""
    L = rfm.lib()
    out = rfm.RfmIqCorrection()
    h = np.zeros((16, 2), dtype=np.int16)
    p = h.ctypes.data_as(C.c_void_p)
    for fmt, ptr, n, dev, why in ((4, p, 16, 0, b"format"), (-1, p, 16, 0, b"format"), (2, p, 0, 0, b"empty"),
                                  (2, p, (1 << 32) + 1, 1, b"2^32"), (2, C.c_void_p(0x1002), 16, 1, b"aligned"),
                                  (3, C.c_void_p(0x1004), 16, 1, b"aligned")):
        assert L.rfm_iq_estimate(fmt, ptr, n, dev, -1, C.byref(out)) == RFM_ERR_INVALID
        assert why in L.rfm_last_error(), (fmt, n, L.rfm_last_error())
    assert L.rfm_iq_estimate(2, p, 16, 0, -1, None) == RFM_ERR_INVALID


def test_apply_is_the_float32_expression():
    x = np.array([[0.5, -0.25], [1.0, 0.75], [-1.0, 0.0]], dtype=np.float32)
    y = iqcorr.apply(x, 0.25, -0.25, 1.5, -0.125)
    r = np.float32([0.25, 0.75, -1.25])
    q = np.float32([0.0, 1.0, 0.25])
    assert np.array_equal(y[:, 0], r)
    assert np.array_equal(y[:, 1], np.float32(1.5) * q + np.float32(-0.125) * r)
    # each step is rounded to float32 on its own (no double intermediate)
    x = np.array([[1.0000001, 0.3]], dtype=np.float32)
    y = iqcorr.apply(x, np.float32(1e-8), np.float32(0.1), np.float32(1.0123), np.float32(-0.0523))
    r = np.float32(np.float32(1.0000001) - np.float32(1e-8))
    q = np.float32(np.float32(0.3) - np.float32(0.1))
    want = np.float32(np.float32(np.float32(1.0123) * q) + np.float32(np.float32(-0.0523) * r))
    assert y[0, 0] == r and y[0, 1] == want


def test_binding_types(rfm):
    assert C.sizeof(rfm.RfmIqCorrection) == 20
    c = rfm.IqCorrection(np.float32(0.01), np.float32(-0.02), np.float32(1.1), np.float32(-0.05), True)
    assert rfm.IqCorrection._from_c(c._c()) == c
    with pytest.raises(TypeError):
        rfm._corr_arg((0.0, 0.0, 1.0, 0.0))
    assert rfm._corr_arg(None) is None
    for bad in (np.zeros((8, 2), dtype=np.int32), np.zeros((8, 2), dtype=np.float64)):
        with pytest.raises(ValueError):
            rfm.estimate_iq_correction(bad)
    with pytest.raises(ValueError):
        rfm.estimate_iq_correction(0x1000)          # a device pointer needs its format and length


# ---------------------------------------------------------------------------------------------------------------------
# the motivating check: mirror images and the DC line of a zero-IF cs8 window, before and after the correction
# ---------------------------------------------------------------------------------------------------------------------
FS = 2.4e6
STATIONS = [300e3, -600e3, 900e3]   # mirrors at -300, +600, -900 kHz: 200 kHz from any station


def _window(n: int, seed: int = 5) -> np.ndarray:
    """Three FM carriers (random 15 kHz-band modulation, 75 kHz deviation) with free mirror channels, equal power."""
    rng = np.random.default_rng(seed)
    acc = np.zeros(n, dtype=np.complex128)
    for f in STATIONS:
        m = np.convolve(rng.standard_normal(n + 255), np.hanning(256) / np.hanning(256).sum(), mode="valid")[:n]
        m /= np.max(np.abs(m))
        acc += np.exp(1j * (2 * np.pi * 75e3 / FS * np.cumsum(m) + 2 * np.pi * f * np.arange(n) / FS))
    return 0.9 * acc / np.max(np.abs(acc))


def test_correction_removes_mirror_and_dc_in_a_cs8_window():
    n = 1 << 19
    x = imbalanced(_window(n), 1.0, 3.0, dc=(0.02, 0.015))
    cap = quantise(x, "s8")
    bins = scan.channel_bins(FS, -1.1e6, 100e3, 23)
    j = {f: int(round((f + 1.1e6) / 100e3)) for f in STATIONS + [-f for f in STATIONS] + [0.0]}

    def powers(y):
        return scan.channel_powers(scan.welch_psd_cf(y[:, 0].astype(np.float64) + 1j * y[:, 1]), bins)

    before = powers(to_cf32(cap))
    c = iqcorr.estimate(cap)
    after = powers(iqcorr.apply(to_cf32(cap), *c[:4]))
    db = lambda v: 10 * np.log10(v)
    for f in STATIONS:
        rej0, rej1 = db(before[j[f]] / before[j[-f]]), db(after[j[f]] / after[j[-f]])
        print(f"[mirror] station {f / 1e3:+.0f} kHz: {rej0:.1f} dB over its mirror before, {rej1:.1f} dB after")
        assert 22.0 < rej0 < 26.0, rej0                 # 1 dB / 3 degrees: about 24 dB image rejection
        assert rej1 > 45.0, rej1
    assert db(before[j[0.0]] / before[j[STATIONS[0]]]) > -30.0
    assert db(after[j[0.0]] / after[j[STATIONS[0]]]) < -45.0
    # the corrected window's candidates are the stations alone
    assert sorted(-1.1e6 + 100e3 * k for k in scan.candidates(after)) == sorted(STATIONS)
    assert set(j[-f] for f in STATIONS) | {j[0.0]} <= set(scan.candidates(before))


def build_iqcorr_driver(tmp_path) -> str:
    lib_dir = os.path.join(ROOT, "pvr.rtl.radiofm_b200")
    exe = str(tmp_path / "host_iqcorr_driver")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
                           os.path.join(ROOT, "tests", "cpp", "host_iqcorr_driver.cpp"), "-o", exe,
                           "-L", lib_dir, "-lradiofm_b200", f"-Wl,-rpath,{lib_dir}",
                           "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath,/usr/local/cuda/lib64"])
    return exe


def test_iqcorr_driver_compiles_against_the_c_abi(rfm, tmp_path):
    exe = build_iqcorr_driver(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "usage" in out.stderr
