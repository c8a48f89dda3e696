"""TEST INFRASTRUCTURE -- restatement of the band scan's spectrum and channel decisions (rfm_scan_*, include/radiofm_b200.h):

    welch_psd        float64 Welch spectrum: N = 4096 periodic-Hann segments, hop N/2, of x = float(u / 127.5 - 1)
                     (RTL_SDR_Source.cpp:207-211); P[k] = sum_s |X_s[k]|^2 / (S N sum w^2), centred
    channel_bins     raster point j owns the bins with f_j - step/2 <= f < f_j + step/2, f = (k - N/2) Fs / N
    channel_powers   C_j = sum of its bins' P, in double, in bin order
    noise_floor      the sorted C at index (count - 1) // 4
    candidates       C_j >= floor * 10^(min_snr_db / 10), C_j > C_{j-1}, C_j >= C_{j+1} (where the neighbours exist)
    check_spectrum   a spectrum with a NaN or Inf bin has no floor, no sort order and no candidates: ValueError, as
                     rfm_scan_run returns RFM_ERR_INVALID before any decision (channel_powers and noise_floor apply it)

The channel part takes the product's own float32 spectrum and evaluates the same double expressions as the product, so
its channel powers and candidates are bit-for-bit the product's.  Only tests/ and bench scripts may import this.
"""
from __future__ import annotations

import numpy as np

N = 4096
HOP = N // 2


def u8_to_float(capture_u8: np.ndarray) -> np.ndarray:
    """[n, 2] u8 -> complex128 of the float32 values the reference's conversion makes."""
    v = (np.arange(256, dtype=np.float64) / 127.5 - 1.0).astype(np.float32).astype(np.float64)
    c = np.asarray(capture_u8, dtype=np.uint8).reshape(-1, 2)
    return v[c[:, 0]] + 1j * v[c[:, 1]]


def window() -> np.ndarray:
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(N) / N)


def welch_psd_cf(x: np.ndarray, chunk: int = 512) -> np.ndarray:
    """Complex samples (float64) -> centred P[k], float64."""
    x = np.asarray(x, dtype=np.complex128)
    n_seg = (x.size - N) // HOP + 1
    w = window()
    acc = np.zeros(N, dtype=np.float64)
    for s0 in range(0, n_seg, chunk):
        s1 = min(n_seg, s0 + chunk)
        idx = (np.arange(s0, s1) * HOP)[:, None] + np.arange(N)[None, :]
        X = np.fft.fft(x[idx] * w[None, :], axis=1)
        acc += np.sum(X.real ** 2 + X.imag ** 2, axis=0)
    return np.fft.fftshift(acc / (n_seg * N * np.sum(w * w)))


def welch_psd(capture_u8: np.ndarray) -> np.ndarray:
    return welch_psd_cf(u8_to_float(capture_u8))


def bin_freqs(fs: float) -> np.ndarray:
    return (np.arange(N) - N // 2).astype(np.float64) * fs / N


def channel_bins(fs: float, first: float, step: float, count: int) -> list[np.ndarray]:
    f = bin_freqs(fs)
    out = []
    for j in range(count):
        fj = first + float(j) * step
        out.append(np.nonzero((fj - step / 2 <= f) & (f < fj + step / 2))[0])
    return out


def check_spectrum(p: np.ndarray) -> None:
    bad = np.flatnonzero(~np.isfinite(np.asarray(p, dtype=np.float64)))
    if bad.size:
        raise ValueError(f"bin {int(bad[0])} of {np.asarray(p).size} is not finite: the scan makes no decision")


def channel_powers(psd: np.ndarray, bins: list[np.ndarray]) -> np.ndarray:
    p = np.asarray(psd)
    check_spectrum(p)
    out = np.zeros(len(bins), dtype=np.float64)
    for j, b in enumerate(bins):
        acc = 0.0
        for k in b:                      # sequential, in bin order
            acc += float(p[k])
        out[j] = acc
    return out


def noise_floor(c: np.ndarray) -> float:
    c = np.asarray(c, dtype=np.float64)
    check_spectrum(c)
    return float(np.sort(c)[(c.size - 1) // 4])


def candidates(c: np.ndarray, min_snr_db: float = 10.0) -> list[int]:
    c = [float(v) for v in np.asarray(c, dtype=np.float64)]
    thr = noise_floor(np.asarray(c)) * 10.0 ** (min_snr_db / 10.0)
    out = []
    for j, v in enumerate(c):
        if v >= thr and (j == 0 or v > c[j - 1]) and (j + 1 == len(c) or v >= c[j + 1]):
            out.append(j)
    return out
