"""TEST INFRASTRUCTURE -- restatement of the IQ correction (rfm_iq_correction, rfm_iq_estimate; include/radiofm_b200.h):

    estimate   means m_I, m_Q and centred moments v_I, v_Q, c = E[I0 Q0] of the capture; dc = (m_I, m_Q),
               a = sqrt(v_I / (v_Q - c^2 / v_I)), b = -a c / v_I, every value in double, rounded to float once;
               v_I <= 0, v_I v_Q - c^2 <= 0 or a non-finite result: a = 1, b = 0, imbalance_valid = 0
                 u8 / s8 / s16  integer sums of codes, squares and cross products (Python ints), centred moments
                                n S_xy - S_x S_y exactly, then the same double expressions as rfm_iqcorr.cu: the product's
                                coefficients are bit-identical to these
                 cf32           exactly rounded float64 sums (math.fsum); the product sums in double in its own fixed
                                order, so it agrees to about 1e-15 relative before the rounding to float
    apply      float32, after the format conversion: r = I - dc_i, q = Q - dc_q, y = r + j (a q + b r), each operation
               rounded on its own -- bit-exact to the kernels (rfm_iq_correct, rfm_dsp.cuh)

Only tests/ and bench scripts may import this.
"""
from __future__ import annotations

import math

import numpy as np

U8, S8, S16, CF32 = 0, 1, 2, 3
MAX_N = 1 << 32


def _fmt(a: np.ndarray) -> int:
    return {np.dtype(np.uint8): U8, np.dtype(np.int8): S8, np.dtype(np.int16): S16,
            np.dtype(np.float32): CF32}[a.dtype]


def _as_pairs(capture) -> np.ndarray:
    a = np.asarray(capture)
    if a.dtype == np.complex64:
        a = np.ascontiguousarray(a).view(np.float32)
    return a.reshape(-1, 2)


def integer_sums(capture) -> tuple[int, int, int, int, int, int]:
    """(n, S_I, S_Q, S_II, S_QQ, S_IQ) of the integer codes of a u8 / s8 / s16 capture, exact."""
    a = _as_pairs(capture)
    assert a.dtype in (np.uint8, np.int8, np.int16), a.dtype
    i = a[:, 0].astype(np.int64)
    q = a[:, 1].astype(np.int64)
    # each sum fits int64 for n <= 2^32 (|code|^2 <= 2^30); Python ints from here on
    return (int(a.shape[0]), int(i.sum()), int(q.sum()), int((i * i).sum()), int((q * q).sum()), int((i * q).sum()))


def _imbalance(vi: float, vq: float, c: float) -> tuple[np.float32, np.float32, bool]:
    ok = vi > 0.0 and vi * vq - c * c > 0.0
    if ok:
        try:
            a = math.sqrt(vi / (vq - c * c / vi))
            b = -a * c / vi
            ok = math.isfinite(a) and math.isfinite(b)
        except (ValueError, ZeroDivisionError):
            ok = False
    if not ok:
        return np.float32(1.0), np.float32(0.0), False
    return np.float32(a), np.float32(b), True


def coefficients_from_integer_sums(fmt: int, sums) -> tuple:
    """(dc_i, dc_q, a, b, imbalance_valid) from integer_sums(): rfm_iqcorr.cu's IqCoefficientsInt, operation by
    operation."""
    n, si, sq, sii, sqq, siq = (int(v) for v in sums)
    vi = n * sii - si * si
    vq = n * sqq - sq * sq
    cc = n * siq - si * sq
    nn = float(n)
    k = 1.0 / 127.5 if fmt == U8 else (2.0 ** -7 if fmt == S8 else 2.0 ** -15)
    k2, n2 = k * k, nn * nn
    if fmt == U8:
        dc = (np.float32(float(si) / nn / 127.5 - 1.0), np.float32(float(sq) / nn / 127.5 - 1.0))
    else:
        dc = (np.float32(float(si) / nn * k), np.float32(float(sq) / nn * k))
    a, b, ok = _imbalance(float(vi) / n2 * k2, float(vq) / n2 * k2, float(cc) / n2 * k2)
    return dc[0], dc[1], a, b, ok


def coefficients_float64(x: np.ndarray) -> tuple:
    """(dc_i, dc_q, a, b, imbalance_valid) of float samples [n, 2] from exactly rounded double sums."""
    x = np.asarray(x).reshape(-1, 2)
    i = x[:, 0].astype(np.float64)
    q = x[:, 1].astype(np.float64)
    nn = float(x.shape[0])
    s = [math.fsum(v) for v in (i, q, i * i, q * q, i * q)]   # products of floats are exact in double
    mi, mq = s[0] / nn, s[1] / nn
    a, b, ok = _imbalance(s[2] / nn - mi * mi, s[3] / nn - mq * mq, s[4] / nn - mi * mq)
    return np.float32(mi), np.float32(mq), a, b, ok


def estimate(capture) -> tuple:
    """What rfm_iq_estimate returns for a host capture (u8 / s8 / s16 exactly; cf32 to about 1e-15 before rounding)."""
    a = _as_pairs(capture)
    if a.shape[0] == 0 or a.shape[0] > MAX_N:
        raise ValueError("n must be 1 .. 2^32")
    f = _fmt(a)
    if f == CF32:
        return coefficients_float64(a)
    return coefficients_from_integer_sums(f, integer_sums(a))


def apply(x_cf32: np.ndarray, dc_i, dc_q, a, b) -> np.ndarray:
    """[.., 2] float32 converted samples -> the corrected float32 samples, bit for bit as the kernels make them."""
    x = np.asarray(x_cf32, dtype=np.float32)
    r = x[..., 0] - np.float32(dc_i)
    q = x[..., 1] - np.float32(dc_q)
    y = np.empty_like(x)
    y[..., 0] = r
    y[..., 1] = np.float32(a) * q + np.float32(b) * r
    return y
