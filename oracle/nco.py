"""TEST INFRASTRUCTURE -- restatement of the phase-accumulator NCO pre-mixer (rfm_downconvert_set_nco;
include/radiofm_b200.h, DESIGN.md section 15):

    word     d = (uint32)(int64) llround(nco_freq / double(in_rate) * 2^32), |nco_freq| <= in_rate / 2; llround rounds
             halves away from zero (neither numpy's nor Python's round does)
    phase    sample i of a call: phi = (phi_start + i d) mod 2^32; phi_start = 0 after set_nco and reset, and
             phi_start += n d mod 2^32 after a call of n samples
    phasor   T0[k] = exp(j 2 pi k / 2^8), T1[k] = exp(j 2 pi k / 2^16), T2[k] = exp(j 2 pi k / 2^24), k < 256, each
             cos / sin computed in double and rounded to float once;
             e = cmul(cmul(T0[phi >> 24], T1[(phi >> 16) & 255]), T2[(phi >> 8) & 255])
    mix      y = cmul(x, e), cmul(u, v) = (u.x v.x - u.y v.y, u.x v.y + u.y v.x), every product and sum rounded to
             float32 on its own -- dc_mix in rfm_downconvert.cu, operand for operand

Only tests/ and bench scripts may import this.
"""
from __future__ import annotations

import math

import numpy as np

TWO32 = 1 << 32
TABLE_BITS = (8, 16, 24)   # T0, T1, T2: the angle step of table m is 2 pi / 2^TABLE_BITS[m]


def llround(x: float) -> int:
    """C's llround: the nearest integer, halves away from zero (exact for any double)."""
    t = math.trunc(x)
    if abs(x - t) >= 0.5:    # x - t is exact
        t += 1 if x > 0 else -1
    return int(t)


def word(nco_freq: float, in_rate) -> int:
    """The frequency word d (uint32).  in_rate is the down-converter's float rate; ValueError out of range."""
    r = float(np.float32(in_rate))
    f = float(nco_freq)
    if not math.isfinite(f) or abs(f) > r / 2:
        raise ValueError(f"nco_freq {f} outside [-in_rate / 2, in_rate / 2]")
    return llround(f / r * 4294967296.0) % TWO32


def phases(d: int, n: int, phi_start: int = 0) -> np.ndarray:
    """phi of samples 0 .. n-1 of a call (uint32)."""
    i = np.arange(n, dtype=np.uint64)
    return ((np.uint64(phi_start) + i * np.uint64(d)) % np.uint64(TWO32)).astype(np.uint32)


def advance(phi_start: int, d: int, n: int) -> int:
    """phi_start of the next call after a call of n samples."""
    return (phi_start + n * d) % TWO32


def table_angle(m: int, k: int) -> float:
    """The double argument of entry k of table m (the host evaluates the same expression)."""
    return 2.0 * math.pi * k / float(1 << TABLE_BITS[m])


def tables() -> np.ndarray:
    """[3, 256, 2] float32: T0, T1, T2."""
    t = np.empty((3, 256, 2), dtype=np.float32)
    for m in range(3):
        for k in range(256):
            a = table_angle(m, k)
            t[m, k] = (np.float32(math.cos(a)), np.float32(math.sin(a)))
    return t


def cmul(u: np.ndarray, v: np.ndarray) -> np.ndarray:
    """[.., 2] float32 x [.., 2] float32, each product and sum rounded to float32 on its own."""
    u = np.asarray(u, dtype=np.float32)
    v = np.asarray(v, dtype=np.float32)
    out = np.empty(np.broadcast_shapes(u.shape, v.shape), dtype=np.float32)
    out[..., 0] = u[..., 0] * v[..., 0] - u[..., 1] * v[..., 1]
    out[..., 1] = u[..., 0] * v[..., 1] + u[..., 1] * v[..., 0]
    return out


_TABLES = None


def phasor(phi: np.ndarray) -> np.ndarray:
    """uint32 phases -> [.., 2] float32 phasors, bit for bit as the kernels make them."""
    global _TABLES
    if _TABLES is None:
        _TABLES = tables()
    p = np.asarray(phi, dtype=np.uint32)
    t0 = _TABLES[0][p >> np.uint32(24)]
    t1 = _TABLES[1][(p >> np.uint32(16)) & np.uint32(255)]
    t2 = _TABLES[2][(p >> np.uint32(8)) & np.uint32(255)]
    return cmul(cmul(t0, t1), t2)


class Nco:
    """One row's NCO: mix() calls of any length continue one phase sequence."""

    def __init__(self, nco_freq: float, in_rate):
        self.d = word(nco_freq, in_rate)
        self.phi = 0

    def reset(self):
        self.phi = 0

    def mix(self, x_cf32: np.ndarray) -> np.ndarray:
        """[n, 2] float32 (converted, corrected) samples -> cmul(x, e) for the next n phases."""
        x = np.asarray(x_cf32, dtype=np.float32).reshape(-1, 2)
        y = cmul(x, phasor(phases(self.d, x.shape[0], self.phi)))
        self.phi = advance(self.phi, self.d, x.shape[0])
        return y


def mix(x_cf32: np.ndarray, nco_freq: float, in_rate, phi_start: int = 0) -> np.ndarray:
    """One call's mixed samples from phase phi_start."""
    n = Nco(nco_freq, in_rate)
    n.phi = phi_start
    return n.mix(x_cf32)
