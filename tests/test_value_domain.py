"""The chain over sample VALUES, on the CPU: the input classes every value-domain case shares, and the proof that they
reach the replay paths of the lane kernels.

The hot path is exact by construction only inside value windows (rfm_math.cuh): rfm_div_unsafe and
rfm_div_unsafe_below (division operands), rfm_atan2f_special (atan2 operands), rfm_f2d_bits / rfm_d2f_bits (normal
floats only), the wrap domains [-6, 12.5) and the |phase| < 16 sincos core, plus the speculative pilot sincos'
rounding margin.  Outside a window the step raises a sticky flag and the kernel replays the 32-sample tile with the
exact routine.  An RTL-SDR u8 capture never leaves the windows (its samples are 1/255 .. 1 in magnitude, never 0);
cs8 / cs16 / cf32 captures do: exact zeros, rail codes, any float magnitude, subnormals, Inf and NaN.

1. Input classes (seeded), also used by test_gpu_value_domain.py:
     Z  zero runs of 1, 31, 32, 33, 384 samples and a whole block, at a block start, mid-block, across a block boundary
        and across a demodulator chunk boundary, inside a station; in cf32 as +0.0, -0.0 and mixed-sign pairs.
     R  rail codes (s8 -128 / 127, s16 -32768 / 32767) in I and in Q, a station overdriven by 6 dB and clipped to the
        container, and a stream that holds every code in I and in Q.
     M  a cf32 station times 2^k (exact: powers of two change no mantissa bits, except into the subnormals), and one
        whose amplitude ramps across 2^-95 inside a block.
     N  one NaN sample, one +Inf sample, a 32-sample NaN burst.
2. Coverage (rfm_steps.cuh compiled for the host like test_host_steps.py): the oracle's demod_in and baseband taps of
   Z, R, M (and N) through the fast steps with the kernels' tile replay; which window family raised each flag is
   recorded, every family must fire, and fast + replay must equal the oracle bit for bit (NaN-equivalent after N).
3. The scan's refusal rule in oracle/scan.py and the IQ estimate's restatement on degenerate classes.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import RATES, ROOT, station
from oracle import iqcorr, scan
from test_iq_formats import to_cf32

CHUNK = 384                  # RFM_DEMOD_CHUNK: demodulator time chunk, baseband samples (rfm_kernels.cu)
M_EXPONENTS = (-140, -100, -64, -31, 40, 61, 97, 126)
N_BLOCKS = 6


def assert_subnormals_kept():
    """The in-process oracle shares the SSE control state with numpy: if a library had set flush-to-zero /
    denormals-are-zero, the oracle would no longer compute what the reference computes on subnormal inputs."""
    assert np.float32(2.0 ** -140) * np.float32(0.5) != 0
    assert np.float32(2.0 ** -126) / np.float32(4.0) != 0


@pytest.fixture(autouse=True)
def _subnormals_kept():
    assert_subnormals_kept()


def nan_equal(a, b) -> bool:
    """NaN at the same positions and the other values bit-equal (x86 and the GPU make different NaN bit patterns)."""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32)))


# ---------------------------------------------------------------------------------------------------------------------
# 1. input classes
# ---------------------------------------------------------------------------------------------------------------------
def requantise(u8: np.ndarray, fmt: str, seed: int = 0, gain: float = 1.0) -> np.ndarray:
    """A u8 station in fmt's container, `gain` times louder, clipped to the container (never wrapped)."""
    v = (u8.astype(np.float64) - 127.5) * gain
    rng = np.random.default_rng(seed)
    if fmt == "s8":
        return np.clip(np.rint(v), -128, 127).astype(np.int8)
    if fmt == "s16":
        return np.clip(np.rint(v * 256 + rng.uniform(-0.5, 0.5, v.shape)), -32768, 32767).astype(np.int16)
    assert fmt == "cf32"
    return (to_cf32(u8).astype(np.float64) * gain).astype(np.float32)


def zero_runs(blk: int, ds: int) -> list[tuple[int, int]]:
    """(start, length) of the Z runs in a stream of N_BLOCKS blocks: 1 at a block start, 31 mid-block, 32 across a
    block boundary, 33 across a demodulator chunk boundary, 384 mid-block, and the whole of block 4."""
    c = 2 * CHUNK * ds                       # input sample of the second chunk boundary of block 3
    return [(blk, 1), (blk + blk // 3, 31), (2 * blk - 16, 32), (3 * blk + c - 16, 33), (3 * blk + blk // 2, 384),
            (4 * blk, blk)]


def with_zero_runs(x: np.ndarray, blk: int, ds: int) -> np.ndarray:
    """Class Z: x [n, 2] with the zero runs; float runs alternate +0.0, -0.0 and mixed-sign (+0, -0) / (-0, +0)."""
    y = x.copy()
    signs = [(0.0, 0.0), (-0.0, -0.0), (0.0, -0.0), (-0.0, 0.0)]
    for r, (p, n) in enumerate(zero_runs(blk, ds)):
        if y.dtype == np.float32:
            y[p:p + n] = np.array(signs[r % 4], dtype=np.float32)
        else:
            y[p:p + n] = 0
    return y


def with_rails(x: np.ndarray, blk: int) -> np.ndarray:
    """Class R: rail codes in I, in Q and in both, in runs of 1, 32 and 384 samples."""
    lo, hi = np.iinfo(x.dtype).min, np.iinfo(x.dtype).max
    y = x.copy()
    codes = [(lo, None), (None, hi), (hi, None), (None, lo), (lo, lo), (hi, hi), (lo, hi), (hi, lo)]
    for r, (i, q) in enumerate(codes):
        for n in (1, 32, 384):
            p = (r + 1) * blk // 2 + 7 * n + 3
            if i is not None:
                y[p:p + n, 0] = i
            if q is not None:
                y[p:p + n, 1] = q
    return y


def every_code(fmt: str, n: int, seed: int = 0) -> np.ndarray:
    """Every code of the container in I and in Q, in a seeded order, repeated to n samples."""
    rng = np.random.default_rng(seed)
    codes = np.arange(-128, 128) if fmt == "s8" else np.arange(-32768, 32768)
    reps = -(-n // codes.size)
    i = np.concatenate([rng.permutation(codes) for _ in range(reps)])[:n]
    q = np.concatenate([rng.permutation(codes) for _ in range(reps)])[:n]
    out = np.stack([i, q], axis=1).astype(np.int8 if fmt == "s8" else np.int16)
    assert n < codes.size or np.unique(out[:, 0]).size == codes.size == np.unique(out[:, 1]).size
    return out


def scaled(x: np.ndarray, k: int) -> np.ndarray:
    """Class M: x * 2^k in float32 (computed in float64, rounded once: exact unless it lands in the subnormals)."""
    return (x.astype(np.float64) * 2.0 ** k).astype(np.float32)


def ramp_across(x: np.ndarray, blk: int, e: int = -95) -> np.ndarray:
    """Class M: block 2 ramps the amplitude from 2^(e-4) to 2^(e+4) (powers of two per 1/16 of the block), the other
    blocks stay at 2^e."""
    g = np.full(x.shape[0], 2.0 ** e)
    steps = np.arange(blk) * 128 // blk                  # 0 .. 127
    g[2 * blk:3 * blk] = 2.0 ** (e - 4 + steps // 16)
    return (x.astype(np.float64) * g[:, None]).astype(np.float32)


def non_finite(x: np.ndarray, blk: int, kind: str, pos: int | None = None) -> tuple[np.ndarray, int]:
    """Class N: one NaN, one +Inf or a 32-sample NaN burst in a cf32 stream; returns it and the first bad sample."""
    y = x.copy()
    p = pos if pos is not None else 2 * blk + blk // 3
    if kind == "nan":
        y[p, 0] = np.nan
    elif kind == "inf":
        y[p, 1] = np.inf
    else:
        assert kind == "nan32"
        y[p:p + 32] = np.nan
    return y, p


def decoder_classes(rate: str, fmt: str, ds: int | None = None) -> dict[str, np.ndarray]:
    """One batch of the decoder cases: stream 0 a clean station, then one class per stream ([n, 2] in fmt).  rate
    names the synthetic station and its block length (conftest.RATES); ds places the chunk-boundary zero run."""
    _, ds0, blk = RATES[rate]
    ds = ds or ds0
    n = N_BLOCKS * blk
    u8 = [station(rate, N_BLOCKS, stream_id=40 + s)[0][:n] for s in range(3)]
    out = {"clean": requantise(u8[0], fmt, seed=1)}
    out["Z"] = with_zero_runs(requantise(u8[1], fmt, seed=2), blk, ds)
    if fmt == "cf32":
        base = requantise(u8[2], "cf32")
        for k in M_EXPONENTS:
            out[f"M 2^{k}"] = scaled(base, k)
        out["M ramp 2^-95"] = ramp_across(base, blk)
    else:
        out["R"] = with_rails(requantise(u8[2], fmt, seed=3), blk)
        out["R +6 dB clipped"] = requantise(u8[2], fmt, seed=4, gain=2.0)
        out["R every code"] = every_code(fmt, n, seed=5)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# 2. coverage of the replay paths
# ---------------------------------------------------------------------------------------------------------------------
FAMILIES = ("atan2_special", "div", "div_below", "bits", "wrap", "phase16", "spec")

SHIM = r'''
#include <string.h>
#include "rfm_steps.cuh"
using namespace rfm;
enum { F_ATAN = 1, F_DIV = 2, F_BELOW = 4, F_BITS = 8, F_WRAP = 16, F_PH16 = 32, F_SPEC = 64 };
static const unsigned kTile = 32;

// demod_step_fast's arithmetic with every window predicate evaluated on its own; returns the families that fired
static unsigned demod_flags(DemodState& st, float xr, float xi, const DemodConst& k) {
  unsigned f = 0;
  if (!(absf(st.phase) < 16.0f)) f |= F_PH16;
  float Sin, Cos;
  rfm_sincos_core(st.phase, &Sin, &Cos);
  const float dre = subf(mulf(Cos, xr), mulf(Sin, xi));
  const float dim = addf(mulf(Cos, xi), mulf(Sin, xr));
  const bool special = rfm_atan2f_special(dim, dre);
  bool b = false;
  const float err = negf(rfm_atan2f_fast(dim, dre, b));
  if (special) f |= F_ATAN;
  if (b && !special) f |= F_DIV;               // rfm_div_unsafe on y / x or on the reduced num / den
  const float incr = fminf(fmaxf(addf(st.incr, mulf(k.beta, err)), k.lo), k.hi);
  const float p = addf(st.phase, addf(incr, mulf(k.alpha, err)));
  bool w = false;
  st.incr = incr;
  st.phase = rfm_wrap_demod_fast(p, w);
  if (w) f |= F_WRAP;
  return f;
}

// pilot_step_fast (XUFREE = false)'s arithmetic, likewise
static unsigned pilot_flags(PilotState& st, float x, const PilotConstDev& k, const SinCosRegs& R) {
  unsigned f = 0;
  if (!(absf(st.phase) < 16.0f)) f |= F_PH16;
  float ps, pc;
  rfm_sincos_core_a(st.phase, R, &ps, &pc);
  float pi = mulf(ps, x), pq = mulf(pc, x);
  pi = subf(subf(mulf(k.b0, pi), mulf(k.a1, st.i1)), mulf(k.a2, st.i2));
  pq = subf(subf(mulf(k.b0, pq), mulf(k.a1, st.q1)), mulf(k.a2, st.q2));
  st.i2 = st.i1; st.i1 = pi; st.q2 = st.q1; st.q1 = pq;
  const bool use_div = pi > absf(pq);
  if (use_div && rfm_div_unsafe_below(pq, pi)) f |= F_BELOW;
  const float err = use_div ? rfm_div_fast(pq, pi) : ((pq > 0.0f) ? 1.0f : -1.0f);
  st.level = fminf(pi, st.level);
  const float freq = fmaxf(fminf(addf(st.freq, addf(mulf(k.lb0, err), mulf(k.lb1, st.x1))), k.maxfreq), k.minfreq);
  st.x1 = err; st.freq = freq;
  bool w = false;
  st.phase = rfm_wrap_pilot_fast(addf(st.phase, freq), w);
  if (w) f |= F_WRAP;
  return f;
}

extern "C" {
// k_demod_spec / k_demod_repair: 32-sample tiles of demod_step_fast, a flagged tile replayed with demod_step; then
// k_bb_lanes' output stage: tiles of demod_output_bits, a flagged tile replayed with demod_output.
// tiles[f] = tiles on which family f fired; mism[0] = steps where the predicates disagree with the real fast step's
// flag, mism[1] = unflagged steps whose state differs from the real fast step's
void run_demod(const float* z, unsigned n, const float* k5, float* bb, unsigned* tiles, unsigned* mism) {
  DemodConst k = {k5[0], k5[1], k5[2], k5[3], k5[4]};
  DemodState st = {0, 0};
  float dc = 0;
  for (unsigned t0 = 0; t0 < n; t0 += kTile) {
    const unsigned tn = (n - t0 < kTile) ? n - t0 : kTile;
    const DemodState start = st;
    unsigned fam = 0;
    bool bad = false;
    float incr[kTile];
    for (unsigned i = 0; i < tn; ++i) {
      DemodState a = st, b = st;
      const unsigned f = demod_flags(a, z[2*(t0+i)], z[2*(t0+i)+1], k);
      bool fb = false;
      demod_step_fast(b, z[2*(t0+i)], z[2*(t0+i)+1], k, fb);
      if ((f != 0) != fb) ++mism[0];
      if (!fb && memcmp(&a, &b, sizeof(a)) != 0) ++mism[1];
      fam |= f; bad = bad || fb;
      st = b;
      incr[i] = st.incr;
    }
    if (bad) {
      st = start;
      for (unsigned i = 0; i < tn; ++i) { demod_step(st, z[2*(t0+i)], z[2*(t0+i)+1], k); incr[i] = st.incr; }
    }
    for (unsigned b = 0; b < 7; ++b) if (fam & (1u << b)) ++tiles[b];
    const float dc0 = dc;
    bool ob = false;
    for (unsigned i = 0; i < tn; ++i) bb[t0+i] = demod_output_bits(incr[i], dc, k.gain, ob);
    if (ob) {
      ++tiles[3];
      dc = dc0;
      for (unsigned i = 0; i < tn; ++i) bb[t0+i] = demod_output(incr[i], dc, k.gain);
    }
  }
}

// k_bb_lanes' pilot: a tile of pilot_step_spec; if flagged, the tile again with pilot_step_fast; if flagged, with
// pilot_step (the kernel's back-off only decides how often the speculation is tried, not the result)
void run_pilot(const float* x, unsigned n, const float* k8, float freq0, float* out, unsigned* tiles, unsigned* mism) {
  PilotConstDev k = {k8[0], k8[1], k8[2], k8[3], k8[4], k8[5], k8[6], k8[7], 0};
  PilotState st = {0, freq0, 0, 0, 0, 0, 0, 1000.f};
  const SinCosRegs R = rfm_sincos_regs();
  PilotCarry sc;
  rfm_sincos(st.phase, &sc.ps, &sc.pc);
  for (unsigned t0 = 0; t0 < n; t0 += kTile) {
    const unsigned tn = (n - t0 < kTile) ? n - t0 : kTile;
    const PilotState start = st;
    const PilotCarry sc0 = sc;
    bool bad = false;
    for (unsigned i = 0; i < tn; ++i) out[t0+i] = pilot_step_spec(st, sc, x[t0+i], k, R, bad);
    if (!bad) continue;
    ++tiles[6];
    st = start; sc = sc0; bad = false;
    unsigned fam = 0;
    for (unsigned i = 0; i < tn; ++i) {
      PilotState a = st;
      const unsigned f = pilot_flags(a, x[t0+i], k, R);
      bool fb = false;
      out[t0+i] = pilot_step_fast(st, x[t0+i], k, R, fb);
      if ((f != 0) != fb) ++mism[0];
      if (!fb && memcmp(&a, &st, sizeof(a)) != 0) ++mism[1];
      fam |= f; bad = bad || fb;
    }
    for (unsigned b = 0; b < 6; ++b) if (fam & (1u << b)) ++tiles[b];
    if (bad) {
      st = start;
      for (unsigned i = 0; i < tn; ++i) out[t0+i] = pilot_step(st, x[t0+i], k);
    }
    rfm_sincos(st.phase, &sc.ps, &sc.pc);
  }
}
}
'''


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("valueshim")
    (d / "shim.cpp").write_text(SHIM)
    so = d / "shim.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I",
                           os.path.join(ROOT, "pvr.rtl.radiofm_b200", "csrc"), str(d / "shim.cpp"), "-o", str(so),
                           "-lm"])
    L = C.CDLL(str(so))
    f32p, u32p = C.POINTER(C.c_float), C.POINTER(C.c_uint)
    L.run_demod.argtypes = [f32p, C.c_uint, f32p, f32p, u32p, u32p]
    L.run_pilot.argtypes = [f32p, C.c_uint, f32p, C.c_float, f32p, u32p, u32p]
    L.run_demod.restype = L.run_pilot.restype = None
    return L


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _u(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint))


def _oracle_taps(port, rate: str, x: np.ndarray):
    fs, ds, blk = RATES[rate]
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    c = o.constants()                    # before any call: they include the pilot's starting frequency
    z, bb, p38 = [], [], []
    xf = to_cf32(x)
    for b in range(x.shape[0] // blk):
        o.process_cf32(xf[b * blk:(b + 1) * blk])
        z.append(o.tap("demod_in"))
        bb.append(o.tap("baseband"))
        p38.append(o.tap("pilot38"))
    o.close()
    return np.ascontiguousarray(np.concatenate(z)), np.concatenate(bb), np.concatenate(p38), c


def _coverage_inputs(rate: str):
    fs, ds, blk = RATES[rate]
    out = {}
    for fmt in ("s8", "s16", "cf32"):
        for name, x in decoder_classes(rate, fmt).items():
            if name != "clean" or fmt == "cf32":
                out[f"{fmt} {name}"] = x
    base = requantise(station(rate, N_BLOCKS, stream_id=42)[0][:N_BLOCKS * blk], "cf32")
    for kind in ("nan", "inf", "nan32"):
        out[f"cf32 N {kind}"] = non_finite(base, blk, kind)[0]
    return out


def test_value_classes_reach_every_replay_family(shim, port, capsys):
    """Every window family of the fast steps fires on some tile of the value classes, and fast + tile replay gives
    the oracle's demodulator output and pilot bit for bit (NaN-equivalent once a NaN has entered the state)."""
    rate = "1.0M"
    totals = dict.fromkeys(FAMILIES, 0)
    per_input = {}
    for name, x in _coverage_inputs(rate).items():
        z, bb, p38, c = _oracle_taps(port, rate, x)
        k5 = np.array([c[3], c[4], c[5], c[6], c[7]], dtype=np.float32)
        k8 = np.array([c[9], c[10], c[11], c[12], c[13], c[14], c[15], c[17]], dtype=np.float32)
        tiles, mism = np.zeros(7, dtype=np.uint32), np.zeros(2, dtype=np.uint32)
        out = np.zeros(z.shape[0], dtype=np.float32)
        shim.run_demod(_f(z), z.shape[0], _f(k5), _f(out), _u(tiles), _u(mism))
        assert nan_equal(out, bb), (name, "baseband")
        if not np.isnan(bb).any():
            assert np.array_equal(out.view(np.uint32), bb.view(np.uint32)), name
        x38 = np.ascontiguousarray(bb)
        o38 = np.zeros_like(x38)
        shim.run_pilot(_f(x38), x38.size, _f(k8), float(np.float32(c[16])), _f(o38), _u(tiles), _u(mism))
        assert nan_equal(o38, p38), (name, "pilot38")
        assert mism[0] == 0 and mism[1] == 0, (name, "the predicates disagree with the fast steps", mism)
        per_input[name] = {f: int(v) for f, v in zip(FAMILIES, tiles) if v}
        for f, v in zip(FAMILIES, tiles):
            totals[f] += int(v)
    # The pilot divides only while its I arm exceeds |Q|, so rfm_div_unsafe_below needs that arm below 2^-30: the
    # 19 kHz filter ringing down after its input has become exactly zero.  A decoder's baseband never stays exactly
    # zero after it has moved (the DC tracker leaves a residue), so none of the classes gets there; a tone burst and
    # silence through the oracle's stand-alone pilot (the same loop, test_host_steps.py) does.
    fs_bb = RATES[rate][0] / RATES[rate][1]
    t = np.arange(24000)
    burst = np.where(t < 2000, 0.1 * np.sin(2 * np.pi * 19000.0 / fs_bb * t), 0.0).astype(np.float32)
    L = port.lib()
    h = L.rfo_pilot_create(np.float32(19000.0 / fs_bb), np.float32(50.0 / fs_bb), np.float32(0.04))
    want = np.zeros_like(burst)
    L.rfo_pilot_process(h, _f(burst), _f(want), burst.size)
    L.rfo_pilot_destroy(h)
    c = port.OracleFmDecoder(RATES[rate][0], -0.15 * RATES[rate][0], downsample=RATES[rate][1]).constants()
    k8 = np.array([c[9], c[10], c[11], c[12], c[13], c[14], c[15], c[17]], dtype=np.float32)
    tiles, mism = np.zeros(7, dtype=np.uint32), np.zeros(2, dtype=np.uint32)
    got = np.zeros_like(burst)
    shim.run_pilot(_f(burst), burst.size, _f(k8), float(np.float32(c[16])), _f(got), _u(tiles), _u(mism))
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)) and mism[0] == 0 and mism[1] == 0
    per_input["pilot: tone burst, then silence"] = {f: int(v) for f, v in zip(FAMILIES, tiles) if v}
    for f, v in zip(FAMILIES, tiles):
        totals[f] += int(v)
    with capsys.disabled():
        print("\n[value domain] tiles flagged per window family:", totals)
        for name, d in per_input.items():
            print(f"  {name:32s} {d}")
    assert all(v > 0 for v in totals.values()), totals
    # finite samples reach the atan2, division and speculation windows; the wrap domains, the |phase| < 16 core and
    # the integer-pipe conversions of the DC tracker are left only once a NaN has entered the demodulator's state
    finite = {f: sum(d.get(f, 0) for n, d in per_input.items() if " N " not in n) for f in FAMILIES}
    assert all(finite[f] > 0 for f in ("atan2_special", "div", "div_below", "spec")), finite
    nonfinite = {f: sum(d.get(f, 0) for n, d in per_input.items() if " N " in n) for f in FAMILIES}
    assert all(nonfinite[f] > 0 for f in ("bits", "wrap", "phase16")), nonfinite


# ---------------------------------------------------------------------------------------------------------------------
# 3. the scan's refusal and the estimate on degenerate classes (restatements)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.filterwarnings("ignore::RuntimeWarning")
def test_scan_restatement_refuses_a_non_finite_spectrum():
    fs, raster = 2.4e6, (-1.0e6, 200000.0, 11)
    bins = scan.channel_bins(fs, *raster)
    rng = np.random.default_rng(3)
    x = (rng.standard_normal(3 * scan.N) + 1j * rng.standard_normal(3 * scan.N)) * 0.1
    psd = scan.welch_psd_cf(x)
    c = scan.channel_powers(psd, bins)
    assert np.all(np.isfinite(c)) and scan.candidates(c, 200.0) == []
    for bad in (np.nan, np.inf, -np.inf):
        y = x.copy()
        y[scan.N + 5] = bad
        p = scan.welch_psd_cf(y)
        assert not np.all(np.isfinite(p))
        with pytest.raises(ValueError, match="not finite"):
            scan.channel_powers(p.astype(np.float32), bins)
        with pytest.raises(ValueError, match="not finite"):
            scan.candidates(np.where(np.arange(c.size) == 3, bad, c))
    # a finite capture whose float32 spectrum overflows: |X|^2 of a coherent tone at 1e30 is about 1e67
    t = 1e30 * np.exp(2j * np.pi * 0.1 * np.arange(3 * scan.N))
    p32 = (scan.welch_psd_cf(t) * float(scan.N) * np.sum(scan.window() ** 2)).astype(np.float32)
    assert np.isinf(p32).any()
    with pytest.raises(ValueError):
        scan.channel_powers(p32, bins)


def test_iq_estimate_restatement_on_degenerate_classes():
    n = 4096
    # all zero: no DC, no statistics for the imbalance
    for dt in (np.int8, np.int16, np.float32):
        r = iqcorr.estimate(np.zeros((n, 2), dtype=dt))
        assert r[:4] == (0.0, 0.0, 1.0, 0.0) and not r[4], (dt, r)
    # a constant rail: the DC is the rail, the variances are zero
    for dt, v in ((np.int8, -128), (np.int16, -32768), (np.int8, 127), (np.int16, 32767)):
        r = iqcorr.estimate(np.full((n, 2), v, dtype=dt))
        assert r[0] == r[1] == np.float32(v / (128.0 if dt == np.int8 else 32768.0)), (dt, v, r)
        assert r[2:4] == (1.0, 0.0) and not r[4]
    # cf32 at the M scales: the float64 restatement of the sums stays finite and scales with the capture
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((n, 2)) * 0.3 + [0.01, -0.02]).astype(np.float32)
    x[:, 1] = (0.9 * x[:, 1] + 0.1 * x[:, 0]).astype(np.float32)
    r0 = iqcorr.coefficients_float64(x)
    for k in (-100, -64, 40, 97):
        r = iqcorr.coefficients_float64(scaled(x, k))
        assert abs(r[0] - r0[0] * 2.0 ** k) <= 1e-12 * abs(r0[0] * 2.0 ** k)
        assert abs(r[2] - r0[2]) <= 1e-9 and abs(r[3] - r0[3]) <= 1e-9, (k, r, r0)
    # non-finite cf32: a non-finite dc, the imbalance forced to the identity and reported invalid
    for bad in (np.nan, np.inf):
        y = x.copy()
        y[17, 0] = bad
        r = iqcorr.estimate(y)
        assert not np.isfinite(r[0]) and r[2:4] == (1.0, 0.0) and not r[4], (bad, r)


def test_class_generators():
    fs, ds, blk = RATES["1.0M"]
    runs = zero_runs(blk, ds)
    assert [n for _, n in runs] == [1, 31, 32, 33, 384, blk]
    assert runs[0][0] % blk == 0                                       # at a block start
    assert runs[2][0] // blk != (runs[2][0] + 31) // blk               # across a block boundary
    p, n = runs[3]
    assert (p // ds) // CHUNK != ((p + n) // ds) // CHUNK             # across a demodulator chunk boundary
    x = decoder_classes("1.0M", "cf32")
    z = x["Z"]
    assert np.sum(z == 0) >= 2 * (blk + 1 + 31 + 32 + 33 + 384)
    assert np.signbit(z[z == 0]).any() and (~np.signbit(z[z == 0])).any()
    assert np.min(np.abs(x["M 2^-140"][x["M 2^-140"] != 0])) < np.finfo(np.float32).tiny
    assert np.max(np.abs(x["M 2^126"])) >= 2.0 ** 125
    for fmt in ("s8", "s16"):
        y = decoder_classes("1.0M", fmt)
        info = np.iinfo(y["R"].dtype)
        for col in (0, 1):
            assert (y["R"][:, col] == info.min).any() and (y["R"][:, col] == info.max).any()
            assert (y["R +6 dB clipped"][:, col] == info.min).sum() > 100
            assert np.unique(y["R every code"][:, col]).size == info.max - info.min + 1
    assert_subnormals_kept()
