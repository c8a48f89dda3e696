// rfm_dsp.cuh -- device building blocks shared by the chain kernels (rfm_kernels.cu) and the stand-alone primitives
// (rfm_downconvert.cu): exact u8 / s8 / s16 -> float conversions, the decimate-by-2 stage bodies of CRDSDownConvert.
#pragma once

#include <cuda_runtime.h>

#include "rfm_math.cuh"

namespace rfm
{

// float(double(u) / 127.5 - 1.0) (RTL_SDR_Source.cpp:207-211) without a table: t = u * 0x1.01p-7 - 1 is exact, the
// second FMA adds the low part of 1/127.5 and rounds once.  Equal to the reference expression for all 256 codes
// (tests/test_abi_host.py::test_u8_conversion_formula, and the GPU parity tests through the whole chain).
__device__ __forceinline__ float rfm_u8_to_float(unsigned word, unsigned byte_sel)
{
  const float m = __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7540u + byte_sel)); // 2^23 + u
  const float u = __fsub_rn(m, 8388608.0f);
  const float t = __fmaf_rn(u, 0x1.01p-7f, -1.0f);
  return __fmaf_rn(u, 0x1.010102p-23f, t);
}

// Formats of the caller's IQ (rfm_iq_format in include/radiofm_b200.h): interleaved I,Q, little-endian.
enum IqFormat : int
{
  kIqU8 = 0,  // RTL-SDR offset binary, rfm_u8_to_float
  kIqS8 = 1,  // cs8 (HackRF): v * 2^-7
  kIqS16 = 2, // cs16 (SoapySDR / UHD host format): v * 2^-15
  kIqCF32 = 3
};
__host__ __device__ constexpr unsigned IqBytes(int f) { return f == kIqCF32 ? 8u : f == kIqS16 ? 4u : 2u; }

// Signed byte byte_sel of word -> v * 2^-7.  Flipping the sign bit makes v + 128 an unsigned byte, which lands in the
// mantissa of 2^23 as for the u8 form; every step is exact, so the result is (float)v * 2^-7 for all 256 codes.
__device__ __forceinline__ float rfm_s8_to_float(unsigned word, unsigned byte_sel)
{
  const float m = __uint_as_float(__byte_perm(word ^ 0x80808080u, 0x4B000000u, 0x7540u + byte_sel)); // 2^23 + v + 128
  return __fmul_rn(__fsub_rn(m, 8388736.0f), 0x1p-7f);
}

// Signed half hi (0: bits 0-15, 1: bits 16-31) of word -> v * 2^-15, exact for all 65536 codes (same construction).
__device__ __forceinline__ float rfm_s16_to_float(unsigned word, unsigned hi)
{
  const float m = __uint_as_float(__byte_perm(word ^ 0x80008000u, 0x4B000000u, hi ? 0x7632u : 0x7610u)); // 2^23 + v + 2^15
  return __fmul_rn(__fsub_rn(m, 8421376.0f), 0x1p-15f);
}

// One byte-sized component of a u8 or s8 word
template <int F>
__device__ __forceinline__ float rfm_iq8_to_float(unsigned word, unsigned byte_sel)
{
  return F == kIqS8 ? rfm_s8_to_float(word, byte_sel) : rfm_u8_to_float(word, byte_sel);
}

// Frequency-flat IQ correction (rfm_iq_correction, include/radiofm_b200.h), applied right after the format conversion:
// r = I - dc_i, q = Q - dc_q, y = r + j (a q + b r).  Two products and one sum, each rounded on its own, so a float32
// restatement on the host (oracle/iqcorr.py) is bit-exact.  Passed to the kernels by value, never re-read from memory.
struct IqCorr
{
  float dc_i, dc_q, a, b;
};

__device__ __forceinline__ float2 rfm_iq_correct(float2 x, const IqCorr& c)
{
  const float r = subf(x.x, c.dc_i);
  const float q = subf(x.y, c.dc_q);
  return make_float2(r, addf(mulf(c.a, q), mulf(c.b, r)));
}

// OscGn = 1.95 - (re^2 + im^2) of the NCO_OSC rotating vector (DownConvert.cpp:441): the double literal makes it
// float(1.95 - double(q)).  For q in [0.5, 1.69] -- the oscillator's amplitude never leaves it -- the same value comes
// out of five dependent float additions: s + e = 1.95f - q exactly (Fast2Sum), then the low part of the constant,
// 1.95 - 1.95f = -0x1.99999ap-25 (to float precision), joins the error term before the last rounding.  The margins to
// the rounding boundaries (>= 0.05 * 2^-24) dwarf the 2^-48 error of that last term; checked against the double
// expression for every one of the 14 176 749 floats of the domain on the host (tests/test_host_math.py) and on the
// device (math probe 13).  20 cycles of dependent latency instead of 45 through the FP64 pipe, no predicates -- this
// sits on the oscillator's critical path.
__device__ __forceinline__ float rfm_osc_gain_exact(float q) { return d2f(subd(1.95, (double)q)); }
__device__ __forceinline__ bool rfm_osc_gain_domain(float q) { return q >= 0.5f && q <= 1.69f; }
__device__ __forceinline__ float rfm_osc_gain_fast(float q) // valid where rfm_osc_gain_domain(q)
{
  const float s = subf(1.95f, q);
  const float e = subf(subf(1.95f, s), q);
  return addf(s, addf(e, -0x1.99999ap-25f));
}
__device__ __forceinline__ float rfm_osc_gain(float q)
{
  return rfm_osc_gain_domain(q) ? rfm_osc_gain_fast(q) : rfm_osc_gain_exact(q);
}

// --------------------------------------------------------------------------------------------------
// Decimate-by-2 stages over an interleaved V buffer [history | new samples]: DownConvert.cpp:516-550 (generic
// half-band: even taps + centre, tap 0 counted twice), :589-688 (fixed 11-tap), :709-727 (CIC3).
// --------------------------------------------------------------------------------------------------
template <int L>
__device__ __forceinline__ float2 hb_generic(const float* h, const float2* V, unsigned k)
{
  const float2* x = V + 2 * k;
  float2 acc;
  acc.x = mulf(x[0].x, h[0]);
  acc.y = mulf(x[0].y, h[0]);
#pragma unroll
  for (int j = 0; j < L; j += 2)
  {
    acc.x = addf(acc.x, mulf(x[j].x, h[j]));
    acc.y = addf(acc.y, mulf(x[j].y, h[j]));
  }
  constexpr int c = (L - 1) / 2;
  acc.x = addf(acc.x, mulf(x[c].x, h[c]));
  acc.y = addf(acc.y, mulf(x[c].y, h[c]));
  return acc;
}

__device__ __forceinline__ float2 hb_out(int kind, unsigned L, const float* h, const float2* V, unsigned k)
{
  float2 acc;
  if (kind == 0)
  {
    switch (L) // the lengths of filtercoef.h's tables, unrolled
    {
      case 11: return hb_generic<11>(h, V, k);
      case 15: return hb_generic<15>(h, V, k);
      case 19: return hb_generic<19>(h, V, k);
      case 23: return hb_generic<23>(h, V, k);
      case 27: return hb_generic<27>(h, V, k);
      case 31: return hb_generic<31>(h, V, k);
      case 35: return hb_generic<35>(h, V, k);
      case 39: return hb_generic<39>(h, V, k);
      case 43: return hb_generic<43>(h, V, k);
      case 47: return hb_generic<47>(h, V, k);
      case 51: return hb_generic<51>(h, V, k);
      default: break;
    }
    const unsigned i = 2 * k;
    float2 x = V[i];
    acc.x = mulf(x.x, h[0]);
    acc.y = mulf(x.y, h[0]);
    for (unsigned j = 0; j < L; j += 2)
    {
      x = V[i + j];
      acc.x = addf(acc.x, mulf(x.x, h[j]));
      acc.y = addf(acc.y, mulf(x.y, h[j]));
    }
    const unsigned c = (L - 1) / 2;
    x = V[i + c];
    acc.x = addf(acc.x, mulf(x.x, h[c]));
    acc.y = addf(acc.y, mulf(x.y, h[c]));
  }
  else if (kind == 1)
  {
    const unsigned i = 2 * k;
    const int idx[7] = {0, 2, 4, 5, 6, 8, 10};
    float2 x = V[i];
    acc.x = mulf(h[0], x.x);
    acc.y = mulf(h[0], x.y);
#pragma unroll
    for (int t = 1; t < 7; ++t)
    {
      x = V[i + idx[t]];
      acc.x = addf(acc.x, mulf(h[idx[t]], x.x));
      acc.y = addf(acc.y, mulf(h[idx[t]], x.y));
    }
  }
  else
  {
    const float2 xeven = V[2 * k], xodd = V[2 * k + 1], even = V[2 * k + 2], odd = V[2 * k + 3];
    acc.x = d2f(muld(.125, addd((double)addf(odd.x, xeven.x), muld(3.0, (double)addf(xodd.x, even.x)))));
    acc.y = d2f(muld(.125, addd((double)addf(odd.y, xeven.y), muld(3.0, (double)addf(xodd.y, even.y)))));
  }
  return acc;
}

// --------------------------------------------------------------------------------------------------
// The generic half-band over DE-INTERLEAVED V buffers -- E[m] = V[2m], O[m] = V[2m+1] -- so that output
// o = sum_j h[2j] E[o + j] + h[c] O[o + (c-1)/2] reads consecutive entries: a thread makes R consecutive outputs from
// (L+1)/2 + R - 1 even and R odd samples held in registers, the taps are kernel parameters.  Same products, same
// summation order as hb_generic (DownConvert.cpp:528-540).  Used by the wideband chain (rfm_downconvert.cu) and by the
// RDS front (rfm_kernels.cu), both through the packed form hb_deint_pk below.
// --------------------------------------------------------------------------------------------------
template <int L>
struct DcTaps
{
  float h[L];
};

// the taps as pairs (h, h): even taps e[j] = h[2 j], centre tap c, and the two constants of the packed arithmetic
template <int L>
struct DcTapsPk
{
  unsigned long long e[(L + 1) / 2], c;
  PairConst pk;
};

template <int L>
inline DcTapsPk<L> MakeDcTapsPk(const DcTaps<L>& t)
{
  DcTapsPk<L> o;
  for (int j = 0; j < (L + 1) / 2; ++j)
    o.e[j] = rfm_pair_bits(t.h[2 * j], t.h[2 * j]);
  o.c = rfm_pair_bits(t.h[(L - 1) / 2], t.h[(L - 1) / 2]);
  o.pk = kPairConst;
  return o;
}

#ifdef __CUDACC__
// (re, im) of a sample is one 64-bit operand, every product and every sum one FFMA2 (exact: rfm_math.cuh) -- 2 issue
// slots per tap instead of 4 (FMUL, FMUL, FADD, FADD), same products, same order
template <int L, int R>
__device__ __forceinline__ void hb_deint_pk(const DcTapsPk<L>& t, const f32x2* E, const f32x2* O, f32x2 (&acc)[R])
{
  constexpr int NE = (L + 1) / 2;
  constexpr int C = (L - 1) / 2;
#pragma unroll
  for (int m = 0; m < NE + R - 1; ++m)
  {
    const f32x2 v = E[m];
#pragma unroll
    for (int r = 0; r < R; ++r)
    {
      const int j = m - r;
      if (j == 0)
        acc[r] = pk_mul(v, t.e[0], t.pk);                          // DownConvert.cpp:528-529
      if (j >= 0 && j < NE)
        acc[r] = pk_add(pk_mul(v, t.e[j], t.pk), acc[r], t.pk);    // :533-534 (j = 0 again: tap 0 is counted twice)
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r)
    acc[r] = pk_add(pk_mul(O[r + (C - 1) / 2], t.c, t.pk), acc[r], t.pk); // :537-540
}
#endif

} // namespace rfm
