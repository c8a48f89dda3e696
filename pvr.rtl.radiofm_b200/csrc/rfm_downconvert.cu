// rfm_downconvert.cu -- CRDSDownConvert (DownConvert.h:68-169, DownConvert.cpp:271-727) on the GPU, batched over rows
// (one row per station of a wideband capture, or per stream), optionally fused with the u8 -> float conversion of
// cRtlSdrSource::ReadAsyncCB (RTL_SDR_Source.cpp:207-211) or the exact s8 / s16 -> float conversions (rfm_dsp.cuh).
//
//   SetFrequency      -> per-row NCO_OSC rotation constants (DownConvert.cpp:311-320)
//   SetDataRate /
//   SetWfmDataRate    -> the decimate-by-2 stage list (rfm_plan.cpp: PlanDecimationChain, :327-399)
//   ProcessData       -> k_dc_osc (the amplitude-stabilised rotating-vector oscillator, :438-442: a nonlinear float
//                        recurrence, one lane per row; a row whose state enters a cycle of period <= 4 -- every row at
//                        0 Hz does after ~120 samples -- is finished in parallel) and k_dc_chain* (mix :464-465 + every
//                        stage :473-481 fused in shared memory; nothing intermediate touches HBM).
//
// Time parallelism: FIR stages carry only a finite history, so a long call is cut into chunks handled by different
// CTAs; a chunk other than the first re-derives the stage histories by running the `warm` input samples in front of it
// (sum over stages of hist_k * 2^k, e.g. 6350 for 7 x HB51) and discarding those outputs.  The results are the same
// sums of the same operands in the same order, i.e. bit-identical to the sequential reference.
//
// Restrictions (RFM_ERR_UNSUPPORTED otherwise): n must be a multiple of 2^stages and every stage must see at least
// 2 * (taps - 1) samples per call -- the reference itself silently mis-filters shorter / odd inputs (its in-place
// stages overwrite the samples they later copy into their delay line, DownConvert.cpp:519-520,544-547).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <vector>

#include "../../include/radiofm_b200.h"
#include "rfm_dsp.cuh"
#include "rfm_kernels.cuh"
#include "rfm_math.cuh"
#include "rfm_plan.h"

using namespace rfm;

namespace rfm
{
extern std::atomic<uint64_t> g_launches;
void SetLastError(const std::string& m);
}

namespace
{
constexpr unsigned kDcMaxStages = 9;   // MAX_DECSTAGES - 1, DownConvert.h:63
constexpr unsigned kDcThreads = 512;
#ifndef RFM_DC_THREADS
#define RFM_DC_THREADS 256
#endif
constexpr unsigned kDcThreadsFast = RFM_DC_THREADS; // uniform half-band kernel: 256 threads x 2 CTAs per SM, every thread two groups
                                                    // of 5 outputs in the first stage (1.75 ms against 1.86 with 512: profiles/r02_c5_dc_chain_ab.txt)
constexpr unsigned kDcTileGeneric = 2048; // input samples per tile, generic kernel
#ifndef RFM_DC_TILE
#define RFM_DC_TILE 5120
#endif
constexpr unsigned kDcTileFast = RFM_DC_TILE; // uniform half-band kernel (multiple of 2^9; 5120 = 5 * 2 * 512: whole groups)

struct DcStage
{
  int kind;              // 0 generic half-band, 1 fixed 11-tap, 2 CIC3
  unsigned len, hist;
  const float* h;        // device taps (nullptr for CIC3)
};

struct DcParams
{
  const void* in;        // [rows][in_stride] samples of the kernel's IQ format, or one shared capture [n] (SHARED)
  size_t in_stride;      // samples
  const float2* osc;     // NCO phasors [rows][osc_stride] (osc_stride == 0: one table for every row)
  size_t osc_stride;
  unsigned n, rows, nst;
  DcStage st[kDcMaxStages];
  const float2* tails_in; // [rows][tail_stride]: V-order histories of every stage, from the previous call
  float2* tails_out;
  size_t tail_stride;
  unsigned tail_off[kDcMaxStages];
  float2* out;           // [rows][out_stride]
  size_t out_stride;
  unsigned chunk, warm, nchunks;
  // optional pre-mixer: sample i of the call is first multiplied by pre[row][(pre_pos + i) mod pre_period] -- the
  // (cos, sin) sequence of a cFreqShift that is Reset() every pre_period samples (FreqShift.cpp:55-69)
  const float2* pre;
  size_t pre_stride;
  unsigned pre_period, pre_pos;
};

// F: IqFormat.  A shared cf32 capture is read as rows of stride 0 (no instantiation of its own).
template <int F, bool SHARED>
__device__ __forceinline__ float2 dc_convert(const DcParams& p, unsigned row, unsigned i)
{
  if (F == kIqCF32)
    return reinterpret_cast<const float2*>(p.in)[(size_t)row * p.in_stride + i];
  if (F == kIqS16)
  {
    const unsigned w = reinterpret_cast<const unsigned*>(p.in)[(SHARED ? 0 : (size_t)row * p.in_stride) + i];
    return make_float2(rfm_s16_to_float(w, 0u), rfm_s16_to_float(w, 1u));
  }
  const unsigned char* b = reinterpret_cast<const unsigned char*>(p.in) + 2 * ((!SHARED ? (size_t)row * p.in_stride : 0) + i);
  const unsigned w = *reinterpret_cast<const unsigned short*>(b);
  return make_float2(rfm_iq8_to_float<F>(w, 0u), rfm_iq8_to_float<F>(w, 1u));
}

// CORR: the IQ correction follows the conversion (rfm_iq_correct)
template <int F, bool SHARED, bool CORR>
__device__ __forceinline__ float2 dc_load(const DcParams& p, const IqCorr& corr, unsigned row, unsigned i)
{
  const float2 x = dc_convert<F, SHARED>(p, row, i);
  return CORR ? rfm_iq_correct(x, corr) : x;
}

// DownConvert.cpp:464-465 (and FreqShift.cpp:63-69: the same four products, one subtraction, one addition)
__device__ __forceinline__ float2 dc_mix(float2 d, float2 o)
{
  float2 r;
  r.x = subf(mulf(d.x, o.x), mulf(d.y, o.y));
  r.y = addf(mulf(d.x, o.y), mulf(d.y, o.x));
  return r;
}

// Phase-accumulator NCO pre-mixer (rfm_downconvert_set_nco; restated in oracle/nco.py).  Row r's phase at sample i of
// a call is phi = (pos + i) d[r] mod 2^32, pos = samples since set_nco / reset mod 2^32 -- the same value as carrying
// phi_start += n d from call to call, but every sample's phase is one integer multiply-add from its index, so time
// chunks and their warm-up samples need no hand-over.  The phasor is the product of three 256-entry tables of
// exp(j 2 pi k / 2^8), exp(j 2 pi k / 2^16) and exp(j 2 pi k / 2^24) (the lowest 8 phase bits are dropped), copied
// into shared memory in front of the kernel's own buffers.
struct DcNco
{
  const float2* tab;   // [3][256] T0, T1, T2
  const unsigned* d;   // [rows] frequency words
  unsigned pos;
};
constexpr unsigned kNcoTab = 3 * 256;                          // float2 entries
constexpr unsigned kNcoSmem = kNcoTab * sizeof(float2);        // 6 KB

// one row's NCO inside a CTA: the shared tables, phi_start of the call and the word
struct NcoRow
{
  const float2* tab;
  unsigned phi0, d;
};

__device__ __forceinline__ float2 nco_phasor(const NcoRow& n, unsigned i)
{
  const unsigned phi = n.phi0 + i * n.d;
  const float2 t0 = n.tab[phi >> 24], t1 = n.tab[256 + ((phi >> 16) & 255u)], t2 = n.tab[512 + ((phi >> 8) & 255u)];
  return dc_mix(dc_mix(t0, t1), t2);
}

// copy the tables into shared memory (the caller's next barrier publishes them) and set up the row
template <unsigned THREADS>
__device__ __forceinline__ NcoRow nco_row(const DcNco& nco, float2* s_tab, unsigned row, unsigned tid)
{
  for (unsigned i = tid; i < kNcoTab; i += THREADS)
    s_tab[i] = nco.tab[i];
  const unsigned d = nco.d[row];
  return NcoRow{s_tab, nco.pos * d, d};
}

// input sample i of this call for `row`, pre-mixed (by the table if one is set, or by the phasor NCO), times the
// NCO_OSC phasor
template <int F, bool SHARED, bool CORR, bool NCO>
__device__ __forceinline__ float2 dc_sample(const DcParams& p, const IqCorr& corr, const NcoRow& nco, const float2* osc,
                                            unsigned row, unsigned i)
{
  float2 d = dc_load<F, SHARED, CORR>(p, corr, row, i);
  if (NCO)
    d = dc_mix(d, nco_phasor(nco, i));
  else if (p.pre)
    d = dc_mix(d, p.pre[(size_t)row * p.pre_stride + (p.pre_pos + i) % p.pre_period]);
  return dc_mix(d, osc[i]);
}

// L2 prefetch of the global operands of tile [pos, pos + tn) (issued a tile ahead: the loads then hit L2)
template <int F, bool SHARED>
__device__ __forceinline__ void dc_prefetch(const DcParams& p, const float2* osc, unsigned row, unsigned pos, unsigned tn,
                                            unsigned tid)
{
  const unsigned i = tid * 16; // 16 float2 = one 128-byte line
  if (i >= tn)
    return;
  if (p.osc_stride)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(osc + pos + i));
  if (F == kIqCF32)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const float2*>(p.in) + (size_t)row * p.in_stride + pos + i));
  if (!SHARED && (F == kIqU8 || F == kIqS8) && (i & 63u) == 0)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const unsigned char*>(p.in) + 2 * ((size_t)row * p.in_stride + pos + i)));
  if (!SHARED && F == kIqS16 && (i & 31u) == 0)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const unsigned char*>(p.in) + 4 * ((size_t)row * p.in_stride + pos + i)));
}

// --------------------------------------------------------------------------------------------------
// NCO_OSC table, DownConvert.cpp:438-442: one lane per row, sequential.  Dependent chain per sample: a*a -> + -> gain
// (round-down / round-up subtraction, select, add) -> * : ~40 cycles; the rotation and the store run beside it.  Each
// lane stores its own entries (8 bytes per sample per row: the L2 merges them into full sectors).  The gain's float
// form is valid on [0.5, 1.69]; a 32-sample tile in which any row leaves that range is replayed with the double form.
// --------------------------------------------------------------------------------------------------
// rows per warp: a store instruction whose lanes hit 32 different rows costs the LSU ~64 cycles, more than the 32-cycle
// recurrence step it accompanies; with 4 rows per warp (the other lanes idle) the stores disappear behind the chain
constexpr unsigned kOscRows = 4;

template <bool FAST>
__device__ __forceinline__ void osc_step(float& a, float& b, float c, float s, float2* dst, bool store, bool& bad)
{
  const float orr = subf(mulf(a, c), mulf(b, s));
  const float oi = addf(mulf(b, c), mulf(a, s));
  const float q = addf(mulf(a, a), mulf(b, b));
  float gn;
  if (FAST)
  {
    gn = rfm_osc_gain_fast(q);
    bad |= !rfm_osc_gain_domain(q);
  }
  else
    gn = rfm_osc_gain(q);
  if (store)
    *dst = make_float2(orr, oi);
  a = mulf(gn, orr);
  b = mulf(gn, oi);
}

__global__ void __launch_bounds__(32) k_dc_osc(const float* cosv, const float* sinv, float* osc1, float2* table,
                                               size_t stride, unsigned n, unsigned rows, unsigned* cyc_t0)
{
  const unsigned lane = threadIdx.x;
  const unsigned r = blockIdx.x * kOscRows + lane;
  const bool valid = lane < kOscRows && r < rows;
  const float c = valid ? cosv[r] : 1.0f, s = valid ? sinv[r] : 0.0f;
  float a = valid ? osc1[2 * r] : 1.0f, b = valid ? osc1[2 * r + 1] : 0.0f;
  // the last four states, h0 oldest
  float2 h0 = make_float2(__int_as_float(0x7fc00001), 0.f), h1 = h0, h2 = h0, h3 = h0;
  float2* row = valid ? table + (size_t)r * stride : nullptr;
  unsigned t0 = 0;
  bool cyc = false;
  for (; t0 < n && !cyc; t0 += 32)
  {
    const unsigned tn = min(32u, n - t0);
    bool per = false;
    if (tn == 32)
    {
      const float a0 = a, b0 = b;
      bool bad = false;
      float2* dst = row + t0; // idle lanes: never dereferenced
#pragma unroll
      for (unsigned k = 0; k < 32; ++k)
      {
        if (k == 28) h0 = make_float2(a, b); // state before sample t0 + 28
        if (k == 29) h1 = make_float2(a, b);
        if (k == 30) h2 = make_float2(a, b);
        if (k == 31) h3 = make_float2(a, b);
        osc_step<true>(a, b, c, s, dst + k, valid, bad);
      }
      if (__any_sync(0xffffffffu, bad))
      {
        a = a0; b = b0;
        for (unsigned k = 0; k < 32; ++k)
        {
          if (k == 28) h0 = make_float2(a, b);
          if (k == 29) h1 = make_float2(a, b);
          if (k == 30) h2 = make_float2(a, b);
          if (k == 31) h3 = make_float2(a, b);
          osc_step<false>(a, b, c, s, dst + k, valid, bad);
        }
      }
      // the state after the tile equals the state four samples earlier: periodic from here on
      per = (__float_as_uint(a) == __float_as_uint(h0.x)) && (__float_as_uint(b) == __float_as_uint(h0.y));
    }
    else
    {
      bool bad = false;
      for (unsigned k = 0; k < tn; ++k)
        osc_step<false>(a, b, c, s, row + t0 + k, valid, bad);
    }
    // every row of this warp is in a short cycle (checked at a tile boundary): the rest is completed in parallel
    cyc = tn == 32 && __all_sync(0xffffffffu, per || !valid);
  }
  if (valid)
    cyc_t0[r] = (cyc && t0 < n) ? t0 : n; // k_dc_osc_fill completes osc[i] = osc[i - 4] for i >= t0
  if (cyc && t0 < n)
  {
    // here the state (a, b) == h0, the state before sample t0 - 4: osc[i] = osc[i - 4] for i >= t0, and the state after
    // sample n - 1 is the one (n - t0) mod 4 steps after h0: h0, h1, h2, h3 in turn
    const unsigned m = (n - t0) & 3u;
    const float2 e = m == 0 ? h0 : (m == 1 ? h1 : (m == 2 ? h2 : h3));
    a = m == 0 ? a : e.x;
    b = m == 0 ? b : e.y;
  }
  if (valid)
  {
    osc1[2 * r] = a;
    osc1[2 * r + 1] = b;
  }
}

__global__ void __launch_bounds__(256) k_dc_osc_fill(float2* table, size_t stride, unsigned n, const unsigned* cyc_t0)
{
  float2* row = table + (size_t)blockIdx.y * stride;
  const unsigned t0 = cyc_t0[blockIdx.y];
  if (t0 >= n)
    return;
  const unsigned i0 = t0 + (blockIdx.x * 256 + threadIdx.x) * 4; // four consecutive entries = one period
  if (i0 >= n)
    return;
  const float2 v0 = row[t0 - 4], v1 = row[t0 - 3], v2 = row[t0 - 2], v3 = row[t0 - 1];
  for (unsigned i = i0; i < n; i += gridDim.x * 1024)
  {
    row[i] = v0;
    if (i + 1 < n) row[i + 1] = v1;
    if (i + 2 < n) row[i + 2] = v2;
    if (i + 3 < n) row[i + 3] = v3;
  }
}

// --------------------------------------------------------------------------------------------------
// generic chain: any stage kinds, interleaved V buffers (the k_rds_front scheme without the LP)
// --------------------------------------------------------------------------------------------------
template <int F, bool SHARED, bool CORR, bool NCO>
__global__ void __launch_bounds__(kDcThreads) k_dc_chain(DcParams p, IqCorr corr, DcNco nco)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_h = reinterpret_cast<float*>(smem_raw + (NCO ? kNcoSmem : 0u));
  unsigned hoff[kDcMaxStages];
  unsigned acc_f = 0;
  for (unsigned k = 0; k < p.nst; ++k)
  {
    hoff[k] = acc_f;
    acc_f += (p.st[k].len + 1u) & ~1u;
  }
  float2* vbuf = reinterpret_cast<float2*>(s_h + acc_f);
  float2* B[kDcMaxStages];
  {
    unsigned off = 0, n = kDcTileGeneric;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      B[k] = vbuf + off;
      off += p.st[k].hist + n;
      n >>= 1;
    }
  }
  const unsigned tid = threadIdx.x;
  const unsigned c = blockIdx.x, row = blockIdx.y;
  const unsigned c_lo = c * p.chunk;
  if (c_lo >= p.n)
    return;
  const unsigned c_hi = min(p.n, c_lo + p.chunk);
  for (unsigned k = 0; k < p.nst; ++k)
    for (unsigned i = tid; i < p.st[k].len; i += kDcThreads)
      s_h[hoff[k] + i] = p.st[k].h ? p.st[k].h[i] : 0.0f;
  const float2* tin = p.tails_in + (size_t)row * p.tail_stride;
  for (unsigned k = 0; k < p.nst; ++k)
    for (unsigned i = tid; i < p.st[k].hist; i += kDcThreads)
      B[k][i] = (c == 0) ? tin[p.tail_off[k] + i] : make_float2(0.f, 0.f);
  NcoRow nrow = {};
  if (NCO)
    nrow = nco_row<kDcThreads>(nco, reinterpret_cast<float2*>(smem_raw), row, tid);
  __syncthreads();
  const float2* osc = p.osc + (size_t)row * p.osc_stride;
  float2* out = p.out + (size_t)row * p.out_stride;
  unsigned pos = (c == 0) ? 0u : c_lo - p.warm;
  while (pos < c_hi)
  {
    const bool store = pos >= c_lo;
    const unsigned tn = min(kDcTileGeneric, (store ? c_hi : c_lo) - pos);
    for (unsigned i = tid; i < tn; i += kDcThreads)
      B[0][p.st[0].hist + i] = dc_sample<F, SHARED, CORR, NCO>(p, corr, nrow, osc, row, pos + i);
    __syncthreads();
    unsigned n = tn;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      const unsigned nout = n >> 1;
      const bool last = k + 1 == p.nst;
      float2* dst = last ? out + (pos >> p.nst) : B[k + 1] + p.st[last ? k : k + 1].hist;
      if (!last || store)
        for (unsigned o = tid; o < nout; o += kDcThreads)
          dst[o] = hb_out(p.st[k].kind, p.st[k].len, s_h + hoff[k], B[k], o);
      __syncthreads();
      n = nout;
    }
    // carry the histories: last `hist` entries of [hist | n_k] to the front
    {
      unsigned nk = tn;
      for (unsigned k = 0; k < p.nst; ++k)
      {
        const unsigned hist = p.st[k].hist;
        float2 v0 = make_float2(0.f, 0.f);
        if (tid < hist)
          v0 = B[k][nk + tid];
        __syncthreads();
        if (tid < hist)
          B[k][tid] = v0;
        nk >>= 1;
      }
    }
    __syncthreads();
    pos += tn;
  }
  if (c + 1 == p.nchunks)
  {
    float2* tout = p.tails_out + (size_t)row * p.tail_stride;
    for (unsigned k = 0; k < p.nst; ++k)
      for (unsigned i = tid; i < p.st[k].hist; i += kDcThreads)
        tout[p.tail_off[k] + i] = B[k][i];
  }
}

// --------------------------------------------------------------------------------------------------
// uniform chain: every stage is the same generic half-band of L taps (SetWfmDataRate: all HB51).  The V buffers are
// kept de-interleaved -- E[m] = V[2m], O[m] = V[2m+1] -- so that output o = sum_j h[2j] E[o + j] + h[c] O[o + (c-1)/2]
// reads consecutive entries; a thread makes R = 5 consecutive outputs from 26 + 4 even and 5 odd samples held in
// registers (7 LDS.64 per output instead of 27; lane stride 5 float2 = 10 banks: conflict-free).  The arithmetic is on
// packed (re, im) pairs -- hb_deint_pk: every exact product and every exact sum one FFMA2, two issue slots per tap
// instead of four (the kernel is issue-bound with the fma pipe a third full).  Same products, same summation order as
// hb_generic.
// --------------------------------------------------------------------------------------------------
// one stage over a tile: groups of R consecutive outputs per thread; dstO == nullptr: last stage, dstE is the output row
// (natural order), else output o goes to the next stage's E / O by parity
template <int L, int R>
__device__ __forceinline__ void dc_stage(const DcTapsPk<L>& taps, const float2* E, const float2* O, float2* dstE, float2* dstO,
                                         unsigned nout, unsigned tid)
{
  for (unsigned g = tid; g * R < nout; g += kDcThreadsFast)
  {
    const unsigned o0 = g * R;
    f32x2 acc[R];
    hb_deint_pk<L, R>(taps, reinterpret_cast<const f32x2*>(E + o0), reinterpret_cast<const f32x2*>(O + o0), acc);
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (o0 + r < nout)
      {
        const unsigned o = o0 + r;
        if (!dstO)
          reinterpret_cast<f32x2*>(dstE)[o] = acc[r];
        else
          reinterpret_cast<f32x2*>((o & 1u) ? dstO : dstE)[o >> 1] = acc[r];
      }
  }
}

template <int F, bool SHARED, int L, bool CORR, bool NCO>
__global__ void __launch_bounds__(kDcThreadsFast) k_dc_chain_uniform(DcParams p, DcTapsPk<L> taps, IqCorr corr, DcNco nco)
{
  constexpr int R = 5;                 // largest group: sizes the slack behind each buffer
  constexpr unsigned HH = (L - 1) / 2; // history entries in each of E and O
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* vbuf = reinterpret_cast<float2*>(smem_raw + (NCO ? kNcoSmem : 0u));
  // buffer offsets in closed form (every stage has the same history, the tile halves from stage to stage): arrays
  // indexed with the run-time stage number would live in local memory
  //   E(k) starts at sum_{j<k} 2 (HH + (T >> j) / 2 + R) = 2 k (HH + R) + 2 T - (T >> (k - 1)),  O(k) follows E(k)
  auto eo = [&](unsigned k) { return 2u * k * (HH + R) + (k ? 2u * kDcTileFast - (kDcTileFast >> (k - 1)) : 0u); };
  auto oo = [&](unsigned k) { return eo(k) + HH + (kDcTileFast >> (k + 1)) + R; };
#define E_(k) (vbuf + eo(k))
#define O_(k) (vbuf + oo(k))
  const unsigned tid = threadIdx.x;
  const unsigned c = blockIdx.x, row = blockIdx.y;
  const unsigned c_lo = c * p.chunk;
  if (c_lo >= p.n)
    return;
  const unsigned c_hi = min(p.n, c_lo + p.chunk);
  const float2* tin = p.tails_in + (size_t)row * p.tail_stride;
  for (unsigned k = 0; k < p.nst; ++k)
  {
    for (unsigned i = tid; i < 2 * HH; i += kDcThreadsFast)
    {
      const float2 v = (c == 0) ? tin[p.tail_off[k] + i] : make_float2(0.f, 0.f);
      ((i & 1u) ? O_(k) : E_(k))[i >> 1] = v;
    }
    // slack entries: defined values (they are read into registers by the last partial group, never accumulated)
    for (unsigned i = tid; i < (unsigned)R; i += kDcThreadsFast)
    {
      const unsigned e = HH + (kDcTileFast >> (k + 1));
      E_(k)[e + i] = make_float2(0.f, 0.f);
      O_(k)[e + i] = make_float2(0.f, 0.f);
    }
  }
  NcoRow nrow = {};
  if (NCO)
    nrow = nco_row<kDcThreadsFast>(nco, reinterpret_cast<float2*>(smem_raw), row, tid);
  __syncthreads();
  const float2* osc = p.osc + (size_t)row * p.osc_stride;
  float2* out = p.out + (size_t)row * p.out_stride;
  unsigned pos = (c == 0) ? 0u : c_lo - p.warm;
  while (pos < c_hi)
  {
    const bool store = pos >= c_lo;
    const unsigned tn = min(kDcTileFast, (store ? c_hi : c_lo) - pos);
    // mix; V index 2 * HH + i: even i -> E[HH + i / 2], odd i -> O[HH + i / 2]
    if (!NCO && p.pre)
    {
      // the pre-mixer's table index walks with the sample: one modulo per tile and thread instead of one per sample
      const float2* pre = p.pre + (size_t)row * p.pre_stride;
      const unsigned step = kDcThreadsFast % p.pre_period;
      unsigned pi = (unsigned)(((unsigned long long)p.pre_pos + pos + tid) % p.pre_period);
      for (unsigned i = tid; i < tn; i += kDcThreadsFast)
      {
        const float2 d = dc_mix(dc_load<F, SHARED, CORR>(p, corr, row, pos + i), pre[pi]);
        ((i & 1u) ? O_(0) : E_(0))[HH + (i >> 1)] = dc_mix(d, osc[pos + i]);
        pi += step;
        pi = pi >= p.pre_period ? pi - p.pre_period : pi;
      }
    }
    else
      for (unsigned i = tid; i < tn; i += kDcThreadsFast)
        ((i & 1u) ? O_(0) : E_(0))[HH + (i >> 1)] = dc_sample<F, SHARED, CORR, NCO>(p, corr, nrow, osc, row, pos + i);
    __syncthreads();
    // operands of the next tile on their way into L2 while this one is filtered
    {
      const unsigned npos = pos + tn;
      if (npos < c_hi)
        dc_prefetch<F, SHARED>(p, osc, row, npos, min(kDcTileFast, ((npos >= c_lo) ? c_hi : c_lo) - npos), tid);
    }
    unsigned n = tn;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      const unsigned nout = n >> 1;
      const bool last = k + 1 == p.nst;
      if (!last || store)
      {
        float2* dstE = last ? out + (pos >> p.nst) : E_(k + 1) + HH;
        float2* dstO = last ? nullptr : O_(k + 1) + HH;
        // outputs per thread: 5 while that keeps every warp busy, fewer for the short late stages (latency-bound)
        if (nout >= 2 * kDcThreadsFast)
          dc_stage<L, 5>(taps, E_(k), O_(k), dstE, dstO, nout, tid);
        else if (nout >= kDcThreadsFast / 2)
          dc_stage<L, 3>(taps, E_(k), O_(k), dstE, dstO, nout, tid);
        else
          dc_stage<L, 1>(taps, E_(k), O_(k), dstE, dstO, nout, tid);
      }
      __syncthreads();
      n = nout;
    }
    // carry: E[i] = E[n_k / 2 + i], O likewise, i < HH.  Warp w takes stages w, w + warps, ..: all stages are read into
    // registers at once, one barrier, all are written (the stage loop above ended with a barrier; the one below closes
    // the tile) -- two barriers per tile instead of two per stage
    {
      constexpr unsigned NW = kDcThreadsFast / 32, PER = (kDcMaxStages + NW - 1) / NW;
      static_assert(HH <= 32, "one lane per history entry");
      const unsigned w = tid >> 5, l = tid & 31u;
      float2 ve[PER], vo[PER];
#pragma unroll
      for (unsigned q = 0; q < PER; ++q)
      {
        const unsigned k = w + q * NW;
        if (k < p.nst && l < HH)
        {
          ve[q] = E_(k)[(tn >> (k + 1)) + l];
          vo[q] = O_(k)[(tn >> (k + 1)) + l];
        }
      }
      __syncthreads();
#pragma unroll
      for (unsigned q = 0; q < PER; ++q)
      {
        const unsigned k = w + q * NW;
        if (k < p.nst && l < HH)
        {
          E_(k)[l] = ve[q];
          O_(k)[l] = vo[q];
        }
      }
    }
    __syncthreads();
    pos += tn;
  }
  if (c + 1 == p.nchunks)
  {
    float2* tout = p.tails_out + (size_t)row * p.tail_stride;
    for (unsigned k = 0; k < p.nst; ++k)
      for (unsigned i = tid; i < 2 * HH; i += kDcThreadsFast)
        tout[p.tail_off[k] + i] = ((i & 1u) ? O_(k) : E_(k))[i >> 1];
  }
}
#undef E_
#undef O_

template <typename T>
cudaError_t DevAlloc(T** p, size_t n)
{
  return cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(n, 1) * sizeof(T));
}
} // namespace

struct rfm_downconvert
{
  unsigned rows = 0, cap = 0, nst = 0;
  int device = 0, sm_count = 148;
  float in_rate = 0.f, max_bw = 0.f, out_rate = 0.f;
  bool wfm = false, uniform51 = false, osc_shared = false;
  std::vector<HalfBandStage> stages;
  std::vector<float> freq;
  unsigned hist[kDcMaxStages] = {0}, tail_off[kDcMaxStages] = {0};
  unsigned tail_stride = 0, warm = 0, min_n = 0;
  int tails_cur = 0;
  float* d_taps[kDcMaxStages] = {nullptr};
  float *d_cos = nullptr, *d_sin = nullptr, *d_osc1 = nullptr;
  unsigned* d_cyc = nullptr;
  const float2* pre = nullptr;
  size_t pre_stride = 0;
  unsigned pre_period = 0, pre_pos = 0;
  float2 *d_osc = nullptr, *d_tails[2] = {nullptr, nullptr};
  // host-pointer entry points: staging
  float2 *d_in = nullptr, *d_out = nullptr;
  uint8_t* d_raw = nullptr;   // u8 / s8 / s16 input, raw_bytes
  size_t raw_bytes = 0;
  DcTaps<51> taps51;
  bool corr_on = false;      // rfm_downconvert_set_iq_correction
  IqCorr corr = {0.f, 0.f, 1.f, 0.f};
  bool nco_on = false;       // rfm_downconvert_set_nco
  unsigned* d_nco_d = nullptr;  // [rows] frequency words
  float2* d_nco_tab = nullptr;  // [3][256] phasor tables
  uint32_t nco_pos = 0;      // samples since set_nco / reset, mod 2^32
};

namespace
{
int DcFail(int code, const std::string& m)
{
  rfm::SetLastError(m);
  return code;
}

int UploadFrequencies(rfm_downconvert* d)
{
  std::vector<float> c(d->rows), s(d->rows);
  d->osc_shared = true;
  for (unsigned r = 0; r < d->rows; ++r)
  {
    const NcoOsc o = PlanNcoOsc(d->freq[r], d->in_rate); // SetFrequency, DownConvert.cpp:311-320
    c[r] = o.cosv;
    s[r] = o.sinv;
    if (c[r] != c[0] || s[r] != s[0])
      d->osc_shared = false;
  }
  if (cudaMemcpy(d->d_cos, c.data(), d->rows * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(d->d_sin, s.data(), d->rows * 4, cudaMemcpyHostToDevice) != cudaSuccess)
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert: upload of the NCO constants failed");
  return RFM_OK;
}

int ResetState(rfm_downconvert* d)
{
  std::vector<float> o1(2 * (size_t)d->rows, 0.0f);
  for (unsigned r = 0; r < d->rows; ++r)
    o1[2 * r] = 1.0f; // DownConvert.cpp:283-284
  bool ok = cudaMemcpy(d->d_osc1, o1.data(), o1.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess;
  for (int b = 0; b < 2; ++b)
    ok = ok && cudaMemset(d->d_tails[b], 0, (size_t)d->rows * d->tail_stride * sizeof(float2)) == cudaSuccess;
  d->tails_cur = 0;
  return ok ? RFM_OK : DcFail(RFM_ERR_CUDA, "rfm_downconvert: state reset failed");
}

template <int F, bool SHARED, bool CORR, bool NCO>
void LaunchChain(rfm_downconvert* d, const DcParams& p, const DcNco& nco, cudaStream_t st)
{
  dim3 grid(p.nchunks, p.rows);
  if (d->uniform51)
  {
    size_t smem = NCO ? kNcoSmem : 0;
    unsigned n = kDcTileFast;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      smem += 2 * (size_t)(25 + n / 2 + 5) * sizeof(float2);
      n >>= 1;
    }
    EnsureDynSmem(k_dc_chain_uniform<F, SHARED, 51, CORR, NCO>, smem);
    k_dc_chain_uniform<F, SHARED, 51, CORR, NCO><<<grid, kDcThreadsFast, smem, st>>>(p, MakeDcTapsPk(d->taps51), d->corr,
                                                                                     nco);
  }
  else
  {
    size_t floats = 0, f2 = 0;
    unsigned n = kDcTileGeneric;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      floats += (p.st[k].len + 1u) & ~1u;
      f2 += p.st[k].hist + n;
      n >>= 1;
    }
    const size_t smem = (NCO ? kNcoSmem : 0) + floats * sizeof(float) + f2 * sizeof(float2);
    EnsureDynSmem(k_dc_chain<F, SHARED, CORR, NCO>, smem);
    k_dc_chain<F, SHARED, CORR, NCO><<<grid, kDcThreads, smem, st>>>(p, d->corr, nco);
  }
}

template <int F, bool SHARED>
void LaunchChain(rfm_downconvert* d, const DcParams& p, const DcNco& nco, cudaStream_t st)
{
  if (d->corr_on)
    d->nco_on ? LaunchChain<F, SHARED, true, true>(d, p, nco, st) : LaunchChain<F, SHARED, true, false>(d, p, nco, st);
  else
    d->nco_on ? LaunchChain<F, SHARED, false, true>(d, p, nco, st) : LaunchChain<F, SHARED, false, false>(d, p, nco, st);
}

// fmt: IqFormat; shared: one capture for every row (a shared cf32 capture is read as rows of stride 0)
int Run(rfm_downconvert* d, int fmt, bool shared, const void* d_in, size_t in_stride, float2* d_out, size_t out_stride,
        uint32_t n, uint32_t* n_out, cudaStream_t st)
{
  if (n_out)
    *n_out = 0;
  if (n == 0)
    return RFM_OK;
  if (n > d->cap)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert: n exceeds max_len");
  if (n % (1u << d->nst) != 0 || n < d->min_n)
    return DcFail(RFM_ERR_UNSUPPORTED,
                  "rfm_downconvert: n must be a multiple of 2^stages and give every stage >= 2*(taps-1) samples "
                  "(the reference mis-filters such inputs, DownConvert.cpp:519-520,544-547)");
  const unsigned orows = d->osc_shared ? 1u : d->rows;
  // every row the same frequency: one table, the carried phasor lives in row 0
  k_dc_osc<<<(orows + kOscRows - 1) / kOscRows, 32, 0, st>>>(d->d_cos, d->d_sin, d->d_osc1, d->d_osc, d->cap, n, orows, d->d_cyc);
  k_dc_osc_fill<<<dim3(std::min(64u, (n + 1023) / 1024), orows), 256, 0, st>>>(d->d_osc, d->cap, n, d->d_cyc);
  DcParams p;
  memset(&p, 0, sizeof(p));
  p.in = d_in; p.in_stride = (shared && fmt == kIqCF32) ? 0 : in_stride;
  p.osc = d->d_osc; p.osc_stride = d->osc_shared ? 0 : d->cap;
  p.n = n; p.rows = d->rows; p.nst = d->nst;
  for (unsigned k = 0; k < d->nst; ++k)
  {
    const HalfBandStage& hs = d->stages[k];
    p.st[k].kind = hs.len == 3 ? 2 : (hs.fixed11 ? 1 : 0);
    p.st[k].len = (unsigned)hs.len;
    p.st[k].hist = d->hist[k];
    p.st[k].h = d->d_taps[k];
    p.tail_off[k] = d->tail_off[k];
  }
  p.tails_in = d->d_tails[d->tails_cur];
  p.tails_out = d->d_tails[d->tails_cur ^ 1];
  p.tail_stride = d->tail_stride;
  p.out = d_out; p.out_stride = out_stride;
  // chunking: the chunk count that minimises (waves of CTAs) x (chunk + warm-up) -- full waves on the device's SMs with
  // two resident CTAs each, warm-up overhead kept small (the time is flat within 3 % from 10 to 25 chunks)
  const unsigned gran = 1u << d->nst;
  unsigned nchunks = 1, chunk = n;
  {
    static const int kslots = KnobInt(RFM_KNOB("RFM_DC_SLOTS"), 0);
    const unsigned slots = kslots > 0 ? (unsigned)kslots : 2u * (unsigned)d->sm_count;
    double best = 1e300;
    const unsigned max_chunks = d->warm ? std::max(1u, n / (4 * d->warm)) : 1u;
    static const int kforce = KnobInt(RFM_KNOB("RFM_DC_CHUNKS"), 0);
    for (unsigned c = 1; c <= std::min(max_chunks, 64u); ++c)
    {
      if (kforce > 0 && c != (unsigned)kforce)
        continue;
      unsigned len = (n + c - 1) / c;
      len = (len + gran - 1) / gran * gran;
      if (d->uniform51 && len >= kDcTileFast) // whole tiles: a partial last tile costs nearly a full one (its barriers)
        len = (len + kDcTileFast - 1) / kDcTileFast * kDcTileFast;
      const unsigned cnt = (n + len - 1) / len;
      const unsigned waves = (cnt * d->rows + slots - 1) / slots;
      const double cost = (double)waves * (len + (cnt > 1 ? d->warm : 0));
      if (cost < best * 0.999)
      {
        best = cost;
        nchunks = cnt;
        chunk = len;
      }
    }
  }
  p.chunk = chunk; p.warm = d->warm; p.nchunks = nchunks;
  p.pre = d->pre; p.pre_stride = d->pre_stride; p.pre_period = d->pre_period ? d->pre_period : 1; p.pre_pos = d->pre_pos;
  if (d->pre)
    d->pre_pos = (unsigned)(((uint64_t)d->pre_pos + n) % d->pre_period);
  const DcNco nco = {d->d_nco_tab, d->d_nco_d, d->nco_pos};
  if (d->nco_on)
    d->nco_pos += n; // mod 2^32: phi_start of the next call is nco_pos * d, i.e. phi_start + n d mod 2^32
  switch (fmt)
  {
    case kIqU8: shared ? LaunchChain<kIqU8, true>(d, p, nco, st) : LaunchChain<kIqU8, false>(d, p, nco, st); break;
    case kIqS8: shared ? LaunchChain<kIqS8, true>(d, p, nco, st) : LaunchChain<kIqS8, false>(d, p, nco, st); break;
    case kIqS16: shared ? LaunchChain<kIqS16, true>(d, p, nco, st) : LaunchChain<kIqS16, false>(d, p, nco, st); break;
    default: LaunchChain<kIqCF32, false>(d, p, nco, st); break;
  }
  d->tails_cur ^= 1;
  rfm::g_launches += 3;
  if (n_out)
    *n_out = n >> d->nst;
  return cudaGetLastError() == cudaSuccess ? RFM_OK : DcFail(RFM_ERR_CUDA, "rfm_downconvert: kernel launch failed");
}
} // namespace

extern "C"
{

int rfm_downconvert_create(uint32_t rows, const float* nco_freq, float in_rate, float max_bw, int wfm, uint32_t max_len,
                           int device, rfm_downconvert** out)
{
  if (!out || !nco_freq || rows == 0 || max_len == 0 || !(in_rate > 0) || !(max_bw > 0))
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_create: invalid argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return DcFail(RFM_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
  if (device < 0)
    cudaGetDevice(&device);
  if (cudaSetDevice(device) != cudaSuccess)
    return DcFail(RFM_ERR_CUDA, "cudaSetDevice failed");
  rfm_downconvert* d = new rfm_downconvert;
  d->rows = rows; d->cap = max_len; d->device = device;
  if (cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || d->sm_count <= 0)
    d->sm_count = 148;
  d->in_rate = in_rate; d->max_bw = max_bw; d->wfm = wfm != 0;
  d->freq.assign(nco_freq, nco_freq + rows);
  d->out_rate = PlanDecimationChain(in_rate, max_bw, d->wfm, &d->stages);
  d->nst = (unsigned)d->stages.size();
  if (d->nst == 0 || d->nst > kDcMaxStages)
  {
    delete d;
    return DcFail(RFM_ERR_UNSUPPORTED, "rfm_downconvert_create: the planned chain has no stage (or more than 9)");
  }
  unsigned off = 0;
  d->uniform51 = true;
  d->min_n = 0;
  d->warm = 0;
  for (unsigned k = 0; k < d->nst; ++k)
  {
    const HalfBandStage& hs = d->stages[k];
    d->hist[k] = hs.len == 3 ? 2u : (unsigned)hs.len - 1;
    d->tail_off[k] = off;
    off += d->hist[k];
    if (hs.len != 51 || hs.fixed11)
      d->uniform51 = false;
    const unsigned need = hs.len == 3 ? 4u : (hs.fixed11 ? 20u : 2u * ((unsigned)hs.len - 1));
    d->min_n = std::max(d->min_n, need << k);
    d->warm += d->hist[k] << k;
  }
  const unsigned gran = 1u << d->nst;
  d->warm = (d->warm + gran - 1) / gran * gran;
  d->tail_stride = (off + 15u) & ~15u;
  if (d->uniform51)
    memcpy(d->taps51.h, d->stages[0].h, 51 * sizeof(float));
  bool ok = DevAlloc(&d->d_cos, rows) == cudaSuccess && DevAlloc(&d->d_sin, rows) == cudaSuccess &&
            DevAlloc(&d->d_osc1, 2 * (size_t)rows) == cudaSuccess && DevAlloc(&d->d_cyc, rows) == cudaSuccess &&
            DevAlloc(&d->d_tails[0], (size_t)rows * d->tail_stride) == cudaSuccess &&
            DevAlloc(&d->d_tails[1], (size_t)rows * d->tail_stride) == cudaSuccess;
  for (unsigned k = 0; ok && k < d->nst; ++k)
    if (d->stages[k].h)
      ok = DevAlloc(&d->d_taps[k], (size_t)d->stages[k].len) == cudaSuccess &&
           cudaMemcpy(d->d_taps[k], d->stages[k].h, d->stages[k].len * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok)
    ok = UploadFrequencies(d) == RFM_OK;
  // the oscillator table: one row when every row has the same frequency, else one per row
  if (ok)
    ok = DevAlloc(&d->d_osc, (size_t)(d->osc_shared ? 1 : rows) * max_len) == cudaSuccess;
  if (ok)
    ok = ResetState(d) == RFM_OK;
  if (!ok)
  {
    rfm_downconvert_destroy(d);
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert_create: device allocation failed");
  }
  *out = d;
  return RFM_OK;
}

void rfm_downconvert_destroy(rfm_downconvert* d)
{
  if (!d)
    return;
  cudaSetDevice(d->device);
  cudaFree(d->d_cos); cudaFree(d->d_sin); cudaFree(d->d_osc1); cudaFree(d->d_osc); cudaFree(d->d_cyc);
  cudaFree(d->d_tails[0]); cudaFree(d->d_tails[1]);
  cudaFree(d->d_in); cudaFree(d->d_out); cudaFree(d->d_raw);
  cudaFree(d->d_nco_d); cudaFree(d->d_nco_tab);
  for (auto* t : d->d_taps)
    cudaFree(t);
  delete d;
}

float rfm_downconvert_output_rate(const rfm_downconvert* d) { return d ? d->out_rate : 0.0f; }

uint32_t rfm_downconvert_stages(const rfm_downconvert* d, uint32_t* taps, uint32_t max)
{
  if (!d)
    return 0;
  for (unsigned k = 0; taps && k < d->nst && k < max; ++k)
    taps[k] = (uint32_t)d->stages[k].len;
  return d->nst;
}

int rfm_downconvert_set_frequency(rfm_downconvert* d, const float* nco_freq)
{
  if (!d || !nco_freq)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_frequency: invalid argument");
  cudaSetDevice(d->device);
  const bool was_shared = d->osc_shared;
  d->freq.assign(nco_freq, nco_freq + d->rows);
  int rc = UploadFrequencies(d);
  if (rc != RFM_OK)
    return rc;
  if (was_shared != d->osc_shared)
  {
    // table shape changes; the carried phasors: shared -> per row copies row 0's, per row -> shared keeps row 0's
    std::vector<float> o1(2 * (size_t)d->rows);
    if (cudaMemcpy(o1.data(), d->d_osc1, o1.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess)
      return DcFail(RFM_ERR_CUDA, "rfm_downconvert_set_frequency: state read failed");
    if (was_shared)
      for (unsigned r = 1; r < d->rows; ++r) { o1[2 * r] = o1[0]; o1[2 * r + 1] = o1[1]; }
    cudaFree(d->d_osc);
    d->d_osc = nullptr;
    if (cudaMemcpy(d->d_osc1, o1.data(), o1.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
        DevAlloc(&d->d_osc, (size_t)(d->osc_shared ? 1 : d->rows) * d->cap) != cudaSuccess)
      return DcFail(RFM_ERR_CUDA, "rfm_downconvert_set_frequency: reallocation failed");
  }
  return RFM_OK;
}

int rfm_downconvert_reset(rfm_downconvert* d)
{
  if (!d)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_reset: null handle");
  cudaSetDevice(d->device);
  d->pre_pos = 0;
  d->nco_pos = 0;
  return ResetState(d);
}

int rfm_downconvert_set_premix(rfm_downconvert* d, const float* d_table, size_t row_stride, uint32_t period)
{
  if (!d || (d_table && (period == 0 || row_stride < period)))
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_premix: invalid argument");
  if (d_table && d->nco_on)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_premix: the phasor NCO is set (one pre-mixer at a time)");
  d->pre = reinterpret_cast<const float2*>(d_table);
  d->pre_stride = row_stride;
  d->pre_period = d_table ? period : 0;
  d->pre_pos = 0;
  return RFM_OK;
}

int rfm_downconvert_set_iq_correction(rfm_downconvert* d, const rfm_iq_correction* c)
{
  if (!d)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_iq_correction: null handle");
  if (c && !(isfinite(c->dc_i) && isfinite(c->dc_q) && isfinite(c->a) && isfinite(c->b)))
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_iq_correction: coefficients must be finite");
  d->corr_on = c != nullptr;
  d->corr = c ? IqCorr{c->dc_i, c->dc_q, c->a, c->b} : IqCorr{0.f, 0.f, 1.f, 0.f};
  return RFM_OK;
}

int rfm_downconvert_set_nco(rfm_downconvert* d, const double* nco_freq)
{
  if (!d)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_nco: null handle");
  if (!nco_freq)
  {
    d->nco_on = false;
    d->nco_pos = 0;
    return RFM_OK;
  }
  if (d->pre)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_nco: a pre-mix table is set (one pre-mixer at a time)");
  const double rate = (double)d->in_rate;
  std::vector<unsigned> w(d->rows);
  for (unsigned r = 0; r < d->rows; ++r)
  {
    if (!(isfinite(nco_freq[r]) && fabs(nco_freq[r]) <= rate / 2))
      return DcFail(RFM_ERR_INVALID, "rfm_downconvert_set_nco: every frequency must be finite and within +-in_rate / 2");
    w[r] = (uint32_t)(int64_t)llround(nco_freq[r] / rate * 4294967296.0);
  }
  cudaSetDevice(d->device);
  if (!d->d_nco_tab)
  {
    // T0, T1, T2: exp(j 2 pi k / 2^8), exp(j 2 pi k / 2^16), exp(j 2 pi k / 2^24), double cos / sin rounded once.  No
    // entry's double value lies within 2^-40 (relative) of a float rounding midpoint (tests/test_nco.py), so any
    // faithfully rounded libm gives these floats.
    std::vector<float2> t(kNcoTab);
    const unsigned bits[3] = {8, 16, 24};
    for (unsigned m = 0; m < 3; ++m)
      for (unsigned k = 0; k < 256; ++k)
      {
        const double a = 2.0 * M_PI * k / (double)(1u << bits[m]);
        t[m * 256 + k] = make_float2((float)cos(a), (float)sin(a));
      }
    if (DevAlloc(&d->d_nco_tab, kNcoTab) != cudaSuccess ||
        cudaMemcpy(d->d_nco_tab, t.data(), kNcoSmem, cudaMemcpyHostToDevice) != cudaSuccess)
      return DcFail(RFM_ERR_CUDA, "rfm_downconvert_set_nco: table upload failed");
  }
  if ((!d->d_nco_d && DevAlloc(&d->d_nco_d, d->rows) != cudaSuccess) ||
      cudaMemcpy(d->d_nco_d, w.data(), d->rows * sizeof(unsigned), cudaMemcpyHostToDevice) != cudaSuccess)
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert_set_nco: upload of the frequency words failed");
  d->nco_on = true;
  d->nco_pos = 0;
  return RFM_OK;
}

int rfm_downconvert_process_cf32(rfm_downconvert* d, const float* iq, uint32_t n, float* out, uint32_t* n_out)
{
  if (!d || !iq || !out)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_process_cf32: invalid argument");
  cudaSetDevice(d->device);
  if (!d->d_in && (DevAlloc(&d->d_in, (size_t)d->rows * d->cap) != cudaSuccess))
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert: staging allocation failed");
  if (!d->d_out && (DevAlloc(&d->d_out, (size_t)d->rows * (d->cap / 2 + 1)) != cudaSuccess))
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert: staging allocation failed");
  if (n > d->cap)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert: n exceeds max_len");
  if (cudaMemcpy(d->d_in, iq, (size_t)d->rows * n * 8, cudaMemcpyHostToDevice) != cudaSuccess)
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert: H2D copy failed");
  uint32_t m = 0;
  int rc = Run(d, kIqCF32, false, d->d_in, n, d->d_out, n >> d->nst, n, &m, 0);
  if (rc == RFM_OK && m && cudaMemcpy(out, d->d_out, (size_t)d->rows * m * 8, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = DcFail(RFM_ERR_CUDA, "rfm_downconvert: D2H copy failed");
  if (n_out)
    *n_out = m;
  return rc;
}

int rfm_downconvert_process_iq(rfm_downconvert* d, int format, int shared_capture, const void* iq, uint32_t n, float* out,
                               uint32_t* n_out)
{
  const uint32_t esz = rfm_iq_format_bytes(format);
  if (!d || !iq || !out || esz == 0)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_process_iq: invalid argument");
  if (format == RFM_IQ_CF32 && !shared_capture)
    return rfm_downconvert_process_cf32(d, static_cast<const float*>(iq), n, out, n_out);
  cudaSetDevice(d->device);
  if (n > d->cap)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert: n exceeds max_len");
  // u8 and s8 fit the staging the u8 path has always allocated (rows x max_len x 2 bytes); s16 / cf32 grow it
  const size_t need = std::max<size_t>((size_t)d->rows * d->cap * 2, (size_t)(shared_capture ? 1 : d->rows) * n * esz);
  if (d->raw_bytes < need)
  {
    cudaFree(d->d_raw);
    d->d_raw = nullptr;
    d->raw_bytes = 0;
    if (DevAlloc(&d->d_raw, need) != cudaSuccess)
      return DcFail(RFM_ERR_CUDA, "rfm_downconvert: staging allocation failed");
    d->raw_bytes = need;
  }
  if (!d->d_out && (DevAlloc(&d->d_out, (size_t)d->rows * (d->cap / 2 + 1)) != cudaSuccess))
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert: staging allocation failed");
  if (cudaMemcpyAsync(d->d_raw, iq, (size_t)(shared_capture ? 1 : d->rows) * n * esz, cudaMemcpyHostToDevice, 0) != cudaSuccess)
    return DcFail(RFM_ERR_CUDA, "rfm_downconvert: H2D copy failed");
  uint32_t m = 0;
  int rc = Run(d, format, shared_capture != 0, d->d_raw, n, d->d_out, n >> d->nst, n, &m, 0);
  if (rc == RFM_OK && m &&
      (cudaMemcpyAsync(out, d->d_out, (size_t)d->rows * m * 8, cudaMemcpyDeviceToHost, 0) != cudaSuccess ||
       cudaStreamSynchronize(0) != cudaSuccess))
    rc = DcFail(RFM_ERR_CUDA, "rfm_downconvert: D2H copy failed");
  if (n_out)
    *n_out = m;
  return rc;
}

int rfm_downconvert_process_u8(rfm_downconvert* d, const uint8_t* iq, int shared_capture, uint32_t n, float* out,
                               uint32_t* n_out)
{
  return rfm_downconvert_process_iq(d, RFM_IQ_U8, shared_capture, iq, n, out, n_out);
}

int rfm_downconvert_process_iq_device(rfm_downconvert* d, int format, int shared_capture, const void* d_in,
                                      size_t in_stride, float* d_out, size_t out_stride, uint32_t n, uint32_t* n_out,
                                      void* cuda_stream)
{
  const uint32_t esz = rfm_iq_format_bytes(format);
  if (!d || !d_in || !d_out || esz == 0)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_process_iq_device: invalid argument");
  if (reinterpret_cast<uintptr_t>(d_in) % esz != 0)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_process_iq_device: d_in must be aligned to the sample size "
                                   "(2 / 2 / 4 / 8 bytes for u8 / s8 / s16 / cf32)");
  cudaSetDevice(d->device);
  return Run(d, format, shared_capture != 0, d_in, in_stride, reinterpret_cast<float2*>(d_out), out_stride, n, n_out,
             static_cast<cudaStream_t>(cuda_stream));
}

int rfm_downconvert_process_device(rfm_downconvert* d, int mode, const void* d_in, size_t in_stride, float* d_out,
                                   size_t out_stride, uint32_t n, uint32_t* n_out, void* cuda_stream)
{
  if (!d || !d_in || !d_out || mode < 0 || mode > 2)
    return DcFail(RFM_ERR_INVALID, "rfm_downconvert_process_device: invalid argument");
  cudaSetDevice(d->device);
  return Run(d, mode == 0 ? kIqCF32 : kIqU8, mode == 1, d_in, in_stride, reinterpret_cast<float2*>(d_out), out_stride, n,
             n_out, static_cast<cudaStream_t>(cuda_stream));
}

} // extern "C"
